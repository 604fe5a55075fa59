"""GPU tests of the two matrix-product engines of stages 2 and 3, each against a plain exact or high-precision reference:

* the FP64 DMMA GEMM (tp_gemm / dgemm_kernel, csrc/gemm.cu): every layout and tile config, the symmetric mirror-on-store,
  deterministic split-K, the alpha / beta / gamma epilogue and the correlation epilogue (EPI_CORR, epi_row0);
* stage 2 on non-integer matrices and on counts >= 2^20 (rowstats_kernel + the DMMA correlation), through the public
  context path, against a longdouble reference with a bound derived from the arithmetic;
* the sliced int8 operator application of stage 3 (tp_iop_apply / io_gemm_kernel, csrc/igemm.cu): 5 and 8 digit planes,
  64- and 32-column tiles, row ranges that start off a 128-row boundary, the Chebyshev epilogue, and the column-maximum
  scratch that io_colmax_kernel keeps between applications.

The hooks upload every operand with its padding columns set to NaN and hand the output back whole, so a kernel that
reads past an edge, or writes outside its block, fails here; production padding is zero and would hide both."""
from fractions import Fraction

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

U = 2.0 ** -53                      # unit roundoff of binary64
SENT = -1.2345e300                  # sentinel of the output elements a launch must not touch
CFGS = (10, 11, 12)                 # TADPOLE_GEMM_CFG: 32x64, 64x64, 128x128 tiles
LAYOUTS = [(1, 1), (1, 0), (0, 1), (0, 0)]      # (a_kc, b_kc)


@pytest.fixture
def restore(ctx):
    """context settings a test changes, put back to their defaults afterwards (the ctx fixture lives for the session)"""
    defaults = {"igemm_min_n": 1024, "io_bn32": -1}
    yield
    for k, v in defaults.items():
        ctx.set(k, v)


def _operands(a, b, a_kc, b_kc):
    """the logical A (M x K) and B (K x N) in the storage the layout flags describe"""
    return (a if a_kc else np.ascontiguousarray(a.T)), (np.ascontiguousarray(b.T) if b_kc else b)


def _gemm(ctx, a, b, a_kc, b_kc, ldd_extra=3, **kw):
    """D = tp_gemm(A, B, ...) of logical A (M x K), B (K x N) in the given layout; D of M x (N + ldd_extra) starts at SENT.
    Returns the M x N block after asserting the rest was left alone."""
    m, n = a.shape[0], b.shape[1]
    sa, sb = _operands(a, b, a_kc, b_kc)
    d = ctx.test_gemm(sa, sb, np.full((m, n + ldd_extra), SENT), a_kc=a_kc, b_kc=b_kc, **kw)
    assert (d[:, n:] == SENT).all(), "tp_gemm wrote outside the M x N block"
    return d[:, :n]


# ======================================================================================================================
# A. DMMA, bit-exact: integer operands with K max|a| max|b| < 2^53 -- every partial sum in any order is exact
# ======================================================================================================================
_EDGE = [1, 3, 8, 31, 33, 64, 127, 129, 600]
# each edge value appears as M, as N and as K (cyclic shifts), then the production shapes: the Gram Y^T B (b, b, n),
# the rotation Y R (n, b, b), the two-GEMM operator / correlation (n, b, n) with b in {32, 96, 288, 704}, n in
# {200, 1031, 2000}
EXACT_SHAPES = [(_EDGE[i], _EDGE[(i + 1) % 9], _EDGE[(i + 2) % 9]) for i in range(9)] + [
    (32, 32, 2000), (96, 96, 1031), (288, 288, 200), (704, 704, 1031),
    (200, 704, 704), (1031, 32, 32), (2000, 288, 288), (1031, 96, 96),
    (200, 704, 200), (1031, 96, 1031), (2000, 32, 2000), (1031, 288, 1031),
]
_exact_cache = {}


def _int_operands(m, n, k, seed, bits=52):
    """integer A (M x K), B (K x N) with K max|a| max|b| < 2^bits, and A B in int64"""
    key = (m, n, k, seed, bits)
    if key not in _exact_cache:
        rng = np.random.default_rng(seed)
        amax = int(np.sqrt(2.0 ** bits / k))
        a = rng.integers(-amax, amax + 1, size=(m, k))
        b = rng.integers(-amax, amax + 1, size=(k, n))
        _exact_cache[key] = (a.astype(np.float64), b.astype(np.float64), a @ b)
    return _exact_cache[key]


@pytest.mark.parametrize("cfg", CFGS)
@pytest.mark.parametrize("a_kc,b_kc", LAYOUTS)
def test_dmma_exact_every_layout_and_tile(ctx, monkeypatch, cfg, a_kc, b_kc):
    monkeypatch.setenv("TADPOLE_GEMM_CFG", str(cfg))
    for (m, n, k) in EXACT_SHAPES:
        a, b, ref = _int_operands(m, n, k, seed=m * 7 + n * 3 + k)
        d = _gemm(ctx, a, b, a_kc, b_kc)
        assert np.array_equal(d, ref.astype(np.float64)), (m, n, k)


@pytest.mark.parametrize("cfg", CFGS)
@pytest.mark.parametrize("a_kc,b_kc", LAYOUTS)
def test_dmma_exact_epilogue(ctx, monkeypatch, cfg, a_kc, b_kc):
    """alpha, beta, gamma powers of two and integer E1, E2: with |A B| < 2^44 and |E| < 2^44 every product and sum of
    the epilogue is exact in binary64 (4 (alpha AB + beta E1 + gamma E2) is an integer below 2^49)"""
    monkeypatch.setenv("TADPOLE_GEMM_CFG", str(cfg))
    rng = np.random.default_rng(cfg)
    for (m, n, k) in [(33, 129, 600), (129, 31, 64), (704, 96, 288), (1, 600, 127)]:
        a, b, ref = _int_operands(m, n, k, seed=k, bits=44)
        e1 = rng.integers(-2 ** 44, 2 ** 44, size=(m, n))
        e2 = rng.integers(-2 ** 44, 2 ** 44, size=(m, n))
        d = _gemm(ctx, a, b, a_kc, b_kc, alpha=2.0, e1=e1.astype(float), beta=-0.5, e2=e2.astype(float), gamma=0.25)
        exact = (8 * ref - 2 * e1 + e2).astype(np.float64) / 4.0
        assert np.array_equal(d, exact), (m, n, k)


@pytest.mark.parametrize("cfg", CFGS)
@pytest.mark.parametrize("a_kc,b_kc", LAYOUTS)
def test_dmma_exact_symmetric(ctx, monkeypatch, cfg, a_kc, b_kc):
    """sym = 1 (B = A^T, tiles below the diagonal skipped and mirrored on store): exact and bitwise symmetric"""
    monkeypatch.setenv("TADPOLE_GEMM_CFG", str(cfg))
    for (m, k) in [(1, 3), (33, 127), (129, 600), (600, 64), (1031, 200)]:
        a, _, _ = _int_operands(m, 1, k, seed=m + k)
        ref = a.astype(np.int64) @ a.astype(np.int64).T
        d = _gemm(ctx, a, np.ascontiguousarray(a.T), a_kc, b_kc, sym=True)
        assert np.array_equal(d, ref.astype(np.float64)), (m, k)
        assert np.array_equal(d, d.T)


@pytest.mark.parametrize("splitk", [8, 32])
@pytest.mark.parametrize("cfg", CFGS)
def test_dmma_exact_split_k(ctx, monkeypatch, cfg, splitk):
    """split-K through the workspace and splitk_reduce_kernel, K divisible by the split count or not (1031 = 64 k-tiles
    of 16 + 7; 600 = 37 + 8/16; 2000 = 125 k-tiles), with and without the epilogue"""
    monkeypatch.setenv("TADPOLE_GEMM_CFG", str(cfg))
    rng = np.random.default_rng(splitk)
    for (m, n, k) in [(96, 96, 1031), (288, 288, 600), (32, 32, 2000), (3, 8, 1031)]:
        a, b, ref = _int_operands(m, n, k, seed=k + 1, bits=44)
        for a_kc, b_kc in LAYOUTS:
            d = _gemm(ctx, a, b, a_kc, b_kc, splitk=splitk)
            assert np.array_equal(d, ref.astype(np.float64)), (m, n, k, a_kc, b_kc)
        e1 = rng.integers(-2 ** 44, 2 ** 44, size=(m, n))
        d = _gemm(ctx, a, b, 0, 0, splitk=splitk, alpha=-2.0, e1=e1.astype(float), beta=0.5)
        assert np.array_equal(d, (-4 * ref + e1).astype(np.float64) / 2.0), (m, n, k)


# ======================================================================================================================
# B. DMMA, rounding bound: |D - R| <= gamma_{K+4} (|alpha| |A||B| + |beta E1| + |gamma E2|)
#    K products accumulated by fused multiply-adds (or, with split-K, ceil(K / splits) of them and at most splits - 1
#    additions of the partial sums: fewer than K + 4 in all), the alpha product and two epilogue additions.
# ======================================================================================================================
def _scaled_normals(m, n, k, seed):
    rng = np.random.default_rng(seed)
    ls = lambda size: 10.0 ** rng.uniform(-8, 8, size=size)
    a = rng.standard_normal((m, k)) * ls((m, 1)) * ls((1, k))
    b = rng.standard_normal((k, n)) * ls((k, 1)) * ls((1, n))
    return a, b


def _assert_rounding_bound(d, a, b, k, alpha=1.0, e1=None, beta=0.0, e2=None, gamma=0.0):
    al, bl = a.astype(np.longdouble), b.astype(np.longdouble)
    r = np.longdouble(alpha) * (al @ bl)
    mag = abs(alpha) * (np.abs(a) @ np.abs(b))
    if e1 is not None:
        r = r + np.longdouble(beta) * e1.astype(np.longdouble)
        mag = mag + np.abs(beta * e1)
    if e2 is not None:
        r = r + np.longdouble(gamma) * e2.astype(np.longdouble)
        mag = mag + np.abs(gamma * e2)
    g = (k + 4) * U / (1 - (k + 4) * U)
    err = np.abs(d.astype(np.longdouble) - r).astype(np.float64)
    bound = g * mag * (1 + 1e-12)          # (the bound's own float64 evaluation: relative 1e-13 at most)
    assert (err <= bound).all(), float((err / np.maximum(bound, 1e-300)).max())


@pytest.mark.parametrize("cfg", CFGS)
def test_dmma_rounding_bound(ctx, monkeypatch, cfg):
    monkeypatch.setenv("TADPOLE_GEMM_CFG", str(cfg))
    rng = np.random.default_rng(100 + cfg)
    for i, (m, n, k) in enumerate([(129, 96, 1031), (600, 33, 600), (33, 600, 127), (200, 288, 200)]):
        a, b = _scaled_normals(m, n, k, seed=i)
        a_kc, b_kc = LAYOUTS[i % 4]
        _assert_rounding_bound(_gemm(ctx, a, b, a_kc, b_kc), a, b, k)
        e1 = rng.standard_normal((m, n)) * (np.abs(a) @ np.abs(b))
        e2 = rng.standard_normal((m, n)) * (np.abs(a) @ np.abs(b))
        kw = dict(alpha=0.3, e1=e1, beta=-1.7, e2=e2, gamma=0.45)
        _assert_rounding_bound(_gemm(ctx, a, b, a_kc, b_kc, **kw), a, b, k, **kw)
    # symmetric launch
    a, _ = _scaled_normals(288, 1, 600, seed=9)
    d = _gemm(ctx, a, np.ascontiguousarray(a.T), 1, 1, sym=True)
    _assert_rounding_bound(d, a, a.T, 600)
    assert np.array_equal(d, d.T)


@pytest.mark.parametrize("splitk", [8, 32])
def test_dmma_rounding_bound_split_k_and_determinism(ctx, splitk):
    a, b = _scaled_normals(96, 96, 2000, seed=splitk)
    rng = np.random.default_rng(splitk)
    e1 = rng.standard_normal((96, 96)) * (np.abs(a) @ np.abs(b))
    for kw in (dict(), dict(alpha=-0.7, e1=e1, beta=1.3)):
        d1 = _gemm(ctx, a, b, 0, 0, splitk=splitk, **kw)
        _assert_rounding_bound(d1, a, b, 2000, **kw)
        d2 = _gemm(ctx, a, b, 0, 0, splitk=splitk, **kw)
        assert np.array_equal(d1, d2), "split-K is documented as deterministic"


# ======================================================================================================================
# C. EPI_CORR, bit-exact against the kernel's own expression
# ======================================================================================================================
def _fma(x, y, z):
    """correctly rounded x * y + z elementwise (exact rational arithmetic, one rounding)"""
    x, y, z = np.broadcast_arrays(x, y, z)
    out = [float(Fraction(p) * Fraction(q) + Fraction(r)) for p, q, r in zip(x.ravel().tolist(), y.ravel().tolist(),
                                                                              z.ravel().tolist())]
    return np.array(out).reshape(x.shape)


def _corr_epilogue(v, mean_r, mean_c, sd_r, sd_c, nrows):
    """(v - nrows (m_i m_j)) / (nrows - 1) / (sd_i sd_j), NaN -> 0, in the kernels' order.  nvcc contracts the
    subtraction and the nrows product into one fused multiply-add (the SASS of dgemm_kernel and ig_gram_kernel:
    DMUL m_i m_j, then DFMA -p * nrows + v), so the reference rounds it once too."""
    p = np.multiply.outer(mean_r, mean_c)
    t = _fma(-p, nrows, v)
    with np.errstate(divide="ignore", invalid="ignore"):
        t = t / (nrows - 1.0)
        t = t / np.multiply.outer(sd_r, sd_c)
    t[np.isnan(t)] = 0.0
    return t


@pytest.mark.parametrize("cfg", CFGS)
def test_dmma_corr_epilogue_bit_exact(ctx, monkeypatch, cfg):
    """Integer-valued X (n x K): the Gram matrix is exact, so the result must be the epilogue evaluated on it to the
    last bit, for caller-supplied mean / sd (one sd is 0: its row and column become NaN -> 0 or +-inf, as the expression
    says); a row block launched with A = X[r0:r1], epi_row0 = r0 must give the same bits as the symmetric launch."""
    monkeypatch.setenv("TADPOLE_GEMM_CFG", str(cfg))
    rng = np.random.default_rng(cfg)
    n, k = 331, 200
    x = rng.integers(0, 3000, size=(n, k)).astype(np.float64)
    x[17] = 0.0                                              # zero row: v = 0 and m = 0 -> 0 / 0 -> NaN -> 0
    mean = x.mean(axis=1) * (1 + 1e-3 * rng.standard_normal(n))
    sd = x.std(axis=1) * rng.uniform(0.5, 2.0, n)
    sd[5] = 0.0
    sd[17] = 0.0
    v = (x.astype(np.int64) @ x.astype(np.int64).T).astype(np.float64)
    ref = _corr_epilogue(v, mean, mean, sd, sd, float(k))
    kw = dict(mean=mean, sd=sd, nrows=float(k))
    full = _gemm(ctx, x, np.ascontiguousarray(x.T), 1, 1, sym=True, **kw)
    assert np.array_equal(full, ref)
    assert (full[17] == 0).all() and (full[:, 17] == 0).all()
    assert np.array_equal(full, full.T)
    for r0, r1 in [(64, 331), (128, 192), (256, 300)]:
        blk = _gemm(ctx, x[r0:r1], np.ascontiguousarray(x.T), 1, 1, epi_row0=r0, **kw)
        assert np.array_equal(blk, full[r0:r1]), (r0, r1)


# ======================================================================================================================
# D. Stage 2 on non-integer matrices (and counts >= 2^20), through ctx.set_filtered + ctx.correlation
# ======================================================================================================================
def _normalised_like(n, seed, counts_scale=None):
    """symmetric n x n with distance decay: Poisson counts x b_i b_j with log-normal biases b (a balanced / normalised
    Hi-C matrix), or -- counts_scale given -- the integer counts times counts_scale.  Columns 3, 10, 40 are near-constant
    (relative spreads 1e-2, 1e-4, 1e-6 around an integer level), column 7 is exactly constant (that integer)."""
    rng = np.random.default_rng(seed)
    d = np.abs(np.subtract.outer(np.arange(n), np.arange(n)))
    c = rng.poisson(200.0 / (1.0 + d) ** 0.8)
    c = np.triu(c) + np.triu(c, 1).T
    if counts_scale is None:
        bias = np.exp(rng.normal(0.0, 0.5, n))
        x = c * np.outer(bias, bias)
    else:
        x = (c * counts_scale).astype(np.float64)
    base = float(np.round(3.0 * x.mean())) + 1.0
    for j, spread in ((3, 1e-2), (10, 1e-4), (40, 1e-6)):
        col = base * (1.0 + spread * rng.standard_normal(n))
        if counts_scale is not None:
            col = np.round(col)
        x[:, j] = col
        x[j, :] = col
    x[:, 7] = base
    x[7, :] = base
    assert np.array_equal(x, x.T)
    return x


def _exact_corr_columns(x, cols):
    """the reference's correlation (R/TADpole.R:94-100) of columns `cols` against all columns, in longdouble from the
    exact mean (centred: algebraically the reference's one-pass formula, without its cancellation), plus the terms of the
    bound: (|X|^T |X|)_ij, kappa_j = sum_k x_kj^2 / ((n - 1) var_j)"""
    n = x.shape[0]
    xl = x.astype(np.longdouble)
    m = xl.sum(axis=0) / n
    xc = xl - m
    var = (xc * xc).sum(axis=0) / (n - 1)
    cov = xc.T @ xc[:, cols] / (n - 1)
    sd = np.sqrt(var)
    with np.errstate(divide="ignore", invalid="ignore"):
        rho = cov / np.outer(sd, sd[cols])
        kappa = ((xl * xl).sum(axis=0) / ((n - 1) * var)).astype(np.float64)
    return rho, m.astype(np.float64), sd.astype(np.float64), kappa, np.abs(x).T @ np.abs(x[:, cols])


@pytest.mark.parametrize("kind", ["normalised", "counts_2p20"])
@pytest.mark.parametrize("n", [200, 601, 1100, 1500])
def test_correlation_non_integer_rounding_bound(ctx, n, kind):
    """Bound of the computed correlation rho^ = fl[(v^ - n m^_i m^_j) / (n - 1) / (sd^_i sd^_j)] for NON-NEGATIVE X
    (u = 2^-53, T_ij = (|X|^T |X|)_ij + n |m_i m_j|, kappa_i = sum_k x_ki^2 / ((n - 1) var_i) >= 1):
      means   m^ = fl(sum / n), relative error <= (n + 1) u (every summand has the sign of the sum);
      Gram    |v^ - v| <= n u (|X|^T |X|)_ij (n fused multiply-adds; exact on the int8 path);
      numer.  one FMA over n fl(m^_i m^_j): |t^ - t| <= (n + 1) u (|X|^T|X|)_ij + (2n + 4) u n |m_i m_j| <= (2n + 4) u T_ij;
      sd      (n - 1) var^ = q^ - n m^^2 with |q^ - q| <= n u sum x^2 and n m^2 <= sum x^2: relative error of var^
              <= (3n + 4) u kappa + 2u, of sd^ half of that + 2u;
      rho     two divisions and the sd product: 3 more u.
    To first order |rho^ - rho| <= (2n + 4) u T_ij / ((n - 1) sd_i sd_j) + |rho_ij| ((3n + 4) u (kappa_i + kappa_j) / 2 + 8u),
    which c n' u [T_ij / ((n - 1) sd_i sd_j) + |rho_ij| (kappa_i + kappa_j) / 2] with n' = n + 2 covers at c = 3 (kappa >= 1
    absorbs the 8u); c = 4 leaves room for the second-order terms while (3n + 4) u kappa <= 0.04, i.e. on every column
    with kappa n u <= 1e-2, where the bound is asserted.  Columns past that (spread 1e-6 of the mean) are beyond what
    the one-pass formula resolves, in the reference as here: only NaN never escapes.  Where kappa n u < 1e-3 on both
    sides, an entry is zeroed (NaN -> 0) exactly when the exact formula zeroes it.  The exactly constant column (sd = 0)
    gives 0 / 0 -> 0 on the diagonal and (rounding residue) / 0 elsewhere, i.e. 0 or +-inf, as in the reference."""
    x = _normalised_like(n, seed=n, counts_scale=None if kind == "normalised" else 2 ** 14)
    if kind == "counts_2p20":
        assert x.max() >= 2 ** 20 and np.array_equal(x, np.round(x))
    ctx.set_filtered(x)
    ctx.correlation()
    cor = ctx.get_correlation(n)
    assert not np.isnan(cor).any()
    assert np.array_equal(cor, cor.T)
    # columns checked: all up to 601 bins; at 1100 and 1500 the special ones, tile edges and a random sample
    if n <= 601:
        cols = np.arange(n)
    else:
        rng = np.random.default_rng(n)
        cols = np.unique(np.r_[0, 3, 7, 10, 40, 31, 32, 63, 64, 127, 128, 129, n - 1, rng.choice(n, 100, replace=False)])
    rho, m, sd, kappa, xtx = _exact_corr_columns(x, cols)
    cc = cor[:, cols]
    nu = (n + 2) * U
    t = xtx + n * np.abs(np.outer(m, m[cols]))
    with np.errstate(divide="ignore", invalid="ignore", over="ignore"):
        bound = 4 * nu * (t / ((n - 1) * np.outer(sd, sd[cols])) +
                          np.abs(rho.astype(np.float64)) * np.add.outer(kappa, kappa[cols]) / 2)
    ok_r, ok_c = kappa * n * U <= 1e-2, kappa[cols] * n * U <= 1e-2
    sel = np.outer(ok_r, ok_c)
    err = np.abs(cc.astype(np.longdouble) - rho).astype(np.float64)
    assert sel.sum() > 0.9 * sel.size
    assert (err[sel] <= bound[sel]).all(), float((err[sel] / bound[sel]).max())
    # zeroing agrees with the exact formula where the one-pass sd is accurate
    z_r, z_c = kappa * n * U < 1e-3, kappa[cols] * n * U < 1e-3
    zsel = np.outer(z_r, z_c)
    exact_zero = ~np.isfinite(rho) | (rho == 0)
    assert np.array_equal((cc == 0)[zsel], exact_zero[zsel])
    # the constant column: 0 / 0 -> 0 on the diagonal, elsewhere 0 or +-inf
    assert cor[7, 7] == 0.0
    assert ((cor[7] == 0) | np.isinf(cor[7])).all()
    # a near-constant column inside the checked range must be among the checked ones
    assert ok_r[3] and ok_r[10]


def test_correlation_same_bits_on_both_engines(ctx, restore):
    """Integer counts at 1100 bins: the tcgen05 int8 Gram (default) and the FP64 DMMA GEMM (igemm_min_n = 0) both sum
    exactly and apply the same epilogue expression (gemm.cu:143-145, igemm.cu:246-248): the same bits."""
    x = _normalised_like(1100, seed=11, counts_scale=1)
    assert float(np.abs(x).max()) < 2 ** 20
    ctx.set_filtered(x)
    ctx.profile(1)
    ctx.correlation()
    prof = ctx.profile(0)
    assert prof["igemm"][1] > 0
    tc = ctx.get_correlation(1100)
    ctx.set("igemm_min_n", 0)
    ctx.set_filtered(x)
    ctx.profile(1)
    ctx.correlation()
    prof = ctx.profile(0)
    assert prof["igemm"][1] == 0 and prof["dgemm"][1] > 0
    assert np.array_equal(ctx.get_correlation(1100), tc)


# ======================================================================================================================
# E. Operator application, bit-exact
# ======================================================================================================================
def _digit_matrix(rows, cols, rng, ndig):
    """integers s = sum_{t < ndig} d_t 128^(ndig - 1 - t), digits in [-63, 63], the leading one +-63 somewhere in every
    row; some entries one digit only, some zero"""
    d = rng.integers(-63, 64, size=(ndig, rows, cols))
    d[1:] *= rng.random((ndig - 1, rows, cols)) < 0.7          # entries with a single (leading) digit
    d[:, rng.random((rows, cols)) < 0.05] = 0                  # zeros
    lead = rng.integers(0, cols, size=rows)
    d[0, np.arange(rows), lead] = rng.choice([-63, 63], size=rows)
    s = np.zeros((rows, cols), dtype=np.int64)
    for t in range(ndig):
        s = s * 128 + d[t]
    return s


_iop_cache = {}


def _iop_exact_case(n, b):
    """S = 2^(e_i - 6 - 7 (NDIG - 1)) s (rows), Y = 2^(f_j - 6 - 7 (NDIG - 1)) y (columns) with three base-128 digits
    each: the largest entry of every row / column has its leading digit +-63, so the kernels' exponent (max < 2^e) is
    e_i / f_j and the digit planes hold exactly the digits of s and y.  Every digit pair has s + t <= 4 <= NP - 1, the
    INT32 sums stay below 2^31 (3 n 63^2), and |S Y| scaled back is an integer below 2^51: the FP64 recombination is
    exact.  The int64 product is computed once per (n, b)."""
    if (n, b) not in _iop_cache:
        rng = np.random.default_rng(n * 1009 + b)
        s = _digit_matrix(n, n, rng, 3)
        y = _digit_matrix(b, n, rng, 3).T.copy()
        e = rng.integers(-30, 31, size=n)
        f = rng.integers(-30, 31, size=b)
        sh = 6 + 14
        S = np.ldexp(s.astype(np.float64), (e - sh)[:, None])
        Y = np.ldexp(y.astype(np.float64), (f - sh)[None, :])
        e1 = rng.integers(-2 ** 40, 2 ** 40, size=(n, b))
        e2 = rng.integers(-2 ** 40, 2 ** 40, size=(n, b))
        p = s @ y
        assert np.abs(8 * p).max() + 3 * 2 ** 40 < 2 ** 53          # the epilogue case below stays exact
        _iop_cache[(n, b)] = (S, Y, p, e1, e2, np.add.outer(e, f) - 2 * sh)
    return _iop_cache[(n, b)]


# each n in {64, 200, 1000, 1031, 2000} and each b in {32, 96, 256, 288, 704, 1024} at least once
IOP_EXACT = [(64, 1024), (200, 704), (1000, 256), (1031, 288), (2000, 32), (2000, 96)]


@pytest.mark.parametrize("bn32", [0, 1])
@pytest.mark.parametrize("np_", [5, 8])
@pytest.mark.parametrize("n,b", IOP_EXACT)
def test_iop_exact(ctx, restore, n, b, np_, bn32):
    ctx.set("io_bn32", bn32)
    S, Y, p, e1, e2, sc = _iop_exact_case(n, b)
    ranges = [(0, n)] + ([(64, n)] if n > 64 else []) + ([(128, 1000)] if n >= 1000 else [])
    for r0, r1 in ranges:
        # plain product, then the epilogue with powers of two: E_k = 2^(e_i + f_j - 40) int, every sum exact
        d = ctx.test_iop(S, [Y], [np.full((n, b), SENT)], np_=np_, row_begin=r0, row_end=r1)[0]
        assert (d[:r0] == SENT).all() and (d[r1:] == SENT).all()
        assert np.array_equal(d[r0:r1], np.ldexp(p.astype(np.float64), sc)[r0:r1]), (r0, r1)
        E1, E2 = np.ldexp(e1.astype(np.float64), sc), np.ldexp(e2.astype(np.float64), sc)
        d = ctx.test_iop(S, [Y], [np.full((n, b), SENT)], np_=np_, row_begin=r0, row_end=r1,
                         alpha=-2.0, e1=[E1], beta=0.5, e2=[E2], gamma=-0.25)[0]
        exact = np.ldexp((-8 * p + 2 * e1 - e2).astype(np.float64), sc - 2)
        assert (d[:r0] == SENT).all() and (d[r1:] == SENT).all()
        assert np.array_equal(d[r0:r1], exact[r0:r1]), (r0, r1)


# ======================================================================================================================
# F. Operator application, rounding bound
# ======================================================================================================================
def _corr_like(n, seed):
    """shaped like M = Xc Xc^T: unit-ish diagonal, small entries of both signs, a zero row, a tiny row, a huge row
    (test_gpu_igemm._centred_corr_like); not symmetric after the row scaling -- the kernel multiplies rows of S"""
    rng = np.random.default_rng(seed)
    a = rng.normal(0.0, 0.03, size=(n, n))
    a = 0.5 * (a + a.T) + np.eye(n) * 0.9
    a -= a.mean(axis=0, keepdims=True)
    a[3, :] = 0.0
    a[5, :] *= 1e-9
    a[7, :] *= 1e6
    return a


def _expo(mx):
    """the kernels' exponent: max < 2^e (frexp), 0 for a zero maximum"""
    e = np.frexp(mx)[1]
    return np.where(mx > 0, e, 0)


@pytest.mark.parametrize("np_", [5, 8])
@pytest.mark.parametrize("n,b", [(64, 96), (200, 32), (1000, 288)])
def test_iop_rounding_bound(ctx, restore, n, b, np_):
    """|D - R| <= |alpha| n 16 2^(-7 NP) 2^(e_i + f_j) + (NP + 4) u (|alpha| |S||Y| + |beta E1| + |gamma E2|): the digit
    pairs left out and the operand digits cut after NP are below (NP + 1) 2^(-7 NP) 2^(e_i + f_j) per product; the FP64
    recombination of NP accumulators, the scaling by alpha and the two epilogue additions round NP + 3 times.  At 64 and
    200 bins the first term is within a few times the rms contribution of the smallest accumulator (scale NP - 1), so an
    application that dropped it fails here at NP = 8 too."""
    rng = np.random.default_rng(n + np_)
    S = _corr_like(n, seed=n)
    Y = rng.standard_normal((n, b)) * 10.0 ** rng.uniform(-12, 12, size=b)
    Y[:, 1] = 0.0
    sig, sig2, e, c = 0.8, 1.3, 0.37, 0.55                   # Chebyshev step: alpha = 2 sig2 / e, beta = -alpha c, gamma
    alpha, beta, gamma = 2 * sig2 / e, -2 * sig2 * c / e, -sig * sig2
    Y0 = rng.standard_normal((n, b)) * np.abs(Y).max(axis=0)
    ef = np.add.outer(_expo(np.abs(S).max(axis=1)), _expo(np.abs(Y).max(axis=0))).astype(np.float64)
    for kw in (dict(), dict(alpha=alpha, e1=[Y], beta=beta, e2=[Y0], gamma=gamma)):
        a = kw.get("alpha", 1.0)
        r = np.longdouble(a) * (S.astype(np.longdouble) @ Y.astype(np.longdouble))
        mag = abs(a) * (np.abs(S) @ np.abs(Y))
        if kw:
            r = r + np.longdouble(beta) * Y + np.longdouble(gamma) * Y0
            mag = mag + np.abs(beta * Y) + np.abs(gamma * Y0)
        bound = abs(a) * n * 16 * np.exp2(-7.0 * np_ + ef) + (np_ + 4) * U * mag
        for bn32 in (0, 1):
            ctx.set("io_bn32", bn32)
            d = ctx.test_iop(S, [Y], [np.full((n, b), SENT)], np_=np_, **kw)[0]
            err = np.abs(d.astype(np.longdouble) - r).astype(np.float64)
            assert (err <= bound).all(), (bn32, bool(kw), float((err / np.maximum(bound, 1e-300)).max()))
            if not kw:
                assert (d[3] == 0.0).all()                   # the zero row of S


# ======================================================================================================================
# G. Operator application, state kept across applications (io_colmax_kernel's maxima and ticket)
# ======================================================================================================================
@pytest.mark.parametrize("bn32", [0, 1])
def test_iop_state_across_applications(ctx, restore, bn32):
    """A sequence of applications on one prepared operator whose column magnitudes fall by 1e12 each time while b
    shrinks and grows (704 -> 64 -> 288), then a second prepare with another n: every application must equal, bit for
    bit, the same application done first on a freshly prepared operator.  A column maximum left over from an earlier
    application would give a later column too large an exponent (digits lost silently); a ticket left over would leave
    the exponents unwritten."""
    ctx.set("io_bn32", bn32)
    for n, seq in ((1000, (704, 64, 288)), (600, (96, 1024, 32))):
        rng = np.random.default_rng(n + bn32)
        S = _corr_like(n, seed=n + 1)
        ys = [rng.standard_normal((n, b)) * 10.0 ** (-12 * i) for i, b in enumerate(seq)]
        for np_ in (5, 8):
            got = ctx.test_iop(S, ys, [np.full(y.shape, SENT) for y in ys], np_=np_)
            for i, y in enumerate(ys):
                fresh = ctx.test_iop(S, [y], [np.full(y.shape, SENT)], np_=np_)[0]
                assert np.array_equal(got[i], fresh), (n, np_, i)
