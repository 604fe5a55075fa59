"""CPU tests of coarsening (DESIGN S0e): the pixel-by-pixel reference and its vectorised restatement
(tests/coarsen_oracle.py), the host logic of LoadedGenome.coarsen on a stand-in genome, the C ABI symbol and the R
routine's argument checks under the stand-in R runtime of tests/mock_r."""
import ctypes
import os
import re
import sys

import numpy as np
import pytest

from tadpole_b200 import _lib
from tadpole_b200.batch import LoadedGenome, _CtxRef

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tests"))
import coarsen_oracle as C  # noqa: E402

SIZES = [37, 1, 20, 8]                       # chromosome 3 holds no pixel


def _genome(seed=0, fractional=False):
    """Duplicates, zeros, NaN counts, negative pairs that cancel, trans and below-diagonal pixels; shuffled."""
    rng = np.random.default_rng(seed)
    starts = np.concatenate(([0], np.cumsum(SIZES)))
    b1, b2, v = [], [], []
    for c in (0, 1, 2):
        n = SIZES[c]
        i = rng.integers(0, n, 300)
        j = np.minimum(n - 1, i + rng.integers(0, 9, i.size))
        x = rng.integers(0, 6, i.size).astype(float)
        if fractional:
            x = x * rng.random(i.size)
        b1.append(starts[c] + i); b2.append(starts[c] + j); v.append(x)
    b1.append([starts[0] + 3, starts[0] + 3, 2, starts[2] + 9, starts[0] + 30, starts[0] + 30])
    b2.append([starts[0] + 4, starts[0] + 5, starts[2] + 1, starts[2] + 4, starts[0] + 31, starts[0] + 31])
    v.append([np.nan, np.nan, 4.0, 6.0, 5.0, -5.0])       # NaN, a trans pixel, one below, a cell that sums to 0 at factor 1
    b1, b2, v = np.concatenate(b1), np.concatenate(b2), np.concatenate(v)
    p = rng.permutation(v.size)
    return b1[p].astype(np.int32), b2[p].astype(np.int32), v[p]


def _global(out, sizes):
    """the per-chromosome (I, J, count) of a reference result as a global pixel list over `sizes`"""
    starts = np.concatenate(([0], np.cumsum(sizes)))
    return (np.concatenate([i + starts[c] for c, (i, _, _) in enumerate(out)]),
            np.concatenate([j + starts[c] for c, (_, j, _) in enumerate(out)]),
            np.concatenate([x for _, _, x in out]))


def _same(a, b):
    return len(a) == len(b) and all(np.array_equal(x[0], y[0]) and np.array_equal(x[1], y[1]) and
                                    np.array_equal(x[2].view(np.uint64), y[2].view(np.uint64)) for x, y in zip(a, b))


FACTORS = [1, 2, 3, 7, 36, 37, 38, 10 ** 6]


@pytest.mark.parametrize("factor", FACTORS)
def test_loop_and_vectorised_reference_agree(factor):
    for seed in range(3):
        b1, b2, v = _genome(seed)
        loop, tr, bl = C.coarsen_pixels(SIZES, b1, b2, v, factor)
        vec, tr2, bl2 = C.coarsen_pixels_np(SIZES, b1, b2, v, factor)
        assert (tr, bl) == (tr2, bl2) == (1, 1)
        assert _same(loop, vec), (seed, factor)
        assert loop[3][0].size == 0
        for (i, j, _), n in zip(loop, C.coarse_bins(SIZES, factor)):
            assert np.all((0 <= i) & (i <= j) & (j < n))
        b1f, b2f, vf = _genome(seed, fractional=True)
        loop, _, _ = C.coarsen_pixels(SIZES, b1f, b2f, vf, factor)
        vec, _, _ = C.coarsen_pixels_np(SIZES, b1f, b2f, vf, factor)
        assert all(np.array_equal(x[0], y[0]) and np.array_equal(x[1], y[1]) and np.allclose(x[2], y[2], rtol=1e-13)
                   for x, y in zip(loop, vec))


def test_zero_sums_and_nan_counts():
    b1, b2, v = np.array([0, 0, 1, 2]), np.array([1, 1, 2, 2]), np.array([5.0, -5.0, np.nan, 3.0])
    out, _, _ = C.coarsen_pixels([4], b1, b2, v, 1)
    assert out[0][0].tolist() == [2] and out[0][2].tolist() == [3.0]
    out, _, _ = C.coarsen_pixels([4], b1, b2, v, 2)             # (0, 1) -> (0, 0) sums to 0; NaN adds 0 to (0, 1)
    assert list(zip(out[0][0].tolist(), out[0][1].tolist(), out[0][2].tolist())) == [(1, 1, 3.0)]


def _dense(out, sizes, c):
    n = sizes[c]
    m = np.zeros((n, n))
    i, j, x = out[c]
    np.add.at(m, (i, j), x)
    return m


@pytest.mark.parametrize("factor", [2, 3, 7, 40])
def test_dense_coarse_matrix_is_a_block_sum_of_the_fine_upper_triangle(factor):
    b1, b2, v = _genome(4)
    fine, _, _ = C.coarsen_pixels(SIZES, b1, b2, v, 1)
    coarse, _, _ = C.coarsen_pixels(SIZES, b1, b2, v, factor)
    cb = C.coarse_bins(SIZES, factor)
    for c, n in enumerate(SIZES):
        f = _dense(fine, SIZES, c)
        pad = np.zeros((cb[c] * factor, cb[c] * factor))
        pad[:n, :n] = f
        want = pad.reshape(cb[c], factor, cb[c], factor).sum(axis=(1, 3))
        assert np.array_equal(_dense(coarse, cb, c), want)
        assert not np.tril(want, -1).any()


@pytest.mark.parametrize("a,b", [(2, 3), (3, 2), (2, 2), (5, 7), (1, 4)])
def test_composition_equals_the_product(a, b):
    b1, b2, v = _genome(5)
    first, _, _ = C.coarsen_pixels(SIZES, b1, b2, v, a)
    mid = C.coarse_bins(SIZES, a)
    two, _, _ = C.coarsen_pixels(mid, *_global(first, mid), b)
    once, _, _ = C.coarsen_pixels(SIZES, b1, b2, v, a * b)
    assert C.coarse_bins(mid, b) == C.coarse_bins(SIZES, a * b)
    assert _same(two, once)


def test_a_factor_of_at_least_n_gives_one_bin():
    b1, b2, v = _genome(6)
    for factor in (37, 38, 10 ** 6):
        out, _, _ = C.coarsen_pixels(SIZES, b1, b2, v, factor)
        assert C.coarse_bins(SIZES, factor) == [1, 1, 1, 1]
        for c, (i, j, x) in enumerate(out[:3]):
            per, _, _ = C.coarsen_pixels(SIZES, b1, b2, v, 1)
            assert i.tolist() == [0] and j.tolist() == [0] and x[0] == per[c][2].sum()


# ---- host logic on a stand-in genome --------------------------------------------------------------------------------

class _FakeGenome:
    def __init__(self, chrom_bins, log):
        self.chrom_bins = np.array(chrom_bins, dtype=np.int32)
        self.log = log

    def coarsen(self, factor):
        self.log.append(("coarsen", factor))
        return _FakeGenome(-(-self.chrom_bins // factor), self.log)

    def downsample(self, contacts, seed):
        self.log.append(("downsample", contacts))
        return _FakeGenome(self.chrom_bins, self.log)

    def depth(self):
        return np.array([10, 10], dtype=np.uint64)

    def close(self):
        pass


class _FakeCtx:
    closed = False

    def close(self):
        self.closed = True


def test_coarsen_factor_bookkeeping_and_argument_errors():
    log = []
    ctx = _FakeCtx()
    g = LoadedGenome(_FakeGenome([10, 5], log), ["chrA", "chrB"], _CtxRef(ctx, True))
    assert g.factor == 1
    c2 = g.coarsen(2)
    assert c2.factor == 2 and c2.chrom_bins.tolist() == [5, 3] and c2.names == g.names and c2.ctx is g.ctx
    c6 = c2.coarsen(np.int64(3))
    assert c6.factor == 6 and c6.chrom_bins.tolist() == [2, 1]
    assert c2.coarsen(3.0).factor == 6
    assert c6.downsample(contacts=5).factor == 6
    assert log == [("coarsen", 2), ("coarsen", 3), ("coarsen", 3), ("downsample", 5)]
    for bad in (0, -1, True, False, 2.5, float("nan"), float("inf"), "2", None, 2 ** 31):
        with pytest.raises(ValueError, match="factor must be an integer"):
            g.coarsen(bad)
    assert len(log) == 4
    g.close()
    with pytest.raises(ValueError, match="closed"):
        g.coarsen(2)
    assert not ctx.closed                          # c2 and c6 still use the context
    c2.close()
    c6.close()
    assert ctx.closed


# ---- ABI and R ------------------------------------------------------------------------------------------------------

def test_symbol_is_declared_and_bound():
    with open(os.path.join(ROOT, "include", "tadpole_b200.h")) as fh:
        assert re.search(r"\bint tp_genome_coarsen\(tp_ctx \*ctx, const tp_genome \*src, int factor, tp_genome \*\*out\);",
                         fh.read())
    assert "tp_genome_coarsen" in _lib.EXPORTED
    lib = _lib.load()
    assert lib.tp_version() >= 108
    out = ctypes.c_void_p()
    for args in ((None, None, 2, ctypes.byref(out)), (None, None, 0, ctypes.byref(out)), (None, None, 2, None)):
        assert lib.tp_genome_coarsen(*args) == _lib.TP_ERR_ARG
        assert "null argument" in lib.tp_last_error().decode()


@pytest.fixture(scope="module")
def R():
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import __graft_entry__ as g
    g.build()
    from mock_r.driver import MockR
    r = MockR()
    yield r
    r.reset()


def test_r_routine_is_registered_and_checks_its_arguments(R):
    from mock_r.driver import RError
    assert R.registered("C_tp_genome_coarsen") == 4
    with pytest.raises(RError, match="takes 4 arguments"):
        R.call("C_tp_genome_coarsen", 0, 0, 1)
    for bad in (0.0, -2.0, 1.5, float("nan"), 2.0 ** 31):
        with pytest.raises(RError, match="factor must be a whole number"):
            R.call("C_tp_genome_coarsen", 0, 0, 1, bad)
    with pytest.raises(RError, match="GPU context has been released"):
        R.call("C_tp_genome_coarsen", 0, 0, 1, 2.0)


def test_r_function_is_exported_and_carries_the_factor():
    pkg = os.path.join(ROOT, "r-package", "TADpoleB200")
    with open(os.path.join(pkg, "NAMESPACE")) as fh:
        assert "export(genome_coarsen)" in fh.read().split("\n")
    with open(os.path.join(pkg, "R", "tadpole.R")) as fh:
        src = fh.read()
    body = src[src.index("genome_coarsen <- function(g, factor)"):]
    body = body[:body.index("\n}\n")]
    assert "ceiling(attr(g, \"n\") / factor)" in body and 'attr(g, "factor") * factor' in body
    assert "stop(\"factor must be a whole number >= 1\")" in body
    down = src[src.index("genome_downsample <- function("):]
    assert '.tp_loaded(p[[1L]], tab, attr(g, "ctx"), attr(g, "factor"))' in down[:down.index("\n}\n")]
