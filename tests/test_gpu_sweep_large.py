"""GPU tests of the n_pcs sweep above the size where each candidate's dSS array fits in one SM's shared memory (~27 700
good bins): there the leaf level of the array lives in the candidate's row of d0 in HBM (coniss_sweep_kernel<...,
DSS_GLOBAL>), the min tree and the live-boundary bitmap stay in shared memory.  Checked through

  * the global leaf array forced at any size (TADPOLE_SWEEP_DSS=global) against the shared-memory path on the same
    scores: n_cluster, the whole score matrix with its NaN pattern, seqdist and merge order of several candidates are
    the same bits                                                             (same arithmetic, only where d is stored)
  * the C oracle (Lance-Williams CONISS on a full distance matrix) on 30 000-bin scores: identical merge order
                                                                                             (rioja::chclust, R/TADpole.R:108)
  * last CONISS height = total sum of squares of the clustered columns                       (chclust)
  * broken-stick level count and Calinski-Harabasz recomputed on the host from the returned dendrogram
                                                                                              (R/TADpole.R:111-120)
  * TAD tables partition the good bins of a 47 000-bin call (n^2 > 2^31)                      (R/TADpole.R:470-497)
and, when the box has >= 2 GPUs, a 2-device context call at 32 000 bins equals the one-GPU call bit for bit.
"""
import threading

import numpy as np
import pytest

from oracle import tadpole_oracle as O

pytestmark = pytest.mark.gpu


def _structured_scores(n, k, seed, nblocks=None):
    """Seeded stand-in for PC scores: block means (TAD-like stretches) plus noise, columns of decreasing scale, centred."""
    rng = np.random.default_rng(seed)
    nblocks = nblocks or max(2, n // 60)
    cuts = np.sort(rng.choice(np.arange(1, n), nblocks - 1, replace=False))
    lab = np.zeros(n, np.int64)
    lab[cuts] = 1
    lab = np.cumsum(lab)
    means = rng.standard_normal((nblocks, k)) * 3.0
    s = (means[lab] + rng.standard_normal((n, k))) * (1.0 + np.arange(k)) ** -0.5
    return s - s.mean(axis=0)


def _sweep(ctx, pcs, k, **kw):
    """(n_cluster, scores) of one sweep on these scores, or None for both when some candidate has no significant level"""
    ctx.set_scores(pcs)
    try:
        return ctx.sweep(k, **kw)
    except Exception:
        return None, None                       # (a candidate without a significant level: the dendrograms exist)


def _same_bits(ctx, monkeypatch, pcs, cands, **kw):
    """default plan, then the global leaf array forced, on the same scores: everything the sweep returns is identical"""
    n, k = pcs.shape
    monkeypatch.delenv("TADPOLE_SWEEP_DSS", raising=False)
    ncl_a, sc_a = _sweep(ctx, pcs, k, **kw)
    ref = {i: ctx.dendro(i - 1, n) for i in cands}
    monkeypatch.setenv("TADPOLE_SWEEP_DSS", "global")
    ncl_b, sc_b = _sweep(ctx, pcs, k, **kw)
    monkeypatch.delenv("TADPOLE_SWEEP_DSS")
    assert (ncl_a is None) == (ncl_b is None)
    if ncl_a is not None:
        assert np.array_equal(ncl_a, ncl_b) and np.array_equal(sc_a, sc_b, equal_nan=True)
    for i, (seq, order) in ref.items():
        seq_b, order_b = ctx.dendro(i - 1, n)
        assert np.array_equal(order, order_b), f"merge order differs at {i} PCs"
        assert np.array_equal(seq, seq_b), f"seqdist differs at {i} PCs"
        assert sorted(order_b.tolist()) == list(range(n - 1))
    return ref


def test_global_leaves_links_path_2k(ctx, monkeypatch):
    """~2 000 bins: the default plan keeps the dSS array, link arrays and reciprocal table in shared memory"""
    pcs = _structured_scores(2000, 200, seed=1)
    ref = _same_bits(ctx, monkeypatch, pcs, (1, 2, 9, 77, 200))
    for i in (1, 9):
        assert np.array_equal(ref[i][1], O.coniss_lw(pcs[:, :i])[1])


def test_global_leaves_bitmap_path_20k(ctx, monkeypatch):
    """~20 000 bins: the default plan uses the live-boundary bitmap beside the shared dSS array"""
    _same_bits(ctx, monkeypatch, _structured_scores(20000, 200, seed=2), (1, 3, 50, 199, 200))


def test_global_leaves_structural_ties(ctx, monkeypatch):
    """the inputs of test_sweep_structural_ties_follow_the_reference: identical rows, runs, far-apart duplicates"""
    rng = np.random.default_rng(7)
    n, k = 900, 24
    pcs = np.cumsum(rng.standard_normal((n, k)), axis=0) * (1.0 + np.arange(k)) ** -0.7
    v = rng.standard_normal(k) * 3.0
    w = rng.standard_normal(k) * 0.5
    pcs[[5, 40, 41, 42, 43, 100, 123, 124, 300, 301, 302, 500, 520, 521, 640, 641, 642, 643, 644, 777, 898]] = v
    pcs[[200, 230, 231, 260]] = w
    pcs[600:606] = pcs[600]
    pcs -= pcs.mean(0)
    ref = _same_bits(ctx, monkeypatch, pcs, (1, 2, 7, 24))
    for i in (1, 24):
        assert np.array_equal(ref[i][1], O.coniss_lw(pcs[:, :i])[1])


def test_global_leaves_zero_variance_families(ctx, monkeypatch):
    """every zero-variance bin gets the same row of scores (quirk Q9): families of exactly tied increases, 0 included"""
    rng = np.random.default_rng(11)
    n, k = 3000, 60
    pcs = _structured_scores(n, k, seed=11)
    zero = np.concatenate([rng.choice(n, 90, replace=False), np.arange(1200, 1240), np.arange(n - 5, n)])
    pcs[zero] = pcs[zero[0]]
    ones = rng.choice(n, 30, replace=False)
    pcs[ones] = rng.standard_normal(k) * 0.1
    ref = _same_bits(ctx, monkeypatch, pcs, (1, 2, 30, 60))
    assert np.array_equal(ref[2][1], O.coniss_lw(pcs[:, :2])[1])


def test_global_leaves_candidate_sharding(ctx, monkeypatch):
    """a rank of a candidate-sharded sweep (cand_begin = 1, cand_stride = 2)"""
    _same_bits(ctx, monkeypatch, _structured_scores(2500, 200, seed=3), (2, 4, 100, 200), cand_begin=1, cand_stride=2)


def _check_levels(seq, s, row, i):
    """last height, n_cluster and three CH values of candidate i (1-based) from its dendrogram `seq`"""
    pcs = s[:, :i]
    tss = ((pcs - pcs.mean(axis=0)) ** 2).sum()
    assert seq.max() == pytest.approx(tss, rel=1e-9)
    disp, bs = O.bstick_table(seq)
    ncl = O.first_true_run(disp > bs)
    levels = np.flatnonzero(~np.isnan(row)) + 1
    assert ncl == levels[-1]                                 # broken stick + first-TRUE-run rule (quirk Q1)
    n = s.shape[0]
    tot = ((s - s.mean(axis=0)) ** 2).sum()                  # CH on ALL k columns (quirk Q2)
    for lv in (levels[0], levels[len(levels) // 2], levels[-1]):
        lab = O.cutree(seq, int(lv))
        edges = np.flatnonzero(np.diff(lab)) + 1
        w = sum(((blk - blk.mean(axis=0)) ** 2).sum() for blk in np.split(s, edges))
        assert row[lv - 1] == pytest.approx((n - lv) * (tot - w) / ((lv - 1) * w), rel=1e-8)


def test_sweep_30k_scores_against_the_c_oracle(ctx):
    """nf = 30 000, k = 40: above the shared-memory dSS array, so the default plan takes the global leaf array"""
    n, k = 30000, 40
    s = _structured_scores(n, k, seed=5, nblocks=400)
    ctx.set_scores(s)
    ncl, sc = ctx.sweep(k)
    for cand in range(1, k + 1):
        seq, order = ctx.dendro(cand - 1, n)
        assert sorted(order.tolist()) == list(range(n - 1))
        pcs = s[:, :cand]
        assert seq.max() == pytest.approx(((pcs - pcs.mean(axis=0)) ** 2).sum(), rel=1e-9)
    for cand in (1, 12):                                     # the full distance matrix: 7.2 GB on the host, seconds
        seq, order = ctx.dendro(cand - 1, n)
        oseq, oorder = O.coniss_lw(s[:, :cand])
        assert np.array_equal(order, oorder), f"merge order differs from the oracle's at {cand} PCs"
        np.testing.assert_allclose(seq, oseq, rtol=1e-11)
    for cand in (1, 12, 40):
        _check_levels(ctx.dendro(cand - 1, n)[0], s, sc[cand - 1], cand)


class _PeakMemory:
    """highest device memory in use (all processes) seen by a polling thread while the block runs"""
    def __init__(self, device=0, period=0.005):
        self.device, self.period, self.peak = device, period, 0

    def _poll(self):
        import torch
        while not self._stop.is_set():
            free, total = torch.cuda.mem_get_info(self.device)
            self.peak = max(self.peak, total - free)
            self._stop.wait(self.period)

    def __enter__(self):
        self._stop = threading.Event()
        self._t = threading.Thread(target=self._poll, daemon=True)
        self._t.start()
        return self

    def __exit__(self, *exc):
        self._stop.set()
        self._t.join()


def test_47k_chromosome_call_device_resident():
    """n = 47 000 > 46 341 (n^2 > 2^31): the whole call on a device-resident matrix (what TADpole() runs for a matrix
    already in HBM: Context.call, then the object packer), checked without any n x n host matrix.  Device peak, the
    17.7 GB input included: 105.2 GB of the 180 GB of one B200 (1000 W power limit), seen by this test's polling thread.
    Eigen-residuals are left out here: tp_pca consumes the correlation matrix and the library hands out no device
    pointer to it, so checking them would mean a 17.7 GB host copy; test_gpu_chromosome checks them at 25 000 bins."""
    import torch
    from tadpole_b200 import Context, api
    from tadpole_b200.synth import synth_hic_gpu
    api.QUIET = True
    n = 47000
    d = synth_hic_gpu(n, seed=13, device=0)
    torch.cuda.synchronize()
    torch.cuda.empty_cache()
    ctx = Context(0)                     # its own context: the ~100 GB it holds go back when the test ends
    try:
        with _PeakMemory() as pm:
            res = ctx.call(device_ptr=d.data_ptr(), n=n, colmajor=0)
        del d
        torch.cuda.empty_cache()
        print(f"47k call: device peak {pm.peak / 1e9:.1f} GB")
        _check_47k(ctx, res, n)
    finally:
        ctx.close()


def _check_47k(ctx, res, n):
    from tadpole_b200 import api
    tp = api._tadpole_from_result(res, ctx)
    nf, bad = res["nf"], res["bad"]
    assert nf > 46341 and 1 <= tp.n_pcs <= 200
    for key, tab in tp.clusters.items():
        assert np.all(tab[:, 0] <= tab[:, 1]) and np.all(tab[1:, 0] > tab[:-1, 1]) and tab.shape[0] <= int(key)
        covered = np.zeros(n, bool)
        covered[np.concatenate([np.arange(a - 1, b) for a, b in tab])] = True
        assert covered[~bad].all()
    s = ctx.get_scores(nf, res["k"])
    for cand in sorted({tp.n_pcs, 2, 150}):
        seq, order = ctx.dendro(cand - 1, nf)
        assert sorted(order.tolist()) == list(range(nf - 1))
        assert np.all(np.diff(seq[order]) >= 0)
        _check_levels(seq, s, tp.scores[cand - 1], cand)
    assert np.array_equal(ctx.dendro(tp.n_pcs - 1, nf)[0], tp.dendro.seqdist)


@pytest.mark.skipif("__import__('tadpole_b200')._lib.device_count() < 2", reason="needs >= 2 GPUs")
def test_two_device_context_32k_equals_one_gpu():
    """one context over 2 devices (sharded Gram, operator applications and dealt-out sweep) at 32 000 bins"""
    import torch
    from tadpole_b200 import Context, api
    from tadpole_b200.synth import synth_hic_gpu
    api.QUIET = True
    n = 32000
    d = synth_hic_gpu(n, seed=17, device=0)
    torch.cuda.synchronize()
    torch.cuda.empty_cache()
    c1 = Context(0)
    try:
        one = c1.call(device_ptr=d.data_ptr(), n=n, colmajor=0)
    finally:
        c1.close()
    m2 = Context([0, 1])
    try:
        two = m2.call(device_ptr=d.data_ptr(), n=n, colmajor=0)
    finally:
        m2.close()
    del d
    torch.cuda.empty_cache()
    assert (one["n_pcs"], one["n_clusters"], one["nf"]) == (two["n_pcs"], two["n_clusters"], two["nf"])
    assert np.array_equal(one["bad"], two["bad"])
    assert np.array_equal(one["seqdist"], two["seqdist"])
    assert np.array_equal(one["scores"], two["scores"], equal_nan=True)
