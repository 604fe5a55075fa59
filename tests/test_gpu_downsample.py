"""GPU tests of equal-depth subsampling (csrc/downsample.cu, DESIGN S0d: tp_genome_depth, tp_genome_downsample,
tp_genome_pixels; LoadedGenome, equal_depth).  Small genomes are compared bit for bit with the read-by-read oracle
(tests/downsample_oracle.py); a genome of about 10^8 reads checks reproducibility and the hypergeometric
spread; calls on a subsample must equal calls on its exported pixels."""
import os
import sys

import numpy as np
import pytest


ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tests"))
pytestmark = pytest.mark.gpu

import downsample_oracle as G  # noqa: E402

SIZES = [400, 1, 300, 5]                     # chromosome 3 holds no pixel
BIG_CELL = 5_000_000


def _small(seed=3):
    """Duplicated cells, zero counts, trans and below-diagonal pixels, one cell of BIG_CELL reads; shuffled."""
    rng = np.random.default_rng(seed)
    starts = np.concatenate(([0], np.cumsum(SIZES)))
    b1, b2, v = [], [], []
    for c in (0, 1, 2):
        n = SIZES[c]
        i = rng.integers(0, n, 6000)
        j = np.minimum(n - 1, i + rng.integers(0, 40, i.size))
        b1.append(starts[c] + i); b2.append(starts[c] + j); v.append(rng.geometric(0.1, i.size).astype(float) - 1.0)
    b1.append([starts[2] + 7, 2, starts[2] + 20]); b2.append([starts[2] + 9, 420, starts[2] + 10])
    v.append([BIG_CELL, 4.0, 6.0])                                     # the big cell, a trans pixel, one below
    b1, b2, v = np.concatenate(b1), np.concatenate(b2), np.concatenate(v)
    p = rng.permutation(v.size)
    return b1[p].astype(np.int32), b2[p].astype(np.int32), v[p]


def _names(sizes):
    return [f"chr{c + 1}" for c in range(len(sizes))]


def _load(b1, b2, v, sizes=SIZES, ctx=None):
    from tadpole_b200 import GenomePixels
    return GenomePixels(b1, b2, v, bins=list(zip(_names(sizes), sizes))).load(ctx=ctx)


def _pixels(g):
    return [g.pixels(nm) for nm in g.names]


def _same_pixels(a, b):
    return all(np.array_equal(x[0], y[0]) and np.array_equal(x[1], y[1]) and np.array_equal(x[2], y[2])
               for x, y in zip(a, b))


@pytest.fixture(scope="module")
def small():
    b1, b2, v = _small()
    c, i, j, n = G.merged_cells(SIZES, b1, b2, v)
    return dict(b1=b1, b2=b2, v=v, total=int(n.sum()), cells=(c, i, j, n))


def test_depth_and_stats(ctx, small):
    with _load(small["b1"], small["b2"], small["v"], ctx=ctx) as g:
        c, _, _, n = small["cells"]
        want = [int(n[c == k].sum()) for k in range(len(SIZES))]
        assert list(g.depth().values()) == want and g.total_depth == small["total"] > BIG_CELL
        assert want[3] == 0
        sub = g.downsample(contacts=small["total"] // 2, seed=1)
        cis, trans, below = sub.stats()
        assert cis.tolist() == [p[0].size for p in _pixels(sub)]
        assert (trans, below) == g.stats()[1:] == (1, 1)
        assert sub.total_depth == small["total"] // 2
        sub.close()


@pytest.mark.parametrize("seed", [0, 12345, 2 ** 32 + 7])
def test_bit_equal_to_the_oracle(ctx, small, seed):
    T = small["total"]
    with _load(small["b1"], small["b2"], small["v"], ctx=ctx) as g:
        for N in (0, 1, T // 2, T - 1, T):
            with g.downsample(contacts=N, seed=seed) as sub:
                got = _pixels(sub)
            want = G.downsample(SIZES, small["b1"], small["b2"], small["v"], N, seed)
            assert sum(int(k.sum()) for _, _, k in got) == N
            for ch, ((gi, gj, gv), (wi, wj, wv)) in enumerate(zip(got, want)):
                assert np.array_equal(gi, wi) and np.array_equal(gj, wj) and np.array_equal(gv, wv), (seed, N, ch)


def test_order_and_duplicate_splitting_do_not_matter(ctx, small):
    b1, b2, v = small["b1"], small["b2"], small["v"]
    N = small["total"] // 3
    with _load(b1, b2, v, ctx=ctx) as g, g.downsample(contacts=N, seed=99) as s:
        ref = _pixels(s)
    p = np.random.default_rng(1).permutation(v.size)
    part = np.floor(v / 3)
    for args in ((b1[p], b2[p], v[p]), (np.concatenate((b1, b1)), np.concatenate((b2, b2)), np.concatenate((part, v - part)))):
        with _load(*args, ctx=ctx) as g, g.downsample(contacts=N, seed=99) as s:
            assert _same_pixels(_pixels(s), ref)


def test_errors_and_freeing_the_source_first(ctx, small):
    from tadpole_b200 import TadpoleError
    b1, b2, v = small["b1"].copy(), small["b2"], small["v"].copy()
    bad = int(np.flatnonzero((v > 0) & (b1 < 400) & (b1 <= b2))[0])
    v[bad] = 2.5
    with _load(b1, b2, v, ctx=ctx) as g:
        for call in (lambda: g.depth(), lambda: g._g.downsample(1, 0)):
            with pytest.raises(TadpoleError, match=r"chromosome 0 \(0-based\), bins \(%d, %d\).*count 2\.5 is not an integer"
                               % (b1[bad], b2[bad])):
                call()
    with _load(np.array([0, 0, 1], np.int32), np.array([0, 0, 2], np.int32), np.array([2.0 ** 31, 2.0 ** 31, 1.0]),
               sizes=[3]) as g:
        with pytest.raises(TadpoleError, match=r"bins \(0, 0\).*2\^32 reads or more"):
            g._g.downsample(1, 0)
    g = _load(small["b1"], small["b2"], small["v"], ctx=ctx)
    with pytest.raises(TadpoleError, match="contacts asked for"):
        g._g.downsample(small["total"] + 1, 0)
    sub = g.downsample(fraction=0.25, seed=5)
    want = G.downsample(SIZES, small["b1"], small["b2"], small["v"], small["total"] // 4, 5)
    g.close()
    got = _pixels(sub)
    assert all(np.array_equal(a[2], b[2]) and np.array_equal(a[0], b[0]) for a, b in zip(got, want))
    sub.close()


# ---- about 10^8 reads ---------------------------------------------------------------------------------------------------

@pytest.fixture(scope="module")
def big():
    from genome_timing import GRCH38
    from tadpole_b200.synth import synth_sparse_genome_pixels
    sizes = [-(-ln // 50000) for _, ln in GRCH38]
    b1, b2, v = synth_sparse_genome_pixels(sizes, band=100, mean_count=16.0, seed=3)
    return sizes, b1, b2, v


def test_large_genome_is_reproducible_and_hypergeometric(ctx, big):
    sizes, b1, b2, v = big
    seed = 2 ** 40 + 1
    with _load(b1, b2, v, sizes, ctx) as g:
        depth = np.array(list(g.depth().values()), dtype=np.float64)
        T = int(depth.sum())
        assert T == int(v.sum()) > 9e7
        N = T // 2
        with g.downsample(contacts=N, seed=seed) as s1, g.downsample(contacts=N, seed=seed) as s2:
            ref = _pixels(s1)
            assert _same_pixels(_pixels(s2), ref)
            kept = np.array(list(s1.depth().values()), dtype=np.float64)
    assert kept.sum() == N
    p = depth / T
    sd = np.sqrt(N * p * (1 - p) * (T - N) / (T - 1))
    assert np.all(np.abs(kept - N * p) <= 6 * sd), (kept - N * p) / sd
    perm = np.random.default_rng(2).permutation(v.size)
    part = np.floor(v / 2)
    for args in ((b1[perm], b2[perm], v[perm]), (np.concatenate((b1, b1)), np.concatenate((b2, b2)), np.concatenate((part, v - part)))):
        with _load(*args, sizes=sizes, ctx=ctx) as g, g.downsample(contacts=N, seed=seed) as s:
            assert _same_pixels(_pixels(s), ref)


# ---- calls on a subsample -------------------------------------------------------------------------------------------------

CALL_SIZES = [320, 260, 300]


@pytest.fixture(scope="module")
def callable_genome():
    from tadpole_b200.synth import synth_genome_pixels
    names, (b1, b2, v), _ = synth_genome_pixels(CALL_SIZES, seed=5, trans_per_chrom=20, centromere=[0, 1, 2])
    assert np.array_equal(v, np.floor(v))
    return b1, b2, v


def _exported(sub, sizes):
    from tadpole_b200 import GenomePixels
    starts = np.concatenate(([0], np.cumsum(sizes)))
    parts = _pixels(sub)
    b1 = np.concatenate([i + starts[c] for c, (i, _, _) in enumerate(parts)])
    b2 = np.concatenate([j + starts[c] for c, (_, j, _) in enumerate(parts)])
    return GenomePixels(b1, b2, np.concatenate([x for _, _, x in parts]), bins=list(zip(_names(sizes), sizes)))


def test_calls_on_a_subsample_equal_calls_on_its_pixels(ctx, callable_genome):
    from genome_timing import same
    from tadpole_b200 import TADpole_genome, api
    api.QUIET = True
    with _load(*callable_genome, sizes=CALL_SIZES, ctx=ctx) as g, g.downsample(fraction=0.5, seed=8) as sub:
        px = _exported(sub, CALL_SIZES)
        a, b = TADpole_genome(sub, max_pcs=20), TADpole_genome(px, max_pcs=20, ctx=ctx)
        assert list(a) == list(b) == _names(CALL_SIZES) and not a.failed
        assert all(same(a[nm], b[nm]) for nm in a)
        a, b = (TADpole_genome(x, max_pcs=20, ctx=ctx, centromere_search=True, centromere_fix=True) for x in (sub, px))
        assert list(a) == list(b) and a.failed == b.failed
        for nm in a:
            if getattr(a[nm], "clusters", None) is None:
                assert all(same(a[nm][arm], b[nm][arm]) for arm in ("p", "q"))
                assert np.array_equal(a[nm].merging_arms, b[nm].merging_arms)
            else:
                assert same(a[nm], b[nm])
        r = TADpole_genome(sub, max_pcs=20, resident=True)
        rr = r.recall(max_pcs=20, min_clusters=3)
        fresh = TADpole_genome(px, max_pcs=20, min_clusters=3, ctx=ctx)
        assert all(same(rr[nm], fresh[nm]) for nm in fresh)
        assert g.total_depth > sub.total_depth > 0


def test_difft_genome_on_two_equal_depth_samples(ctx, callable_genome):
    from tadpole_b200 import TADpole_genome, api, diffT_genome, equal_depth
    from tadpole_b200.synth import synth_genome_pixels
    api.QUIET = True
    _, (c1, c2, cv), _ = synth_genome_pixels(CALL_SIZES, seed=6, trans_per_chrom=20)
    with _load(*callable_genome, sizes=CALL_SIZES, ctx=ctx) as x, _load(c1, c2, cv, sizes=CALL_SIZES, ctx=ctx) as y:
        ex, ey = equal_depth(x, y, seed=4)
        assert ex.total_depth == ey.total_depth == min(x.total_depth, y.total_depth)
        assert (ex is x) != (ey is y)
        out = diffT_genome(TADpole_genome(ex, max_pcs=20), TADpole_genome(ey, max_pcs=20), nperm=50, ctx=ctx)
        assert len(out.chrom) + len(out.skipped) > 0
        assert np.all((out.p_value > 0) & (out.p_value <= 1))
        for s in (ex, ey):
            if s is not x and s is not y:
                s.close()


def test_two_devices_equal_one(callable_genome):
    from genome_timing import same
    from tadpole_b200 import Context, TADpole_genome, api
    from tadpole_b200._lib import device_count
    if device_count() < 2:
        pytest.skip("needs 2 GPUs")
    api.QUIET = True
    one, two = Context(0), Context([0, 1])
    try:
        results = []
        for c in (one, two):
            with _load(*callable_genome, sizes=CALL_SIZES, ctx=c) as g, g.downsample(fraction=0.5, seed=8) as sub:
                results.append((_pixels(sub), TADpole_genome(sub, max_pcs=20)))
        assert _same_pixels(results[0][0], results[1][0])
        assert all(same(results[0][1][nm], results[1][1][nm]) for nm in results[0][1])
    finally:
        one.close(); two.close()


def test_mock_r_routines_drive_the_library(small):
    from mock_r.driver import MockR, RError
    R = MockR()
    try:
        rctx = R.call("C_tp_ctx", 0, raw=True)
        handle, cis, tb = R.call("C_tp_genome", rctx, np.array(SIZES, np.int32), small["b1"], small["b2"], small["v"], 0)
        c, _, _, n = small["cells"]
        depth = R.call("C_tp_genome_depth", rctx, handle, len(SIZES))
        assert depth.tolist() == [float(n[c == k].sum()) for k in range(len(SIZES))]
        N = small["total"] // 2
        h2, cis2, tb2 = R.call("C_tp_genome_downsample", rctx, handle, len(SIZES), float(N), 77.0)
        want = G.downsample(SIZES, small["b1"], small["b2"], small["v"], N, 77)
        assert cis2.tolist() == [float(w[0].size) for w in want] and tb2.tolist() == tb.tolist()
        for ch, (wi, wj, wv) in enumerate(want):
            i, j, x = R.call("C_tp_genome_pixels", rctx, h2, ch, len(SIZES))
            o = np.lexsort((j, i))
            assert np.array_equal(i[o], wi) and np.array_equal(j[o], wj) and np.array_equal(x[o], wv)
        with pytest.raises(RError, match="contacts asked for"):
            R.call("C_tp_genome_downsample", rctx, handle, len(SIZES), float(small["total"] + 1), 0.0)
        with pytest.raises(RError, match="whole number"):
            R.call("C_tp_genome_downsample", rctx, handle, len(SIZES), 1.5, 0.0)
        with pytest.raises(RError, match="out of range"):
            R.call("C_tp_genome_pixels", rctx, h2, len(SIZES), len(SIZES))
    finally:
        R.reset()
