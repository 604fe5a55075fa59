"""GPU tests of coarsening (csrc/coarsen.cu, DESIGN S0e: tp_genome_coarsen; LoadedGenome.coarsen).  Small genomes are
compared bit for bit with the pixel-by-pixel reference (tests/coarsen_oracle.py), a GRCh38-sized 10 kb genome with the
vectorised one; calls on a coarse genome must equal calls on a fresh ingest of the reference's coarse pixels."""
import math
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tests"))
pytestmark = pytest.mark.gpu

import coarsen_oracle as C  # noqa: E402
from oracle.genome_oracle import split_genome_pixels  # noqa: E402

SIZES = [400, 1, 300, 5, 7]                   # chromosome 4 holds no pixel
NMAX = max(SIZES)


def _small(seed=3, fractional=False):
    """Duplicated cells, zero and NaN counts, a pair that cancels, trans and below-diagonal pixels; shuffled."""
    rng = np.random.default_rng(seed)
    starts = np.concatenate(([0], np.cumsum(SIZES)))
    b1, b2, v = [], [], []
    for c in (0, 1, 2, 3):
        n = SIZES[c]
        i = rng.integers(0, n, 6000)
        j = np.minimum(n - 1, i + rng.integers(0, 40, i.size))
        x = rng.geometric(0.1, i.size).astype(float) - 1.0
        if fractional:
            x = x * rng.random(i.size) + 1e-3
        b1.append(starts[c] + i); b2.append(starts[c] + j); v.append(x)
    if not fractional:
        v[0][:50] = np.nan
        b1.append([2, starts[2] + 20, 5, 5]); b2.append([420, starts[2] + 10, 399, 399]); v.append([4.0, 6.0, 7.0, -7.0])
    else:
        b1.append([2, starts[2] + 20]); b2.append([420, starts[2] + 10]); v.append([4.0, 6.0])
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
    return len(a) == len(b) and all(np.array_equal(x[0], y[0]) and np.array_equal(x[1], y[1]) and
                                    np.array_equal(np.asarray(x[2]).view(np.uint64), np.asarray(y[2]).view(np.uint64))
                                    for x, y in zip(a, b))


@pytest.fixture(scope="module")
def small():
    return _small()


@pytest.mark.parametrize("factor", [1, 2, 3, 7, NMAX - 1, NMAX, NMAX + 1, 10 ** 6])
def test_bit_equal_to_the_oracle(ctx, small, factor):
    want, trans, below = C.coarsen_pixels(SIZES, *small, factor)
    with _load(*small, ctx=ctx) as g, g.coarsen(factor) as cg:
        assert cg.factor == factor
        assert cg.chrom_bins.tolist() == C.coarse_bins(SIZES, factor)
        got = _pixels(cg)
        assert _same_pixels(got, want), factor
        cis, tr, bl = cg.stats()
        assert cis.tolist() == [w[0].size for w in want] and (tr, bl) == (trans, below) == g.stats()[1:] == (1, 1)
    assert want[4][0].size == 0


def test_integer_sums_just_below_2_53_are_exact(ctx):
    big = 2.0 ** 52
    parts = [big, big / 2, big / 4, big / 8, 1.0, 2.0, 3.0]          # with fill: eight cells of coarse cell (0, 0)
    total = sum(parts)
    fill = float(2 ** 53 - 1) - total                              # the cell's sum is 2^53 - 1
    assert 0 < fill < big and fill == int(fill)
    b1 = np.array([0, 1, 2, 3, 0, 1, 2, 3, 9], np.int32)
    b2 = np.array([0, 1, 2, 3, 3, 2, 3, 3, 9], np.int32)
    v = np.array(parts + [fill, 5.0])
    p = np.random.default_rng(0).permutation(v.size)
    with _load(b1[p], b2[p], v[p], sizes=[12], ctx=ctx) as g, g.coarsen(4) as cg:
        i, j, x = cg.pixels("chr1")
    assert i.tolist() == [0, 2] and j.tolist() == [0, 2] and x.tolist() == [float(2 ** 53 - 1), 5.0]


def test_fractional_counts_are_within_the_summation_bound(ctx):
    b1, b2, v = _small(7, fractional=True)
    u = 2.0 ** -53
    for factor in (2, 7, NMAX):
        want, _, _ = C.coarsen_pixels(SIZES, b1, b2, v, factor)
        with _load(b1, b2, v, ctx=ctx) as g, g.coarsen(factor) as cg:
            got = _pixels(cg)
        split, _, _ = split_genome_pixels(b1, b2, v, SIZES)
        for c, ((gi, gj, gx), (wi, wj, _), (fi, fj, fv)) in enumerate(zip(got, want, split)):
            assert np.array_equal(gi, wi) and np.array_equal(gj, wj), (factor, c)
            cells = {}
            for a, b, x in zip(fi.tolist(), fj.tolist(), fv.tolist()):
                cells.setdefault((a // factor, b // factor), []).append(x)
            for a, b, x in zip(gi.tolist(), gj.tolist(), gx.tolist()):
                vals = cells[(a, b)]
                m = len(vals)
                gam = (m - 1) * u / (1 - (m - 1) * u)
                assert abs(x - math.fsum(vals)) <= gam * sum(abs(t) for t in vals), (factor, c, a, b)


def test_composition_and_depth(ctx, small):
    b1, b2, v = small
    keep = ~np.isnan(v)                                             # depth needs integer counts
    b1, b2, v = b1[keep], b2[keep], np.abs(v[keep])
    with _load(b1, b2, v, ctx=ctx) as g:
        depth = g.depth()
        for a, b in ((2, 3), (3, 2), (7, 60), (1, 5)):
            with g.coarsen(a) as ga, ga.coarsen(b) as gab, g.coarsen(a * b) as gp:
                assert gab.factor == gp.factor == a * b
                assert gab.chrom_bins.tolist() == gp.chrom_bins.tolist()
                assert _same_pixels(_pixels(gab), _pixels(gp))
                assert ga.depth() == gab.depth() == depth
        N = g.total_depth // 3
        with g.coarsen(3) as g3, g3.downsample(contacts=N, seed=4) as d3, g.downsample(contacts=N, seed=4) as d, \
                d.coarsen(3) as c3:
            assert d3.total_depth == c3.total_depth == N
            assert d3.factor == c3.factor == 3


# ---- calls on a coarse genome ------------------------------------------------------------------------------------------

CALL_SIZES = [600, 480, 540]


@pytest.fixture(scope="module")
def callable_genome():
    from tadpole_b200.synth import synth_genome_pixels
    _, (b1, b2, v), _ = synth_genome_pixels(CALL_SIZES, seed=5, trans_per_chrom=20, centromere=[0, 1, 2])
    return b1, b2, v


def _fresh(b1, b2, v, factor):
    """GenomePixels of the reference's coarse pixels over the coarse bin table"""
    from tadpole_b200 import GenomePixels
    out, _, _ = C.coarsen_pixels_np(CALL_SIZES, b1, b2, v, factor)
    cb = C.coarse_bins(CALL_SIZES, factor)
    starts = np.concatenate(([0], np.cumsum(cb)))
    gb1 = np.concatenate([i + starts[c] for c, (i, _, _) in enumerate(out)]).astype(np.int32)
    gb2 = np.concatenate([j + starts[c] for c, (_, j, _) in enumerate(out)]).astype(np.int32)
    return GenomePixels(gb1, gb2, np.concatenate([x for _, _, x in out]), bins=list(zip(_names(CALL_SIZES), cb)))


@pytest.mark.parametrize("factor", [2, 3])
def test_calls_on_a_coarse_genome_equal_calls_on_a_fresh_ingest(ctx, callable_genome, factor):
    from genome_timing import same
    from tadpole_b200 import TADpole_genome, api
    api.QUIET = True
    with _load(*callable_genome, sizes=CALL_SIZES, ctx=ctx) as g, g.coarsen(factor) as cg:
        px = _fresh(*callable_genome, factor)
        a, b = TADpole_genome(cg, max_pcs=20), TADpole_genome(px, max_pcs=20, ctx=ctx)
        assert list(a) == list(b) == _names(CALL_SIZES) and not a.failed
        assert all(same(a[nm], b[nm]) for nm in a)
        a, b = (TADpole_genome(x, max_pcs=20, ctx=ctx, centromere_search=True, centromere_fix=True) for x in (cg, px))
        assert list(a) == list(b) and a.failed == b.failed
        split = 0
        for nm in a:
            if getattr(a[nm], "clusters", None) is None:
                split += 1
                assert all(same(a[nm][arm], b[nm][arm]) for arm in ("p", "q"))
                assert np.array_equal(a[nm].merging_arms, b[nm].merging_arms)
            else:
                assert same(a[nm], b[nm])
        assert split > 0
        r = TADpole_genome(cg, max_pcs=20, resident=True)
        rr = r.recall(max_pcs=20, min_clusters=3)
        fresh = TADpole_genome(px, max_pcs=20, min_clusters=3, ctx=ctx)
        assert all(same(rr[nm], fresh[nm]) for nm in fresh)


def test_difft_genome_on_two_equal_depth_coarse_samples(ctx, callable_genome):
    from tadpole_b200 import TADpole_genome, api, diffT_genome, equal_depth
    from tadpole_b200.synth import synth_genome_pixels
    api.QUIET = True
    _, (c1, c2, cv), _ = synth_genome_pixels(CALL_SIZES, seed=6, trans_per_chrom=20)
    with _load(*callable_genome, sizes=CALL_SIZES, ctx=ctx) as x, _load(c1, c2, cv, sizes=CALL_SIZES, ctx=ctx) as y:
        ex, ey = equal_depth(x, y, seed=4)
        with ex.coarsen(2) as cx, ey.coarsen(2) as cy:
            assert cx.total_depth == cy.total_depth == min(x.total_depth, y.total_depth)
            out = diffT_genome(TADpole_genome(cx, max_pcs=20), TADpole_genome(cy, max_pcs=20), nperm=50, ctx=ctx)
            assert len(out.chrom) + len(out.skipped) > 0
            assert np.all((out.p_value > 0) & (out.p_value <= 1))
        for s in (ex, ey):
            if s is not x and s is not y:
                s.close()


# ---- GRCh38 at 10 kb -----------------------------------------------------------------------------------------------------

def test_grch38_at_10kb_coarsened_by_5_equals_the_vectorised_reference(ctx):
    from genome_timing import GRCH38
    from tadpole_b200.synth import synth_sparse_genome_pixels
    sizes = [-(-ln // 10000) for _, ln in GRCH38]
    b1, b2, v = synth_sparse_genome_pixels(sizes, band=50, seed=1)
    assert v.size > 15_000_000
    want, _, _ = C.coarsen_pixels_np(sizes, b1, b2, v, 5)
    with _load(b1, b2, v, sizes=sizes, ctx=ctx) as g, g.coarsen(5) as cg:
        assert cg.chrom_bins.tolist() == C.coarse_bins(sizes, 5)
        assert _same_pixels(_pixels(cg), want)
        assert cg.total_depth == g.total_depth


# ---- errors and lifetime -------------------------------------------------------------------------------------------------

def test_errors_and_freeing_either_genome_first(ctx, small):
    from tadpole_b200 import TadpoleError
    want, _, _ = C.coarsen_pixels(SIZES, *small, 3)
    g = _load(*small, ctx=ctx)
    with pytest.raises(ValueError, match="factor must be an integer"):
        g.coarsen(0)
    with pytest.raises(TadpoleError, match="factor must be >= 1"):
        g._g.coarsen(0)
    c = g.coarsen(3)
    g.close()                                            # the source first
    with pytest.raises(ValueError, match="closed"):
        g.coarsen(2)
    assert _same_pixels(_pixels(c), want)
    g = _load(*small, ctx=ctx)
    c2 = g.coarsen(3)
    c2.close()                                           # the result first
    with g.coarsen(3) as c3:
        assert _same_pixels(_pixels(c3), want)
    g.close()
    c.close()


def test_a_context_without_the_handles_device_is_rejected(small):
    import ctypes
    from tadpole_b200 import Context
    from tadpole_b200._lib import TP_ERR_ARG, device_count
    if device_count() < 2:
        pytest.skip("needs 2 GPUs")
    zero, one = Context(0), Context(1)
    try:
        with _load(*small, ctx=zero) as g:
            out = ctypes.c_void_p()
            assert one.lib.tp_genome_coarsen(one._h, g._g._h, 2, ctypes.byref(out)) == TP_ERR_ARG
            assert "not a device of the context" in one.lib.tp_last_error().decode()
            assert not out.value
    finally:
        zero.close(); one.close()


def test_mock_r_routines_drive_the_library(ctx, callable_genome):
    from mock_r.driver import MockR
    from tadpole_b200 import TADpole_genome, api
    api.QUIET = True
    b1, b2, v = callable_genome
    R = MockR()
    try:
        rctx = R.call("C_tp_ctx", 0, raw=True)
        handle, _, tb = R.call("C_tp_genome", rctx, np.array(CALL_SIZES, np.int32), b1, b2, v, 0)
        h2, cis2, tb2 = R.call("C_tp_genome_coarsen", rctx, handle, len(CALL_SIZES), 2.0)
        with _load(b1, b2, v, sizes=CALL_SIZES, ctx=ctx) as g, g.coarsen(2) as cg:
            want = _pixels(cg)
            assert cis2.tolist() == [float(w[0].size) for w in want] and tb2.tolist() == tb.tolist()
            depth = R.call("C_tp_genome_depth", rctx, h2, len(CALL_SIZES))
            assert depth.tolist() == [float(x) for x in cg.depth().values()]
            for ch, (wi, wj, wv) in enumerate(want):
                i, j, x = R.call("C_tp_genome_pixels", rctx, h2, ch, len(CALL_SIZES))
                o = np.lexsort((j, i))
                assert np.array_equal(i[o], wi) and np.array_equal(j[o], wj) and np.array_equal(x[o], wv)
            sel = np.arange(len(CALL_SIZES), dtype=np.int32)
            out = R.call("C_tp_call_genome", rctx, h2, sel, 20, 2, 0.01, 4, True)
            py = TADpole_genome(cg, max_pcs=20)
            for item, nm in zip(out, cg.names):
                bad, npcs, ncl, seq, scores, levels, tables = item
                assert npcs[0] == py[nm].n_pcs and ncl[0] == py[nm].optimal_n_clusters
                assert np.array_equal(np.asarray(seq).view(np.uint64), py[nm].dendro.seqdist.view(np.uint64))
    finally:
        R.reset()
