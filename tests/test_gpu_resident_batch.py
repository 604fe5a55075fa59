"""GPU tests of the resident batch handle (csrc/group.cu: "batch_resident", tp_batch_recall, tp_batch_dendro,
tp_batch_resident_bytes) through TADpole_batch / TADpole_genome(resident=True), Tadpole.recall / dendro_for and
GenomeResult.recall.  A recall runs the same sweep and CH kernels on the same PC scores as tp_recall on the context of a
single call, so every comparison here is bit for bit: against the genome call itself at the same max_pcs, and against
TADpole() on the chromosome's dense matrix followed by its own recall() / dendro_for()."""
import ctypes
import gc

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

# five chromosomes of 300-2500 bins, one of 64 bins and one of 2 bins, which fails
SIZES = [1200, 300, 2, 2500, 64, 800, 1700]
CEN_SIZES = [900, 1500, 700, 1100]
CEN = [0, 1, 3]                        # drawn with a centromere; chromosome 2 does not split


def same(a, b):
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    return a.shape == b.shape and np.array_equal(np.isnan(a), np.isnan(b)) and \
        np.array_equal(a.view(np.uint64)[~np.isnan(a)], b.view(np.uint64)[~np.isnan(b)])


def same_tables(a, b):
    assert sorted(a) == sorted(b)
    for k in a:
        assert np.array_equal(a[k], b[k]), f"level {k}"


def same_whole(a, b):
    assert (a.n_pcs, a.optimal_n_clusters) == (b.n_pcs, b.optimal_n_clusters)
    assert same(a.dendro.seqdist, b.dendro.seqdist) and np.array_equal(a.dendro.labels, b.dendro.labels)
    assert same(a.scores, b.scores)
    same_tables(a.clusters, b.clusters)


def same_obj(a, b):
    if b.get("p") is None:
        same_whole(a, b)
        return
    for arm in ("p", "q"):
        x, y = a[arm], b[arm]
        assert (x.n_pcs, x.optimal_n_clusters) == (y.n_pcs, y.optimal_n_clusters)
        assert same(x.dendro.seqdist, y.dendro.seqdist) and np.array_equal(x.dendro.labels, y.dendro.labels)
        same_tables(x.cluster, y.cluster)
        assert (x.scores is None) == (y.scores is None) and (x.scores is None or same(x.scores, y.scores))
    assert np.array_equal(a.merging_arms, b.merging_arms)


def same_genome(a, b):
    assert list(a) == list(b) and a.failed == b.failed and a.stats == b.stats
    for nm in b:
        same_obj(a[nm], b[nm])


def _pixels(sizes, seed, centromere=None):
    from tadpole_b200 import GenomePixels
    from tadpole_b200.synth import synth_genome_pixels
    names, (b1, b2, v), _ = synth_genome_pixels(sizes, seed=seed, centromere=centromere)
    return GenomePixels(b1, b2, v, bins=list(zip(names, sizes)))


@pytest.fixture(scope="module")
def px():
    return _pixels(SIZES, 3)


@pytest.fixture(scope="module")
def pxc():
    return _pixels(CEN_SIZES, 5, CEN)


def dense_of(ctx, pixels):
    """{name: the dense matrix the genome call sees} (Genome.matrix) of every chromosome of 2 bins or more."""
    g = pixels._ingest(ctx)
    try:
        return {nm: g.matrix(c) for c, (nm, n) in enumerate(zip(pixels.names, pixels.chrom_bins)) if n >= 2}
    finally:
        g.close()


@pytest.fixture(autouse=True)
def quiet():
    from tadpole_b200 import api
    api.QUIET = True


def test_genome_recall_equals_fresh_genome_call(ctx, px):
    from tadpole_b200 import TADpole, TADpole_genome
    res = TADpole_genome(px, resident=True, ctx=ctx)
    same_genome(res, TADpole_genome(px, ctx=ctx))                  # resident mode changes no result
    assert "chr3" in res.failed and len(res) == len(SIZES) - 1
    dense = dense_of(ctx, px)
    for m, c in ((200, 3), (50, 2), (17, 2)):
        rec = res.recall(max_pcs=m, min_clusters=c)
        assert rec.failed == res.failed and rec.stats == res.stats
        fresh = TADpole_genome(px, max_pcs=m, min_clusters=c, ctx=ctx)
        if m == 200:
            same_genome(rec, fresh)
        else:
            # a fresh call with fewer PCs runs its PCA with a narrower block: the same decomposition, not the same bits;
            # what the user reads off it agrees
            assert list(rec) == list(fresh) and rec.failed == fresh.failed
            for nm in fresh:
                assert (rec[nm].n_pcs, rec[nm].optimal_n_clusters) == (fresh[nm].n_pcs, fresh[nm].optimal_n_clusters), nm
        # fewer PCs: what tp_recall gives on the context of a single call with the same max_pcs as the genome call
        for nm in res:
            same_whole(rec[nm], TADpole(dense[nm], ctx=ctx).recall(max_pcs=m, min_clusters=c))
        if m == 50:
            same_genome(rec.recall(max_pcs=17, min_clusters=2), res.recall(max_pcs=17, min_clusters=2))   # recall of a recall
    sub = res.recall(max_pcs=40, chroms=["chr6", "chr1"])
    assert list(sub) == ["chr6", "chr1"]
    same_whole(sub["chr1"], res["chr1"].recall(max_pcs=40))


def test_objects_equal_single_call_handles(ctx, px):
    from tadpole_b200 import TADpole, TADpole_batch, TADpole_genome
    dense = dense_of(ctx, px)
    res = TADpole_genome(px, resident=True, ctx=ctx, chroms=["chr4", "chr2", "chr5"])
    mats = [dense[nm] for nm in ("chr1", "chr6", "chr2")]
    batch = TADpole_batch(mats, resident=True, ctx=ctx)
    for obj, m in [(res[nm], dense[nm]) for nm in res] + list(zip(batch, mats)):
        ref = TADpole(m, ctx=ctx)
        same_whole(obj, ref)
        k = min(200, ref.dendro.labels.size)
        for n in (1, ref.n_pcs, k):
            assert same(obj.dendro_for(n).seqdist, ref.dendro_for(n).seqdist), n
            assert np.array_equal(obj.dendro_for(n).labels, ref.dendro.labels)
        rec, rref = obj.recall(max_pcs=40, min_clusters=3), ref.recall(max_pcs=40, min_clusters=3)
        same_whole(rec, rref)
        for n in (1, rec.n_pcs, min(40, k)):
            assert same(rec.dendro_for(n).seqdist, rref.dendro_for(n).seqdist), n
        same_whole(obj.recall(), TADpole(m, ctx=ctx))               # the source object is not used up by a recall


@pytest.mark.parametrize("fix", [False, True])
def test_arms(ctx, pxc, fix):
    from tadpole_b200 import TADpole_genome
    kw = dict(centromere_search=True, centromere_fix=fix, ctx=ctx)
    res = TADpole_genome(pxc, resident=True, **kw)
    same_genome(res, TADpole_genome(pxc, **kw))
    assert "merging_arms" in res["chr1"] and "merging_arms" in res["chr2"]
    for c in (3, 2):
        same_genome(res.recall(max_pcs=200, min_clusters=c), TADpole_genome(pxc, min_clusters=c, **kw))
    dense = dense_of(ctx, pxc)
    for nm, obj in res.items():
        if obj.get("p") is None:                                    # centromere_fix, not split: a whole call
            continue
        with pytest.raises(ValueError, match="arms"):
            obj.dendro_for(1)
        ctx.filter(mat=dense[nm])
        for arm in ("p", "q"):
            a = obj[arm]
            keep = a.dendro.labels.astype(np.int32) - 1
            fresh = ctx.call_arm(keep)
            k = fresh["k"]
            for n in (1, a.n_pcs, k):
                seq, _ = ctx.dendro(n - 1, keep.size)
                assert same(a.dendro_for(n).seqdist, seq), (nm, arm, n)
            assert same(a.dendro_for(a.n_pcs).seqdist, a.dendro.seqdist)


def test_errors(ctx, px):
    from tadpole_b200 import TADpole_batch, TADpole_genome, _lib
    res = TADpole_genome(px, max_pcs=60, resident=True, ctx=ctx)
    rec = res.recall(max_pcs=100)
    over = [nm for nm in res if res[nm].dendro.labels.size > 60]
    assert over and set(rec.failed) == set(res.failed) | set(over)
    for nm in over:
        assert "tp_recall: max_pcs = 100 needs" in rec.failed[nm] and "holds 60" in rec.failed[nm]
    for nm in set(res) - set(over):
        assert nm in rec
    with pytest.raises(Exception, match="holds 60"):
        res[over[0]].recall(max_pcs=100)
    # default mode: no handle, as before
    plain = TADpole_genome(px, ctx=ctx, chroms=["chr2"])
    for call in (lambda: plain["chr2"].recall(), lambda: plain["chr2"].dendro_for(2), lambda: plain.recall()):
        with pytest.raises(RuntimeError, match="carries no device handle"):
            call()
    with pytest.raises(RuntimeError, match="carries no device handle"):
        TADpole_batch([dense_of(ctx, px)["chr2"]], ctx=ctx)[0].recall()
    # selections outside the batch fail the library call; a failed item or a missing arm fails that item only
    store = res["chr1"]._resident()["batch"]
    for items, parts in (([99], [-1]), ([0], [2])):
        with pytest.raises(_lib.TadpoleError, match="outside items"):
            store.recall(items, parts)
    out, _ = store.recall([2, 0, 0], [-1, 0, -1], max_pcs=60)
    assert "failed" in str(out[0]) and "does not exist" in str(out[1]) and not isinstance(out[2], Exception)
    assert out[0].code == out[1].code == _lib.TP_ERR_ARG


def test_resident_bytes_and_release(ctx, px):
    import torch
    from tadpole_b200 import TADpole_genome, _lib
    rb = lambda n: (n + 7) // 8 * 8
    # warm the pool's one context to its largest buffers: with streams=1 it runs every item
    TADpole_genome(px, resident=True, ctx=ctx, streams=1).recall(max_pcs=30, streams=1)
    gc.collect()
    free0 = torch.cuda.mem_get_info(0)[0]
    res = TADpole_genome(px, resident=True, ctx=ctx, streams=1)
    store = res["chr1"]._resident()["batch"]
    nfs = [res[nm].dendro.labels.size for nm in res]
    scores = sum(8 * nf * rb(min(200, nf)) for nf in nfs)
    dendros = sum(8 * min(200, nf) * rb(nf - 1) for nf in nfs)
    assert store.nbytes() == scores + dendros                     # 16 bytes per (good bin x PC) plus the padding to 8
    rec = res.recall(max_pcs=30, streams=1)
    assert rec["chr1"]._resident()["batch"].nbytes() == scores + sum(8 * min(30, nf) * rb(nf - 1) for nf in nfs)
    assert torch.cuda.mem_get_info(0)[0] <= free0 - (scores + dendros) + (8 << 20)
    del res, rec, store
    gc.collect()
    assert abs(torch.cuda.mem_get_info(0)[0] - free0) <= 8 << 20
    # "batch_resident" = 0 (the default): no store
    m = np.ascontiguousarray(dense_of(ctx, px)["chr2"])
    h = ctypes.c_void_p()
    ptrs = (ctypes.c_void_p * 1)(m.ctypes.data)
    ns = np.array([m.shape[0]], np.int32)
    _lib.check(ctx.lib.tp_call_batch(ctx._h, 1, ptrs, _lib._ip(ns), 0, 0, 200, 2, 0.01, 1, 1, 0, ctypes.byref(h)))
    try:
        assert ctx.lib.tp_batch_status(h, 0) == _lib.TP_OK and ctx.lib.tp_batch_resident_bytes(h) == 0
        seq = np.zeros(m.shape[0])
        assert ctx.lib.tp_batch_dendro(h, 0, -1, 0, _lib._dp(seq)) == _lib.TP_ERR_ARG
    finally:
        ctx.lib.tp_batch_free(h)


def test_resident_call_without_a_context_holds_only_its_stores(ctx, px):
    """Without ctx the genome call's own context, and the working buffers of its pool, go when the call returns: a live
    result holds its stores only, and each recall runs on a context of its own."""
    import torch
    from tadpole_b200 import TADpole, TADpole_genome
    TADpole_genome(px, resident=True).recall(max_pcs=30)
    gc.collect()
    free0 = torch.cuda.mem_get_info(0)[0]
    res = TADpole_genome(px, resident=True)
    store = res["chr1"]._resident()["batch"]
    assert store.ctx is None and free0 - torch.cuda.mem_get_info(0)[0] <= store.nbytes() + (16 << 20)
    rec = res.recall(min_clusters=3)
    same_genome(rec, TADpole_genome(px, min_clusters=3, ctx=ctx))
    held = store.nbytes() + rec["chr1"]._resident()["batch"].nbytes()
    assert free0 - torch.cuda.mem_get_info(0)[0] <= held + (16 << 20)
    same_whole(res["chr4"].recall(max_pcs=40), TADpole(dense_of(ctx, px)["chr4"], ctx=ctx).recall(max_pcs=40))
    del res, rec, store
    gc.collect()
    assert abs(torch.cuda.mem_get_info(0)[0] - free0) <= 8 << 20


def test_resident_call_restores_the_context_key(ctx, px):
    from tadpole_b200 import TADpole_genome
    ctx.set("batch_resident", 1)
    try:
        TADpole_genome(px, ctx=ctx, chroms=["chr2"], resident=True)
        assert ctx.get("batch_resident") == 1
        TADpole_genome(px, ctx=ctx, chroms=["chr2"])
        assert ctx.get("batch_resident") == 1
    finally:
        ctx.set("batch_resident", 0)
    TADpole_genome(px, ctx=ctx, chroms=["chr2"], resident=True)
    assert ctx.get("batch_resident") == 0


@pytest.mark.skipif(__import__("tadpole_b200._lib", fromlist=["x"]).device_count() < 2, reason="needs two GPUs")
def test_two_devices(ctx, px, pxc):
    from tadpole_b200 import Context, TADpole_genome
    two = Context([0, 1])
    for pixels, kw in ((px, {}), (pxc, dict(centromere_search=True, centromere_fix=True))):
        one = TADpole_genome(pixels, resident=True, ctx=ctx, **kw)
        res = TADpole_genome(pixels, resident=True, ctx=two, **kw)
        same_genome(res, one)
        crossed = 0
        for m, c in ((200, 3), (30, 2), (200, 2), (30, 3), (50, 2), (60, 3)):
            rec = res.recall(max_pcs=m, min_clusters=c, streams=2)
            same_genome(rec, one.recall(max_pcs=m, min_clusters=c))
            # which device recalls an item depends on which worker claims it: count the items recalled on the other
            # device than their store (the peer copy)
            for nm, obj in rec.items():
                h = obj._resident()
                for part in ((-1,) if obj.get("p") is None else (0, 1)):
                    sd, dd = h["batch"].devices_of(h["item"], part)
                    crossed += sd != dd
        assert crossed > 0


def test_r_routines_match_the_python_host(ctx, px):
    """C_tp_ctx_set / C_tp_call_batch with "batch_resident" / C_tp_batch_recall / C_tp_batch_dendro through the stand-in R
    runtime (which checks arity and PROTECT balance on every .Call) against TADpole_batch(resident=True)."""
    import os
    import sys
    sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
    from mock_r.driver import MockR, RError, Sexp
    from tadpole_b200 import TADpole_batch
    dense = dense_of(ctx, px)
    mats = [dense["chr1"], dense["chr6"]]
    py = TADpole_batch(mats, resident=True, ctx=ctx)
    R = MockR()
    try:
        rctx = R.call("C_tp_ctx", 0, raw=True)
        assert R.call("C_tp_ctx_set", rctx, "batch_resident", 1.0)[0] == 0
        res = R.call("C_tp_call_batch", rctx, mats, 200, 2, 0.01, 4)
        assert R.call("C_tp_ctx_set", rctx, "batch_resident", 0.0)[0] == 1
        assert len(res) == 3 and isinstance(res[2], Sexp)
        assert len(R.call("C_tp_call_batch", rctx, mats[:1], 200, 2, 0.01, 4)) == 1       # not resident: no batch
        batch = res[2]
        for i, obj in enumerate(py):
            assert res[i][1][0] == obj.n_pcs and same(res[i][3], obj.dendro.seqdist)
            for n in (1, 7, obj.n_pcs):
                assert same(R.call("C_tp_batch_dendro", batch, i, -1, n), obj.dendro_for(n).seqdist)
        with pytest.raises(RError, match="between 1 and"):
            R.call("C_tp_batch_dendro", batch, 0, -1, 201)
        rec = R.call("C_tp_batch_recall", rctx, batch, np.array([1, 0], np.int32), np.array([-1, -1], np.int32), 40, 3)
        assert len(rec) == 3 and isinstance(rec[2], Sexp)
        for r, obj in zip(rec[:2], (py[1], py[0])):
            want = obj.recall(max_pcs=40, min_clusters=3)
            assert r[1][0] == want.n_pcs and r[2][0] == want.optimal_n_clusters and same(r[3], want.dendro.seqdist)
        assert same(R.call("C_tp_batch_dendro", rec[2], 0, -1, 40), py[1].recall(max_pcs=40).dendro_for(40).seqdist)
        bad = R.call("C_tp_batch_recall", rctx, batch, np.array([0], np.int32), np.array([-1], np.int32), 300, 2)
        assert isinstance(bad[0], list) and "holds 200" in bad[0][0]
    finally:
        R.reset()
