"""GPU tests of centromere_search in the batch paths (csrc/group.cu: tp_call_batch_arms, tp_call_genome_arms): every
matrix split at its centromere and both arms called in the library's batch workers must give, bit for bit, what
TADpole(m, centromere_search=True) gives on that matrix -- arms, per-level tables, merging_arms, messages and errors."""
import os
import sys

import numpy as np
import pytest

from oracle import genome_oracle as G
from oracle import tadpole_oracle as O

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
pytestmark = pytest.mark.gpu

MAX_PCS = 40
SIZES = [1500, 2, 700, 1, 2100, 64]
CENTROMERES = [0, 2, 4, 5]                      # the chromosomes of 64 bins and more


def same(a, b):
    a, b = np.asarray(a), np.asarray(b)
    return a.shape == b.shape and np.array_equal(np.isnan(a), np.isnan(b)) and \
        np.array_equal(a.view(np.uint64)[~np.isnan(a)], b.view(np.uint64)[~np.isnan(b)])


@pytest.fixture(scope="module")
def split_mats():
    from tadpole_b200.synth import synth_hic
    mats = [synth_hic(n, seed=20 + n % 7, centromere=True) for n in (600, 1500, 2100)]
    # quirk Q3, the matrix of test_gpu_handle.py::test_centromere_fix_mode: a q-arm bad bin whose original index is past
    # the arm's end, so the reference keeps that bad row in the q arm
    m = synth_hic(700, seed=4, centromere=True)
    q0 = int(O.load_mat_numeric(m, centromere_search=True).centromere[-1])
    assert q0 + 41 > 700 - q0
    m[q0 + 40, :] = 0
    m[:, q0 + 40] = 0
    # quirk Q3 inside the arm: centromere at bins 151..170 (1-based), so the q arm has 530 bins; the bad bin 300 of the q
    # arm makes the reference drop the arm's 300th row (original bin 470) instead
    m2 = synth_hic(700, seed=6)
    m2[150:170, :] = 0
    m2[:, 150:170] = 0
    m2[299, :] = 0
    m2[:, 299] = 0
    lm = O.load_mat_numeric(m2, centromere_search=True)
    assert lm.centromere.tolist() == list(range(151, 171)) and 300 <= 700 - 170
    assert 300 in lm.q.names and 470 not in lm.q.names
    return mats + [m, m2]


@pytest.fixture(scope="module")
def unsplit_mats():
    """TADpole(centromere_search=True, bad_frac=0) does not split these: no bad bin, and a bad stretch at the start."""
    from tadpole_b200.synth import synth_hic
    m2 = synth_hic(300, seed=8, zero_frac=0.0)
    m3 = m2.copy()
    m3[:4, :] = 0
    m3[:, :4] = 0
    return [m2, m3]


def same_arm_obj(a, b, fix):
    assert a.n_pcs == b.n_pcs and a.optimal_n_clusters == b.optimal_n_clusters
    assert same(a.dendro.seqdist, b.dendro.seqdist)
    assert list(a.dendro.labels) == list(b.dendro.labels)
    assert sorted(a.cluster) == sorted(b.cluster)
    assert all(np.array_equal(a.cluster[k], b.cluster[k]) for k in b.cluster)
    assert ("scores" in a) == ("scores" in b) == fix
    if fix:
        assert same(a.scores, b.scores) and sorted(a.clusters) == sorted(b.clusters)


def same_split_obj(a, b, fix):
    for arm in ("p", "q"):
        same_arm_obj(a[arm], b[arm], fix)
    assert np.array_equal(a.merging_arms, b.merging_arms)


def same_whole_obj(a, b):
    assert "p" not in a and a.n_pcs == b.n_pcs and a.optimal_n_clusters == b.optimal_n_clusters
    assert same(a.dendro.seqdist, b.dendro.seqdist) and same(a.scores, b.scores)
    assert sorted(a.clusters) == sorted(b.clusters) and all(np.array_equal(a.clusters[k], b.clusters[k]) for k in b.clusters)


def same_obj(a, b, fix):
    if "p" in b:
        same_split_obj(a, b, fix)
    else:
        same_whole_obj(a, b)


def same_item(item, ref, fix):
    """An item of call_batch(centromere_search=True) against TADpole(centromere_search=True)'s object."""
    from tadpole_b200 import api
    assert item["split"] is True and item["centromere"].size > 0
    for arm in ("p", "q"):
        a, r = item[arm], ref[arm]
        assert a["n_pcs"] == r.n_pcs and a["n_clusters"] == r.optimal_n_clusters
        assert same(a["seqdist"], r.dendro.seqdist)
        assert sorted(str(k) for k in a["tables"]) == sorted(r.cluster)
        assert all(np.array_equal(a["tables"][int(k)], r.cluster[k]) for k in r.cluster)
        if fix:
            assert same(a["scores"], r.scores)
    assert np.array_equal(api._merging_arms(item["p"]["labels"], item["q"]["labels"], item["centromere"].size),
                          ref.merging_arms)


@pytest.mark.parametrize("fix", [False, True])
def test_split_batch_equals_tadpole(ctx, split_mats, fix):
    from tadpole_b200 import TADpole, TADpole_batch, api
    api.QUIET = True
    refs = [TADpole(m, max_pcs=MAX_PCS, centromere_search=True, centromere_fix=fix, ctx=ctx) for m in split_mats]
    items = ctx.call_batch(split_mats, max_pcs=MAX_PCS, inflight=4, centromere_search=True, centromere_fix=fix)
    for m, item, ref in zip(split_mats, items, refs):
        same_item(item, ref, fix)
        assert item["device_ms"] > 0 and item["bad"].size == m.shape[0]
    for tp, ref in zip(TADpole_batch(split_mats, max_pcs=MAX_PCS, centromere_search=True, centromere_fix=fix, ctx=ctx,
                                     streams=3), refs):
        same_split_obj(tp, ref, fix)
    # quirk Q3: the q arms of the last two matrices differ between the two modes
    for m in split_mats[-2:]:
        q_default = TADpole(m, max_pcs=MAX_PCS, centromere_search=True, ctx=ctx).q
        q_fixed = TADpole(m, max_pcs=MAX_PCS, centromere_search=True, centromere_fix=True, ctx=ctx).q
        assert list(q_default.dendro.labels) != list(q_fixed.dendro.labels)


def test_unsplit_batch(ctx, split_mats, unsplit_mats):
    from tadpole_b200 import TADpole, TADpole_batch, TadpoleError, api
    from tadpole_b200._lib import TP_ERR_NOSPLIT
    api.QUIET = True
    items = ctx.call_batch(unsplit_mats, max_pcs=MAX_PCS, bad_frac=0.0, centromere_search=True)
    for m, it in zip(unsplit_mats, items):
        assert isinstance(it, TadpoleError) and it.code == TP_ERR_NOSPLIT
        with pytest.raises(ValueError) as want:
            TADpole(m, max_pcs=MAX_PCS, bad_frac=0.0, centromere_search=True, ctx=ctx)
        with pytest.raises(ValueError) as got:
            TADpole_batch([split_mats[0], m], max_pcs=MAX_PCS, bad_frac=0.0, centromere_search=True, ctx=ctx)
        assert str(got.value) == str(want.value)
    # centromere_fix: processed whole; a batch may mix split and unsplit matrices
    mixed = [unsplit_mats[0], split_mats[0], unsplit_mats[1]]
    refs = [TADpole(m, max_pcs=MAX_PCS, bad_frac=0.0, centromere_search=True, centromere_fix=True, ctx=ctx) for m in mixed]
    items = ctx.call_batch(mixed, max_pcs=MAX_PCS, bad_frac=0.0, centromere_search=True, centromere_fix=True)
    assert items[0]["split"] is False and items[0]["centromere"] is None and items[1]["split"] is True
    assert items[2]["centromere"].tolist() == [1, 2, 3, 4]
    for tp, ref in zip(TADpole_batch(mixed, max_pcs=MAX_PCS, bad_frac=0.0, centromere_search=True, centromere_fix=True,
                                     ctx=ctx), refs):
        same_obj(tp, ref, True)


def test_messages_equal_the_loop_of_tadpole(ctx, split_mats, unsplit_mats, capsys):
    from tadpole_b200 import TADpole, TADpole_batch, api
    was = api.QUIET
    api.QUIET = False
    try:
        capsys.readouterr()
        for fix in (False, True):
            mats = split_mats[:2] + [unsplit_mats[1]] + split_mats[2:]
            want_err = None
            for m in mats:
                try:
                    TADpole(m, max_pcs=MAX_PCS, bad_frac=0.0, centromere_search=True, centromere_fix=fix, ctx=ctx)
                except ValueError as e:
                    want_err = str(e)
                    break
            want = capsys.readouterr().err
            try:
                TADpole_batch(mats, max_pcs=MAX_PCS, bad_frac=0.0, centromere_search=True, centromere_fix=fix, ctx=ctx)
                got_err = None
            except ValueError as e:
                got_err = str(e)
            got = capsys.readouterr().err
            assert got == want and got_err == want_err and (want_err is None) == fix
            assert "Processing arm q" in got and "centromere position" in got
    finally:
        api.QUIET = was


@pytest.fixture(scope="module")
def genome():
    from tadpole_b200.synth import synth_genome_pixels
    names, (b1, b2, v), mats = synth_genome_pixels(SIZES, seed=7, trans_per_chrom=200, centromere=CENTROMERES)
    parts, trans, below = G.split_genome_pixels(b1, b2, v, SIZES)
    dense = [O.coo_to_dense(i, j, x, n)[0] for (i, j, x), n in zip(parts, SIZES)]
    return dict(names=names, b1=b1, b2=b2, v=v, dense=dense)


def test_synth_genome_default_is_unchanged():
    from tadpole_b200.synth import synth_genome_pixels
    a = synth_genome_pixels([50, 1, 40], seed=3, trans_per_chrom=20)
    b = synth_genome_pixels([50, 1, 40], seed=3, trans_per_chrom=20, centromere=[])
    c = synth_genome_pixels([50, 1, 40], seed=3, trans_per_chrom=20, centromere=[2])
    for x, y in zip(a[1], b[1]):
        assert np.array_equal(x, y)
    assert np.array_equal(a[2][0], c[2][0]) and not np.array_equal(a[2][2], c[2][2])


def same_genome(r1, r2, fix=False):
    assert list(r1) == list(r2) and r1.failed == r2.failed
    for k in r1:
        same_obj(r1[k], r2[k], fix)


def test_genome_equals_tadpole_on_each_dense_matrix(ctx, genome):
    from tadpole_b200 import GenomePixels, TADpole, TADpole_genome, TadpoleError, api
    api.QUIET = True
    px = GenomePixels(genome["b1"], genome["b2"], genome["v"], bins=list(zip(genome["names"], SIZES)))
    res = TADpole_genome(px, max_pcs=MAX_PCS, ctx=ctx, centromere_search=True)
    split = 0
    for nm, d in zip(genome["names"], genome["dense"]):
        try:
            ref = TADpole(d, max_pcs=MAX_PCS, centromere_search=True, ctx=ctx)
        except ValueError as e:
            assert res.failed[nm] == str(e) and nm not in res
            continue
        except TadpoleError:
            assert nm in res.failed and nm not in res
            continue
        assert nm not in res.failed
        same_split_obj(res[nm], ref, False)
        split += 1
    assert split >= 3 and "chr2" in res.failed and "chr4" in res.failed
    sel = TADpole_genome(px, chroms=["chr5", "chr2", "chr1"], max_pcs=MAX_PCS, ctx=ctx, centromere_search=True)
    assert list(sel) == ["chr5", "chr1"] and list(sel.failed) == ["chr2"]
    for nm in sel:
        same_split_obj(sel[nm], res[nm], False)
    same_genome(TADpole_genome(px, max_pcs=MAX_PCS, ctx=ctx, streams=1, centromere_search=True), res)
    same_genome(TADpole_genome(px, max_pcs=MAX_PCS, ctx=ctx, streams=8, centromere_search=True), res)
    # centromere_fix: the 2-bin chromosome is called whole, as TADpole(centromere_fix=True) calls it (or fails as it does)
    fixed = TADpole_genome(px, max_pcs=MAX_PCS, ctx=ctx, centromere_search=True, centromere_fix=True)
    for nm, d in zip(genome["names"], genome["dense"]):
        try:
            ref = TADpole(d, max_pcs=MAX_PCS, centromere_search=True, centromere_fix=True, ctx=ctx)
        except (ValueError, TadpoleError):
            assert nm in fixed.failed
            continue
        same_obj(fixed[nm], ref, True)


def test_two_gpus_give_the_one_gpu_bits(split_mats, genome):
    from tadpole_b200 import Context, GenomePixels, TADpole_batch, TADpole_genome, api
    from tadpole_b200._lib import device_count
    if device_count() < 2:
        pytest.skip("needs two GPUs")
    api.QUIET = True
    px = GenomePixels(genome["b1"], genome["b2"], genome["v"], bins=list(zip(genome["names"], SIZES)))
    one = Context(0)
    two = Context([0, 1])
    try:
        for a, b in zip(TADpole_batch(split_mats, max_pcs=MAX_PCS, centromere_search=True, ctx=two, streams=2),
                        TADpole_batch(split_mats, max_pcs=MAX_PCS, centromere_search=True, ctx=one, streams=2)):
            same_split_obj(a, b, False)
        same_genome(TADpole_genome(px, max_pcs=MAX_PCS, ctx=two, streams=2, centromere_search=True),
                    TADpole_genome(px, max_pcs=MAX_PCS, ctx=one, streams=2, centromere_search=True))
    finally:
        two.close()
        one.close()


def same_r_arm(r_arm, w):
    npcs, ncl, seq, scores, keep, badc = r_arm
    assert npcs[0] == w["n_pcs"] and ncl[0] == w["n_clusters"] and same(seq, w["seqdist"])
    assert np.array_equal(np.isnan(scores), np.isnan(w["scores"]))
    assert np.array_equal(scores[~np.isnan(scores)], w["scores"][~np.isnan(scores)])
    assert keep.tolist() == (w["keep"] + 1).tolist()
    assert (badc is None) == (w["bad_columns"] is None)
    assert badc is None or badc.tolist() == w["bad_columns"].tolist()


def test_r_shim_returns_the_binding_values(ctx, split_mats, unsplit_mats, genome):
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from mock_r.driver import MockR
    R = MockR()
    try:
        rctx = R.call("C_tp_ctx", 0, raw=True)
        mats = split_mats[:2] + unsplit_mats[:1]
        out = R.call("C_tp_call_batch_arms", rctx, mats, MAX_PCS, 2, 0.0, 4)
        want = ctx.call_batch(mats, max_pcs=MAX_PCS, bad_frac=0.0, centromere_search=True)
        assert len(out) == 3 and isinstance(out[2][0], str) and isinstance(want[2], Exception)
        for item, w in zip(out[:2], want[:2]):
            bad, cen, p, q = item
            assert np.array_equal(bad, w["bad"]) and cen.tolist() == w["centromere"].tolist()
            same_r_arm(p, w["p"])
            same_r_arm(q, w["q"])
        handle, _, _ = R.call("C_tp_genome", rctx, np.array(SIZES, np.int32), genome["b1"], genome["b2"], genome["v"], 0)
        sel = np.array([4, 1, 0], np.int32)
        g = ctx.genome_ingest(SIZES, genome["b1"], genome["b2"], genome["v"])
        try:
            for fix in (False, True):
                out = R.call("C_tp_call_genome_arms", rctx, handle, sel, MAX_PCS, 2, 0.01, 4, fix)
                want = ctx.call_genome(g, sel, max_pcs=MAX_PCS, centromere_search=True, centromere_fix=fix)
                for item, w in zip(out, want):
                    if isinstance(w, Exception):
                        assert isinstance(item[0], str)
                        continue
                    if not w["split"]:                   # processed whole: the C_tp_call_genome layout
                        assert np.array_equal(item[0], w["bad"]) and same(item[3], w["seqdist"])
                        continue
                    same_r_arm(item[2], w["p"])
                    same_r_arm(item[3], w["q"])
        finally:
            g.close()
    finally:
        R.reset()
