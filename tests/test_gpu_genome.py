"""GPU tests of the genome-wide input (csrc/ingest.cu S0c: tp_genome_ingest[_file]; csrc/group.cu: tp_call_genome):
one pixel list over every chromosome, split by chromosome on the GPU.  Each chromosome's dense matrix must equal, bit for
bit, oracle.coo_to_dense of the local pixels that oracle/genome_oracle.py (split_genome_pixels) gives it, and each
chromosome's call must return what TADpole() returns for that dense matrix."""
import os
import sys

import numpy as np
import pytest

from oracle import genome_oracle as G
from oracle import tadpole_oracle as O

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
pytestmark = pytest.mark.gpu

SIZES = [1500, 2, 700, 1, 2100, 64]


def same(a, b):
    return a.shape == b.shape and np.array_equal(np.isnan(a), np.isnan(b)) and \
        np.array_equal(a.view(np.uint64)[~np.isnan(a)], b.view(np.uint64)[~np.isnan(b)])


@pytest.fixture(scope="module")
def genome():
    """The synthetic genome plus below-diagonal pixels, repeated cells (integer counts) and a NaN count, shuffled; and
    the oracle's split of it."""
    from tadpole_b200.synth import synth_genome_pixels
    names, (b1, b2, v), mats = synth_genome_pixels(SIZES, seed=7, trans_per_chrom=200)
    rng = np.random.default_rng(11)
    starts = np.concatenate(([0], np.cumsum(SIZES)))
    cis = np.flatnonzero((np.searchsorted(starts, b1, "right") == np.searchsorted(starts, b2, "right")) & (b1 < b2))
    low = rng.choice(cis, 300, replace=False)                            # the same cells, named from below the diagonal
    rep = rng.choice(cis, 2000, replace=False)                           # cells named twice
    b1, b2 = (np.concatenate([b1, b2[low], b1[rep]]).astype(np.int32),
              np.concatenate([b2, b1[low], b2[rep]]).astype(np.int32))
    v = np.concatenate([v, v[low], rng.integers(1, 9, rep.size).astype(float)])
    v[cis[5]] = np.nan
    perm = rng.permutation(b1.size)
    b1, b2, v = b1[perm], b2[perm], v[perm]
    parts, trans, below = G.split_genome_pixels(b1, b2, v, SIZES)
    dense = [O.coo_to_dense(i, j, x, n)[0] for (i, j, x), n in zip(parts, SIZES)]
    return dict(names=names, b1=b1, b2=b2, v=v, parts=parts, trans=trans, below=below, dense=dense)


def bins_of(genome):
    return list(zip(genome["names"], SIZES))


def check_matrices_and_stats(g, genome):
    cis, trans, below = g.stats()
    assert cis.tolist() == [p[0].size for p in genome["parts"]]
    assert trans == genome["trans"] > 0 and below == genome["below"] >= 300
    for c, want in enumerate(genome["dense"]):
        assert same(g.matrix(c), want), genome["names"][c]


def test_dense_build_is_bit_identical(ctx, genome):
    g = ctx.genome_ingest(SIZES, genome["b1"], genome["b2"], genome["v"])
    try:
        check_matrices_and_stats(g, genome)
        assert np.isnan(genome["dense"][0]).any() or any(np.isnan(d).any() for d in genome["dense"])
    finally:
        g.close()


def pixel_text(b1, b2, v, header=False):
    def one(x):
        return "NA" if x != x else str(int(x))
    return ("bin1_id\tbin2_id\tcount\n" if header else "") + \
        "".join(f"{a}\t{b}\t{one(c)}\n" for a, b, c in zip(b1.tolist(), b2.tolist(), v.tolist()))


def same_tadpole(a, b):
    assert a.n_pcs == b.n_pcs and a.optimal_n_clusters == b.optimal_n_clusters
    assert same(a.dendro.seqdist, b.dendro.seqdist)
    assert same(np.asarray(a.scores), np.asarray(b.scores))
    assert sorted(a.clusters) == sorted(b.clusters)
    assert all(np.array_equal(a.clusters[k], b.clusters[k]) for k in b.clusters)


def same_results(r1, r2):
    assert list(r1) == list(r2) and sorted(r1.failed) == sorted(r2.failed)
    for k in r1:
        same_tadpole(r1[k], r2[k])


def test_hicpro_and_cooler_text_give_the_array_results(ctx, genome, tmp_path):
    from tadpole_b200 import GenomePixels, TADpole_genome
    b1, b2, v, names = genome["b1"], genome["b2"], genome["v"], genome["names"]
    # HiC-Pro: 1-based ids, tab, no header; the *_abs.bed bin table
    mat = tmp_path / "sample_50000.matrix"
    mat.write_text(pixel_text(b1 + 1, b2 + 1, v))
    bed = tmp_path / "sample_50000_abs.bed"
    rows = [(nm, i) for nm, n in zip(names, SIZES) for i in range(n)]
    bed.write_text("".join(f"{nm}\t{i * 50000}\t{(i + 1) * 50000}\t{k + 1}\n" for k, (nm, i) in enumerate(rows)))
    # cooler dump -t pixels --header / -t bins --header: 0-based ids
    pix = tmp_path / "pixels.tsv"
    pix.write_text(pixel_text(b1, b2, v, header=True))
    cbins = tmp_path / "bins.tsv"
    cbins.write_text("chrom\tstart\tend\n" + "".join(f"{nm}\t{i * 50000}\t{(i + 1) * 50000}\n" for nm, i in rows))
    forms = [GenomePixels(path=str(mat), bins=str(bed)), GenomePixels(path=str(pix), bins=str(cbins), index_base=0)]
    for src in forms:
        assert src.names == names and src.chrom_bins.tolist() == SIZES
        g = src._ingest(ctx)
        try:
            check_matrices_and_stats(g, genome)
        finally:
            g.close()
    want = TADpole_genome(GenomePixels(b1, b2, v, bins=bins_of(genome)), max_pcs=40, ctx=ctx)
    for src in forms:
        same_results(TADpole_genome(src, max_pcs=40, ctx=ctx), want)


def test_calls_equal_tadpole_on_each_dense_matrix(ctx, genome):
    from tadpole_b200 import GenomePixels, TADpole, TADpole_genome, TadpoleError
    px = GenomePixels(genome["b1"], genome["b2"], genome["v"], bins=bins_of(genome))
    res = TADpole_genome(px, max_pcs=40, ctx=ctx)
    assert res.stats["trans"] == genome["trans"] and res.stats["below"] == genome["below"]
    assert res.stats["cis"] == {nm: p[0].size for nm, p in zip(genome["names"], genome["parts"])}
    assert "chr4" in res.failed and "at least 2" in res.failed["chr4"]         # the 1-bin chromosome
    ran = 0
    for nm, d in zip(genome["names"], genome["dense"]):
        try:
            ref = TADpole(d, max_pcs=40, ctx=ctx)
        except TadpoleError:
            assert nm in res.failed and nm not in res
            continue
        assert nm not in res.failed
        same_tadpole(res[nm], ref)
        ran += 1
    assert ran >= 3 and list(res) == [nm for nm in genome["names"] if nm in res]
    # chroms= selects and orders; the number of calls in flight does not change a bit
    sel = TADpole_genome(px, chroms=["chr5", "chr1", "chr4"], max_pcs=40, ctx=ctx)
    assert list(sel) == ["chr5", "chr1"] and list(sel.failed) == ["chr4"]
    for nm in sel:
        same_tadpole(sel[nm], res[nm])
    same_results(TADpole_genome(px, max_pcs=40, ctx=ctx, streams=1), res)
    same_results(TADpole_genome(px, max_pcs=40, ctx=ctx, streams=8), res)


def test_two_gpus_give_the_one_gpu_bits(genome):
    from tadpole_b200 import Context, GenomePixels, TADpole_genome
    from tadpole_b200._lib import device_count
    if device_count() < 2:
        pytest.skip("needs two GPUs")
    px = GenomePixels(genome["b1"], genome["b2"], genome["v"], bins=bins_of(genome))
    one = Context(0)
    two = Context([0, 1])
    try:
        same_results(TADpole_genome(px, max_pcs=40, ctx=two, streams=2), TADpole_genome(px, max_pcs=40, ctx=one, streams=2))
    finally:
        two.close()
        one.close()


def test_errors(ctx, tmp_path):
    from tadpole_b200 import GenomePixels, TADpole_genome, TadpoleError
    with pytest.raises(TadpoleError, match=r"entry 3 is \(2, 9\): outside the 6 bins of the bin table"):
        ctx.genome_ingest([4, 2], [0, 1, 2], [3, 4, 9], [1.0, 1.0, 1.0])
    p = tmp_path / "g.matrix"
    p.write_text("1\t2\t3\n2\t7\t1\n")
    with pytest.raises(TadpoleError, match="row 2 names a bin outside the 6 bins"):
        ctx.genome_ingest([4, 2], path=str(p), index_base=1)
    px = GenomePixels([0], [1], [1.0], bins=[("chr1", 4), ("chr2", 2)])
    with pytest.raises(ValueError, match="chr3"):
        TADpole_genome(px, chroms=["chr1", "chr3"], ctx=ctx)
    with pytest.raises(TadpoleError, match="chromosomes"):
        ctx.genome_ingest([], [0], [0], [1.0])


def test_r_shim_returns_the_binding_values(ctx, genome, tmp_path):
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from mock_r.driver import MockR
    R = MockR()
    try:
        rctx = R.call("C_tp_ctx", 0, raw=True)
        handle, cis, tb = R.call("C_tp_genome", rctx, np.array(SIZES, np.int32), genome["b1"], genome["b2"], genome["v"], 0)
        assert cis.tolist() == [p[0].size for p in genome["parts"]] and tb.tolist() == [genome["trans"], genome["below"]]
        sel = np.array([4, 3, 0], np.int32)
        out = R.call("C_tp_call_genome", rctx, handle, sel, 40, 2, 0.01, 4, True)
        g = ctx.genome_ingest(SIZES, genome["b1"], genome["b2"], genome["v"])
        try:
            want = ctx.call_genome(g, sel, max_pcs=40)
        finally:
            g.close()
        assert len(out) == 3 and isinstance(out[1][0], str) and isinstance(want[1], Exception)
        for item, w in ((out[0], want[0]), (out[2], want[2])):
            bad, npcs, ncl, seq, scores, levels, tables = item
            assert np.array_equal(bad, w["bad"]) and npcs[0] == w["n_pcs"] and ncl[0] == w["n_clusters"]
            assert same(seq, w["seqdist"])
            assert np.array_equal(np.isnan(scores), np.isnan(w["scores"]))
            assert np.array_equal(scores[~np.isnan(scores)], w["scores"][~np.isnan(scores)])
            assert sorted(int(l) for l in levels) == sorted(w["tables"])
            for lv, t in zip(levels, tables):
                assert np.array_equal(t, w["tables"][int(lv)])
        # the file routine: the same stats (HiC-Pro text, 1-based)
        p = tmp_path / "g.matrix"
        p.write_text(pixel_text(genome["b1"] + 1, genome["b2"] + 1, genome["v"]))
        _, cis2, tb2 = R.call("C_tp_genome_file", rctx, np.array(SIZES, np.int32), str(p), 1)
        assert np.array_equal(cis2, cis) and np.array_equal(tb2, tb)
    finally:
        R.reset()
