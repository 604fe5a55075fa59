"""GPU tests of the read-pair ingest (csrc/pairs.cu, DESIGN S0f: tp_genome_ingest_pairs_file; GenomePairs).  Small files
in the three layouts are compared bit for bit with the line-by-line reference (tests/pairs_oracle.py), also through
windows of a few hundred bytes (many windows, lines straddling them, many table growths) and as several files; a
GRCh38-sized file at 10 kb with the vectorised reference.  Calls on a pairs genome must equal calls on the reference's
cells ingested as pixels."""
import gzip
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tests"))
pytestmark = pytest.mark.gpu

import pairs_oracle as P  # noqa: E402

SIZES = [("chr1", 50000), ("chr10", 30001), ("chr2", 7770), ("chr3", 5), ("chrX", 120)]
BIN = 100


def _pixels(g):
    return [g.pixels(nm) for nm in g.names]


def _same(a, b):
    return len(a) == len(b) and all(np.array_equal(x[0], y[0]) and np.array_equal(x[1], y[1]) and
                                    np.array_equal(np.asarray(x[2], np.float64).view(np.uint64),
                                                   np.asarray(y[2], np.float64).view(np.uint64)) for x, y in zip(a, b))


def _check(g, want, counts):
    assert g.pair_counts == counts
    assert _same(_pixels(g), want)
    cis, trans, below = g.stats()
    assert cis.tolist() == [w[0].size for w in want] and trans == counts["trans"] and below == 0
    assert g.total_depth == counts["cis"]


def _load(paths, ctx, sizes=SIZES, binsize=BIN, layout="4dn", base=1):
    from tadpole_b200 import GenomePairs
    return GenomePairs(paths, sizes, binsize=binsize, columns=P.LAYOUTS[layout], index_base=base).load(ctx=ctx)


@pytest.fixture(scope="module")
def files(tmp_path_factory):
    d = tmp_path_factory.mktemp("pairs")
    out = {}
    for k, (layout, base) in enumerate([("4dn", 1), ("hicpro", 1), ("juicer", 1), ("4dn", 0), ("juicer", 0)]):
        path = str(d / f"{layout}_{base}.txt")
        P.write_pairs(path, layout, SIZES, 20000, 1500, 500, seed=10 + k, index_base=base, quirks=True)
        out[(layout, base)] = path
    return out


@pytest.mark.parametrize("layout,base", [("4dn", 1), ("hicpro", 1), ("juicer", 1), ("4dn", 0), ("juicer", 0)])
@pytest.mark.parametrize("window", [None, 300])
def test_bit_equal_to_the_line_reference(ctx, files, monkeypatch, layout, base, window):
    path = files[(layout, base)]
    want, counts = P.bin_pairs_text([path], SIZES, BIN, P.LAYOUTS[layout], base)
    assert counts["trans"] and counts["unplaced"] and all(w[0].size for w in want)
    if window:
        monkeypatch.setenv("TADPOLE_PAIRS_WINDOW", str(window))
    with _load(path, ctx, layout=layout, base=base) as g:
        assert g.binsize == BIN and g.chrom_bins.tolist() == P.n_bins(SIZES, BIN)
        _check(g, want, counts)
    if window:
        assert ctx.ingest_stats()["host_fields"] > os.path.getsize(path) / window / 2     # slot 3: the windows


@pytest.mark.parametrize("window", [None, 256])
def test_several_files_equal_their_concatenation_in_either_order(ctx, files, tmp_path, monkeypatch, window):
    a, b = files[("hicpro", 1)], str(tmp_path / "b.txt")
    P.write_pairs(b, "hicpro", SIZES, 5000, 100, 100, seed=99, quirks=True)
    cat = tmp_path / "ab.txt"
    cat.write_bytes(open(a, "rb").read() + open(b, "rb").read())
    want, counts = P.bin_pairs_text([str(cat)], SIZES, BIN, P.LAYOUTS["hicpro"])
    if window:
        monkeypatch.setenv("TADPOLE_PAIRS_WINDOW", str(window))
    for order in ([a, b], [b, a], [str(cat)]):
        with _load(order, ctx, layout="hicpro") as g:
            _check(g, want, counts)


def test_coarsen_composition_and_depth(ctx, files):
    from tadpole_b200 import GenomePairs
    path = files[("juicer", 1)]
    for b, f in ((10, 3), (100, 7), (1, 250)):
        with _load(path, ctx, binsize=b, layout="juicer") as fine, fine.coarsen(f) as cf, \
                _load(path, ctx, binsize=f * b, layout="juicer") as direct:
            assert cf.binsize == direct.binsize == f * b
            assert cf.chrom_bins.tolist() == direct.chrom_bins.tolist()
            assert _same(_pixels(cf), _pixels(direct))
            assert sum(fine.depth().values()) == fine.pair_counts["cis"] == cf.total_depth
    g = GenomePairs(path, SIZES, binsize=BIN, columns=P.LAYOUTS["juicer"]).load(ctx=ctx)
    with g, g.downsample(contacts=100, seed=1) as d:
        assert d.binsize == BIN and d.total_depth == 100 and d.pair_counts is None


# ---- calls ------------------------------------------------------------------------------------------------------------

CALL_SIZES = [("chrA", 6_000_000), ("chrB", 4_800_000), ("chrC", 5_400_000)]


@pytest.fixture(scope="module")
def call_file(tmp_path_factory):
    path = str(tmp_path_factory.mktemp("call") / "call.pairs")
    P.write_pairs(path, "4dn", CALL_SIZES, 3_000_000, 20_000, 5_000, seed=21)
    return path


def test_calls_on_a_pairs_genome_equal_calls_on_the_references_pixels(ctx, call_file):
    from genome_timing import same
    from tadpole_b200 import GenomePairs, GenomePixels, TADpole_genome, api
    api.QUIET = True
    want, _ = P.bin_pairs_np([call_file], CALL_SIZES, 10_000)
    nb = P.n_bins(CALL_SIZES, 10_000)
    starts = np.concatenate(([0], np.cumsum(nb)))
    px = GenomePixels(np.concatenate([i + starts[c] for c, (i, _, _) in enumerate(want)]).astype(np.int32),
                      np.concatenate([j + starts[c] for c, (_, j, _) in enumerate(want)]).astype(np.int32),
                      np.concatenate([x for _, _, x in want]), bins=[(nm, n) for (nm, _), n in zip(CALL_SIZES, nb)])
    pairs = GenomePairs(call_file, binsize=10_000)              # the table from the '#chromsize:' header
    a, b = TADpole_genome(pairs, max_pcs=20, ctx=ctx), TADpole_genome(px, max_pcs=20, ctx=ctx)
    assert list(a) == list(b) == [nm for nm, _ in CALL_SIZES] and not a.failed
    assert all(same(a[nm], b[nm]) for nm in a)
    with pairs.load(ctx=ctx) as g:
        a, b = (TADpole_genome(x, max_pcs=20, ctx=ctx, centromere_search=True, centromere_fix=True) for x in (g, px))
        assert list(a) == list(b) and a.failed == b.failed
        for nm in a:
            if getattr(a[nm], "clusters", None) is None:
                assert all(same(a[nm][arm], b[nm][arm]) for arm in ("p", "q"))
            else:
                assert same(a[nm], b[nm])
        r = TADpole_genome(g, max_pcs=20, resident=True)
        rr = r.recall(max_pcs=20, min_clusters=3)
        fresh = TADpole_genome(px, max_pcs=20, min_clusters=3, ctx=ctx)
        assert all(same(rr[nm], fresh[nm]) for nm in fresh)


# ---- errors -------------------------------------------------------------------------------------------------------------

# (text of the second file, index_base, window, the reference's line, the library's message)
ERRORS = [
    (b"r chr1 10 chr1 20\n#c\nr chr1 10 chr1\nr chr1 x chr1 3\n", 1, None, 3, "line 3: fewer fields"),
    (b"r chr1 10 chr1 20\r\nr chr1 1a chr1 3\n", 1, None, 2, "line 2: a position is not 1 to 18 digits"),
    (b"\n\nr chr1 1 chr1 2\nr chr1 0 chr1 3\n", 1, None, 4, "line 4: a position lies outside its chromosome"),
    (b"r chr1 0 chr1 3\nr chrX 0 chrX 120\n", 0, None, 2, "line 2: a position lies outside its chromosome"),
    (b"r chr1 3 chrM 0\nr chrX 121 chrM 5\n", 1, None, 2, "line 2: a position lies outside its chromosome"),
    (b"r chr1 1 chr1 2\n" * 20 + b"r chr1 3 chr1 4 " + b"y" * 400 + b"\nr chr1 x chr1 1\n", 1, 300, 21,
     "line 21 is longer than the device window"),
    (b"r chr1 1 chr1 2\n" * 20 + b"r chr1 3 chr1\n" + b"r chr1 3 chr1 4 " + b"y" * 400 + b"\n", 1, 300, 21,
     "line 21: fewer fields"),
    (b"", 1, None, 0, "holds no pair lines"),
    (b"# header\n\n  \t\r\n", 1, None, 0, "holds no pair lines"),
]


@pytest.mark.parametrize("k", range(len(ERRORS)))
def test_errors_name_the_file_and_the_lowest_line(ctx, tmp_path, monkeypatch, k):
    from tadpole_b200 import TadpoleError
    text, base, window, line, msg = ERRORS[k]
    good, bad = str(tmp_path / "good.pairs"), str(tmp_path / "bad.pairs")
    open(good, "wb").write(b"r chr1 10 chr1 20\n")
    open(bad, "wb").write(text)
    with pytest.raises(P.PairsError) as ref:
        P.bin_pairs_text([good, bad], SIZES, BIN, index_base=base, window=window or P.WINDOW)
    assert (ref.value.path, ref.value.line) == (bad, line)
    if window:
        monkeypatch.setenv("TADPOLE_PAIRS_WINDOW", str(window))
    with pytest.raises(TadpoleError) as e:
        _load([good, bad], ctx, base=base)
    assert f"'{bad}'" in str(e.value) and msg in str(e.value), str(e.value)
    with _load(good, ctx) as g:                              # the context is still usable
        assert g.pair_counts["cis"] == 1


def test_gzip_input_is_refused(ctx, tmp_path):
    from tadpole_b200 import TadpoleError
    path = str(tmp_path / "x.pairs.gz")
    open(path, "wb").write(gzip.compress(b"r chr1 10 chr1 20\n"))
    with pytest.raises(TadpoleError, match="compressed input is not read"):
        _load(path, ctx)


# ---- GRCh38 at 10 kb -----------------------------------------------------------------------------------------------------

def test_grch38_at_10kb_equals_the_vectorised_reference(ctx, tmp_path):
    from genome_timing import GRCH38
    path = str(tmp_path / "grch38.pairs")
    P.write_pairs(path, "4dn", GRCH38, 20_000_000, 1_500_000, 300_000, seed=3)
    want, counts = P.bin_pairs_np([path], GRCH38, 10_000)
    assert counts["lines"] > 20_000_000
    with _load(path, ctx, sizes=GRCH38, binsize=10_000) as g:
        assert g.pair_counts == counts
        assert _same(_pixels(g), want)
    os.unlink(path)


# ---- R -----------------------------------------------------------------------------------------------------------------

def test_mock_r_routine_drives_the_library(ctx, files):
    from mock_r.driver import MockR
    from test_pairs_host import _strings
    path = files[("hicpro", 1)]
    R = MockR()
    try:
        rctx = R.call("C_tp_ctx", 0, raw=True)
        names = [nm for nm, _ in SIZES]
        lay = np.array(list(P.LAYOUTS["hicpro"]) + [1], np.int32)
        h, cis, tb, cnt = R.call("C_tp_genome_pairs_file", rctx, _strings(R, [path]), _strings(R, names),
                                 np.array([float(ln) for _, ln in SIZES]), float(BIN), lay)
        with _load(path, ctx, layout="hicpro") as g:
            want = _pixels(g)
            c = g.pair_counts
            assert cnt.tolist() == [float(c["lines"]), float(c["cis"]), float(c["trans"]), float(c["unplaced"])]
            assert cis.tolist() == [float(w[0].size) for w in want] and tb.tolist() == [float(c["trans"]), 0.0]
            for ch, (wi, wj, wv) in enumerate(want):
                i, j, x = R.call("C_tp_genome_pixels", rctx, h, ch, len(SIZES))
                o = np.lexsort((j, i))
                assert np.array_equal(i[o], wi) and np.array_equal(j[o], wj) and np.array_equal(x[o], wv)
    finally:
        R.reset()
