"""CPU tests of the read-pair ingest (DESIGN S0f): the line-by-line and vectorised references (tests/pairs_oracle.py)
agree and keep the spec's properties, GenomePairs checks its arguments and reads every form of the chromosome table, the
C ABI symbol and version, and the R routine's registration and argument checks under the stand-in R runtime of
tests/mock_r."""
import ctypes
import gzip
import os
import re
import sys

import numpy as np
import pytest

from tadpole_b200 import _lib
from tadpole_b200.batch import GenomePairs, LoadedGenome, _CtxRef, read_chromsizes

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tests"))
import pairs_oracle as P  # noqa: E402
import coarsen_oracle as C  # noqa: E402

SIZES = [("chr1", 5000), ("chr10", 3001), ("chr2", 777), ("chrX", 12)]


def _same(a, b):
    return len(a) == len(b) and all(np.array_equal(x[0], y[0]) and np.array_equal(x[1], y[1]) and
                                    np.array_equal(np.asarray(x[2]).view(np.uint64), np.asarray(y[2]).view(np.uint64))
                                    for x, y in zip(a, b))


@pytest.mark.parametrize("layout", sorted(P.LAYOUTS))
@pytest.mark.parametrize("base", [0, 1])
def test_line_and_vectorised_references_agree(tmp_path, layout, base):
    path = tmp_path / "p.txt"
    P.write_pairs(path, layout, SIZES, 3000, 300, 100, seed=5, index_base=base, quirks=True)
    for binsize in (1, 7, 100, 5000, 10 ** 6):
        a, ca = P.bin_pairs_text([path], SIZES, binsize, P.LAYOUTS[layout], base)
        b, cb = P.bin_pairs_np([path], SIZES, binsize, P.LAYOUTS[layout], base)
        assert ca == cb and ca["lines"] == ca["cis"] + ca["trans"] + ca["unplaced"]
        assert ca["trans"] > 0 and ca["unplaced"] >= 2 * len(P.UNPLACED)
        assert _same(a, b), binsize
        for (i, j, x), n in zip(a, P.n_bins(SIZES, binsize)):
            assert np.all((0 <= i) & (i <= j) & (j < n)) and np.all(x >= 1)
        assert sum(float(x.sum()) for _, _, x in a) == ca["cis"]


def test_swapped_pairs_land_in_the_same_cell(tmp_path):
    names, c1, p1, c2, p2 = P.synth_pairs(SIZES, 500, 50, 20, seed=2)
    one, two = tmp_path / "a.pairs", tmp_path / "b.pairs"
    one.write_bytes(P.pair_lines("4dn", names, c1, p1, c2, p2))
    two.write_bytes(P.pair_lines("4dn", names, c2, p2, c1, p1))
    a, ca = P.bin_pairs_text([one], SIZES, 50)
    b, cb = P.bin_pairs_text([two], SIZES, 50)
    assert ca == cb and _same(a, b)


def _global(out, nb):
    starts = np.concatenate(([0], np.cumsum(nb)))
    return (np.concatenate([i + starts[c] for c, (i, _, _) in enumerate(out)]),
            np.concatenate([j + starts[c] for c, (_, j, _) in enumerate(out)]),
            np.concatenate([x for _, _, x in out]))


@pytest.mark.parametrize("b,f", [(1, 7), (10, 3), (100, 50), (37, 1000)])
def test_pairs_at_b_then_coarsen_f_equal_pairs_at_fb(tmp_path, b, f):
    path = tmp_path / "p.txt"
    P.write_pairs(path, "hicpro", SIZES, 4000, 100, 50, seed=7, quirks=True)
    fine, _ = P.bin_pairs_text([path], SIZES, b, P.LAYOUTS["hicpro"])
    nb = P.n_bins(SIZES, b)
    coarse, _, _ = C.coarsen_pixels_np(nb, *_global(fine, nb), f)
    assert C.coarse_bins(nb, f) == P.n_bins(SIZES, f * b)
    direct, _ = P.bin_pairs_text([path], SIZES, f * b, P.LAYOUTS["hicpro"])
    assert _same(coarse, direct)


def test_several_files_equal_their_concatenation_in_any_order(tmp_path):
    a, b = tmp_path / "a.txt", tmp_path / "b.txt"
    P.write_pairs(a, "juicer", SIZES, 800, 40, 20, seed=1, quirks=True)
    P.write_pairs(b, "juicer", SIZES, 600, 30, 10, seed=2)
    cat = tmp_path / "ab.txt"
    cat.write_bytes(a.read_bytes() + b.read_bytes())
    want = P.bin_pairs_text([cat], SIZES, 64, P.LAYOUTS["juicer"])
    for order in ([a, b], [b, a]):
        got, counts = P.bin_pairs_text(order, SIZES, 64, P.LAYOUTS["juicer"])
        assert counts == want[1] and _same(got, want[0])


def _errors(tmp_path, text, base=1, window=P.WINDOW):
    path = tmp_path / "e.pairs"
    path.write_bytes(text)
    with pytest.raises(P.PairsError) as e:
        P.bin_pairs_text([path], SIZES, 10, index_base=base, window=window)
    return e.value.line, e.value.kind


def test_reference_errors_name_the_lowest_line(tmp_path):
    ok = b"r chr1 10 chr1 20\n"
    assert _errors(tmp_path, b"#h\n" + ok + b"r chr1 10 chr1\n" + b"r chr1 x chr1 3\n") == (3, "fewer fields than the columns need")
    assert _errors(tmp_path, ok + b"r chr1 1x chr1 3\n")[0] == 2
    assert _errors(tmp_path, ok + b"r chr1 1234567890123456789 chrM 3\n")[1] == "a position is not 1 to 18 digits"
    assert _errors(tmp_path, ok * 3 + b"r chr1 0 chr1 3\n") == (4, "a position lies outside its chromosome")
    assert _errors(tmp_path, ok + b"r chrX 1 chrX 13\n")[0] == 2
    assert _errors(tmp_path, ok + b"r chrX 0 chrX 12\n", base=0)[0] == 2
    assert _errors(tmp_path, ok + b"r chr1 3 chrM 0\n" + ok + b"r chr1 1 chr1 5001\n")[0] == 4
    assert _errors(tmp_path, ok + b"r chr1 2 chr1 3 " + b"x" * 100 + b"\n", window=60) == (2, "longer than the device window")
    assert _errors(tmp_path, b"") == (0, "holds no pair lines")
    assert _errors(tmp_path, b"# only\n\n \t\r\n") == (0, "holds no pair lines")
    assert _errors(tmp_path, gzip.compress(ok)) == (0, "compressed input is not read")
    # the edges pass: positions index_base and length - 1 + index_base, a last line without '\n', a line of exactly
    # the window's bytes
    path = tmp_path / "k.pairs"
    path.write_bytes(b"r chr1 1 chr1 5000\nr chrX 12 chrX 1")
    out, counts = P.bin_pairs_text([path], SIZES, 10)
    assert counts["cis"] == 2 and out[0][1].tolist() == [499] and out[3][1].tolist() == [1]
    path.write_bytes(ok)
    assert P.bin_pairs_text([path], SIZES, 10, window=len(ok))[1]["cis"] == 1


# ---- host logic --------------------------------------------------------------------------------------------------------

def test_chromsizes_in_all_its_forms(tmp_path):
    want = [("chr1", 5000), ("chr10", 3001), ("chr2", 777), ("chrX", 12)]
    sizes = tmp_path / "g.chrom.sizes"
    sizes.write_text("chr1\t5000\nchr10\t3001\n\nchr2 777\nchrX\t12\textra\n")
    assert read_chromsizes(str(sizes)) == want
    assert read_chromsizes(want) == want
    assert read_chromsizes([list(x) for x in want]) == want
    assert read_chromsizes(dict(want)) == want
    assert read_chromsizes([("chr1", np.int64(5000)), ("chr10", 3001.0), ("chr2", "777"), ("chrX", 12)]) == want
    pairs = tmp_path / "h.pairs"
    P.write_pairs(pairs, "4dn", want, 10, 1, 1, seed=1)
    assert read_chromsizes(None, str(pairs)) == want
    g = GenomePairs(str(pairs), binsize=100)
    assert g.names == [n for n, _ in want] and g.chrom_bins.tolist() == [50, 31, 8, 1]
    assert g.columns == (1, 2, 3, 4) and g.index_base == 1 and g.paths == [str(pairs)]
    g = GenomePairs([pairs, pairs], dict(want), binsize=np.int64(3001), columns=[1, 2, 4, 5], index_base=0)
    assert g.chrom_bins.tolist() == [2, 1, 1, 1] and g.columns == (1, 2, 4, 5) and g.index_base == 0
    bare = tmp_path / "bare.pairs"
    P.write_pairs(bare, "hicpro", want, 10, 1, 1, seed=1)
    with pytest.raises(ValueError, match="no '#chromsize:' header lines"):
        GenomePairs(bare, binsize=10)


@pytest.mark.parametrize("kw,msg", [
    (dict(binsize=0), "binsize must be an integer >= 1"),
    (dict(binsize=None), "binsize must be an integer >= 1"),
    (dict(binsize=2.5), "binsize must be an integer >= 1"),
    (dict(binsize=True), "binsize must be an integer >= 1"),
    (dict(columns=(1, 2, 3)), "columns must be four different"),
    (dict(columns=(1, 2, 3, 3)), "columns must be four different"),
    (dict(columns=(1, 2, 3, 64)), "columns must be four different"),
    (dict(columns=(-1, 2, 3, 4)), "columns must be four different"),
    (dict(index_base=2), "index_base must be 0 or 1"),
    (dict(chromsizes=[("chr1", 10), ("chr1", 20)]), "appears twice"),
    (dict(chromsizes=[("", 10)]), "empty or contains whitespace"),
    (dict(chromsizes=[("chr 1", 10)]), "empty or contains whitespace"),
    (dict(chromsizes=[("chr1", 0)]), "a whole number >= 1"),
    (dict(chromsizes=[("chr1", 10.5)]), "a whole number >= 1"),
    (dict(chromsizes=[("chr1", "ten")]), "a whole number >= 1"),
    (dict(chromsizes=[]), "the chromosome table is empty"),
    (dict(chromsizes=[("chr1", 2 ** 31), ("chr2", 10)], binsize=1), "at most 2\\^31 - 2"),
])
def test_argument_errors(tmp_path, kw, msg):
    args = dict(chromsizes=SIZES, binsize=10)
    args.update(kw)
    with pytest.raises(ValueError, match=msg):
        GenomePairs(str(tmp_path / "x.pairs"), **args)
    with pytest.raises(ValueError, match="one or more file paths"):
        GenomePairs([], SIZES, binsize=10)


class _FakeGenome:
    def __init__(self, chrom_bins):
        self.chrom_bins = np.array(chrom_bins, dtype=np.int32)

    def coarsen(self, factor):
        return _FakeGenome(-(-self.chrom_bins // factor))

    def downsample(self, contacts, seed):
        return _FakeGenome(self.chrom_bins)

    def depth(self):
        return np.array([10, 10], dtype=np.uint64)

    def close(self):
        pass


class _FakeCtx:
    def close(self):
        pass


def test_binsize_and_pair_counts_bookkeeping():
    counts = dict(lines=9, cis=5, trans=3, unplaced=1)
    g = LoadedGenome(_FakeGenome([10, 5]), ["a", "b"], _CtxRef(_FakeCtx(), True), binsize=1000, pair_counts=counts)
    assert g.binsize == 1000 and g.pair_counts == counts
    c = g.coarsen(3)
    assert c.binsize == 3000 and c.factor == 3 and c.pair_counts is None
    assert c.downsample(contacts=4).binsize == 3000
    px = LoadedGenome(_FakeGenome([10, 5]), ["a", "b"], _CtxRef(_FakeCtx(), True))
    assert px.binsize is None and px.pair_counts is None and px.coarsen(2).binsize is None


# ---- ABI and R -----------------------------------------------------------------------------------------------------------

def test_symbol_is_declared_and_bound():
    with open(os.path.join(ROOT, "include", "tadpole_b200.h")) as fh:
        assert re.search(r"\bint tp_genome_ingest_pairs_file\(tp_ctx \*ctx, const char \*const \*paths, int npaths, "
                         r"const char \*const \*names,\s+const int64_t \*lengths, int nchrom, int64_t binsize, "
                         r"const int cols\[4\], int index_base,\s+unsigned long long counts_out\[4\], tp_genome \*\*out\);",
                         fh.read())
    assert "tp_genome_ingest_pairs_file" in _lib.EXPORTED
    lib = _lib.load()
    assert lib.tp_version() >= 109
    out = ctypes.c_void_p()
    assert lib.tp_genome_ingest_pairs_file(None, None, 0, None, None, 0, 1, None, 1, None, ctypes.byref(out)) == _lib.TP_ERR_ARG
    assert "null argument" in lib.tp_last_error().decode()


@pytest.fixture(scope="module")
def R():
    import __graft_entry__ as g
    g.build()
    from mock_r.driver import MockR
    r = MockR()
    yield r
    r.reset()


def _strings(R, items):
    """a character vector of the mock R runtime"""
    from mock_r.driver import STRSXP, Sexp
    L = R.lib
    elts = [L.mock_elt(L.mock_string(s.encode()), 0) for s in items]
    arr = (ctypes.c_void_p * max(len(elts), 1))(*elts)
    return Sexp(L.mock_vector(STRSXP, len(elts), ctypes.cast(arr, ctypes.c_void_p)))


def test_r_routine_is_registered_and_checks_its_arguments(R):
    from mock_r.driver import RError
    assert R.registered("C_tp_genome_pairs_file") == 6
    with pytest.raises(RError, match="takes 6 arguments"):
        R.call("C_tp_genome_pairs_file", 0, 0, 1)
    paths, names = _strings(R, ["a.pairs"]), _strings(R, ["chr1", "chr2"])
    lay = np.array([1, 2, 3, 4, 1], np.int32)
    good = np.array([100.0, 200.0])
    with pytest.raises(RError, match="at least one pairs file"):
        R.call("C_tp_genome_pairs_file", 0, _strings(R, []), names, good, 10.0, lay)
    with pytest.raises(RError, match="as many numeric lengths"):
        R.call("C_tp_genome_pairs_file", 0, paths, names, np.array([100.0]), 10.0, lay)
    with pytest.raises(RError, match="as many numeric lengths"):
        R.call("C_tp_genome_pairs_file", 0, paths, names, np.array([100, 200], np.int32), 10.0, lay)
    for bad in (0.0, 1.5, float("nan")):
        with pytest.raises(RError, match="lengths must be whole numbers"):
            R.call("C_tp_genome_pairs_file", 0, paths, names, np.array([100.0, bad]), 10.0, lay)
        with pytest.raises(RError, match="binsize must be a whole number"):
            R.call("C_tp_genome_pairs_file", 0, paths, names, good, bad, lay)
    with pytest.raises(RError, match="layout must be"):
        R.call("C_tp_genome_pairs_file", 0, paths, names, good, 10.0, lay[:4])
    with pytest.raises(RError, match="GPU context has been released"):
        R.call("C_tp_genome_pairs_file", 0, paths, names, good, 10.0, lay)


def test_r_function_is_exported_and_carries_the_binsize():
    pkg = os.path.join(ROOT, "r-package", "TADpoleB200")
    with open(os.path.join(pkg, "NAMESPACE")) as fh:
        assert "export(genome_load_pairs)" in fh.read().split("\n")
    with open(os.path.join(pkg, "R", "tadpole.R")) as fh:
        src = fh.read()
    body = src[src.index("genome_load_pairs <- function(paths, chromsizes = NULL, binsize, columns = 2:5, index_base = 1L)"):]
    body = body[:body.index("\n}\n")]
    assert "C_tp_genome_pairs_file" in body and "as.integer(c(columns - 1L, index_base))" in body
    assert 'attr(g, "binsize") <- binsize' in body and 'attr(g, "pairs")' in body
    coarse = src[src.index("genome_coarsen <- function("):]
    assert 'attr(out, "binsize") <- attr(g, "binsize") * factor' in coarse[:coarse.index("\n}\n")]
