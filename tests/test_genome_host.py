"""CPU tests of the genome-wide input's host side: bin tables become chromosome names and bins per chromosome
(tadpole_b200.read_bins), and oracle/genome_oracle.py (split_genome_pixels), the checker of the GPU route kernel, splits
a pixel list the way a vectorised restatement does."""
import numpy as np
import pytest

from oracle import genome_oracle as G


def test_hicpro_abs_bed(tmp_path):
    from tadpole_b200 import read_bins
    p = tmp_path / "sample_50000_abs.bed"
    rows = [("chr1", i) for i in range(3)] + [("chr2", i) for i in range(2)] + [("chrX", 0)]
    p.write_text("".join(f"{c}\t{i * 50000}\t{(i + 1) * 50000}\t{k + 1}\n" for k, (c, i) in enumerate(rows)))
    names, n = read_bins(str(p))
    assert names == ["chr1", "chr2", "chrX"] and n.tolist() == [3, 2, 1] and n.dtype == np.int32


def test_cooler_bins_with_header(tmp_path):
    from tadpole_b200 import read_bins
    p = tmp_path / "bins.tsv"
    p.write_text("chrom\tstart\tend\tweight\n" + "".join(f"chr{c}\t{i}\t{i + 1}\t0.5\n" for c, k in ((1, 4), (2, 1), (10, 2))
                                                          for i in range(k)))
    names, n = read_bins(p)
    assert names == ["chr1", "chr2", "chr10"] and n.tolist() == [4, 1, 2]
    # the same without the header line
    p.write_text("".join(f"chr{c}\t{i}\t{i + 1}\n" for c, k in ((1, 4), (2, 1), (10, 2)) for i in range(k)))
    assert read_bins(p)[1].tolist() == [4, 1, 2]


def test_tables_and_name_count_lists():
    from tadpole_b200 import read_bins
    names, n = read_bins([("chr1", 5), ("chr2", 1), ("chrM", 2)])
    assert names == ["chr1", "chr2", "chrM"] and n.tolist() == [5, 1, 2]
    assert read_bins(np.array([["a", "0"], ["a", "1"], ["b", "0"]]))[1].tolist() == [2, 1]
    assert read_bins(["a", "a", "a", "b"]) == (["a", "b"], pytest.approx(np.array([3, 1])))
    pd = pytest.importorskip("pandas")
    assert read_bins(pd.DataFrame({"chrom": ["x", "y", "y"], "start": [0, 0, 1]}))[1].tolist() == [1, 2]


def test_non_contiguous_chromosome_is_an_error(tmp_path):
    from tadpole_b200 import GenomePixels, read_bins
    with pytest.raises(ValueError, match="reappears"):
        read_bins(["chr1", "chr1", "chr2", "chr1"])
    with pytest.raises(ValueError, match="reappears"):
        read_bins([("chr1", 2), ("chr2", 2), ("chr1", 1)])
    p = tmp_path / "abs.bed"
    p.write_text("chr1\t0\t10\t1\nchr2\t0\t10\t2\nchr1\t10\t20\t3\n")
    with pytest.raises(ValueError, match="chr1"):
        read_bins(str(p))
    with pytest.raises(ValueError, match="bin table"):
        GenomePixels([0], [0], [1.0])


def test_genome_pixels_index_base_defaults():
    from tadpole_b200 import GenomePixels
    assert GenomePixels([0], [0], [1.0], bins=[("a", 2)]).index_base == 0
    assert GenomePixels(path="x.matrix", bins=[("a", 2)]).index_base == 1
    assert GenomePixels(path="x.matrix", bins=[("a", 2)], index_base=0).index_base == 0


def split_vectorised(b1, b2, v, chrom_bins, base):
    starts = np.concatenate(([0], np.cumsum(chrom_bins)))
    x, y = np.asarray(b1, np.int64) - base, np.asarray(b2, np.int64) - base
    cx, cy = np.searchsorted(starts, x, "right") - 1, np.searchsorted(starts, y, "right") - 1
    cis = cx == cy
    up = cis & (x <= y)
    parts = [(x[up & (cx == c)] - starts[c], y[up & (cx == c)] - starts[c], np.asarray(v)[up & (cx == c)])
             for c in range(len(chrom_bins))]
    return parts, int((~cis).sum()), int((cis & (x > y)).sum())


@pytest.mark.parametrize("base", [0, 1])
def test_split_genome_pixels_against_vectorised_split(base):
    rng = np.random.default_rng(base + 3)
    chrom_bins = [40, 1, 2, 17, 300, 5]
    total = sum(chrom_bins)
    b1 = rng.integers(0, total, 5000) + base
    b2 = rng.integers(0, total, 5000) + base
    v = rng.poisson(3.0, 5000).astype(float)
    v[::41] = np.nan
    got, trans, below = G.split_genome_pixels(b1, b2, v, chrom_bins, base)
    want, wt, wb = split_vectorised(b1, b2, v, chrom_bins, base)
    assert (trans, below) == (wt, wb) and trans > 0 and below > 0
    for (i, j, x), (wi, wj, wx) in zip(got, want):
        assert np.array_equal(i, wi) and np.array_equal(j, wj) and np.array_equal(x, wx, equal_nan=True)
    assert sum(p[0].size for p in got) + trans + below == b1.size


def test_split_genome_pixels_small_case_and_errors():
    parts, trans, below = G.split_genome_pixels([0, 2, 3, 4, 1], [1, 4, 3, 3, 2], [1.0, 2.0, 3.0, 4.0, 5.0], [2, 3])
    assert trans == 1 and below == 1                 # (0, 1) cis on chr A; (2, 4) and (3, 3) cis on B; (4, 3) below; (1, 2) trans
    assert parts[0][0].tolist() == [0] and parts[0][1].tolist() == [1]
    assert parts[1][0].tolist() == [0, 1] and parts[1][1].tolist() == [2, 1] and parts[1][2].tolist() == [2.0, 3.0]
    with pytest.raises(ValueError, match="entry 2 is outside the 5 bins"):
        G.split_genome_pixels([0, 5], [0, 0], [1.0, 1.0], [2, 3])
