"""CPU tests of diffT_genome's host side: which (chromosome, level) problems are built from two genome-wide calls, with
which padded labels, bad positions and seeds, and why the others are skipped.  The library call itself is replaced by a
stand-in context, so nothing here needs a GPU; tests/test_gpu_difft_genome.py checks the numbers on the device."""
import numpy as np
import pytest

from oracle import tadpole_oracle as O


def tadpole_like(tables, kept):
    """A Tadpole-like dict: clusters {str(level): [rows, 2] start / end} and a dendrogram whose labels are the kept bins."""
    return {"clusters": {str(k): np.asarray(t, dtype=np.int64) for k, t in tables.items()},
            "dendro": {"labels": np.asarray(kept, dtype=np.int64)}}


class FakeCtx:
    """Stands in for Context.difft_multi: records the arguments and returns recognisable values."""

    def __init__(self, refuse=()):
        self.refuse = set(refuse)
        self.args = None

    def difft_multi(self, off, lx, ly, pad_left, pad_right, ntads, bad_off, bad, seed=0, nperm=1000, want_curves=True):
        self.args = dict(off=np.asarray(off), lx=np.asarray(lx), ly=np.asarray(ly), pad_left=list(pad_left),
                         pad_right=list(pad_right), ntads=list(ntads), bad_off=np.asarray(bad_off), bad=np.asarray(bad),
                         seed=seed, nperm=nperm)
        nprob = len(off) - 1
        totals = np.arange(nprob, dtype=np.float64) * 10
        null = np.tile(np.arange(nperm, dtype=np.float64) * 3, (nprob, 1))
        status = np.array([1 if p in self.refuse else 0 for p in range(nprob)], dtype=np.int32)
        null[status != 0] = np.nan
        curves = np.arange(off[-1], dtype=np.float64)
        return dict(curves=curves, totals=totals, null_totals=null, status=status)


def genome_pair():
    # chr1: levels 2, 3 and 5 in control, 2, 3 and 4 in case; the case's tables start at bin 3 and miss bins 7 and 8
    c1 = tadpole_like({2: [[1, 10], [11, 20]], 3: [[1, 5], [6, 12], [13, 20]], 5: [[1, 4], [5, 8], [9, 12], [13, 16], [17, 20]]},
                      np.arange(1, 21))
    k1 = tadpole_like({2: [[3, 9], [10, 22]], 3: [[3, 6], [9, 14], [15, 22]], 4: [[3, 6], [9, 12], [13, 16], [17, 22]]},
                      [b for b in range(3, 23) if b not in (7, 8)])
    # chr2: unequal row counts at level 2 (the reference's stop), equal at level 3
    c2 = tadpole_like({2: [[1, 5], [6, 9]], 3: [[1, 3], [4, 6], [7, 9]]}, np.arange(1, 10))
    k2 = tadpole_like({2: [[1, 3], [4, 6], [7, 9]], 3: [[1, 2], [3, 7], [8, 9]]}, np.arange(1, 10))
    arms = {"p": {}, "q": {}, "merging_arms": np.zeros((0, 2))}
    return c1, k1, c2, k2, arms


def test_problems_levels_padding_and_bad_positions():
    from tadpole_b200.batch import _difft_genome_problems
    c1, k1, c2, k2, _ = genome_pair()
    probs, skipped = _difft_genome_problems({"chr1": c1, "chr2": c2}, {"chr2": k2, "chr1": k1})
    assert [(p["chrom"], p["level"]) for p in probs] == [("chr1", 2), ("chr1", 3), ("chr2", 3)]   # control's order
    assert skipped == {("chr2", 2): "Both calls must have the same number of TADs."}
    for p in probs:
        x = c1 if p["chrom"] == "chr1" else c2
        y = k1 if p["chrom"] == "chr1" else k2
        bx, by = x["clusters"][str(p["level"])], y["clusters"][str(p["level"])]
        tx, ty = O.difft_labels(bx, by)
        assert np.array_equal(p["tx"], tx) and np.array_equal(p["ty"], ty)
        sx, sy, ex, ey = bx[0, 0], by[0, 0], bx[-1, 1], by[-1, 1]
        assert (p["pad_left"], p["pad_right"], p["ntads"]) == (max(0, sy - sx), max(0, ex - ey), by.shape[0])
        # the y part of the padded extent is bin_index of y itself
        size = ey - sy + 1
        assert np.array_equal(p["ty"][p["pad_left"]:p["pad_left"] + size], O.bin_index(by, size))
    # bad positions: the case's filtered bins 7, 8 inside its extent 3..22, as positions within start:end
    assert probs[0]["bad"].tolist() == [5, 6] and probs[1]["bad"].tolist() == [5, 6]
    assert probs[2]["bad"].size == 0


def test_requested_levels_and_skipped_reasons():
    from tadpole_b200.batch import GenomeResult, _difft_genome_problems
    c1, k1, c2, k2, arms = genome_pair()
    control = GenomeResult(chr1=c1, chr2=c2, chr3=arms, chr5=c2)
    control.failed = {"chr4": "no significant level"}
    case = GenomeResult(chr1=k1, chr3=arms, chr4=k2, chr6=k2)
    case.failed = {"chr2": "TADpole error", "chr7": "elsewhere"}
    probs, skipped = _difft_genome_problems(control, case, levels=[4, 3, 5, 3])
    assert [(p["chrom"], p["level"]) for p in probs] == [("chr1", 3)]
    assert skipped[("chr1", 4)] == "level 4 is not scored in control"
    assert skipped[("chr1", 5)] == "level 5 is not scored in case"
    assert skipped["chr2"] == "failed in case: TADpole error"
    assert skipped["chr3"].startswith("centromere_search result")
    assert skipped["chr4"] == "failed in control: no significant level"
    assert skipped["chr5"] == "missing from case"
    assert skipped["chr6"] == "missing from control"
    assert skipped["chr7"] == "failed in case: elsewhere"
    assert len(skipped) == 8


def test_library_call_seeds_and_result_packing():
    from tadpole_b200.batch import diffT_genome
    c1, k1, c2, k2, _ = genome_pair()
    fake = FakeCtx(refuse={1})
    seed = 2 ** 64 - 2
    res = diffT_genome({"chr1": c1, "chr2": c2}, {"chr1": k1, "chr2": k2}, nperm=7, seed=seed, ctx=fake)
    a = fake.args
    lens = [15 + 7, 15 + 7, 9]                                  # chr1: extent 1..22 at both levels; chr2: 9 bins
    assert a["off"].tolist() == [0, 22, 44, 53] and a["seed"] == seed and a["nperm"] == 7
    assert a["lx"].size == sum(lens) and a["bad_off"].tolist() == [0, 2, 4, 4] and a["bad"].tolist() == [5, 6, 5, 6]
    assert a["ntads"] == [2, 3, 3] and a["pad_left"] == [2, 2, 0] and a["pad_right"] == [0, 0, 0]
    # problem 1 was refused: it is skipped with the reason, the others keep their own seed seed + p (mod 2^64)
    assert res.chrom == ["chr1", "chr2"] and res.level.tolist() == [2, 3]
    assert res.seed == [seed, (seed + 2) % 2 ** 64] == [2 ** 64 - 2, 0]
    assert "refused" in res.skipped[("chr1", 3)] and "2 borders" in res.skipped[("chr1", 3)]
    assert res.total.tolist() == [0.0, 20.0]
    assert res.null_totals.shape == (2, 7)
    # p_value = (1 + #{null <= total}) / (nperm + 1); null = 0, 3, ..., 18
    assert res.p_value.tolist() == [2 / 8, 8 / 8]
    assert np.array_equal(res.curves[0], np.arange(0, 22)) and np.array_equal(res.curves[1], np.arange(44, 53))


def test_nothing_to_compare():
    from tadpole_b200.batch import diffT_genome
    c1, k1, *_ = genome_pair()
    fake = FakeCtx()
    res = diffT_genome({"chr1": c1}, {"chr2": k1}, nperm=5, ctx=fake)
    assert fake.args is None and res.chrom == [] and res.null_totals.shape == (0, 5)
    assert res.skipped == {"chr1": "missing from case", "chr2": "missing from control"}
