"""GPU tests of tp_difft_multi and diffT_genome: ragged diffT comparisons, each with its own null distribution drawn and
scored on the device in one call.  Integer work: every curve and total is compared bit for bit with the single calls
(tp_difft_batch, tp_difft_null) and with the oracle."""
import os
import sys

import numpy as np
import pytest

from oracle import tadpole_oracle as O

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tests"))
pytestmark = pytest.mark.gpu


def exact_total(tx, ty):
    """Sum of the per-bin diffT scores: sum cx^2 + sum cy^2 - 2 sum J^2 over non-zero labels (integer)."""
    tx, ty = np.asarray(tx, np.int64), np.asarray(ty, np.int64)
    sq = lambda a: int((np.unique(a, return_counts=True, axis=0)[1].astype(np.int64) ** 2).sum()) if len(a) else 0
    both = (tx != 0) & (ty != 0)
    return sq(tx[tx != 0]) + sq(ty[ty != 0]) - 2 * sq(np.stack([tx[both], ty[both]], axis=1))


def partition(rng, start, end, ntads):
    cuts = np.sort(rng.choice(np.arange(start + 1, end + 1), ntads - 1, replace=False))
    return np.stack([np.concatenate(([start], cuts)), np.concatenate((cuts - 1, [end]))], axis=1)


def ragged_mix():
    """(x bed, y bed, bad positions) of a ragged mix: 1 to 30 000 bins, 1 to 1 200 TADs, pads on either side, gaps and
    overwritten rows in x, and one problem random_bed refuses (in the middle)."""
    rng = np.random.default_rng(11)
    mix = []
    mix.append((np.array([[1, 1]]), np.array([[1, 1]]), []))                                   # L = 1, one TAD
    mix.append((partition(rng, 1, 500, 1), partition(rng, 1, 500, 1), [3, 4]))                 # ntads = 1
    x = partition(rng, 5, 2000, 40)
    x[::3, 1] -= 2                                                                              # zero gaps in x
    mix.append((x, partition(rng, 1, 1980, 40), [1, 2, 50, 700]))                              # pad left of x, right of y
    mix.append((partition(rng, 1, 30000, 1200), partition(rng, 3, 30010, 1200), [9, 10, 11]))  # overflows the shared table
    x = partition(rng, 1, 800, 20)
    x[10] = [x[8, 0] + 3, x[8, 0] + 5]                                                          # row 11 splits row 9 in two
    x[14] = [x[13, 1], x[13, 0]]                                                                # a reversed row (seq counts down)
    mix.append((x, partition(rng, 1, 800, 20), []))                                            # non-contiguous x labels
    mix.append((partition(rng, 1, 30, 10), partition(rng, 1, 30, 10), list(range(2, 29))))    # refused: 9 borders, 1 bin
    mix.append((partition(rng, 1, 5000, 60), partition(rng, 1, 5000, 60), list(range(100, 300))))
    mix.append((partition(rng, 1, 3, 3), partition(rng, 1, 3, 3), []))                         # every candidate taken
    mix.append((partition(rng, 100, 1400, 1100), partition(rng, 90, 1390, 1100), [5]))         # 1 100 TADs, pads both sides
    return mix


def multi_args(mix):
    labs = [O.difft_labels(x, y) for x, y, _ in mix]
    off = np.concatenate(([0], np.cumsum([tx.size for tx, _ in labs])))
    pl = [max(0, int(y[0, 0] - x[0, 0])) for x, y, _ in mix]
    pr = [max(0, int(x[-1, 1] - y[-1, 1])) for x, y, _ in mix]
    nt = [y.shape[0] for _, y, _ in mix]
    boff = np.concatenate(([0], np.cumsum([len(b) for *_, b in mix])))
    bad = np.concatenate([np.asarray(b, np.int32) for *_, b in mix]).astype(np.int32)
    return labs, off, pl, pr, nt, boff, bad


def test_ragged_mix_equals_the_single_calls(ctx):
    mix = ragged_mix()
    labs, off, pl, pr, nt, boff, bad = multi_args(mix)
    nperm, seed = 48, 2 ** 64 - 3                                    # the per-problem seed wraps at 2^64
    ctx.profile(1)
    r = ctx.difft_multi(off, np.concatenate([a for a, _ in labs]), np.concatenate([b for _, b in labs]), pl, pr, nt, boff,
                        bad, seed=seed, nperm=nperm)
    ctx.profile(0)
    assert r["status"].tolist() == [0, 0, 0, 0, 0, 1, 0, 0, 0]
    for p, ((x, y, b), (tx, ty)) in enumerate(zip(mix, labs)):
        curve = r["curves"][off[p]:off[p + 1]]
        assert np.array_equal(curve, ctx.difft_batch(tx[None], ty[None])[0]), p
        assert r["totals"][p] == exact_total(tx, ty), p
        if r["status"][p]:
            assert np.isnan(r["null_totals"][p]).all()
            continue
        s = (seed + p) % 2 ** 64
        single = ctx.difft_null(tx, nt[p], nperm, pad_left=pl[p], pad_right=pr[p], bad_positions=b, seed=s,
                                want_curves=False)
        assert np.array_equal(r["null_totals"][p], single["totals"]), p
        if tx.size <= 2000:                                          # the oracle's generator and O(L^2) loop
            for perm in (0, 17, nperm - 1):
                rb = O.random_bed(y, bad_columns=b or None, seed=s, perm=perm)
                assert r["null_totals"][p, perm] == O.difft(x, rb, raw=True)[-1], (p, perm)
    # the 1 200-TAD pair has more label keys (x, y and joint) than the 4 096 slots of the shared table and the 1 100-TAD
    # pair fewer: the shared-table launch and the overflow launch both ran in this one call
    keys = lambda tx, ty: np.unique(tx).size + np.unique(ty).size + np.unique(np.stack([tx, ty]), axis=1).shape[1]
    assert keys(*labs[3]) > 4096 > keys(*labs[8])


def test_refused_problem_raises_in_the_single_call(ctx):
    mix = ragged_mix()
    x, y, b = mix[5]
    tx, _ = O.difft_labels(x, y)
    from tadpole_b200 import TadpoleError
    with pytest.raises(TadpoleError, match="sample larger than the population"):
        ctx.difft_null(tx, y.shape[0], 4, bad_positions=b)


def test_arguments_are_checked(ctx):
    from tadpole_b200 import TadpoleError
    one = np.ones(4, np.int32)
    with pytest.raises(TadpoleError, match="1-based"):
        ctx.difft_multi([0, 4], one, one, [0], [0], [2], [0, 1], [0], nperm=2)
    with pytest.raises(TadpoleError, match="extent"):
        ctx.difft_multi([0, 4], one, one, [2], [2], [2], [0, 0], [], nperm=2)
    with pytest.raises(TadpoleError, match="L_p"):
        ctx.difft_multi(np.array([0, 4, 4]), one, one, [0, 0], [0, 0], [1, 1], [0, 0, 0], [], nperm=2)


def test_launches_do_not_grow_with_the_number_of_problems(ctx):
    rng = np.random.default_rng(3)

    def run(n):
        mix = [(partition(rng, 1, L, T), partition(rng, 1, L, T), [])
               for L, T in zip(rng.integers(50, 400, n), rng.integers(1, 20, n))]
        labs, off, pl, pr, nt, boff, bad = multi_args(mix)
        before = ctx.launches
        r = ctx.difft_multi(off, np.concatenate([a for a, _ in labs]), np.concatenate([b for _, b in labs]), pl, pr, nt,
                            boff, bad, seed=1, nperm=20)
        assert (r["status"] == 0).all() and r["null_totals"].shape == (n, 20)
        return ctx.launches - before

    assert run(3) == run(300) == 2                                   # observed pairs + fused null draws


def genome_inputs(sizes, redraw=(), seed=1):
    """GenomePixels of a seeded genome (synth_genome_pixels' matrices, cis pixels only); chromosomes in `redraw` get the
    matrix of another seed."""
    from tadpole_b200 import GenomePixels
    from tadpole_b200.synth import synth_genome_pixels, synth_hic
    names, _, mats = synth_genome_pixels(sizes, seed=seed, trans_per_chrom=0)
    mats = [synth_hic(n, seed=seed + 1000 + c) if c in redraw else m for c, (n, m) in enumerate(zip(sizes, mats))]
    starts = np.concatenate(([0], np.cumsum(sizes)))
    b1, b2, v = [], [], []
    for c, m in enumerate(mats):
        i, j = np.triu_indices(m.shape[0])
        s = m[i, j] != 0
        b1.append(i[s] + starts[c]); b2.append(j[s] + starts[c]); v.append(m[i, j][s])
    return GenomePixels(np.concatenate(b1).astype(np.int32), np.concatenate(b2).astype(np.int32), np.concatenate(v),
                        bins=list(zip(names, sizes)))


def case_bad(case, chrom, y):
    start, end = int(y[0, 0]), int(y[-1, 1])
    span = np.arange(start, end + 1)
    return (span[~np.isin(span, case[chrom].dendro.labels)] - start + 1).tolist()


@pytest.fixture(scope="module")
def genomes(ctx):
    from tadpole_b200 import TADpole_genome, api
    api.QUIET = True
    sizes = [420, 300, 380, 260]
    control = TADpole_genome(genome_inputs(sizes), ctx=ctx)
    case = TADpole_genome(genome_inputs(sizes, redraw=(1, 3)), ctx=ctx)
    assert not control.failed and not case.failed
    return control, case


def test_identical_samples(ctx, genomes):
    from tadpole_b200 import diffT_genome
    g, _ = genomes
    res = diffT_genome(g, g, nperm=50, seed=9, ctx=ctx)
    assert len(res.chrom) == sum(len(t.clusters) for t in g.values()) and not res.skipped
    assert (res.total == 0).all() and all((c == 0).all() for c in res.curves)            # quirk Q10: an all-zero curve
    assert np.array_equal(res.p_value, (1 + (res.null_totals == 0).sum(axis=1)) / 51)


def test_end_to_end_equals_the_loop_of_single_calls(ctx, genomes):
    from tadpole_b200 import diffT, diffT_genome, diffT_null
    control, case = genomes
    res = diffT_genome(control, case, nperm=100, seed=5, ctx=ctx)
    assert not res.skipped and len(res.chrom) > 8
    p = 0
    for chrom in control:
        for k in sorted(set(int(k) for k in control[chrom].clusters) & set(int(k) for k in case[chrom].clusters)):
            x, y = control[chrom].clusters[str(k)], case[chrom].clusters[str(k)]
            assert (res.chrom[p], res.level[p], res.seed[p]) == (chrom, k, 5 + p)
            assert np.array_equal(res.curves[p], diffT(x, y, ctx=ctx))
            tx, ty = O.difft_labels(x, y)
            assert res.total[p] == exact_total(tx, ty)
            null = diffT_null(x, y, nperm=100, bad_columns=case_bad(case, chrom, y) or None, seed=5 + p, ctx=ctx)
            assert np.array_equal(res.null_totals[p], null.totals)
            assert res.p_value[p] == (1 + (null.totals <= res.total[p]).sum()) / 101
            if chrom in ("chr1", "chr3"):                                                   # not redrawn
                assert res.total[p] == 0
            p += 1
    assert p == len(res.chrom)
    assert any(res.total[i] > 0 for i, c in enumerate(res.chrom) if c in ("chr2", "chr4"))


def test_r_shim_equals_python(ctx, genomes):
    from mock_r.driver import MockR
    from tadpole_b200.batch import _difft_genome_problems
    control, case = genomes
    probs, _ = _difft_genome_problems(control, case)
    off = np.concatenate(([0], np.cumsum([p["tx"].size for p in probs])))
    boff = np.concatenate(([0], np.cumsum([p["bad"].size for p in probs])))
    args = (np.concatenate([p["tx"] for p in probs]).astype(np.int32), np.concatenate([p["ty"] for p in probs]).astype(np.int32),
            np.array([p["pad_left"] for p in probs], np.int32), np.array([p["pad_right"] for p in probs], np.int32),
            np.array([p["ntads"] for p in probs], np.int32))
    bad = np.concatenate([p["bad"] for p in probs]).astype(np.int32)
    want = ctx.difft_multi(off, *args, boff, bad, seed=7, nperm=30)
    R = MockR()
    try:
        rctx = R.call("C_tp_ctx", 0, raw=True)
        curves, totals, null, status = R.call("C_tp_difft_multi", rctx, off.astype(np.float64), [args[0], args[1]],
                                              np.stack(args[2:], axis=1), boff.astype(np.float64), bad, 7.0, 30)
    finally:
        R.reset()
    assert np.array_equal(curves, want["curves"]) and np.array_equal(totals, want["totals"])
    assert null.shape == (30, len(probs)) and np.array_equal(null.T, want["null_totals"])
    assert np.array_equal(status, want["status"])


def test_scale_human_like_genome(ctx):
    """BASELINE configs[4] scale: 24 chromosomes (GRCh38 at 200 kb, 15.5k bins), every shared level, 1 000 random
    partitions per comparison; a few permutations spot-checked against the oracle."""
    from tadpole_b200 import TADpole_genome, diffT_genome, api
    from genome_timing import GRCH38
    api.QUIET = True
    sizes = [max(2, -(-ln // 200000)) for _, ln in GRCH38]
    control = TADpole_genome(genome_inputs(sizes, seed=4), ctx=ctx)
    case = TADpole_genome(genome_inputs(sizes, redraw=range(0, 24, 3), seed=4), ctx=ctx)
    res = diffT_genome(control, case, nperm=1000, seed=3, ctx=ctx)
    assert len(set(res.chrom)) >= 20 and len(res.chrom) > 100
    assert res.null_totals.shape == (len(res.chrom), 1000) and np.isfinite(res.null_totals).all()
    for p in (0, len(res.chrom) // 2, len(res.chrom) - 1):
        chrom, k = res.chrom[p], int(res.level[p])
        x, y = control[chrom].clusters[str(k)], case[chrom].clusters[str(k)]
        bad = case_bad(case, chrom, y) or None
        tx, ty = O.difft_labels(x, y)
        assert (res.curves[p] == O.difft_from_labels_c(tx, ty)).all()
        for perm in (0, 999):
            rb = O.random_bed(y, bad_columns=bad, seed=res.seed[p], perm=perm)
            assert res.null_totals[p, perm] == exact_total(*O.difft_labels(x, rb))
            if tx.size <= 1500:
                assert res.null_totals[p, perm] == O.difft(x, rb, raw=True)[-1]
