"""diffT_genome against the per-comparison loop it replaces, on the same context (run on the GPU):

  A  diffT_genome(control, case, nperm): every (chromosome, level) comparison and all its random partitions in one
     library call (tp_difft_multi).
  B  the loop a user writes without it: for each comparison, diffT(x, y) and the null totals of tp_difft_null with the
     same bad columns and seed (Context.difft_null without curves: the totals diffT_genome returns).

Input: two seeded human-like genomes at 50 kb (the 24 GRCh38 chromosomes, 61.8k bins), control and a case in which every
third chromosome is drawn with another seed, each called with TADpole_genome.  Both routes must give the same bits
(observed curves and null totals) before anything is timed.  The routes alternate; device ms is the sum of the diffT
kernels' CUDA-event times (profile class "difft", which covers the observed-pair, random-partition and fused kernels).
Prints one JSON line (also written to --out): problems, sum of L, nperm, wall and device ms of both routes, the card's
name and power limit.

    python tests/difft_genome_timing.py [--steps 3] [--nperm 1000] [--scale 1.0] [--out result.json]
"""
import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

from genome_timing import GRCH38, card  # noqa: E402


def genome(sizes, redraw, seed):
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


def route_b(problems, ctx, nperm, seed):
    from tadpole_b200 import diffT
    curves, null = [], []
    for p, pr in enumerate(problems):
        curves.append(diffT(pr["x"], pr["y"], ctx=ctx))
        r = ctx.difft_null(pr["tx"], pr["ntads"], nperm, pad_left=pr["pad_left"], pad_right=pr["pad_right"],
                           bad_positions=pr["bad"] if pr["bad"].size else None, seed=(seed + p) % 2 ** 64, want_curves=False)
        null.append(r["totals"])
    return curves, np.array(null)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=3, help="timed repetitions of each route (alternating A, B)")
    ap.add_argument("--nperm", type=int, default=1000)
    ap.add_argument("--scale", type=float, default=1.0, help="chromosome sizes x scale (rehearsals at a small size)")
    ap.add_argument("--seed", type=int, default=1)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    from tadpole_b200 import Context, TADpole_genome, api, diffT_genome
    from tadpole_b200.batch import _difft_genome_problems
    api.QUIET = True
    sizes = [max(2, int(round(-(-ln // 50000) * a.scale))) for _, ln in GRCH38]
    ctx = Context(0)
    t = time.perf_counter()
    control = TADpole_genome(genome(sizes, (), a.seed), ctx=ctx)
    case = TADpole_genome(genome(sizes, range(0, 24, 3), a.seed), ctx=ctx)
    call_s = time.perf_counter() - t
    problems, skipped = _difft_genome_problems(control, case)
    # same bits first (and a warm-up of both routes)
    ra = diffT_genome(control, case, nperm=a.nperm, seed=a.seed, ctx=ctx)
    cb, nb = route_b(problems, ctx, a.nperm, a.seed)
    identical = (len(ra.chrom) == len(problems) and np.array_equal(ra.null_totals, nb)
                 and all(np.array_equal(x, y) for x, y in zip(ra.curves, cb)))
    wa, wb, da, db = [], [], [], []
    for _ in range(a.steps):
        ctx.profile(1)
        t = time.perf_counter()
        diffT_genome(control, case, nperm=a.nperm, seed=a.seed, ctx=ctx)
        wa.append((time.perf_counter() - t) * 1e3)
        da.append(ctx.profile(0)["difft"][0])
        ctx.profile(1)
        t = time.perf_counter()
        route_b(problems, ctx, a.nperm, a.seed)
        wb.append((time.perf_counter() - t) * 1e3)
        db.append(ctx.profile(0)["difft"][0])
    ctx.close()
    out = dict(card=card(), chromosomes=len(sizes), bins=int(sum(sizes)), problems=len(problems), skipped=len(skipped),
               sum_L=int(sum(p["tx"].size for p in problems)), nperm=a.nperm, tadpole_genome_s=round(call_s, 1),
               identical=bool(identical), steps=a.steps,
               A_wall_ms=[round(x, 1) for x in wa], A_device_ms=[round(x, 1) for x in da],
               B_wall_ms=[round(x, 1) for x in wb], B_device_ms=[round(x, 1) for x in db])
    line = json.dumps(out)
    print(line)
    if a.out:
        with open(a.out, "w") as fh:
            fh.write(line + "\n")
    if not identical:
        sys.exit("the two routes differ")


if __name__ == "__main__":
    main()
