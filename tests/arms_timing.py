"""centromere_search over a whole genome, two routes on the same input (run on the GPU):

  A  TADpole_genome(GenomePixels(...), centromere_search=True): the pixels are split by chromosome on the GPU and every
     chromosome is split at its centromere and its two arms called in the library's batch workers (tp_call_genome_arms).
  B  the route without it: the pixels split by chromosome on the host into one dense FP64 matrix per chromosome, then a
     Python loop of TADpole(m, centromere_search=True), one call at a time.

Input: the seeded human-like genome of tests/genome_timing.py (the 24 GRCh38 chromosomes at --res bp, sizes x --scale),
every chromosome drawn with a centromere (synth_genome_pixels(centromere=...)).  Both routes must give the same bits for
every chromosome (the script exits non-zero if not).  Prints one JSON line (also written to --out): wall seconds of each
route per step (A and B alternate), A's batch device ms, the card's name and power limit.

    python tests/arms_timing.py [--res 50000] [--scale 1.0] [--steps 2] [--streams 4] [--out result.json]
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


def host_dense(b1, b2, v, sizes):
    """One dense upper-triangle matrix per chromosome from the global pixel list (trans and below-diagonal pixels
    dropped, repeated cells added)."""
    starts = np.concatenate(([0], np.cumsum(sizes)))
    cx, cy = np.searchsorted(starts, b1, "right") - 1, np.searchsorted(starts, b2, "right") - 1
    keep = (cx == cy) & (b1 <= b2)
    x, y, w, cx = b1[keep].astype(np.int64), b2[keep].astype(np.int64), v[keep], cx[keep]
    mats = []
    for c, n in enumerate(sizes):
        s = cx == c
        lin = (x[s] - starts[c]) * n + (y[s] - starts[c])
        mats.append(np.bincount(lin, weights=w[s], minlength=n * n).reshape(n, n))
    return mats


def route_b(b1, b2, v, names, sizes, ctx):
    from tadpole_b200 import TADpole, TadpoleError
    out, failed = {}, {}
    for nm, m in zip(names, host_dense(b1, b2, v, sizes)):
        try:
            out[nm] = TADpole(m, centromere_search=True, ctx=ctx)
        except (ValueError, TadpoleError) as e:
            failed[nm] = str(e)
    return out, failed


def bits(a, b):
    a, b = np.asarray(a), np.asarray(b)
    return a.shape == b.shape and np.array_equal(np.isnan(a), np.isnan(b)) and \
        np.array_equal(a.view(np.uint64)[~np.isnan(a)], b.view(np.uint64)[~np.isnan(b)])


def same(a, b):
    if "p" not in a or "p" not in b or not np.array_equal(a.merging_arms, b.merging_arms):
        return False
    for arm in ("p", "q"):
        x, y = a[arm], b[arm]
        if x.n_pcs != y.n_pcs or x.optimal_n_clusters != y.optimal_n_clusters or not bits(x.dendro.seqdist, y.dendro.seqdist):
            return False
        if sorted(x.cluster) != sorted(y.cluster) or not all(np.array_equal(x.cluster[k], y.cluster[k]) for k in y.cluster):
            return False
    return True


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--res", type=int, default=50000, help="bin size in bp")
    ap.add_argument("--scale", type=float, default=1.0, help="chromosome sizes x scale (rehearsals at a small size)")
    ap.add_argument("--steps", type=int, default=2, help="timed repetitions of each route (alternating A, B)")
    ap.add_argument("--streams", type=int, default=4)
    ap.add_argument("--seed", type=int, default=1)
    ap.add_argument("--out", default=None, help="also write the JSON line to this file")
    a = ap.parse_args()
    from tadpole_b200 import Context, GenomePixels, TADpole_genome, api
    from tadpole_b200.synth import synth_genome_pixels
    api.QUIET = True
    names = [nm for nm, _ in GRCH38]
    sizes = [max(2, int(round(-(-ln // a.res) * a.scale))) for _, ln in GRCH38]
    t = time.perf_counter()
    _, (b1, b2, v), _ = synth_genome_pixels(sizes, seed=a.seed, trans_per_chrom=1000, centromere=range(len(sizes)))
    gen_s = time.perf_counter() - t
    ctx = Context(0)
    px = GenomePixels(b1, b2, v, bins=list(zip(names, sizes)))
    TADpole_genome(px, ctx=ctx, streams=a.streams, centromere_search=True)         # warm-up: modules, pool contexts
    route_b(b1, b2, v, names, sizes, ctx)
    wa, wb, dev_ms = [], [], []
    for _ in range(a.steps):
        t = time.perf_counter()
        ra = TADpole_genome(px, ctx=ctx, streams=a.streams, centromere_search=True)
        wa.append(time.perf_counter() - t)
        dev_ms.append(ctx.last_batch_device_ms)
        t = time.perf_counter()
        rb, fb = route_b(b1, b2, v, names, sizes, ctx)
        wb.append(time.perf_counter() - t)
    ctx.close()
    identical = list(ra) == list(rb) and ra.failed == fb and all(same(ra[k], rb[k]) for k in rb)
    out = dict(card=card(), res_bp=a.res, scale=a.scale, chromosomes=len(sizes), bins=int(sum(sizes)),
               largest=int(max(sizes)), pixels=int(b1.size), split=len(ra), failed=sorted(ra.failed),
               generate_s=round(gen_s, 1), streams=a.streams, steps=a.steps, identical=bool(identical),
               A_wall_s=[round(x, 3) for x in wa], A_batch_device_ms=[round(x, 1) for x in dev_ms],
               B_wall_s=[round(x, 3) for x in wb])
    line = json.dumps(out)
    print(line)
    if a.out:
        with open(a.out, "w") as fh:
            fh.write(line + "\n")
    if not identical:
        sys.exit("the two routes differ")


if __name__ == "__main__":
    main()
