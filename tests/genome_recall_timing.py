"""What the resident genome handle saves (run on the GPU): TADpole_genome(resident=True) once, then GenomeResult.recall
with another min_clusters and with fewer PCs, against the whole genome call.

Input: a seeded human-like genome (the 24 GRCh38 chromosomes at --res bp, synth_genome_pixels).  Each recall is checked
bit for bit against its reference: min_clusters = 3 against TADpole_genome(min_clusters=3); max_pcs = 50 against the
first chromosome's TADpole() followed by recall().  Prints one JSON line (also written to --out): wall seconds and
tp_batch_device_ms of the genome call and of each recall, the resident bytes, the card's name and power limit.

    python tests/genome_recall_timing.py [--res 50000] [--steps 2] [--streams 4] [--scale 1.0] [--out result.json]
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

from genome_timing import GRCH38, card, same  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--res", type=int, default=50000, help="bin size in bp")
    ap.add_argument("--steps", type=int, default=2, help="timed repetitions (genome call, recall, recall)")
    ap.add_argument("--streams", type=int, default=4)
    ap.add_argument("--scale", type=float, default=1.0, help="chromosome sizes x scale (rehearsals at a small size)")
    ap.add_argument("--seed", type=int, default=1)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    from tadpole_b200 import Context, GenomePixels, TADpole, TADpole_genome, api
    from tadpole_b200.synth import synth_genome_pixels
    api.QUIET = True
    names = [nm for nm, _ in GRCH38]
    sizes = [max(2, int(round(-(-ln // a.res) * a.scale))) for _, ln in GRCH38]
    t = time.perf_counter()
    _, (b1, b2, v), _ = synth_genome_pixels(sizes, seed=a.seed, trans_per_chrom=1000)
    gen_s = time.perf_counter() - t
    px = GenomePixels(b1, b2, v, bins=list(zip(names, sizes)))
    ctx = Context(0)

    def timed(fn):
        ctx.sync()
        t0 = time.perf_counter()
        r = fn()
        return r, time.perf_counter() - t0, ctx.last_batch_device_ms

    res = TADpole_genome(px, ctx=ctx, streams=a.streams, resident=True)           # warm-up of every shape
    res.recall(min_clusters=3, streams=a.streams)
    res.recall(max_pcs=50, streams=a.streams)
    rows = []
    for _ in range(a.steps):
        del res
        res, w0, d0 = timed(lambda: TADpole_genome(px, ctx=ctx, streams=a.streams, resident=True))
        r3, w1, d1 = timed(lambda: res.recall(min_clusters=3, streams=a.streams))
        r50, w2, d2 = timed(lambda: res.recall(max_pcs=50, streams=a.streams))
        rows.append(dict(genome_s=w0, genome_device_ms=d0, recall_min_clusters3_s=w1, recall_min_clusters3_device_ms=d1,
                         recall_max_pcs50_s=w2, recall_max_pcs50_device_ms=d2))
    store = next(iter(res.values()))._resident()["batch"]
    # the results the timed calls gave
    fresh3 = TADpole_genome(px, ctx=ctx, streams=a.streams, min_clusters=3)
    ok3 = list(fresh3) == list(r3) and all(same(r3[nm], fresh3[nm]) for nm in fresh3)
    first = names[int(np.argmin(sizes))] if a.scale < 1 else "chr21"
    g = px._ingest(ctx)
    try:
        m = g.matrix(names.index(first))
    finally:
        g.close()
    ok50 = same(r50[first], TADpole(m, ctx=ctx).recall(max_pcs=50))
    # a fresh call with max_pcs = 50 runs its PCA with a narrower block: how many chromosomes still give the same bits
    fresh50 = TADpole_genome(px, ctx=ctx, streams=a.streams, max_pcs=50)
    eq50 = sum(bool(same(r50[nm], fresh50[nm])) for nm in fresh50 if nm in r50)
    line = dict(what="genome_recall_timing", card=card(), res_bp=a.res, scale=a.scale, chromosomes=len(sizes),
                bins=int(sum(sizes)), largest=int(max(sizes)), pixels=int(b1.size), generate_s=gen_s, streams=a.streams,
                resident_bytes=store.nbytes(), failed=sorted(res.failed), steps=rows,
                bit_identical=dict(min_clusters3_vs_genome_call=bool(ok3), max_pcs50_vs_tadpole_recall=bool(ok50),
                                   chromosome_checked=first),
                max_pcs50_chromosomes_equal_to_fresh_max_pcs50_call=f"{eq50} of {len(fresh50)}")
    text = json.dumps(line)
    print(text)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as fh:
            fh.write(text + "\n")


if __name__ == "__main__":
    main()
