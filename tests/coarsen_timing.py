"""What coarsening costs on the GPU (run on the GPU): tp_genome_coarsen at factors 2, 5 and 10 on a GRCh38-sized sparse
synthetic genome.

Input: the 24 GRCh38 chromosomes at --res bp, every cell within --band bins of the diagonal drawn by
synth_sparse_genome_pixels, in chromosome then row order as HiC-Pro and cooler write them, routed into the buckets by
the genome ingest.  Times are CUDA events on the context's stream around each library call (the call ends in a stream
synchronise), --steps repetitions of each factor after one warm-up; every result must equal the first one's pixels.
Compulsory traffic per call: 16 B read per bucket entry, the table cleared and walked twice (3 x 16 B per slot) and 16 B
written per output cell; the table atomics are not counted.  Prints one JSON line (also written to --out) with the
card's name and power limit, read in the same run.

    python tests/coarsen_timing.py [--res 10000] [--band 50] [--steps 5] [--out result.json]
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


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--res", type=int, default=10000, help="bin size in bp")
    ap.add_argument("--band", type=int, default=50, help="cells per row, from the diagonal on")
    ap.add_argument("--mean", type=float, default=32.0, help="mean count of a cell in the band")
    ap.add_argument("--factors", default="2,5,10")
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--seed", type=int, default=1)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    from tadpole_b200 import Context, GenomePixels
    from tadpole_b200.synth import synth_sparse_genome_pixels
    sizes = [-(-ln // a.res) for _, ln in GRCH38]
    t = time.perf_counter()
    b1, b2, v = synth_sparse_genome_pixels(sizes, band=a.band, mean_count=a.mean, seed=a.seed)
    gen_s = time.perf_counter() - t
    ctx = Context(0)
    stream = torch.cuda.ExternalStream(ctx.stream, device=torch.device("cuda", 0))

    def timed(fn):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        out = fn()
        e1.record(stream)
        e1.synchronize()
        return out, e0.elapsed_time(e1)

    g = GenomePixels(b1, b2, v, bins=list(zip([nm for nm, _ in GRCH38], sizes))).load(ctx=ctx)
    ncis = int(g.stats()[0].sum())
    cap = 1024
    while cap < 2 * ncis:
        cap *= 2
    rows = []
    for f in (int(x) for x in a.factors.split(",")):
        ms = []
        first, nout = None, None
        for step in range(a.steps + 1):
            cg, t_ms = timed(lambda: g.coarsen(f))
            px = [cg.pixels(nm) for nm in cg.names[:3]]
            if first is None:
                first, nout = px, int(cg.stats()[0].sum())
            else:
                assert all(np.array_equal(x[k], y[k]) for x, y in zip(px, first) for k in range(3)), "result changed"
            cg.close()
            if step:                                     # step 0 is the warm-up
                ms.append(t_ms)
        traffic = 16 * ncis + 3 * 16 * cap + 16 * nout
        rows.append(dict(factor=f, pixels_in=ncis, pixels_out=nout, table_slots=cap, compulsory_bytes=traffic,
                         coarsen_ms=[round(x, 3) for x in ms], gb_s=round(traffic / (min(ms) / 1e3) / 1e9, 1)))
    g.close()
    ctx.close()
    res = dict(what="tp_genome_coarsen", card=card(), res_bp=a.res, band=a.band,
               steps=a.steps, factors=rows, generate_s=round(gen_s, 2))
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
