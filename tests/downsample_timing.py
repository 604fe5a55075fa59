"""What equal-depth subsampling costs on the GPU (run on the GPU): tp_genome_depth and tp_genome_downsample at N = T / 2 on
a GRCh38-sized sparse synthetic genome.

Input: the 24 GRCh38 chromosomes at --res bp, every cell within --band bins of the diagonal drawn by
synth_sparse_genome_pixels (about 5e8 cis reads at 10 kb with the defaults: the dense generators cannot reach that
depth).  Times are CUDA events on the context's stream around each library call, --steps repetitions after one warm-up;
the subsample of every repetition must equal the first one's pixels.  Philox evaluations = (select passes + 1) x T.
Prints one JSON line (also written to --out) with the card's name and power limit, read in the same run.

    python tests/downsample_timing.py [--res 10000] [--band 50] [--mean 32] [--steps 3] [--out result.json]
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

SELECT_PASSES = 6        # 64-bit keys, 12-bit digits (csrc/downsample.cu)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--res", type=int, default=10000, help="bin size in bp")
    ap.add_argument("--band", type=int, default=50, help="cells per row, from the diagonal on")
    ap.add_argument("--mean", type=float, default=32.0, help="mean count of a cell in the band")
    ap.add_argument("--steps", type=int, default=3)
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
    T = g.total_depth
    N = T // 2
    first = None
    depth_ms, down_ms = [], []
    for step in range(a.steps + 1):
        _, ms_d = timed(g.depth)
        sub, ms_s = timed(lambda: g.downsample(contacts=N, seed=a.seed))
        px = [sub.pixels(nm) for nm in sub.names[:3]]
        if first is None:
            first = px
        else:
            assert all(np.array_equal(x[k], y[k]) for x, y in zip(px, first) for k in range(3)), "subsample changed"
        assert sub.total_depth == N
        sub.close()
        if step:                                     # step 0 is the warm-up
            depth_ms.append(ms_d)
            down_ms.append(ms_s)
    g.close()
    ctx.close()
    res = dict(what="tp_genome_depth / tp_genome_downsample at N = T/2", card=card(), res_bp=a.res, band=a.band,
               pixels=int(v.size), cis_reads=int(T), contacts=int(N), steps=a.steps,
               depth_ms=[round(x, 3) for x in depth_ms], downsample_ms=[round(x, 3) for x in down_ms],
               philox_evaluations=(SELECT_PASSES + 1) * int(T),
               philox_per_s=round((SELECT_PASSES + 1) * T / (min(down_ms) / 1e3), 1), generate_s=round(gen_s, 2))
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
