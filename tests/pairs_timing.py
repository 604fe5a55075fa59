"""What loading read pairs costs on the GPU (run on the GPU): GenomePairs(...).load() at --res bp on a seeded GRCh38-sized
4DN pairs file of several GB, against the raw read of the same file and a host route.

Input: write_pairs (tests/pairs_oracle.py) over the 24 GRCh38 chromosomes, --pairs cis pairs (distance decaying like 1/d)
plus 7.5 % trans and 1.5 % unplaced pairs, about 82 bytes per line, in a temporary directory.  Measured in one run, in
this order, on the file as the page cache holds it after the write:
  * raw read: the file read into one 64 MB buffer after another (readinto), no parsing;
  * GPU load: GenomePairs(...).load() wall time (--steps times after one warm-up), with the library's device time of the
    per-window line-end and parse kernels and its window count (tp_ingest_stats), so device ms per window stands
    against the raw read ms of a window's bytes; peak device memory as the lowest free memory sampled (1 ms) during a
    load, against the free memory before it;
  * host route: pandas + numpy binning (bin_pairs_np) and GenomePixels(...).load() of its cells, whose pixels must be the
    GPU load's bits.
Prints one JSON line (also written to --out) with the card's name and power limit, read in the same run.

    python tests/pairs_timing.py [--pairs 40000000] [--res 10000] [--steps 2] [--out result.json]
"""
import argparse
import json
import os
import shutil
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

from genome_timing import GRCH38, card  # noqa: E402
import pairs_oracle as P  # noqa: E402


def raw_read(path, chunk=64 << 20):
    buf = bytearray(chunk)
    t = time.perf_counter()
    with open(path, "rb", buffering=0) as fh:
        while fh.readinto(buf):
            pass
    return time.perf_counter() - t


class FreeMemory:
    """the lowest free device memory seen while the block runs (sampled every millisecond)"""

    def __init__(self, torch):
        self.torch, self.low, self.stop = torch, None, False

    def __enter__(self):
        self.before = self.low = self.torch.cuda.mem_get_info(0)[0]
        self.th = threading.Thread(target=self._run, daemon=True)
        self.th.start()
        return self

    def _run(self):
        while not self.stop:
            self.low = min(self.low, self.torch.cuda.mem_get_info(0)[0])
            time.sleep(0.001)

    def __exit__(self, *exc):
        self.stop = True
        self.th.join()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--pairs", type=int, default=40_000_000, help="cis pairs")
    ap.add_argument("--res", type=int, default=10000, help="bin size in bp")
    ap.add_argument("--steps", type=int, default=2)
    ap.add_argument("--seed", type=int, default=1)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    from tadpole_b200 import Context, GenomePairs, GenomePixels
    d = tempfile.mkdtemp(prefix="pairs_timing_")
    try:
        path = os.path.join(d, "grch38.pairs")
        t = time.perf_counter()
        P.write_pairs(path, "4dn", GRCH38, a.pairs, int(a.pairs * 0.075), int(a.pairs * 0.015), seed=a.seed)
        write_s = time.perf_counter() - t
        size = os.path.getsize(path)
        read_s = [raw_read(path) for _ in range(2)]
        ctx = Context(0)
        gp = GenomePairs(path, binsize=a.res)
        loads = []
        for step in range(a.steps + 1):
            with FreeMemory(torch) as mem:
                t = time.perf_counter()
                g = gp.load(ctx=ctx)
                wall = time.perf_counter() - t
            st = ctx.ingest_stats()
            loads.append(dict(wall_s=round(wall, 3), device_ms=round(float(st["parse_ms"]), 1),
                              windows=int(st["host_fields"]), peak_device_bytes=int(mem.before - mem.low)))
            if step < a.steps:
                g.close()
        loads = loads[1:]                                   # the first load is the warm-up
        counts = g.pair_counts
        gpu_px = [g.pixels(nm) for nm in g.names]
        t = time.perf_counter()
        want, hcounts = P.bin_pairs_np([path], GRCH38, a.res)
        bin_s = time.perf_counter() - t
        nb = P.n_bins(GRCH38, a.res)
        starts = np.concatenate(([0], np.cumsum(nb)))
        t = time.perf_counter()
        h = GenomePixels(np.concatenate([i + starts[c] for c, (i, _, _) in enumerate(want)]).astype(np.int32),
                         np.concatenate([j + starts[c] for c, (_, j, _) in enumerate(want)]).astype(np.int32),
                         np.concatenate([x for _, _, x in want]),
                         bins=[(nm, n) for (nm, _), n in zip(GRCH38, nb)]).load(ctx=ctx)
        host_load_s = time.perf_counter() - t
        host_px = [h.pixels(nm) for nm in h.names]
        same = hcounts == counts and all(np.array_equal(x[k], y[k]) for x, y in zip(gpu_px, host_px) for k in range(2)) \
            and all(np.array_equal(x[2].view(np.uint64), y[2].view(np.uint64)) for x, y in zip(gpu_px, host_px))
        assert same, "the GPU load and the host route differ"
        cells = int(sum(x[0].size for x in gpu_px))
        g.close()
        h.close()
        ctx.close()
        best = min(loads, key=lambda r: r["wall_s"])
        win = best["windows"]
        res = dict(what="GenomePairs.load", card=card(), res_bp=a.res, file_bytes=size, pair_lines=counts["lines"],
                   counts=counts, cells=cells, write_s=round(write_s, 1), raw_read_s=[round(x, 3) for x in read_s],
                   raw_read_gb_s=round(size / min(read_s) / 1e9, 2), loads=loads,
                   load_gb_s=round(size / best["wall_s"] / 1e9, 2),
                   device_ms_per_window=round(best["device_ms"] / win, 2),
                   raw_read_ms_per_window=round(min(read_s) * 1e3 / win, 2),
                   host_route=dict(pandas_numpy_bin_s=round(bin_s, 2), pixels_load_s=round(host_load_s, 2),
                                   total_s=round(bin_s + host_load_s, 2)),
                   same_bits=bool(same))
        line = json.dumps(res)
        print(line)
        if a.out:
            os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
            with open(a.out, "w") as fh:
                fh.write(line + "\n")
    finally:
        shutil.rmtree(d, ignore_errors=True)


if __name__ == "__main__":
    main()
