"""Genome-wide TAD calling from one HiC-Pro pixel file, two routes on the same input (run on the GPU):

  A  TADpole_genome(GenomePixels(path=..., bins=...)): the text is parsed on the GPU, the pixels are split by chromosome
     there (tp_genome_ingest_file) and each chromosome's dense matrix exists only in HBM while its call runs.
  B  the route without it: read the pixel file on the host (pandas), split the pixels by chromosome, build one dense
     FP64 matrix per chromosome (1.5 GB of doubles at 50 kb) and call TADpole_batch on them.

Input: a seeded human-like genome at 50 kb (the 24 GRCh38 chromosomes, 61.8k bins, largest 4 980), synth_genome_pixels,
written as a HiC-Pro *.matrix (1-based ids, tab) with its *_abs.bed.  Both routes must give the same bits for every
chromosome.  Prints one JSON line (also written to --out when given): wall seconds of each route, the device ms of A's
ingest and of the calls, the card's name and power limit.

    python tests/genome_timing.py [--steps 2] [--streams 4] [--scale 1.0] [--out result.json]
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

# GRCh38 chromosome lengths (bp)
GRCH38 = [("chr1", 248956422), ("chr2", 242193529), ("chr3", 198295559), ("chr4", 190214555), ("chr5", 181538259),
          ("chr6", 170805979), ("chr7", 159345973), ("chr8", 145138636), ("chr9", 138394717), ("chr10", 133797422),
          ("chr11", 135086622), ("chr12", 133275309), ("chr13", 114364328), ("chr14", 107043718), ("chr15", 101991189),
          ("chr16", 90338345), ("chr17", 83257441), ("chr18", 80373285), ("chr19", 58617616), ("chr20", 64444167),
          ("chr21", 46709983), ("chr22", 50818468), ("chrX", 156040895), ("chrY", 57227415)]


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=60).stdout.strip().splitlines()
        return q[0] if q else "unknown"
    except Exception as e:              # the card's name is part of the number; say when it could not be read
        return f"unknown ({e})"


def write_input(d, res_bp, scale, seed):
    import pandas as pd
    from tadpole_b200.synth import synth_genome_pixels
    names = [nm for nm, _ in GRCH38]
    sizes = [max(2, int(round(-(-ln // res_bp) * scale))) for _, ln in GRCH38]
    _, (b1, b2, v), _ = synth_genome_pixels(sizes, seed=seed, trans_per_chrom=1000)
    mat = os.path.join(d, f"genome_{res_bp}.matrix")
    pd.DataFrame({"a": b1 + 1, "b": b2 + 1, "c": v.astype(np.int64)}).to_csv(mat, sep="\t", header=False, index=False)
    bed = os.path.join(d, f"genome_{res_bp}_abs.bed")
    rows = [(nm, i) for nm, n in zip(names, sizes) for i in range(n)]
    pd.DataFrame({"chrom": [r[0] for r in rows], "start": [r[1] * res_bp for r in rows],
                  "end": [(r[1] + 1) * res_bp for r in rows], "id": np.arange(1, len(rows) + 1)}).to_csv(
        bed, sep="\t", header=False, index=False)
    return mat, bed, names, sizes, int(b1.size), os.path.getsize(mat)


def route_b(mat, names, sizes, ctx, streams):
    """The pixel file read on the host, split by chromosome, one dense matrix per chromosome, then TADpole_batch."""
    import pandas as pd
    from tadpole_b200 import TADpole_batch
    t0 = time.perf_counter()
    px = pd.read_csv(mat, sep="\t", header=None, names=["a", "b", "c"], dtype={"a": np.int64, "b": np.int64, "c": np.float64})
    x, y, v = px["a"].to_numpy() - 1, px["b"].to_numpy() - 1, px["c"].to_numpy()
    t1 = time.perf_counter()
    starts = np.concatenate(([0], np.cumsum(sizes)))
    cx, cy = np.searchsorted(starts, x, "right") - 1, np.searchsorted(starts, y, "right") - 1
    keep = (cx == cy) & (x <= y)
    x, y, v, cx = x[keep], y[keep], v[keep], cx[keep]
    mats = []
    for c, n in enumerate(sizes):
        s = cx == c
        lin = (x[s] - starts[c]) * n + (y[s] - starts[c])
        mats.append(np.bincount(lin, weights=v[s], minlength=n * n).reshape(n, n))
    t2 = time.perf_counter()
    tps = TADpole_batch(mats, ctx=ctx, streams=streams)
    t3 = time.perf_counter()
    return dict(zip(names, tps)), dict(read_s=t1 - t0, split_dense_s=t2 - t1, batch_s=t3 - t2,
                                       batch_device_ms=ctx.last_batch_device_ms, host_dense_gb=sum(n * n for n in sizes) * 8 / 1e9)


def same(a, b):
    ok = a.n_pcs == b.n_pcs and a.optimal_n_clusters == b.optimal_n_clusters
    ok = ok and np.array_equal(a.dendro.seqdist.view(np.uint64), b.dendro.seqdist.view(np.uint64))
    sa, sb = np.asarray(a.scores), np.asarray(b.scores)
    ok = ok and sa.shape == sb.shape and np.array_equal(np.isnan(sa), np.isnan(sb)) and np.array_equal(sa[~np.isnan(sa)], sb[~np.isnan(sb)])
    return ok and sorted(a.clusters) == sorted(b.clusters) and all(np.array_equal(a.clusters[k], b.clusters[k]) for k in b.clusters)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=2, help="timed repetitions of each route (alternating A, B)")
    ap.add_argument("--streams", type=int, default=4)
    ap.add_argument("--scale", type=float, default=1.0, help="chromosome sizes x scale (rehearsals at a small size)")
    ap.add_argument("--seed", type=int, default=1)
    ap.add_argument("--out", default=None, help="also write the JSON line to this file")
    a = ap.parse_args()
    from tadpole_b200 import Context, GenomePixels, TADpole_genome, api
    api.QUIET = True
    with tempfile.TemporaryDirectory() as d:
        t = time.perf_counter()
        mat, bed, names, sizes, nnz, nbytes = write_input(d, 50000, a.scale, a.seed)
        gen_s = time.perf_counter() - t
        ctx = Context(0)
        px = GenomePixels(path=mat, bins=bed)
        assert px.names == names and px.chrom_bins.tolist() == sizes
        TADpole_genome(px, ctx=ctx, streams=a.streams)             # warm-up: module loads, pool contexts, buffers
        route_b(mat, names, sizes, ctx, a.streams)
        wa, wb, ingest_ms, parse_ms, calls_ms, parts = [], [], [], [], [], []
        for _ in range(a.steps):
            t = time.perf_counter()
            ra = TADpole_genome(px, ctx=ctx, streams=a.streams)
            wa.append(time.perf_counter() - t)
            st = ctx.ingest_stats()
            ingest_ms.append(st["wall_ms"])
            parse_ms.append(st["parse_ms"])
            calls_ms.append(ctx.last_batch_device_ms)
            t = time.perf_counter()
            rb, pb = route_b(mat, names, sizes, ctx, a.streams)
            wb.append(time.perf_counter() - t)
            parts.append(pb)
        ctx.close()
    identical = list(ra) == list(rb) and not ra.failed and all(same(ra[k], rb[k]) for k in rb)
    out = dict(card=card(), chromosomes=len(sizes), bins=int(sum(sizes)), largest=int(max(sizes)), pixels=nnz,
               text_bytes=nbytes, generate_s=round(gen_s, 1), streams=a.streams, steps=a.steps, identical=bool(identical),
               A_wall_s=[round(x, 3) for x in wa], A_ingest_wall_ms=[round(x, 1) for x in ingest_ms],
               A_ingest_device_ms=[round(x, 1) for x in parse_ms], A_calls_device_ms=[round(x, 1) for x in calls_ms],
               B_wall_s=[round(x, 3) for x in wb], B_parts=[{k: round(v, 3) for k, v in p.items()} for p in parts])
    line = json.dumps(out)
    print(line)
    if a.out:
        with open(a.out, "w") as fh:
            fh.write(line + "\n")
    if not identical:
        sys.exit("the two routes differ")


if __name__ == "__main__":
    main()
