#!/usr/bin/env python
"""bench.py -- TADpole calls/sec on synthetic Hi-C matrices (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path
    python bench.py --impl reference --gpus N --steps K ...  # CPU restatement of the reference
    python bench.py ... --dump-outputs DIR                   # also write the last timed step's results as DIR/*.npy

Workload: BASELINE.json configs[1], synthetic 2,000-bin Hi-C matrices with nested block TADs and power-law decay,
max_pcs = 200.  One TADpole() call = bad-column filter, Pearson correlation, PCA to 200 components, the n_pcs sweep
(CONISS per candidate), broken stick + Calinski-Harabasz, selection.  A "step" is one pass of the hot path over one
BATCH of --batch (16) different matrices -- genome-wide use is one call per chromosome, and a lone 2000-bin call leaves
most of a B200 idle -- handed to the library in one tp_call_batch, which keeps --streams calls in flight with its own
host threads (one Python / R thread just waits).  With N > 1 every rank runs its own batches (no data-path
collective): weak scaling.

value  : calls/s with the input matrices already resident in HBM (device pointers through the C ABI), CUDA events on
         the library's streams (tp_batch_device_ms), max over ranks.
e2e    : the same through the public API TADpole_batch(matrices) with the matrices in pinned HOST memory: H2D copy,
         D2H of the results, per-level tables and object assembly inside the timed (wall clock) region.
single_call : one call at a time (latency); the per-kernel rooflines are taken from that pass (CUDA events around
         every launch of a class).
strong_scaling : ONE chromosome-wide call (BASELINE configs[3], 25,000 bins) spread over all N ranks -- row blocks of
         the symmetric products and of every operator application by their owner + NCCL all-gather, candidates of the
         sweep rank-interleaved -- and the 15,000-bin centromere_search call with the arms on disjoint halves of the ranks
         (configs[2]); at N > 1 rank 0 repeats the call alone and the results must be identical bit for bit.
The step's inputs (16 x 32 MB) are larger than L2, so no step re-reads a warm input.

The reference is a pure-R package and R is not installed here or on the GPU box (probed: `Rscript`), so
`--impl reference` and `cpu_baseline` time oracle/ (numpy + C restatement in the reference's algorithmic shape: full
LAPACK SVD, per-candidate O(N^2) dist + Lance-Williams CONISS, per-level Calinski-Harabasz) on all host cores, every
one of the 200 candidates in full; a reference step is a bounded sample of the GPU arm's step: ONE of the batch's calls.
"""
from __future__ import annotations

import argparse
import json
import os
import shutil
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

N_BINS = 2000
MAX_PCS = 200
METRIC = "tadpole_calls_per_sec"
UNIT = "calls/s"


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--batch", type=int, default=0, help="calls per step (one tp_call_batch of that many different matrices); "
                                                         "0 = twice the calls in flight")
    ap.add_argument("--streams", type=int, default=16, help="calls kept in flight per GPU by the library's own threads "
                                                            "(fewer when the box has under a quarter of a CPU per thread)")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--bins", type=int, default=N_BINS)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--large-n", type=int, default=8000,
                    help="bins of one extra profiled call whose tensor-kernel rooflines are reported beside the workload's "
                         "(N = 1 only; 0 = skip)")
    ap.add_argument("--strong-bins", type=int, default=25000, help="bins of the one call spread over all ranks (0 = skip)")
    ap.add_argument("--arm-bins", type=int, default=15000, help="bins of the centromere_search call, arms sharded (0 = skip)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the timed batch returned in its last step to "
                                                          "DIR/<name>.npy (see dump_outputs)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs needs --impl b200")
    return args


def usable_cpus():
    """CPUs this process may run on (a container's share, not the host's count)."""
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except (AttributeError, OSError):
        return os.cpu_count() or 1


def workload_text(bins):
    return (f"synthetic {bins}-bin Hi-C matrix, nested block TADs, power-law decay, max_pcs=200 "
            "(BASELINE.json configs[1]); one TADpole() call per matrix")


def r_probe():
    """SURVEY 8(c): if Rscript with rioja + fpc ever appears, the real reference supersedes the restatement."""
    rs = shutil.which("Rscript")
    if not rs:
        return {"Rscript": None, "note": "R is not installed: CPU arm = oracle/ port"}
    try:
        ok = subprocess.run([rs, "-e", "stopifnot(requireNamespace('rioja'), requireNamespace('fpc'))"],
                            capture_output=True, timeout=60).returncode == 0
    except Exception:
        ok = False
    return {"Rscript": rs, "rioja_fpc": ok,
            "note": "R found: run tests/golden/make_r_golden.R to pin the oracle to the real reference" if ok
                    else "R found but rioja / fpc are missing"}


# ---------------------------------------------------------------------------------------------
# CPU arm: the oracle, timed (the only place besides tests/ and smoke() that touches oracle/)
# ---------------------------------------------------------------------------------------------
def cpu_full_call(mat, threads):
    """One FULL call of the reference-shaped CPU path: every one of the 200 candidates, all host cores."""
    from oracle import tadpole_oracle as O
    t0 = time.perf_counter()
    n_pcs, n_cl, _, st = O.tadpole_cpu_full(mat, max_pcs=MAX_PCS, threads=threads)
    return time.perf_counter() - t0, dict(front_s=round(st["front_s"], 3), sweep_s=round(st["sweep_s"], 3), k=st["k"],
                                          n_pcs=int(n_pcs), n_clusters=int(n_cl))


def cpu_sample_text(detail, threads):
    return (f"one full call per step (1 of the GPU arm's batch): filter + correlation + full LAPACK SVD ({detail['front_s']} s) "
            f"and ALL {detail['k']} candidates (dist + Lance-Williams CONISS + broken stick + per-level CH, plain C, "
            f"{detail['sweep_s']} s) on {threads} threads; nothing extrapolated")


def run_reference(args, rank, world):
    if rank != 0:
        return
    from tadpole_b200.synth import synth_hic
    threads = usable_cpus()
    mats = [synth_hic(args.bins, seed=1 + s) for s in range(min(4, max(1, args.steps)))]
    if args.warmup > 0:          # ONE untimed call whatever W is: page-in and thread start-up are all this path has to warm,
        cpu_full_call(mats[0], threads)      # and every further warm-up call would cost as much as a timed step
    secs, detail = [], None
    t0 = time.perf_counter()
    for s in range(args.steps):
        sec, detail = cpu_full_call(mats[s % len(mats)], threads)
        secs.append(sec)
    wall = time.perf_counter() - t0
    sec = wall / args.steps
    val = 1.0 / sec
    line = {
        "impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": sec * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": workload_text(args.bins), "bins": args.bins, "max_pcs": MAX_PCS,
                   "calls_per_step": 1,
                   "note": "reference is pure R and R is not installed: CPU restatement (oracle/) in the reference's "
                           "algorithmic shape, every step one full call, runs on rank 0 only"},
        "cpu_baseline": {"value": val, "unit": UNIT, "cores": threads, "kind": "port", "sample": cpu_sample_text(detail, threads)},
        "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0, "r_probe": r_probe(),
    }
    print(json.dumps(line), flush=True)


# ---------------------------------------------------------------------------------------------
# GPU arm
# ---------------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, device):
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        try:
            self.p = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                       "-i", str(device), "-lms", "100"], stdout=self.f, stderr=subprocess.DEVNULL)
        except OSError:
            self.p = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": []}
        if self.p is None:
            return out
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.flush()
        self.f.seek(0)
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in self.f:
            f = [x.strip() for x in line.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for nm, v in zip(names, f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        self.f.close()
        try:
            os.unlink(self.f.name)
        except OSError:
            pass
        if sm:
            out = {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(mx)), "reasons": sorted(reasons),
                   "samples": len(sm)}
        return out


def h2d_bytes(n):
    """bytes tp_filter copies to the device for a row-major n x n host matrix: band copies of the upper triangle
    (csrc/filter.cu): rows [r, r + band) x columns [r, n)"""
    band = max(n // 32, 64)
    return sum((n - r) * 8 * min(band, n - r) for r in range(0, n, band))


DUMP_LIMIT = 64 << 20


def dump_outputs(out_dir, results, prefix=""):
    """Write the per-call results of one step as a caller of tp_call_batch receives them, so that two builds can be
    compared output for output: <prefix>callNN_scores.npy (CH score matrix) with <prefix>callNN_scored.npy (1 where a
    level is scored; the library's NaN marks the others, written as 0 so that every dumped value is finite),
    <prefix>callNN_seqdist.npy (CONISS heights of the chosen candidate), <prefix>callNN_bad.npy (bad-bin mask as 0 / 1)
    and <prefix>counts.npy (one row per call: nf, k, n_pcs, n_clusters), all float64.  Calls are written in batch order
    while the total stays within DUMP_LIMIT bytes; at sizes where it would not, the first calls of the step stand for it."""
    os.makedirs(out_dir, exist_ok=True)
    total, counts = 0, []
    for i, r in enumerate(results):
        if isinstance(r, Exception):
            raise r
        unscored = np.isnan(r["scores"])
        arrays = {"scores": np.where(unscored, 0.0, r["scores"]), "scored": ~unscored, "seqdist": r["seqdist"], "bad": r["bad"]}
        size = sum(a.size * 8 for a in arrays.values()) + 4 * 8
        if total + size > DUMP_LIMIT:
            break
        for name, a in arrays.items():
            np.save(os.path.join(out_dir, f"{prefix}call{i:02d}_{name}.npy"), np.asarray(a, dtype=np.float64))
        counts.append([r["nf"], r["k"], r["n_pcs"], r["n_clusters"]])
        total += size
    np.save(os.path.join(out_dir, f"{prefix}counts.npy"), np.array(counts, dtype=np.float64).reshape(-1, 4))


def measure_fp64_peak(torch):
    """cuBLAS DGEMM TFLOP/s on this box (library GEMM used only as the roofline denominator)."""
    a = torch.randn(4096, 4096, dtype=torch.float64, device="cuda")
    b = torch.randn(4096, 4096, dtype=torch.float64, device="cuda")
    best = 0.0
    for _ in range(6):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); torch.matmul(a, b); e1.record(); torch.cuda.synchronize()
        best = max(best, 2 * 4096 ** 3 / (e0.elapsed_time(e1) * 1e-3) / 1e12)
    return best


def measure_int8_peak(torch):
    """Library int8 GEMM (torch._int_mm -> cuBLASLt, int32 accumulation) 8192^3, best of 10, TOP/s (2 per multiply-add):
    the measured denominator of the tcgen05 kind::i8 kernels.  None when the library call is unavailable."""
    try:
        a = torch.randint(-127, 127, (8192, 8192), dtype=torch.int8, device="cuda")
        b = torch.randint(-127, 127, (8192, 8192), dtype=torch.int8, device="cuda")
        torch._int_mm(a, b)
        best = 0.0
        for _ in range(10):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(); torch._int_mm(a, b); e1.record(); torch.cuda.synchronize()
            best = max(best, 2 * 8192 ** 3 / (e0.elapsed_time(e1) * 1e-3) / 1e12)
        return best
    except Exception:
        return None


def strong_scaling(args, torch, dist, rank, world, local_rank, Context, sharding, api):
    """One chromosome-wide call over all ranks (configs[3]) and the arm-sharded centromere call (configs[2])."""
    from tadpole_b200 import TADpole
    from tadpole_b200.synth import synth_hic_gpu
    out = {}
    ctx = Context(local_rank)
    env = sharding.DistEnv(ctx) if world > 1 else None

    def sync_all():
        ctx.sync(); torch.cuda.synchronize()
        if world > 1:
            dist.barrier()

    for key, bins, cen in (("chr", args.strong_bins, False), ("arms", args.arm_bins, True)):
        if bins <= 0:
            continue
        dev = synth_hic_gpu(bins, seed=7 if cen else 3, device=local_rank, centromere=cen)
        if world > 1:
            sums = env.exchange(float(dev.sum()))
            assert all(v == sums[0] for v in sums), "ranks drew different matrices"
        host = dev.cpu().numpy()                                   # pageable host memory, as an R matrix is
        del dev
        torch.cuda.empty_cache()
        walls, tp = [], None
        for rep in range(3):                                       # first call allocates; the last two are timed
            sync_all()
            t0 = time.perf_counter()
            tp = TADpole(host, max_pcs=MAX_PCS, centromere_search=cen, ctx=ctx, dist=env)
            sync_all()
            walls.append((time.perf_counter() - t0) * 1e3)
        stages = ctx.timings()
        ctx.profile(1)
        TADpole(host, max_pcs=MAX_PCS, centromere_search=cen, ctx=ctx, dist=env)
        prof = ctx.profile(0)
        t = torch.tensor([min(walls[1:]), stages["total_ms"]] + [stages[k] for k in ("filter_ms", "compact_ms", "correlation_ms", "pca_ms", "sweep_ms", "ch_ms")],
                         dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        t = [float(v) for v in t]
        r = {"bins": bins, "centromere_search": cen, "ranks": world,
             "wall_ms": round(t[0], 2), "device_total_ms": round(t[1], 2),
             "stages_ms": dict(zip(("filter", "compact", "correlation", "pca", "sweep", "ch"), (round(v, 2) for v in t[2:]))),
             "stages_sum_ms": round(sum(t[2:]), 2),
             "comm_ms": round(prof["comm"][0], 2), "islice_ms": round(prof["islice"][0], 2),
             "igemm_ms": round(prof["igemm"][0], 2), "sweep_kernel_ms": round(prof["coniss_sweep"][0], 2),
             "pca_applications": int(stages["pca_applications"]), "pca_iterations": int(stages["pca_iterations"]),
             "timing": "max over ranks; wall = host matrix (pageable) in, tadpole object out, best of 2 after one warm call; "
                       "stages = CUDA events on the library stream; comm / islice / igemm / sweep = rank 0 CUDA events around "
                       "every launch of the class in one extra profiled call"}
        if cen:
            r["result"] = {"p": [tp.p.n_pcs, tp.p.optimal_n_clusters], "q": [tp.q.n_pcs, tp.q.optimal_n_clusters],
                           "tads": int(tp.merging_arms.shape[0])}
            summ = tp.merging_arms.tobytes() + tp.p.dendro.seqdist.tobytes() + tp.q.dendro.seqdist.tobytes()
        else:
            r["result"] = {"n_pcs": tp.n_pcs, "optimal_n_clusters": tp.optimal_n_clusters, "levels": len(tp.clusters)}
            summ = tp.scores.tobytes() + tp.dendro.seqdist.tobytes()
        big = max(("comm", "islice", "sweep"), key=lambda k_: {"comm": r["comm_ms"], "islice": r["islice_ms"], "sweep": r["stages_ms"]["sweep"]}[k_])
        r["largest_non_gemm_cost"] = big
        if world > 1:
            every = env.exchange(summ)
            r["all_ranks_identical"] = all(e == every[0] for e in every)
            if rank == 0:                                           # the same call on this GPU alone
                ctx.comm_select(-1)
                ref = TADpole(host, max_pcs=MAX_PCS, centromere_search=cen, ctx=ctx)
                ctx.comm_select(env.world_slot)
                if cen:
                    same = (np.array_equal(ref.merging_arms, tp.merging_arms) and all(
                        np.array_equal(ref[a].dendro.seqdist, tp[a].dendro.seqdist) and ref[a].n_pcs == tp[a].n_pcs for a in "pq"))
                else:
                    same = (ref.n_pcs == tp.n_pcs and ref.optimal_n_clusters == tp.optimal_n_clusters
                            and np.array_equal(ref.dendro.seqdist, tp.dendro.seqdist)
                            and np.array_equal(ref.scores, tp.scores, equal_nan=True))
                r["identical_to_1gpu"] = bool(same)
                r["one_gpu_stages_sum_ms"] = round(sum(ctx.timings()[k] for k in ("filter_ms", "compact_ms", "correlation_ms", "pca_ms", "sweep_ms", "ch_ms")), 2)
            dist.barrier()
        out[key] = r
        del host, tp
    ctx.close()
    return out


def run_b200(args, rank, world, local_rank):
    import torch
    import torch.distributed as dist
    from tadpole_b200 import Context, TADpole_batch, api, sharding
    from tadpole_b200.synth import synth_hic

    api.QUIET = True
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    # every call in flight has a library-owned host thread (asleep on an event most of the time): keep at most 4 per CPU
    S = max(1, min(args.streams, max(8, 4 * usable_cpus() // max(world, 1))))
    B, n = (args.batch if args.batch > 0 else 2 * S), args.bins
    ctx = Context(local_rank)
    # the library's batch threads wait for their streams most of the time; a spinning wait (the CUDA default) needs a core
    # each, so with several ranks on one host they sleep on blocking-sync events instead (tp_call_batch decides this for
    # the threads of ONE process; it cannot see the other ranks)
    ncpu = usable_cpus()
    sync_blocking = world * S > ncpu // 2          # applied to the batch passes only; a single call at a time spins

    # synthetic inputs: B different matrices per rank; pinned host copies for e2e, device copies for value
    host = []
    for s in range(B):
        m = synth_hic(n, seed=1000 * rank + 1 + s)
        t = torch.empty((n, n), dtype=torch.float64, pin_memory=True)
        t.numpy()[:] = m
        host.append(t)
    dev = [t.cuda(non_blocking=False) for t in host]
    torch.cuda.synchronize()
    ptrs = [d.data_ptr() for d in dev]
    host_np = [t.numpy() for t in host]

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- warm-up: the pool's contexts allocate their buffers -----------------------------------------
    for _ in range(max(args.warmup, 3)):
        ctx.call_batch(None, device_ptrs=ptrs, n=n, inflight=S, tables=False, max_pcs=MAX_PCS)
    # ---- single call at a time: latency, per-kernel device times (CUDA events around each launch) ----
    lat_steps = 20
    for i in range(3):
        ctx.call(device_ptr=ptrs[i % B], n=n, colmajor=0, max_pcs=MAX_PCS)
    lstream = torch.cuda.ExternalStream(ctx.stream, device=torch.device("cuda", local_rank))
    clocks = ClockSampler(local_rank) if rank == 0 else None
    barrier()
    ctx.profile(1)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(lstream)
    for i in range(lat_steps):
        res = ctx.call(device_ptr=ptrs[i % B], n=n, colmajor=0, max_pcs=MAX_PCS)
    e1.record(lstream)
    ctx.sync()
    ms_single = e0.elapsed_time(e1)
    prof = ctx.profile(0)
    stage = ctx.timings()
    # ---- value: K steps of B device-resident calls, S in flight ------------------------------------
    if sync_blocking:
        ctx.set("sync_blocking", 1)
    barrier()
    last_step = ctx.call_batch(None, device_ptrs=ptrs * args.steps, n=n, inflight=S, tables=False, max_pcs=MAX_PCS)[-B:]
    ms_thr, launches = ctx.last_batch_device_ms, ctx.last_batch_launches
    barrier()
    clk = clocks.stop() if clocks else None
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, last_step, f"rank{rank}_" if world > 1 else "")
    del last_step
    # ---- e2e: public API, pinned host input, copies + tables + objects inside the timed region ----
    TADpole_batch(host_np, max_pcs=MAX_PCS, ctx=ctx, streams=S)
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        tps = TADpole_batch(host_np, max_pcs=MAX_PCS, ctx=ctx, streams=S)
    ctx.sync()
    t_e2e = time.perf_counter() - t0
    barrier()
    tp = tps[-1]
    d2h = int(n + tp.scores.size * 8 + (res["nf"] - 1) * 8) * B
    # one call at a time through the public API (what a plain TADpole() in a loop costs)
    from tadpole_b200 import TADpole
    ctx.set("sync_blocking", 0)
    t0 = time.perf_counter()
    for i in range(lat_steps):
        TADpole(host_np[i % B], max_pcs=MAX_PCS, ctx=ctx)
    t_e2e_single = time.perf_counter() - t0

    tmax = torch.tensor([ms_thr, t_e2e * 1e3, ms_single, t_e2e_single * 1e3], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
    ms_all, e2e_ms_all, ms_single_all, e2e_single_all = (float(v) for v in tmax)
    ctx.close()

    strong = None
    if args.strong_bins > 0 or args.arm_bins > 0:
        try:
            strong = strong_scaling(args, torch, dist, rank, world, local_rank, Context, sharding, api)
        except Exception as e:                                      # the headline line must still be printed
            if world > 1:
                raise
            strong = {"failed": f"{type(e).__name__}: {e}"}

    if rank == 0:
        ncalls = args.steps * B
        value = world * ncalls / (ms_all * 1e-3)
        e2e_val = world * ncalls / (e2e_ms_all * 1e-3)
        peaks = {}
        try:
            with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as fh:
                peaks = json.load(fh)
        except OSError:
            pass
        hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
        peak_src = "measured (MEASURED_PEAKS.json hbm_gbs)" if peaks else "fallback 6650 GB/s (B200_PROFILING.md)"
        nf, k = res["nf"], res["k"]
        fp64_peak = measure_fp64_peak(torch)
        int8_peak = measure_int8_peak(torch)
        int8_src = ("measured in this run: torch._int_mm (cuBLASLt int8 -> int32) 8192^3, best of 10; executed digit-product "
                    "operations, not FP64 flops")
        if not int8_peak:
            int8_peak, int8_src = 4500.0, "nominal B200 dense int8 (4.5 POP/s): torch._int_mm unavailable"
        b_blk = -(-(k + max(32, k // 4)) // 32) * 32 if nf > 512 else nf      # width of the Rayleigh-Ritz problems
        nlev = float(np.count_nonzero(~np.isnan(res["scores"]))) if res.get("scores") is not None else 0.0

        def roof_of(cls):
            t_ms, cnt = prof[cls]
            if not cnt:
                return None
            per = t_ms / cnt                                   # ms per launch (CUDA events around each launch)
            src = peak_src
            if cls == "dgemm":
                r = {"kernel": "dgemm_kernel (FP64 DMMA mma.sync m8n8k4)", "bound": "tensor",
                     "achieved": prof["gemm_gflop"][0] / t_ms, "peak": fp64_peak, "unit": "TFLOP/s", "traffic": None}
                src = "cuBLAS DGEMM 4096^3 via torch.matmul, best of 6, measured in this run"
            elif cls == "igemm":
                r = {"kernel": "ig_gram_kernel + io_gemm_kernel (tcgen05.mma kind::i8; digit slicing timed apart as islice)", "bound": "tensor",
                     "achieved": prof["igemm_gop"][0] / t_ms, "peak": int8_peak, "unit": "TOP/s", "traffic": None}
                src = int8_src
            else:
                if cls == "coniss_sweep":      # SURVEY 8(d) S4: 8 Nf k(k+1)/2 read + 8 k (Nf-1) written per sweep
                    alg, name = 8.0 * nf * k * (k + 1) / 2 + 8.0 * k * (nf - 1), "coniss_sweep_kernel"
                elif cls == "ch":              # S5: 8 (Nf-1) per candidate + 24 k per scored level
                    alg, name = 8.0 * (nf - 1) * k + 24.0 * k * nlev, "ch_kernel"
                elif cls == "rowmean":         # S1: one pass over the N x N input
                    alg, name = 8.0 * n * n, "rowmean_kernel"
                elif cls == "compact":         # S1: Nf x Nf gather written once
                    alg, name = 8.0 * nf * nf, "compact_kernel"
                elif cls == "chol":            # read G, write L and L^-1 (lower triangles): 3 * 8 * b(b+1)/2
                    alg, name = 12.0 * b_blk * (b_blk + 1), "cholinv8_kernel"
                elif cls == "islice":
                    return None
                else:                          # eigensolver: read T, write V: 2 * 8 * b^2
                    alg, name = 16.0 * b_blk * b_blk, "osj_kernel"
                r = {"kernel": name, "bound": "hbm", "achieved": alg / (per * 1e-3) / 1e9, "peak": hbm_peak,
                     "unit": "GB/s", "traffic": None}
                if cls == "coniss_sweep":
                    r["merges_per_s"] = k * (nf - 1) / (per * 1e-3)
                if cls in ("jacobi", "chol", "coniss_sweep"):
                    r["note"] = "latency-bound: serial dependent steps on L2 / shared-memory resident data"
            r["frac"] = r["achieved"] / r["peak"]
            r["peak_source"] = src
            r["share_of_step"] = t_ms / ms_single          # of the one-call-at-a-time pass the classes were timed in
            r["avg_launch_ms"] = per
            r["launches_per_call"] = cnt / lat_steps
            return r

        classes = ("dgemm", "igemm", "jacobi", "chol", "coniss_sweep", "ch", "rowmean", "compact")
        roofs = {c: roof_of(c) for c in classes}
        roofs = {c: r for c, r in roofs.items() if r}
        for fn in ("r02_traffic.json", "r01_traffic.json"):     # DRAM bytes per launch from the ncu --set full captures
            try:
                with open(os.path.join(ROOT, "profiles", fn)) as fh:
                    traffic = json.load(fh)
            except OSError:
                continue
            if n == 2000:
                for r in roofs.values():
                    key = r["kernel"].split(" ")[0] if r["kernel"].startswith("dgemm_kernel") else (
                        "io_gemm_kernel" if r["kernel"].startswith("ig_gram_kernel + io_gemm_kernel") else r["kernel"])
                    if r["traffic"] is None and key in traffic:
                        r["traffic"] = traffic[key]
                        r["traffic_unit"] = f"bytes per launch (ncu dram__bytes_read.sum + dram__bytes_write.sum, profiles/{fn})"
        top = max(roofs, key=lambda c: roofs[c]["share_of_step"])
        roof = roofs[top]

        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_all / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic",
            "config": {"workload": workload_text(n), "bins": n, "good_bins": nf, "max_pcs": MAX_PCS,
                       "calls_per_step": B, "calls_timed": ncalls * world,
                       "n_pcs_found": res["n_pcs"], "optimal_n_clusters": res["n_clusters"],
                       "l2": f"every step passes over {B} different {n}x{n} f64 matrices ({B * n * n * 8 >> 20} MiB > L2): "
                             "no step re-reads a warm input",
                       "calls_in_flight_per_gpu": S,
                       "host_wait": ("blocking-sync events (threads sleep)" if sync_blocking else "cudaStreamSynchronize (spin)")
                                    + f", {ncpu} logical CPUs for {world * S} batch threads",
                       "parallelism": f"{world} GPU(s) x {S} independent calls in flight, kept in flight by tp_call_batch's own host "
                                      "threads (one context + stream each); no collective on the data path"},
            "e2e": {"value": e2e_val, "unit": UNIT, "h2d_bytes_per_step": h2d_bytes(n) * B, "d2h_bytes_per_step": d2h,
                    "ms_per_step": e2e_ms_all / args.steps,
                    "api": "TADpole_batch(list of pinned host matrices): one host thread -> tp_call_batch; returns tadpole objects"},
            "single_call": {"ms_per_call": ms_single_all / lat_steps, "calls_per_s": world * lat_steps / (ms_single_all * 1e-3),
                            "e2e_ms_per_call": e2e_single_all / lat_steps,
                            "note": "one call at a time per GPU (latency); rooflines and kernel_ms_per_call are from this pass"},
            "gpu_launches": int(launches),
            "clocks": clk,
            "roofline": roof,
            "roofline_all_kernels": roofs,
            "fp64_dgemm_peak_tflops_measured": fp64_peak,
            "int8_peak_tops": int8_peak,
            "stage_ms_last_call": {k_: round(v, 4) for k_, v in stage.items()},
            "kernel_ms_per_call": {c: round(v[0] / lat_steps, 4) for c, v in prof.items() if v[1]},
            "h2d_note": "only the upper triangle of the matrix is uploaded (band copies)",
            "kernel_launches_per_call": {c: v[1] / lat_steps for c, v in prof.items() if v[1]},
            "r_probe": r_probe(),
        }
        if strong is not None:
            line["strong_scaling"] = strong
        if world == 1 and not args.no_cpu_baseline:
            threads = usable_cpus()
            sec, detail = cpu_full_call(host_np[0].copy(), threads)
            line["cpu_baseline"] = {"value": 1.0 / sec, "unit": UNIT, "cores": threads, "kind": "port",
                                    "sample": "oracle/ (numpy + C restatement; R unavailable): " + cpu_sample_text(detail, threads),
                                    "same_result_as_gpu": bool(detail["n_pcs"] == tps[0].n_pcs and detail["n_clusters"] == tps[0].optimal_n_clusters)}
            c0 = Context(local_rank)
            # the tensor-core kernels at a size where they are the step (the 2000-bin workload leaves them 64-CTA grids)
            if args.large_n > 0:
                nl = args.large_n
                ml = synth_hic(nl, seed=77)
                for _ in range(2):
                    rl = c0.call(ml, max_pcs=MAX_PCS)
                c0.profile(1)
                rl = c0.call(ml, max_pcs=MAX_PCS)
                pl = c0.profile(0)
                stl = c0.timings()
                big = {"bins": nl, "good_bins": rl["nf"], "n_pcs_found": rl["n_pcs"],
                       "stage_ms": {k_: round(v, 3) for k_, v in stl.items()},
                       "kernel_ms": {c: round(v[0], 3) for c, v in pl.items() if v[1]},
                       "kernel_launches": {c: v[1] for c, v in pl.items() if v[1]}}
                if pl["igemm"][1]:
                    a = pl["igemm_gop"][0] / pl["igemm"][0]
                    big["igemm_roofline"] = {"kernel": "ig_gram_kernel + io_gemm_kernel<5|8> (tcgen05.mma kind::i8)", "bound": "tensor",
                                             "achieved": a, "peak": int8_peak, "unit": "TOP/s", "frac": a / int8_peak,
                                             "peak_source": int8_src}
                if pl["dgemm"][1]:
                    a = pl["gemm_gflop"][0] / pl["dgemm"][0]
                    big["dgemm_roofline"] = {"kernel": "dgemm_kernel (FP64 DMMA)", "bound": "tensor", "achieved": a, "peak": fp64_peak,
                                             "unit": "TFLOP/s", "frac": a / fp64_peak,
                                             "peak_source": "cuBLAS DGEMM 4096^3 measured in this run"}
                for fn in (f"r02_traffic_n{nl}.json", f"r01_traffic_n{nl}.json"):
                    try:
                        with open(os.path.join(ROOT, "profiles", fn)) as fh:
                            big["traffic_bytes_per_launch_ncu"] = {k_: v for k_, v in json.load(fh).items() if not k_.startswith("_")}
                            big["traffic_source"] = f"profiles/{fn}"
                        break
                    except OSError:
                        pass
                line["large_n_call"] = big
                del ml
            # input side (SURVEY 8f-2): the same call starting from the matrix FILE, text parsed on the GPU
            try:
                hm = host_np[0]
                text = "\n".join("\t".join(map(str, row)) for row in hm.astype(np.int64).tolist()) + "\n"
                with tempfile.NamedTemporaryFile("w", suffix=".tsv", delete=False) as fh:
                    fh.write(text)
                t_file = []
                for _ in range(6):
                    t0 = time.perf_counter()
                    ptr, n_in = c0.ingest_tsv(fh.name)
                    c0.call(device_ptr=ptr, n=n_in, colmajor=0, max_pcs=MAX_PCS)
                    t_file.append((time.perf_counter() - t0) * 1e3)
                ist = c0.ingest_stats()
                os.unlink(fh.name)
                alg = ist["text_bytes"] + 8.0 * n * n            # file bytes read once + the FP64 matrix written once
                line["from_file"] = {
                    "ms_per_call": float(np.median(t_file[1:])), "text_bytes": ist["text_bytes"],
                    "ingest_wall_ms": ist["wall_ms"], "parse_kernels_ms": ist["parse_ms"], "host_converted_fields": ist["host_fields"],
                    "roofline": {"kernel": "newline_* + parse_rows_kernel (ingest.cu)", "bound": "hbm",
                                 "achieved": alg / (ist["parse_ms"] * 1e-3) / 1e9, "peak": hbm_peak, "unit": "GB/s",
                                 "frac": alg / (ist["parse_ms"] * 1e-3) / 1e9 / hbm_peak, "traffic": None,
                                 "note": "event span of 4 launches incl. one host read-back of the row count"},
                    "note": "wall clock from the open() of the TSV file to the returned result, page cache warm"}
            except OSError as e:
                line["from_file"] = {"unavailable": str(e)}
            # ... and from the upper-triangle pixels of the same matrix (cooler-style triplets, tp_ingest_coo)
            hm = host_np[0]
            iu = np.triu_indices(n)
            pv = hm[iu]
            nzp = pv != 0
            pb1, pb2, pv = iu[0][nzp].astype(np.int32), iu[1][nzp].astype(np.int32), np.ascontiguousarray(pv[nzp])
            t_pix = []
            for _ in range(6):
                t0 = time.perf_counter()
                ptr, n_in = c0.ingest_coo(pb1, pb2, pv, n)
                rp = c0.call(device_ptr=ptr, n=n_in, colmajor=0, max_pcs=MAX_PCS)
                t_pix.append((time.perf_counter() - t0) * 1e3)
            ist = c0.ingest_stats()
            alg = 16.0 * pb1.size + 8.0 * n * n                  # 16 B per pixel read + the FP64 matrix written once
            line["from_pixels"] = {
                "ms_per_call": float(np.median(t_pix[1:])), "pixels": int(pb1.size), "pixel_bytes": int(16 * pb1.size),
                "dense_upper_bytes": int(n * (n + 1) // 2 * 8), "ingest_wall_ms": ist["wall_ms"], "scatter_span_ms": ist["parse_ms"],
                "same_result_as_dense": bool(rp["n_pcs"] == tps[0].n_pcs and rp["n_clusters"] == tps[0].optimal_n_clusters),
                "algorithmic_gbs": alg / (ist["parse_ms"] * 1e-3) / 1e9,
                "note": "wall clock from the host pixel arrays to the returned result; the span covers the PCIe copies too"}
            c0.close()
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def main():
    args = parse()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    run_b200(args, rank, world, local_rank)


if __name__ == "__main__":
    main()
