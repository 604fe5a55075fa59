"""Ad-hoc (not a test): chromosome calls above the shared-memory size of the n_pcs sweep, and what the global dSS leaf array
costs.  python tests/large_n_timing.py OUT.json [N ...]

  * per N (default 32 000, 40 000, 50 000 bins; synth_hic_gpu matrix handed over device-resident): wall time of one call
    after a small warm-up call on the same context, tp_ctx_timings per stage, and the peak device memory (all processes,
    the input included) seen by a thread polling cudaMemGetInfo every 5 ms during the call;
  * at 25 000 bins (seeded scores, k = 200): the sweep with the shared-memory dSS array (default there) against the
    global leaf array (TADPOLE_SWEEP_DSS=global), alternating, 3 runs each, then one TADPOLE_SWEEP_TRACE run of each
    for the cycles per merge step.
The card's name and power limit are read in the same run."""
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm,memory.total", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 else "unknown"


class Peak:
    def __init__(self):
        self.peak = 0

    def _poll(self):
        import torch
        while not self.stop.is_set():
            free, total = torch.cuda.mem_get_info(0)
            self.peak = max(self.peak, total - free)
            self.stop.wait(0.005)

    def __enter__(self):
        self.stop = threading.Event()
        self.t = threading.Thread(target=self._poll, daemon=True)
        self.t.start()
        return self

    def __exit__(self, *a):
        self.stop.set()
        self.t.join()


def one_call(n):
    import torch
    from tadpole_b200 import Context
    from tadpole_b200.synth import synth_hic, synth_hic_gpu
    ctx = Context(0)
    try:
        ctx.call(synth_hic(2000, seed=1))                      # warm-up: modules loaded, smem opt-ins done
        d = synth_hic_gpu(n, seed=n)
        torch.cuda.synchronize()
        torch.cuda.empty_cache()
        base = torch.cuda.mem_get_info(0)
        with Peak() as pk:
            t0 = time.perf_counter()
            res = ctx.call(device_ptr=d.data_ptr(), n=n, colmajor=0, want_scores=False)
            wall = (time.perf_counter() - t0) * 1e3
        out = dict(n=n, nf=res["nf"], k=res["k"], n_pcs=res["n_pcs"], n_clusters=res["n_clusters"], wall_ms=wall,
                   peak_device_bytes=int(pk.peak), input_bytes=n * n * 8,
                   used_before_call_bytes=int(base[1] - base[0]), stages=ctx.timings())
        del d
    except Exception as e:                                     # e.g. an allocation the device cannot hold: reported
        out = dict(n=n, error=str(e))
    finally:
        ctx.close()
        torch.cuda.empty_cache()
    return out


def trace_line(fn):
    """run fn with TADPOLE_SWEEP_TRACE set, return the '[sweep trace]' line the library writes to stderr"""
    os.environ["TADPOLE_SWEEP_TRACE"] = "1"
    sys.stderr.flush()
    saved = os.dup(2)
    with tempfile.TemporaryFile(mode="w+") as tf:
        os.dup2(tf.fileno(), 2)
        try:
            fn()
        finally:
            os.dup2(saved, 2)
            os.close(saved)
            del os.environ["TADPOLE_SWEEP_TRACE"]
        tf.seek(0)
        lines = [ln.strip() for ln in tf if ln.startswith("[sweep trace]")]
    return lines[-1] if lines else None


def sweep_compare(n=25000, k=200, reps=3):
    from tadpole_b200 import Context
    from test_gpu_sweep_large import _structured_scores
    s = _structured_scores(n, k, seed=25)
    ctx = Context(0)
    res = dict(n=n, k=k, shared_ms=[], global_ms=[])
    try:
        ctx.set_scores(s)
        ctx.sweep(k)                                           # warm-up
        ref = None
        for r in range(2 * reps):
            mode = "global" if r % 2 else "shared"
            if mode == "global":
                os.environ["TADPOLE_SWEEP_DSS"] = "global"
            ctx.set_scores(s)
            ncl, sc = ctx.sweep(k)
            os.environ.pop("TADPOLE_SWEEP_DSS", None)
            res[mode + "_ms"].append(ctx.timings()["sweep_ms"])
            same = (ncl.tobytes(), np.nan_to_num(sc, nan=-1.0).tobytes())
            ref = ref or same
            assert same == ref, "the two sweeps differ"
        for mode in ("shared", "global"):
            def run():
                if mode == "global":
                    os.environ["TADPOLE_SWEEP_DSS"] = "global"
                ctx.set_scores(s)
                ctx.sweep(k)
                os.environ.pop("TADPOLE_SWEEP_DSS", None)
            res[mode + "_trace"] = trace_line(run)
    finally:
        ctx.close()
    return res


def main():
    if len(sys.argv) < 2:
        sys.exit("usage: python tests/large_n_timing.py OUT.json [N ...]")
    out_path = sys.argv[1]
    sizes = [int(a) for a in sys.argv[2:]] or [32000, 40000, 50000]
    from tadpole_b200 import api
    api.QUIET = True
    out = dict(gpu=gpu_info(), sweep_25k=sweep_compare(), calls=[])
    print(json.dumps(out["sweep_25k"]), flush=True)
    for n in sizes:
        r = one_call(n)
        print(json.dumps(r), flush=True)
        out["calls"].append(r)
    out["gpu_after"] = gpu_info()
    os.makedirs(os.path.dirname(os.path.abspath(out_path)), exist_ok=True)
    with open(out_path, "w") as fh:
        json.dump(out, fh, indent=1)


if __name__ == "__main__":
    main()
