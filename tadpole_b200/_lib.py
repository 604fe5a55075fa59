"""ctypes binding of libtadpole_b200.so (include/tadpole_b200.h).

There is no CPU fallback: if the shared library is missing or no B200 is visible the
product fails loudly.  Nothing under oracle/ is imported here.
"""
from __future__ import annotations

import ctypes
import os
from ctypes import POINTER, c_char_p, c_double, c_int, c_int32, c_longlong, c_uint8, c_void_p

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libtadpole_b200.so")

TP_OK, TP_ERR_ARG, TP_ERR_CUDA, TP_ERR_NOLEVEL, TP_ERR_NOCONV, TP_ERR_NOMEM, TP_ERR_NOSPLIT = range(7)

# every symbol include/tadpole_b200.h declares
EXPORTED = [
    "tp_last_error", "tp_version", "tp_ctx_create", "tp_ctx_destroy", "tp_ctx_sync", "tp_ctx_stream",
    "tp_ctx_launches", "tp_ctx_set", "tp_ctx_timings", "tp_ctx_profile", "tp_filter", "tp_compact", "tp_set_filtered",
    "tp_get_filtered", "tp_correlation", "tp_get_correlation", "tp_set_correlation", "tp_pca",
    "tp_get_scores", "tp_set_scores", "tp_sweep", "tp_get_sweep_scores", "tp_get_dendro", "tp_select", "tp_call", "tp_call_arm",
    "tp_difft_batch", "tp_assemble", "tp_assemble_levels", "tp_test_cholinv", "tp_test_eig", "tp_test_igram", "tp_test_mgram", "tp_test_symshard", "tp_test_ss_need", "tp_test_ss_tile",
    "tp_comm_unique_id", "tp_ctx_comm_init", "tp_ctx_comm_select", "tp_ctx_comm_info",
    "tp_ingest_tsv", "tp_ingest_tsv_file", "tp_ingested", "tp_get_ingested", "tp_ingest_stats", "tp_test_parse_field",
    "tp_ingest_coo", "tp_ingest_coo_file",
    "tp_difft_null", "tp_recall",
    "tp_ctx_create_multi", "tp_device_count", "tp_ctx_devices", "tp_ctx_generation", "tp_ctx_dims", "tp_call_arms", "tp_call_batch",
    "tp_batch_size", "tp_batch_device_ms", "tp_batch_launches", "tp_batch_status", "tp_batch_error", "tp_batch_dims", "tp_batch_get", "tp_batch_free", "tp_find_groups",
    "tp_genome_ingest", "tp_genome_ingest_file", "tp_genome_stats", "tp_genome_matrix", "tp_call_genome", "tp_genome_free",
    "tp_centromere_split", "tp_batch_split",
]


class TadpoleError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"libtadpole_b200 error {code}: {msg}")
        self.code = code


_lib = None


def load():
    """Load the shared library (building is __graft_entry__.build()'s job, not ours)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} not found: build it with `python -m tadpole_b200.build` "
            "(nvcc, sm_100a). tadpole_b200 has no CPU fallback.")
    lib = ctypes.CDLL(LIB_PATH)
    dp, ip, u8p, vp = POINTER(c_double), POINTER(c_int), POINTER(c_uint8), c_void_p
    sig = {
        "tp_last_error": (c_char_p, []),
        "tp_version": (c_int, []),
        "tp_ctx_create": (c_int, [c_int, POINTER(vp)]),
        "tp_ctx_create_multi": (c_int, [ip, c_int, POINTER(vp)]),
        "tp_device_count": (c_int, []),
        "tp_ctx_devices": (c_int, [vp, ip, c_int]),
        "tp_ctx_generation": (c_longlong, [vp]),
        "tp_ctx_dims": (c_int, [vp, ip, ip, ip, ip, ip]),
        "tp_call_arms": (c_int, [vp, ip, c_int, ip, c_int, c_int, c_int, POINTER(vp)]),
        "tp_call_batch": (c_int, [vp, c_int, POINTER(vp), ip, c_int, c_int, c_int, c_int, c_double, c_int, c_int, c_int,
                                  POINTER(vp)]),
        "tp_batch_size": (c_int, [vp]),
        "tp_batch_device_ms": (c_double, [vp]),
        "tp_batch_launches": (c_longlong, [vp]),
        "tp_batch_status": (c_int, [vp, c_int]),
        "tp_batch_error": (c_char_p, [vp, c_int]),
        "tp_batch_dims": (c_int, [vp, c_int, c_int, ip, ip, ip, ip, ip, ip, ip, ip]),
        "tp_batch_get": (c_int, [vp, c_int, c_int, u8p, ip, ip, dp, dp, ip, ip, ip, ip, dp, ip, ip, ip]),
        "tp_batch_free": (c_int, [vp]),
        "tp_batch_split": (c_int, [vp, c_int, ip, ip, ip, u8p]),
        "tp_centromere_split": (c_int, [u8p, c_int, c_int, ip, ip, ip, ip, ip, ip, ip, ip, ip, ip, ip]),
        "tp_genome_ingest": (c_int, [vp, ip, c_int, ip, ip, dp, ctypes.c_size_t, c_int, POINTER(vp)]),
        "tp_genome_ingest_file": (c_int, [vp, ip, c_int, c_char_p, c_int, c_int, POINTER(vp)]),
        "tp_genome_stats": (c_int, [vp, POINTER(ctypes.c_ulonglong), POINTER(ctypes.c_ulonglong), POINTER(ctypes.c_ulonglong)]),
        "tp_genome_matrix": (c_int, [vp, vp, c_int, dp]),
        "tp_call_genome": (c_int, [vp, vp, ip, c_int, c_int, c_int, c_double, c_int, c_int, c_int, POINTER(vp)]),
        "tp_genome_free": (c_int, [vp]),
        "tp_find_groups": (c_int, [dp, c_int, ip]),
        "tp_ctx_destroy": (c_int, [vp]),
        "tp_ctx_sync": (c_int, [vp]),
        "tp_ctx_stream": (vp, [vp]),
        "tp_ctx_launches": (c_longlong, [vp]),
        "tp_ctx_set": (c_int, [vp, c_char_p, c_double]),
        "tp_ctx_timings": (c_int, [vp, dp]),
        "tp_ctx_profile": (c_int, [vp, c_int, dp, POINTER(c_longlong)]),
        "tp_ingest_tsv": (c_int, [vp, c_char_p, ctypes.c_size_t, c_int, ip]),
        "tp_ingest_tsv_file": (c_int, [vp, c_char_p, c_int, ip]),
        "tp_ingested": (c_int, [vp, POINTER(vp), ip]),
        "tp_get_ingested": (c_int, [vp, dp]),
        "tp_ingest_stats": (c_int, [vp, dp]),
        "tp_test_parse_field": (c_int, [c_char_p, c_int, dp]),
        "tp_ingest_coo": (c_int, [vp, ip, ip, dp, ctypes.c_size_t, c_int, c_int, POINTER(ctypes.c_ulonglong)]),
        "tp_ingest_coo_file": (c_int, [vp, c_char_p, c_int, c_int, c_int, ip, POINTER(ctypes.c_ulonglong),
                                       POINTER(ctypes.c_ulonglong)]),
        "tp_filter": (c_int, [vp, vp, c_int, c_int, c_int, c_double, u8p, dp, dp]),
        "tp_compact": (c_int, [vp, ip, c_int]),
        "tp_set_filtered": (c_int, [vp, dp, c_int]),
        "tp_get_filtered": (c_int, [vp, dp]),
        "tp_correlation": (c_int, [vp]),
        "tp_get_correlation": (c_int, [vp, dp]),
        "tp_set_correlation": (c_int, [vp, dp, c_int]),
        "tp_pca": (c_int, [vp, c_int, ip]),
        "tp_comm_unique_id": (c_int, [vp]),
        "tp_ctx_comm_init": (c_int, [vp, vp, c_int, c_int, c_int]),
        "tp_ctx_comm_select": (c_int, [vp, c_int]),
        "tp_ctx_comm_info": (c_int, [vp, ip, ip]),
        "tp_test_cholinv": (c_int, [vp, dp, c_int, c_int, dp, dp, ip]),
        "tp_test_eig": (c_int, [vp, dp, c_int, c_double, dp, dp, ip]),
        "tp_test_igram": (c_int, [vp, dp, c_int, dp, ip]),
        "tp_test_mgram": (c_int, [vp, dp, c_int, c_int, c_int, dp]),
        "tp_test_symshard": (c_int, [vp, dp, c_int, c_int, c_int, c_double, dp]),
        "tp_test_ss_need": (c_int, [c_int, c_int, c_int, c_int]),
        "tp_test_ss_tile": (c_int, [c_int, c_int, c_int, c_int, c_int, c_int]),
        "tp_get_scores": (c_int, [vp, dp]),
        "tp_set_scores": (c_int, [vp, dp, c_int, c_int]),
        "tp_sweep": (c_int, [vp, c_int, c_int, c_int, ip, ip]),
        "tp_get_dendro": (c_int, [vp, c_int, dp, ip]),
        "tp_get_sweep_scores": (c_int, [vp, dp]),
        "tp_select": (c_int, [dp, c_int, c_int, c_int, ip, ip]),
        "tp_call": (c_int, [vp, vp, c_int, c_int, c_int, c_int, c_int, c_double, u8p, ip, ip, ip, ip, ip, dp]),
        "tp_call_arm": (c_int, [vp, ip, c_int, c_int, c_int, ip, ip, ip, ip, dp]),
        "tp_recall": (c_int, [vp, c_int, c_int, ip, ip, ip, ip, dp]),
        "tp_difft_batch": (c_int, [vp, vp, vp, c_int, c_int, c_int, vp]),
        "tp_difft_null": (c_int, [vp, vp, c_int, c_int, c_int, c_int, vp, c_int, ctypes.c_ulonglong, c_int, vp, vp, vp, vp]),
        "tp_assemble": (c_int, [dp, c_int, c_int, ip, ip, c_int, ip, ip, ip, ip]),
        "tp_assemble_levels": (c_int, [dp, c_int, ip, c_int, ip, ip, c_int, ip, ip, ip]),
    }
    for name, (res, args) in sig.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def _nccl_first_from_torch():
    """The library binds NCCL at run time (dlopen) the first time a communicator is made.  If torch is going to be used in
    this process too, its bundled NCCL must be the copy that gets loaded: the dynamic loader keeps ONE library per soname,
    and torch cannot live with the system's older libnccl.so.2.  So import torch first when it is there (an R host has no
    torch and binds the system NCCL)."""
    try:
        import torch  # noqa: F401
    except ImportError:
        pass


def device_count():
    return int(load().tp_device_count())


def check(rc):
    if rc != TP_OK:
        raise TadpoleError(rc, load().tp_last_error().decode("utf-8", "replace"))


def _dp(a):
    return a.ctypes.data_as(POINTER(c_double))


def _ip(a):
    return a.ctypes.data_as(POINTER(c_int))


def _centromere(search, fix):
    """The `centromere` argument of tp_call_batch / tp_call_genome: 0 whole matrices, 1 centromere_search, 2 with
    centromere_fix."""
    return (2 if fix else 1) if search else 0


class Context:
    """One GPU context (device buffers, stream), or -- given a list of devices -- one multi-device context that spreads
    every call over those GPUs from this one host thread (tp_ctx_create_multi).  Thin wrapper over tp_ctx."""

    def __init__(self, device=0):
        self.lib = load()
        self._h = c_void_p()
        if isinstance(device, (list, tuple)):
            _nccl_first_from_torch()
            devs = np.ascontiguousarray(device, dtype=np.int32)
            check(self.lib.tp_ctx_create_multi(_ip(devs), devs.size, ctypes.byref(self._h)))
            self.devices = [int(d) for d in devs]
            self.device = self.devices[0]
        else:
            check(self.lib.tp_ctx_create(int(device), ctypes.byref(self._h)))
            self.device = int(device)
            self.devices = [self.device]

    @property
    def generation(self):
        """changes whenever the state resident in the context is replaced (stale-handle check, tp_ctx_generation)"""
        return int(self.lib.tp_ctx_generation(self._h))

    @generation.setter
    def generation(self, _):
        pass                         # the library counts

    def dims(self):
        v = [c_int(0) for _ in range(5)]
        check(self.lib.tp_ctx_dims(self._h, *[ctypes.byref(x) for x in v]))
        return dict(zip(("n", "nf", "k", "k_full", "maxlev"), (x.value for x in v)))

    def close(self):
        if getattr(self, "_h", None) is not None and self._h:
            self.lib.tp_ctx_destroy(self._h)
            self._h = c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ---- plumbing ----
    def set(self, key, value):
        check(self.lib.tp_ctx_set(self._h, key.encode(), float(value)))

    def sync(self):
        check(self.lib.tp_ctx_sync(self._h))

    @property
    def stream(self):
        return self.lib.tp_ctx_stream(self._h) or 0

    @property
    def launches(self):
        return int(self.lib.tp_ctx_launches(self._h))

    def timings(self):
        out = np.zeros(10)
        check(self.lib.tp_ctx_timings(self._h, _dp(out)))
        keys = ["filter_ms", "compact_ms", "correlation_ms", "pca_ms", "sweep_ms", "ch_ms", "total_ms",
                "pca_iterations", "pca_applications", "jacobi_sweeps"]
        return dict(zip(keys, out.tolist()))

    PROFILE_CLASSES = ["rowmean", "compact", "dgemm", "jacobi", "coniss_sweep", "ch", "difft", "gemm_gflop", "chol", "igemm",
                       "comm", "igemm_gop", "islice", "spare13", "spare14", "spare15"]

    def profile(self, enable=-1):
        """enable: 1 start/reset, 0 stop, -1 read.  Returns {class: (ms, launches)} accumulated so far."""
        ms = np.zeros(16)
        cnt = np.zeros(16, dtype=np.int64)
        check(self.lib.tp_ctx_profile(self._h, int(enable), _dp(ms), cnt.ctypes.data_as(POINTER(c_longlong))))
        return {k: (float(m), int(c)) for k, m, c in zip(self.PROFILE_CLASSES, ms, cnt)}

    # ---- input side ----
    def ingest_tsv(self, src, sep="\t"):
        """Parse a header-less separator-delimited square matrix on the device (R/TADpole.R:17).  src: a path (str /
        os.PathLike) or the text itself (bytes).  Returns (device_ptr, n) for filter()/call() with device_ptr=."""
        n = c_int(0)
        if isinstance(src, (bytes, bytearray, memoryview)):
            buf = bytes(src)
            check(self.lib.tp_ingest_tsv(self._h, buf, len(buf), ord(sep), ctypes.byref(n)))
        else:
            check(self.lib.tp_ingest_tsv_file(self._h, os.fsencode(src), ord(sep), ctypes.byref(n)))
        ptr = c_void_p()
        check(self.lib.tp_ingested(self._h, ctypes.byref(ptr), ctypes.byref(n)))
        return ptr.value, n.value

    def ingest_coo(self, bin1=None, bin2=None, count=None, n=None, index_base=0, path=None, sep="\t"):
        """Upper-triangle pixels (bin1, bin2, count) -> the dense matrix in HBM (tp_ingest_coo), or the same from a
        three-column text file (tp_ingest_coo_file; n=None: largest bin + 1).  Returns (device_ptr, n); the number of
        pixels below the diagonal that were ignored is left in self.last_coo_below."""
        below = ctypes.c_ulonglong(0)
        nn = c_int(0)
        if path is not None:
            nnz = ctypes.c_ulonglong(0)
            check(self.lib.tp_ingest_coo_file(self._h, os.fsencode(path), ord(sep), int(n or 0), int(index_base),
                                              ctypes.byref(nn), ctypes.byref(nnz), ctypes.byref(below)))
            self.last_coo_nnz = int(nnz.value)
        else:
            b1 = np.ascontiguousarray(bin1, dtype=np.int32)
            b2 = np.ascontiguousarray(bin2, dtype=np.int32)
            v = np.ascontiguousarray(count, dtype=np.float64)
            assert b1.ndim == 1 and b1.shape == b2.shape == v.shape, "bin1, bin2, count: equal-length vectors expected"
            check(self.lib.tp_ingest_coo(self._h, _ip(b1), _ip(b2), _dp(v), b1.size, int(n), int(index_base),
                                         ctypes.byref(below)))
            self.last_coo_nnz = int(b1.size)
        self.last_coo_below = int(below.value)
        ptr = c_void_p()
        check(self.lib.tp_ingested(self._h, ctypes.byref(ptr), ctypes.byref(nn)))
        return ptr.value, nn.value

    def get_ingested(self, n):
        out = np.empty((n, n))
        check(self.lib.tp_get_ingested(self._h, _dp(out)))
        return out

    def ingest_stats(self):
        out = np.zeros(4)
        check(self.lib.tp_ingest_stats(self._h, _dp(out)))
        return dict(wall_ms=out[0], parse_ms=out[1], text_bytes=int(out[2]), host_fields=int(out[3]))

    # ---- stage 1 ----
    def filter(self, mat=None, bad_frac=0.01, colmajor=None, device_ptr=None, n=None):
        """mat: numpy n x n float64 (C or F order), or device_ptr + n (+ colmajor)."""
        if device_ptr is None:
            mat = np.asarray(mat)
            if mat.dtype != np.float64 or not (mat.flags.c_contiguous or mat.flags.f_contiguous):
                mat = np.ascontiguousarray(mat, dtype=np.float64)
            assert mat.ndim == 2 and mat.shape[0] == mat.shape[1], "square matrix expected"
            n = mat.shape[0]
            colmajor = 0 if mat.flags.c_contiguous else 1
            ptr, ondev = mat.ctypes.data, 0
        else:
            ptr, ondev, colmajor = int(device_ptr), 1, int(bool(colmajor))
        bad = np.zeros(n, dtype=np.uint8)
        rm = np.zeros(n)
        thr = np.zeros(1)
        check(self.lib.tp_filter(self._h, ptr, n, colmajor, ondev, float(bad_frac),
                                 bad.ctypes.data_as(POINTER(c_uint8)), _dp(rm), _dp(thr)))
        return bad.astype(bool), rm, float(thr[0])

    def compact(self, keep):
        keep = np.ascontiguousarray(keep, dtype=np.int32)
        check(self.lib.tp_compact(self._h, _ip(keep), keep.size))
        return keep.size

    def set_filtered(self, x):
        x = np.ascontiguousarray(x, dtype=np.float64)
        check(self.lib.tp_set_filtered(self._h, _dp(x), x.shape[0]))

    def get_filtered(self, nf):
        out = np.zeros((nf, nf))
        check(self.lib.tp_get_filtered(self._h, _dp(out)))
        return out

    # ---- stage 2 ----
    def correlation(self):
        check(self.lib.tp_correlation(self._h))

    def get_correlation(self, nf):
        out = np.zeros((nf, nf))
        check(self.lib.tp_get_correlation(self._h, _dp(out)))
        return out

    def set_correlation(self, cor):
        cor = np.ascontiguousarray(cor, dtype=np.float64)
        check(self.lib.tp_set_correlation(self._h, _dp(cor), cor.shape[0]))

    # ---- stage 3 ----
    def pca(self, max_pcs=200):
        k = c_int(0)
        check(self.lib.tp_pca(self._h, int(max_pcs), ctypes.byref(k)))
        return k.value

    # ---- multi-GPU ----
    def comm_unique_id(self):
        """128-byte NCCL unique id (call on one rank, ship the bytes to the others)."""
        _nccl_first_from_torch()
        buf = ctypes.create_string_buffer(128)
        check(self.lib.tp_comm_unique_id(ctypes.cast(buf, ctypes.c_void_p)))
        return buf.raw

    def comm_init(self, unique_id, rank, nranks, slot=0):
        _nccl_first_from_torch()
        buf = ctypes.create_string_buffer(bytes(unique_id), 128)
        check(self.lib.tp_ctx_comm_init(self._h, ctypes.cast(buf, ctypes.c_void_p), int(rank), int(nranks), int(slot)))

    def comm_select(self, slot):
        check(self.lib.tp_ctx_comm_select(self._h, int(slot)))

    def comm_info(self):
        r, n = c_int(0), c_int(1)
        check(self.lib.tp_ctx_comm_info(self._h, ctypes.byref(r), ctypes.byref(n)))
        return r.value, n.value

    def test_cholinv(self, g, factor_only=False):
        """(L, Linv or None, bad) of a symmetric positive definite b x b matrix (test hook)."""
        g = np.ascontiguousarray(g, dtype=np.float64)
        b = g.shape[0]
        l = np.zeros((b, b)); li = np.zeros((b, b)); bad = np.zeros(1, dtype=np.int32)
        check(self.lib.tp_test_cholinv(self._h, _dp(g), b, int(factor_only), _dp(l), _dp(li), _ip(bad)))
        return np.tril(l), (None if factor_only else li), int(bad[0])

    def test_eig(self, t, tol=1e-14):
        """(w descending, V, sweeps) of a symmetric positive semi-definite b x b matrix (test hook)."""
        t = np.ascontiguousarray(t, dtype=np.float64)
        b = t.shape[0]
        w = np.zeros(b); v = np.zeros((b, b)); sw = np.zeros(1, dtype=np.int32)
        check(self.lib.tp_test_eig(self._h, _dp(t), b, float(tol), _dp(w), _dp(v), _ip(sw)))
        return w, v, int(sw[0])

    def test_igram(self, x):
        """Exact Gram matrix x @ x.T of a symmetric integer-count matrix (tcgen05 int8 path), or None when the
        input is not integer-valued (test hook)."""
        x = np.ascontiguousarray(x, dtype=np.float64)
        n = x.shape[0]
        g = np.zeros((n, n)); used = np.zeros(1, dtype=np.int32)
        check(self.lib.tp_test_igram(self._h, _dp(x), n, _dp(g), _ip(used)))
        return g if used[0] else None

    def test_mgram(self, a, row_begin=0, row_end=None, fill=0.0):
        """Rows [row_begin, row_end) of a @ a.T through the sliced int8 Gram of tp_pca (test hook); other rows = fill."""
        a = np.ascontiguousarray(a, dtype=np.float64)
        n = a.shape[0]
        g = np.full((n, n), float(fill))
        check(self.lib.tp_test_mgram(self._h, _dp(a), n, int(row_begin), n if row_end is None else int(row_end), _dp(g)))
        return g

    def test_symshard(self, a, nranks, kind, fill=-7.0):
        """a @ a.T as `nranks` ranks of a sharded call compute it (every block pair once + local transpose), emulated on
        this GPU (test hook).  kind 0: exact integer Gram, kind 1: sliced FP64 Gram."""
        a = np.ascontiguousarray(a, dtype=np.float64)
        n = a.shape[0]
        g = np.zeros((n, n))
        check(self.lib.tp_test_symshard(self._h, _dp(a), n, int(nranks), int(kind), float(fill), _dp(g)))
        return g

    def get_scores(self, nf, k):
        out = np.zeros((nf, k))
        check(self.lib.tp_get_scores(self._h, _dp(out)))
        return out

    def set_scores(self, scores):
        scores = np.ascontiguousarray(scores, dtype=np.float64)
        check(self.lib.tp_set_scores(self._h, _dp(scores), scores.shape[0], scores.shape[1]))

    # ---- stages 4 + 5 ----
    def sweep(self, k, min_clusters=2, cand_begin=0, cand_stride=1):
        """Returns (n_cluster[k], scores[k, maxlev] NaN padded)."""
        ncl = np.zeros(k, dtype=np.int32)
        maxlev = c_int(0)
        check(self.lib.tp_sweep(self._h, int(min_clusters), int(cand_begin), int(cand_stride), _ip(ncl), ctypes.byref(maxlev)))
        return ncl, self._sweep_scores(k, maxlev.value)

    def _sweep_scores(self, k, maxlev):
        """tp_get_sweep_scores: the k x maxlev score matrix of the last sweep."""
        sc = np.empty((k, maxlev))
        check(self.lib.tp_get_sweep_scores(self._h, _dp(sc)))
        return sc

    def dendro(self, cand, nf):
        seq = np.zeros(nf - 1)
        order = np.zeros(nf - 1, dtype=np.int32)
        check(self.lib.tp_get_dendro(self._h, int(cand), _dp(seq), _ip(order)))
        return seq, order

    def select(self, scores):
        scores = np.ascontiguousarray(scores, dtype=np.float64)
        oc, ol = c_int(0), c_int(0)
        check(self.lib.tp_select(_dp(scores), scores.shape[0], scores.shape[1], scores.shape[1],
                                 ctypes.byref(oc), ctypes.byref(ol)))
        return oc.value, ol.value

    # ---- one-shot ----
    def call(self, mat=None, max_pcs=200, min_clusters=2, bad_frac=0.01, device_ptr=None, n=None, colmajor=None,
             want_scores=True):
        if device_ptr is None:
            mat = np.asarray(mat)
            if mat.dtype != np.float64 or not (mat.flags.c_contiguous or mat.flags.f_contiguous):
                mat = np.ascontiguousarray(mat, dtype=np.float64)
            n = mat.shape[0]
            colmajor = 0 if mat.flags.c_contiguous else 1
            ptr, ondev = mat.ctypes.data, 0
        else:
            ptr, ondev, colmajor = int(device_ptr), 1, int(bool(colmajor))
        bad = np.zeros(n, dtype=np.uint8)
        nf, k, npcs, ncl, maxlev = c_int(0), c_int(0), c_int(0), c_int(0), c_int(0)
        seq = np.zeros(max(n - 1, 1))
        check(self.lib.tp_call(self._h, ptr, n, colmajor, ondev, int(max_pcs), int(min_clusters), float(bad_frac),
                               bad.ctypes.data_as(POINTER(c_uint8)), ctypes.byref(nf), ctypes.byref(k),
                               ctypes.byref(npcs), ctypes.byref(ncl), ctypes.byref(maxlev), _dp(seq)))
        return dict(bad=bad.astype(bool), nf=nf.value, k=k.value, n_pcs=npcs.value, n_clusters=ncl.value,
                    scores=self._sweep_scores(k.value, maxlev.value) if want_scores else None,
                    seqdist=seq[:nf.value - 1].copy())

    def call_arm(self, keep, max_pcs=200, min_clusters=2):
        keep = np.ascontiguousarray(keep, dtype=np.int32)
        nf = keep.size
        k, npcs, ncl, maxlev = c_int(0), c_int(0), c_int(0), c_int(0)
        seq = np.zeros(nf - 1)
        check(self.lib.tp_call_arm(self._h, _ip(keep), nf, int(max_pcs), int(min_clusters), ctypes.byref(k),
                                   ctypes.byref(npcs), ctypes.byref(ncl), ctypes.byref(maxlev), _dp(seq)))
        return dict(nf=nf, k=k.value, n_pcs=npcs.value, n_clusters=ncl.value,
                    scores=self._sweep_scores(k.value, maxlev.value), seqdist=seq)

    def call_arms(self, keep_p, keep_q, max_pcs=200, min_clusters=2):
        """tp_call_arms: both chromosome arms (on disjoint halves of the devices of a multi-device context).
        Returns (result_p, result_q), each as call_arm returns."""
        kp = np.ascontiguousarray(keep_p, dtype=np.int32)
        kq = np.ascontiguousarray(keep_q, dtype=np.int32)
        h = c_void_p()
        check(self.lib.tp_call_arms(self._h, _ip(kp), kp.size, _ip(kq), kq.size, int(max_pcs), int(min_clusters),
                                    ctypes.byref(h)))
        try:
            items = [self._batch_item(h, a, tables=False) for a in range(2)]
        finally:
            self.lib.tp_batch_free(h)
        return tuple({key: it[key] for key in ("nf", "k", "n_pcs", "n_clusters", "scores", "seqdist")} for it in items)

    def _batch_item(self, h, i, tables, part=-1):
        """Item i of a tp_batch as the dict call() returns, plus 'tables' {level: [rows, 2]} (or None) and 'device_ms'.
        part 0 / 1: the p / q arm of split item i instead, with 'tables', 'keep' (0-based), 'bad_columns' (original 1-based,
        or None) and 'labels' (fixed labels of the optimal level) in place of 'bad' and 'device_ms'."""
        d = [c_int(0) for _ in range(8)]
        check(self.lib.tp_batch_dims(h, i, part, *[ctypes.byref(x) for x in d]))
        nn, nf, k, ml, nlev, nrows, nk, nbad = (x.value for x in d)
        bad = np.zeros(nn, np.uint8); sc = np.empty((k, ml)); seq = np.empty(nf - 1)
        lev = np.zeros(nlev, np.int32); off = np.zeros(nlev + 1, np.int32)
        st = np.zeros(nrows, np.int32); en = np.zeros(nrows, np.int32)
        keep = np.zeros(nk, np.int32); badc = np.zeros(max(nbad, 0), np.int32)
        lab = np.zeros(nf + max(nbad, 0) if part >= 0 else 0, np.int32)
        npcs, ncl, ms = c_int(0), c_int(0), c_double(0.0)
        check(self.lib.tp_batch_get(h, i, part, bad.ctypes.data_as(POINTER(c_uint8)), ctypes.byref(npcs), ctypes.byref(ncl),
                                    _dp(sc), _dp(seq), _ip(lev), _ip(off), _ip(st), _ip(en), ctypes.byref(ms), _ip(keep),
                                    _ip(badc), _ip(lab)))
        tab = np.stack([st, en], axis=1).astype(np.int64)
        item = dict(nf=nf, k=k, n_pcs=npcs.value, n_clusters=ncl.value, scores=sc, seqdist=seq,
                    tables={int(l): tab[off[j]: off[j + 1]] for j, l in enumerate(lev)} if tables else None)
        if part >= 0:
            return dict(keep=keep, bad_columns=badc if nbad >= 0 else None, **item, labels=lab)
        return dict(bad=bad.astype(bool), **item, device_ms=ms.value)

    def call_batch(self, mats, max_pcs=200, min_clusters=2, bad_frac=0.01, inflight=8, tables=True, device_ptrs=None, n=None,
                   centromere_search=False, centromere_fix=False):
        """tp_call_batch: one tp_call per matrix, `inflight` calls per device kept in flight by library-owned threads over
        every device of the context.  mats: list of square float64 arrays (all C or all F order); or device_ptrs + n
        (row-major, single-device contexts).  Returns a list of dicts as call() returns, plus 'tables' {level: [rows, 2]}
        and 'device_ms'; a failed call's entry is the TadpoleError.
        centromere_search: each matrix split at its centromere and its two arms called in the same workers, tables always
        built; a split matrix's entry is dict(split=True, centromere (1-based bins), bad, device_ms, p, q) with p / q as
        _batch_item reads an arm, an unsplit one's (centromere_fix) the dict above plus split=False and centromere, and
        one that does not split without centromere_fix fails with TP_ERR_NOSPLIT."""
        if device_ptrs is None:
            mats = [m if (m.dtype == np.float64 and (m.flags.c_contiguous or m.flags.f_contiguous))
                    else np.ascontiguousarray(m, dtype=np.float64) for m in (np.asarray(m) for m in mats)]
            colmajor = 0 if all(m.flags.c_contiguous for m in mats) else 1
            if colmajor:
                mats = [m if m.flags.f_contiguous else np.asfortranarray(m) for m in mats]
            ptrs = (c_void_p * max(len(mats), 1))(*[m.ctypes.data for m in mats])
            ns = np.array([m.shape[0] for m in mats], dtype=np.int32)
            ondev = 0
        else:
            ptrs = (c_void_p * max(len(device_ptrs), 1))(*[int(p) for p in device_ptrs])
            ns = np.full(len(device_ptrs), int(n), dtype=np.int32)
            colmajor, ondev = 0, 1
        ncalls = int(ns.size)
        h = c_void_p()
        tables = bool(tables or centromere_search)
        check(self.lib.tp_call_batch(self._h, ncalls, ptrs, _ip(ns), colmajor, ondev, int(max_pcs), int(min_clusters),
                                     float(bad_frac), int(inflight), int(tables), _centromere(centromere_search, centromere_fix),
                                     ctypes.byref(h)))
        return self._batch_results(h, ncalls, tables)

    def _split_state(self, h, i, n):
        """(split: -1 / 0 / 1, the longest bad stretch cs..ce (1-based bins) or None, bad flags or None) of item i
        (tp_batch_split)."""
        sp, cs, ce = c_int(0), c_int(0), c_int(0)
        bad = np.zeros(max(n, 1), np.uint8)
        check(self.lib.tp_batch_split(h, i, ctypes.byref(sp), ctypes.byref(cs), ctypes.byref(ce),
                                      bad.ctypes.data_as(POINTER(c_uint8))))
        return (sp.value, np.arange(cs.value, ce.value + 1) if cs.value else None,
                bad[:n].astype(bool) if sp.value >= 0 else None)

    def _batch_results(self, h, ncalls, tables):
        """Every item of a tp_batch (freed here) as call_batch returns them."""
        out = []
        self.last_batch_device_ms = float(self.lib.tp_batch_device_ms(h))
        self.last_batch_launches = int(self.lib.tp_batch_launches(h))
        try:
            for i in range(ncalls):
                rc = self.lib.tp_batch_status(h, i)
                if rc != TP_OK:
                    err = TadpoleError(rc, self.lib.tp_batch_error(h, i).decode("utf-8", "replace"))
                    # a centromere_search item that failed after its filter: split (-1 = not reached), the longest bad
                    # stretch and the bad flags, for load_mat's messages
                    nn = c_int(0)
                    check(self.lib.tp_batch_dims(h, i, -1, ctypes.byref(nn), None, None, None, None, None, None, None))
                    err.split, err.centromere, err.bad = self._split_state(h, i, nn.value)
                    out.append(err)
                    continue
                nn = c_int(0)
                check(self.lib.tp_batch_dims(h, i, -1, ctypes.byref(nn), None, None, None, None, None, None, None))
                split, cen, bad = self._split_state(h, i, nn.value)
                if split == 1:                       # centromere_search, split: the item's bad flags and device time, the arms
                    ms = c_double(0.0)
                    check(self.lib.tp_batch_get(h, i, -1, None, None, None, None, None, None, None, None, None,
                                                ctypes.byref(ms), None, None, None))
                    out.append(dict(split=True, centromere=cen, bad=bad, device_ms=ms.value,
                                    p=self._batch_item(h, i, True, 0), q=self._batch_item(h, i, True, 1)))
                    continue
                item = self._batch_item(h, i, tables)
                if split == 0:                       # centromere_search, not split: processed whole (centromere_fix)
                    item.update(split=False, centromere=cen)
                out.append(item)
        finally:
            self.lib.tp_batch_free(h)
        return out

    # ---- genome-wide input ----
    def genome_ingest(self, chrom_bins, bin1=None, bin2=None, count=None, index_base=0, path=None, sep="\t"):
        """tp_genome_ingest[_file]: pixels over the whole genome (global bin ids over chrom_bins, the bins per chromosome)
        routed into one bucket per chromosome on this context's (first) device.  Returns a Genome handle."""
        cb = np.ascontiguousarray(chrom_bins, dtype=np.int32)
        h = c_void_p()
        if path is not None:
            check(self.lib.tp_genome_ingest_file(self._h, _ip(cb), cb.size, os.fsencode(path), ord(sep), int(index_base),
                                                 ctypes.byref(h)))
        else:
            b1 = np.ascontiguousarray(bin1, dtype=np.int32)
            b2 = np.ascontiguousarray(bin2, dtype=np.int32)
            v = np.ascontiguousarray(count, dtype=np.float64)
            if not (b1.ndim == 1 and b1.shape == b2.shape == v.shape):
                raise ValueError("bin1, bin2, count: equal-length vectors expected")
            check(self.lib.tp_genome_ingest(self._h, _ip(cb), cb.size, _ip(b1), _ip(b2), _dp(v), b1.size, int(index_base),
                                            ctypes.byref(h)))
        return Genome(self, h, cb)

    def call_genome(self, genome, chroms=None, max_pcs=200, min_clusters=2, bad_frac=0.01, inflight=8, tables=True,
                    centromere_search=False, centromere_fix=False):
        """tp_call_genome: one call per selected chromosome (0-based indices, default all), results in that order as
        call_batch returns them (a failed call's entry is the TadpoleError), with centromere_search too."""
        sel = np.arange(genome.chrom_bins.size, dtype=np.int32) if chroms is None else np.ascontiguousarray(chroms, dtype=np.int32)
        h = c_void_p()
        tables = bool(tables or centromere_search)
        check(self.lib.tp_call_genome(self._h, genome._h, _ip(sel), int(sel.size), int(max_pcs), int(min_clusters),
                                      float(bad_frac), int(inflight), int(tables), _centromere(centromere_search, centromere_fix),
                                      ctypes.byref(h)))
        return self._batch_results(h, int(sel.size), tables)

    def recall(self, nf, max_pcs=200, min_clusters=2):
        """tp_recall: the n_pcs sweep and the selection again on the PC scores resident in the context."""
        k, npcs, ncl, maxlev = c_int(0), c_int(0), c_int(0), c_int(0)
        seq = np.zeros(nf - 1)
        check(self.lib.tp_recall(self._h, int(max_pcs), int(min_clusters), ctypes.byref(k), ctypes.byref(npcs),
                                 ctypes.byref(ncl), ctypes.byref(maxlev), _dp(seq)))
        return dict(nf=nf, k=k.value, n_pcs=npcs.value, n_clusters=ncl.value,
                    scores=self._sweep_scores(k.value, maxlev.value), seqdist=seq)

    # ---- stage 6 ----
    def difft_batch(self, lx, ly):
        lx = np.ascontiguousarray(lx, dtype=np.int32)
        ly = np.ascontiguousarray(ly, dtype=np.int32)
        assert lx.shape == ly.shape and lx.ndim == 2
        out = np.empty(lx.shape, dtype=np.float64)
        check(self.lib.tp_difft_batch(self._h, lx.ctypes.data, ly.ctypes.data, lx.shape[1], lx.shape[0], 0,
                                      out.ctypes.data))
        return out

    def difft_null(self, labels_x, ntads, nperm, pad_left=0, pad_right=0, bad_positions=None, seed=0,
                   want_curves=True, want_labels=False):
        """tp_difft_null: nperm random partitions drawn on the device, each scored against labels_x.
        Returns dict(borders [nperm, ntads-1], totals [nperm], curves [nperm, L] or None, labels or None)."""
        lx = np.ascontiguousarray(labels_x, dtype=np.int32)
        L = lx.size
        bad = np.ascontiguousarray(bad_positions if bad_positions is not None else [], dtype=np.int32)
        borders = np.empty((nperm, max(ntads - 1, 0)), dtype=np.int32)
        totals = np.empty(nperm)
        curves = np.empty((nperm, L)) if want_curves else None
        labels = np.empty((nperm, L), dtype=np.int32) if want_labels else None
        check(self.lib.tp_difft_null(self._h, lx.ctypes.data, L, int(pad_left), int(pad_right), int(ntads),
                                     bad.ctypes.data if bad.size else None, int(bad.size), int(seed) & (2 ** 64 - 1), int(nperm),
                                     borders.ctypes.data if borders.size else None,
                                     labels.ctypes.data if want_labels else None,
                                     curves.ctypes.data if want_curves else None, totals.ctypes.data))
        return dict(borders=borders, totals=totals, curves=curves, labels=labels)

    def difft_batch_dev(self, lx_ptr, ly_ptr, L, npairs, out_ptr):
        check(self.lib.tp_difft_batch(self._h, int(lx_ptr), int(ly_ptr), int(L), int(npairs), 1, int(out_ptr)))


class Genome:
    """Handle on the per-chromosome buckets of a genome-wide pixel list (tp_genome), held on its context's device."""

    def __init__(self, ctx, h, chrom_bins):
        self.lib, self.ctx, self._h, self.chrom_bins = ctx.lib, ctx, h, chrom_bins

    def stats(self):
        """(cis pixels per chromosome, trans pixels, pixels below the diagonal)"""
        cis = np.zeros(self.chrom_bins.size, dtype=np.uint64)
        trans, below = ctypes.c_ulonglong(0), ctypes.c_ulonglong(0)
        check(self.lib.tp_genome_stats(self._h, cis.ctypes.data_as(POINTER(ctypes.c_ulonglong)), ctypes.byref(trans),
                                       ctypes.byref(below)))
        return cis.astype(np.int64), int(trans.value), int(below.value)

    def matrix(self, chrom):
        """The dense upper-triangle matrix of chromosome `chrom` (0-based) as the calls see it (tp_genome_matrix)."""
        n = int(self.chrom_bins[chrom])
        out = np.empty((n, n))
        check(self.lib.tp_genome_matrix(self.ctx._h, self._h, int(chrom), _dp(out)))
        return out

    def close(self):
        if getattr(self, "_h", None):
            self.lib.tp_genome_free(self._h)
            self._h = c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def parse_field(text):
    """tp_test_parse_field (host-only hook): (status, value) of one field as the device parser converts it."""
    lib = load()
    b = text.encode() if isinstance(text, str) else bytes(text)
    out = c_double(0.0)
    st = lib.tp_test_parse_field(b, len(b), ctypes.byref(out))
    return st, out.value


def find_groups(seqdist):
    """tp_find_groups: hclust merge matrix [n-1, 2] (R convention) of a chclust dendrogram (rioja's .find.groups rule)."""
    lib = load()
    x = np.ascontiguousarray(seqdist, dtype=np.float64)
    out = np.zeros((2, x.size), dtype=np.int32)          # column-major n1 x 2
    check(lib.tp_find_groups(_dp(x), x.size, _ip(out)))
    return out.T.astype(np.int64)


def assemble(seqdist, n_clusters, names, bad):
    """tp_assemble: start/end table (1-based) and fixed labels for one hierarchical level."""
    lib = load()
    seqdist = np.ascontiguousarray(seqdist, dtype=np.float64)
    names = np.ascontiguousarray(names, dtype=np.int32)
    nf = names.size
    nbad = -1 if bad is None else len(bad)
    badarr = np.ascontiguousarray(bad if bad is not None else [], dtype=np.int32)
    cap = n_clusters + max(nbad, 0) + 2
    start = np.zeros(cap, dtype=np.int32)
    end = np.zeros(cap, dtype=np.int32)
    labels = np.zeros(nf + max(nbad, 0), dtype=np.int32)
    nrows = c_int(0)
    check(lib.tp_assemble(_dp(seqdist), nf, int(n_clusters), _ip(names), _ip(badarr), nbad, _ip(start), _ip(end),
                          ctypes.byref(nrows), _ip(labels)))
    return np.stack([start[:nrows.value], end[:nrows.value]], axis=1).astype(np.int64), labels


def centromere_split(bad, fix=False):
    """tp_centromere_split (host only): load_mat's split of the bad flags at the longest bad stretch (R/TADpole.R:58-86).
    Returns (split, (cs, ce) or None when there is no bad bin, (keep_p, bad_p), (keep_q, bad_q)): keep 0-based, bad
    columns original 1-based or None (NULL); the arms are None when split is False."""
    lib = load()
    b = np.ascontiguousarray(bad, dtype=np.uint8)
    n = b.size
    bufs = [np.zeros(max(n, 1), np.int32) for _ in range(4)]
    v = [c_int(0) for _ in range(7)]
    sp, cs, ce, nkp, nbp, nkq, nbq = v
    check(lib.tp_centromere_split(b.ctypes.data_as(POINTER(c_uint8)), n, int(bool(fix)), ctypes.byref(sp), ctypes.byref(cs),
                                  ctypes.byref(ce), _ip(bufs[0]), ctypes.byref(nkp), _ip(bufs[1]), ctypes.byref(nbp),
                                  _ip(bufs[2]), ctypes.byref(nkq), _ip(bufs[3]), ctypes.byref(nbq)))
    span = (cs.value, ce.value) if cs.value else None
    if not sp.value:
        return False, span, None, None
    arm = lambda k, nk, bb, nb: (k[:nk.value].copy(), bb[:nb.value].copy() if nb.value >= 0 else None)
    return True, span, arm(bufs[0], nkp, bufs[1], nbp), arm(bufs[2], nkq, bufs[3], nbq)


def assemble_levels(seqdist, levels, names, bad):
    """tp_assemble_levels: {level: [rows, 2] start/end table (1-based)} for many hierarchical levels at once."""
    lib = load()
    seqdist = np.ascontiguousarray(seqdist, dtype=np.float64)
    names = np.ascontiguousarray(names, dtype=np.int32)
    levels = np.ascontiguousarray(levels, dtype=np.int32)
    nf = names.size
    nbad = -1 if bad is None else len(bad)
    badarr = np.ascontiguousarray(bad if bad is not None else [], dtype=np.int32)
    cap = int(levels.sum()) + levels.size * (max(nbad, 0) + 2)
    start = np.zeros(max(cap, 1), dtype=np.int32)
    end = np.zeros(max(cap, 1), dtype=np.int32)
    off = np.zeros(levels.size + 1, dtype=np.int32)
    check(lib.tp_assemble_levels(_dp(seqdist), nf, _ip(levels), int(levels.size), _ip(names), _ip(badarr), nbad,
                                 _ip(start), _ip(end), _ip(off)))
    tab = np.stack([start[: off[-1]], end[: off[-1]]], axis=1).astype(np.int64)
    return {int(k): tab[off[i]: off[i + 1]] for i, k in enumerate(levels)}
