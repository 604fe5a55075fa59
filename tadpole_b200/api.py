"""Host-side mirror of the reference's R API (NAMESPACE:3-8) over the C ABI.

    TADpole(mat_file, max_pcs=200, min_clusters=2, bad_frac=0.01, chr, start, end, resol,
            centromere_search=False)                                  R/TADpole.R:344
    load_mat(mat_file, chr, start, end, resol, bad_frac=0.01, centromere_search=False)   :15
    diffT(bed_x, bed_y)                                               R/DiffT.R:19
    random_bed(bed, bad_columns=None)                                 R/DiffT.R:61

R is not available in the build image, so the host language is Python (the reference is an
interpreted-language package; this file plays the role of R/*.R in INTEGRATION.md).  Same
argument names, defaults, messages and error behaviour; chr/start/end/resol are accepted and
ignored exactly as in the reference, where they only label plots.  All numeric work happens in
libtadpole_b200 on the GPU; this file only does what the R wrapper would do: read the file,
integer bookkeeping of bad columns / centromere, and packing the result object.
"""
from __future__ import annotations

import sys

import numpy as np

from . import _lib
from .hclust import Dendro

__all__ = ["TADpole", "load_mat", "diffT", "diffT_null", "random_bed", "random_bed_batch", "bin_index", "Tadpole", "LoadedMatrix", "get_context"]

_CTX = {}
QUIET = False


def message(text):
    """R's message(): diagnostics on stderr."""
    if not QUIET:
        print(text, file=sys.stderr)


def get_context(device=0):
    ctx = _CTX.get(device)
    if ctx is None:
        ctx = _CTX[device] = _lib.Context(device)
    return ctx


class SparseCounts:
    """A contact matrix given by its non-zero upper-triangle pixels, the layout of `cooler dump` / HiC-Pro: either
    SparseCounts(bin1, bin2, count, n_bins) from arrays (a scipy.sparse matrix goes through from_scipy) or
    SparseCounts(path=..., n_bins=None) for a three-column text file.  Accepted wherever a matrix file is: the dense
    matrix the reference would have read (R/TADpole.R:17) is built on the GPU, only the pixels cross PCIe."""

    def __init__(self, bin1=None, bin2=None, count=None, n_bins=None, index_base=0, path=None, sep="\t"):
        if path is None:
            if bin1 is None or bin2 is None or count is None or n_bins is None:
                raise ValueError("SparseCounts needs bin1, bin2, count and n_bins, or a path")
        self.bin1, self.bin2, self.count = bin1, bin2, count
        self.n_bins, self.index_base, self.path, self.sep = n_bins, int(index_base), path, sep

    @classmethod
    def from_scipy(cls, m):
        m = m.tocoo()
        if m.shape[0] != m.shape[1]:
            raise ValueError("square matrix expected")
        return cls(m.row, m.col, m.data, m.shape[0])

    def _ingest(self, ctx):
        return ctx.ingest_coo(self.bin1, self.bin2, self.count, self.n_bins, self.index_base, self.path, self.sep)


def read_matrix(mat_file, ctx=None):
    """bigmemory::read.big.matrix(mat_file, type='double', sep='\\t') (R/TADpole.R:17): header-less
    tab-separated numeric matrix, as a numpy array.  The text is uploaded and parsed on the GPU
    (csrc/ingest.cu); an in-memory square array is passed through."""
    if isinstance(mat_file, np.ndarray):
        return mat_file
    ctx = ctx or get_context()
    if isinstance(mat_file, SparseCounts):
        _, n = mat_file._ingest(ctx)
    else:
        _, n = ctx.ingest_tsv(mat_file)
    return ctx.get_ingested(n)


def _matrix_args(mat_file, ctx):
    """Keyword arguments that hand the input matrix to Context.filter / Context.call: an in-memory array as it is,
    a file through the device-side parser -- the FP64 matrix of a file never exists on the host."""
    if isinstance(mat_file, np.ndarray):
        return dict(mat=mat_file)
    if isinstance(mat_file, SparseCounts):
        ptr, n = mat_file._ingest(ctx)
        return dict(mat=None, device_ptr=ptr, n=n, colmajor=0)
    ptr, n = ctx.ingest_tsv(mat_file)
    return dict(mat=None, device_ptr=ptr, n=n, colmajor=0)


class LoadedMatrix:
    """What load_mat returns: the filtered matrix with its 'bad_columns' attribute
    (R/TADpole.R:88-90), or, when the chromosome was split, the list(p, q, centromere)
    (R/TADpole.R:85).  The matrix itself stays on the GPU; to_numpy() fetches it."""

    def __init__(self, ctx, n_bins, keep, bad_columns, split=None):
        self._ctx = ctx
        self.n_bins = n_bins
        self.keep = keep                    # 0-based original indices of kept bins
        self.names = None if keep is None else keep + 1
        self.bad_columns = bad_columns      # R: character names for the whole matrix, numeric for arms
        self.p = self.q = self.centromere = None
        if split is not None:
            self.p, self.q, self.centromere = split

    @property
    def is_split(self):
        return self.p is not None

    def to_numpy(self):
        self._ctx.compact(self.keep)
        return self._ctx.get_filtered(self.keep.size)

    @property
    def shape(self):
        return (self.keep.size, self.keep.size)


def _split_centromere(bad, fix=False):
    """R/TADpole.R:58-86 on the bad flags (tp_centromere_split).  Returns None when the matrix is not split.
    fix=True removes the q-arm bad columns by their position within the arm (quirk Q3 repaired)."""
    split, span, arm_p, arm_q = _lib.centromere_split(bad, fix)
    cen = None if span is None else np.arange(span[0], span[1] + 1)
    _messages_split(cen, split)
    if not split:
        return None
    as64 = lambda a: None if a is None else a.astype(np.int64)
    return (arm_p[0].astype(np.int64), as64(arm_p[1])), (arm_q[0].astype(np.int64), as64(arm_q[1])), cen


def _messages_split(cen, split):
    """load_mat's messages about the centromere cen = cs..ce (R/TADpole.R:64-70); None: no bad bin, nothing is said."""
    if cen is None:
        return
    message(f"centromere position: {cen[0]} {cen[-1]}")
    if not split:
        message("longest stretch of bad rows/columns at the ends, not splitting the matrix.")


def _messages_bad(bad):
    message(f"{int(bad.sum())} bad columns found at position(s):")
    message(" ".join(str(i) for i in np.flatnonzero(bad) + 1))


# TADpole(centromere_search=TRUE) on a matrix that load_mat does not split: R/TADpole.R:356-359 then does
# mat$centromer / mat[['p']] on a plain matrix and errors (quirk Q4)
NOSPLIT_MESSAGE = ("centromere_search=TRUE but load_mat did not split the matrix "
                   "(no bad columns, or the longest bad stretch touches an end); the reference errors here")


def load_mat(mat_file, chr=None, start=None, end=None, resol=None, bad_frac=0.01, centromere_search=False,
             ctx=None, centromere_fix=False):
    """Load a Hi-C matrix, flag bad columns, optionally split at the centromere (R/TADpole.R:15-92).
    Plots (R/TADpole.R:24-53) are out of scope.  centromere_fix: see TADpole()."""
    ctx = ctx or get_context()
    bad, _, _ = ctx.filter(bad_frac=bad_frac, **_matrix_args(mat_file, ctx))
    return _loaded_from_flags(ctx, bad, centromere_search, centromere_fix)


def _loaded_from_flags(ctx, bad, centromere_search, fix=False):
    n = bad.size
    _messages_bad(bad)
    if bad.any() and centromere_search:
        split = _split_centromere(bad, fix)
        if split is not None:
            (kp, bp), (kq, bq), cen = split
            return LoadedMatrix(ctx, n, None, None, split=(LoadedMatrix(ctx, n, kp.astype(np.int32), bp),
                                                           LoadedMatrix(ctx, n, kq.astype(np.int32), bq), cen))
    keep = np.flatnonzero(~bad).astype(np.int32)
    return LoadedMatrix(ctx, n, keep, np.flatnonzero(bad) + 1)


class _Obj(dict):
    """R list semantics: x$name and x[['name']]."""
    __getattr__ = dict.get

    def __setattr__(self, k, v):
        self[k] = v


class Tadpole(_Obj):
    """The returned 'tadpole' object (R/TADpole.R:463-468; arms :354,376-378,407,442):
    n_pcs, optimal_n_clusters, dendro, clusters (dict keyed by str(k) -> [rows, 2] start/end),
    scores; with centromere_search: p, q (each n_pcs, optimal_n_clusters, dendro, cluster) and
    merging_arms.

    Beyond the reference: a whole-chromosome object is also a handle on the pipeline state that stays in HBM
    (PC scores, all k dendrograms): recall() repeats only the n_pcs sweep for another max_pcs / min_clusters, and
    dendro_for() returns the dendrogram of any candidate number of PCs (what CH_map / plot_hierarchy browse),
    as long as the context has not been used for another matrix since.  The objects of TADpole_batch / TADpole_genome
    with resident=True are such handles too, on stores of their own that no later call replaces; there recall() of a
    centromere_search result recalls both arms, and each arm has dendro_for()."""

    def _resident(self):
        h = object.__getattribute__(self, "__dict__").get("_handle")
        if h is None:
            raise RuntimeError("this tadpole object carries no device handle (centromere_search results do not)")
        if "batch" in h:
            return h
        if h["ctx"].generation != h["generation"]:
            raise RuntimeError("the GPU context has been used for another matrix since this call; its resident state is gone")
        return h

    def recall(self, max_pcs=200, min_clusters=2):
        """TADpole() again on the same matrix with another max_pcs (<= the one computed) / min_clusters, from the
        resident PC scores: same result as a fresh call, without load_mat, cor and prcomp."""
        h = self._resident()
        if "batch" in h:
            res, store = h["batch"].recall([h["item"]], max_pcs=max_pcs, min_clusters=min_clusters, inflight=1)
            return _recalled_object(res[0], store, 0, h["centromere_fix"])
        res = h["ctx"].recall(h["nf"], max_pcs=max_pcs, min_clusters=min_clusters)
        res["bad"] = h["bad"]
        return _tadpole_from_result(res, h["ctx"])       # the sweep state was replaced: this object is now stale

    def dendro_for(self, n_pcs):
        """chclust dendrogram of the candidate that clusters on the first n_pcs PCs (R/TADpole.R:108)."""
        h = self._resident()
        if "batch" in h:
            if "names" not in h:
                raise ValueError("a centromere_search result has no dendrogram of its own: use dendro_for of its arms p / q")
            return Dendro(h["batch"].dendro(h["item"], h["part"], int(n_pcs) - 1, h["nf"]), labels=h["names"])
        seq, _ = h["ctx"].dendro(int(n_pcs) - 1, h["nf"])
        return Dendro(seq, labels=h["names"])


class ResidentArm(_Obj):
    """An arm (p or q) of a centromere_search result of TADpole_batch / TADpole_genome with resident=True: the arm
    object of TADpole(centromere_search=True) plus dendro_for() of any candidate number of PCs."""
    _resident = Tadpole._resident
    dendro_for = Tadpole.dendro_for


def _recalled_object(res, store, i, centromere_fix):
    """The object of item i of a recall (an exception is raised)."""
    if isinstance(res, Exception):
        raise res
    from .batch import _tadpole_from_batch_item
    return _tadpole_from_batch_item(res, centromere_fix, (store, i))


def _levels_table(res, names, bad_cols):
    """for (k in which(!is.na(scores[n_PCs, ]))) ... (R/TADpole.R:381-408,470-497)."""
    row = res["scores"][res["n_pcs"] - 1]
    levels = np.flatnonzero(~np.isnan(row)) + 1
    tabs = _lib.assemble_levels(res["seqdist"], levels, names, bad_cols)
    return {str(int(k)): tabs[int(k)] for k in levels}


def _messages_optimal(res):
    message(f"Optimal number of PCs: {res['n_pcs']}")
    message(f"Optimal number of clusters: {res['n_clusters']}")


def _tadpole_from_result(res, ctx):
    """Packs the whole-chromosome result (R/TADpole.R:463-497) and attaches the device handle."""
    bad = res["bad"]
    _messages_optimal(res)
    names = (np.flatnonzero(~bad) + 1).astype(np.int32)
    bad_cols = (np.flatnonzero(bad) + 1).astype(np.int32)
    tp = Tadpole()
    tp.n_pcs = res["n_pcs"]
    tp.optimal_n_clusters = res["n_clusters"]
    tp.dendro = Dendro(res["seqdist"], labels=names)
    tp.clusters = _levels_table(res, names, bad_cols)
    tp.scores = res["scores"]
    object.__getattribute__(tp, "__dict__")["_handle"] = dict(ctx=ctx, generation=ctx.generation, nf=int(names.size),
                                                             names=names, bad=bad)
    return tp


def TADpole(mat_file, max_pcs=200, min_clusters=2, bad_frac=0.01, chr=None, start=None, end=None, resol=None,
            centromere_search=False, ctx=None, dist=None, centromere_fix=False):
    """Call hierarchical TADs (R/TADpole.R:344-501).

    centromere_fix (default False = the reference's behaviour, quirks included): opt-in repairs of the
    centromere_search path (SURVEY.md quirks Q3, Q4 and the TODO at R/TADpole.R:304): the q-arm's bad columns are
    removed by their position within the arm; a chromosome that load_mat does not split (no bad columns, or the
    longest bad stretch touches an end) is processed whole instead of raising; and every arm also carries its
    `scores` matrix and the `clusters` spelling, so that CH_map-style consumers work on arms.

    dist: a sharding.DistEnv when the call is spread over several GPUs (one process per GPU, every rank calls with
    the same matrix and gets the same object back).  Without centromere_search the whole job works on the one
    matrix; with it the ranks split between the two arms, as the arms are independent (R/TADpole.R:357)."""
    ctx = ctx or get_context()
    mat = _matrix_args(mat_file, ctx)
    if not centromere_search:
        res = ctx.call(max_pcs=max_pcs, min_clusters=min_clusters, bad_frac=bad_frac, **mat)
        _messages_bad(res["bad"])
        return _tadpole_from_result(res, ctx)

    bad, _, _ = ctx.filter(bad_frac=bad_frac, **mat)
    lm = _loaded_from_flags(ctx, bad, True, centromere_fix)
    if not lm.is_split and centromere_fix:
        res = ctx.call_arm(lm.keep, max_pcs=max_pcs, min_clusters=min_clusters)
        res["bad"] = bad
        return _tadpole_from_result(res, ctx)
    if not lm.is_split:
        raise ValueError(NOSPLIT_MESSAGE)
    arm_res = {}
    if dist is not None and dist.world > 1:
        # every rank runs its own arm (collectively with the other ranks of that arm); the small result summaries
        # are then exchanged so that every rank assembles the same object
        dist.select_arm()
        mine = ctx.call_arm(getattr(lm, dist.my_arm).keep, max_pcs=max_pcs, min_clusters=min_clusters)
        dist.select_world()
        every = dist.exchange((dist.my_arm, mine))
        for arm in ("p", "q"):
            arm_res[arm] = every[dist.arms[arm][0]][1]
    else:
        # tp_call_arms: on a multi-device context the two halves of the devices work on the two arms at the same time
        arm_res["p"], arm_res["q"] = ctx.call_arms(lm.p.keep, lm.q.keep, max_pcs=max_pcs, min_clusters=min_clusters)
    tp = Tadpole()
    labels = []
    for arm in ("p", "q"):
        la = getattr(lm, arm)
        names = la.names.astype(np.int32)
        tp[arm] = _arm_object(arm, arm_res[arm], names, _levels_table(arm_res[arm], names, la.bad_columns), centromere_fix)
        labels.append(_arm_labels(arm_res[arm], names, la.bad_columns))
    tp.merging_arms = _merging_arms(labels[0], labels[1], len(lm.centromere))
    return tp


def _arm_object(arm, res, names, tables, centromere_fix, cls=_Obj):
    """One arm of a centromere_search result (R/TADpole.R:376-408): n_pcs, optimal_n_clusters, dendro and the per-level
    tables as `cluster`; with centromere_fix also `clusters` and `scores`."""
    message(f"Processing arm {arm}")
    _messages_optimal(res)
    a = cls()
    a.n_pcs = res["n_pcs"]
    a.optimal_n_clusters = res["n_clusters"]
    a.dendro = Dendro(res["seqdist"], labels=names)
    a.cluster = tables
    if centromere_fix:
        a.clusters, a.scores = a.cluster, res["scores"]
    return a


def _arm_labels(res, names, bad_columns):
    """The optimal level of an arm, bad columns re-inserted, fix_values applied (R/TADpole.R:411-431)."""
    bad_for_merge = bad_columns if bad_columns is not None else np.zeros(0, np.int32)
    return _lib.assemble(res["seqdist"], res["n_clusters"], names, bad_for_merge)[1]


def _merging_arms(labels_p, labels_q, ncen):
    """c(p labels, centromere zeros, q labels) -> start / end of its non-zero runs (R/TADpole.R:432-442)."""
    allv = np.concatenate([labels_p.astype(np.int64), np.zeros(ncen, np.int64), labels_q.astype(np.int64)])
    brk = np.flatnonzero(allv[1:] != allv[:-1]) + 1
    starts = np.concatenate(([0], brk))
    ends = np.concatenate((brk, [allv.size]))
    keep = allv[starts] != 0
    return np.stack([starts[keep] + 1, ends[keep]], axis=1)


# ---- diffT -------------------------------------------------------------------------------------------

def _bed_rows(bed):
    """Accepts a [T,3] table (chrom, start, end), a [T,2] array (start, end) or a path."""
    if isinstance(bed, str):
        rows = []
        with open(bed) as fh:
            for line in fh:
                f = line.split()
                if len(f) >= 3:
                    rows.append((int(f[1]), int(f[2])))
        return np.array(rows, dtype=np.int64)
    if hasattr(bed, "iloc"):
        return bed.iloc[:, 1:3].to_numpy(dtype=np.int64)
    arr = np.asarray(bed)
    if arr.ndim == 2 and arr.shape[1] >= 3:
        return arr[:, 1:3].astype(np.int64)
    return arr.astype(np.int64)


def bin_index(bed, size):
    """bin_index (R/DiffT.R:1-9): TAD label per bin, offsets relative to the first row's start,
    later rows overwrite earlier ones, uncovered bins stay 0."""
    bed = np.asarray(bed, dtype=np.int64)
    tad = np.zeros(int(size), dtype=np.int32)
    off = bed[0, 0]
    for t in range(bed.shape[0]):
        lo, hi = sorted((int(bed[t, 0] - off), int(bed[t, 1] - off)))      # seq(a, b) runs downwards when a > b
        tad[max(lo, 0): hi + 1] = t + 1                                     # tad_index[0] <- x is a no-op in R
    return tad


def _difft_labels(bed_x, bed_y):
    bx, by = _bed_rows(bed_x), _bed_rows(bed_y)
    if bx.shape[0] != by.shape[0]:
        raise ValueError("Both calls must have the same number of TADs.")       # R/DiffT.R:20
    sx, sy, ex, ey = bx[0, 0], by[0, 0], bx[-1, 1], by[-1, 1]
    tx = bin_index(bx, ex - sx + 1)
    ty = bin_index(by, ey - sy + 1)
    tx = np.concatenate((np.ones(max(0, sx - sy), np.int32), tx, np.full(max(0, ey - ex), tx.max(), np.int32)))
    ty = np.concatenate((np.ones(max(0, sy - sx), np.int32), ty, np.full(max(0, ex - ey), ty.max(), np.int32)))
    if tx.size != ty.size:
        raise AssertionError("length(tad_x) == length(tad_y) is not TRUE")       # stopifnot, R/DiffT.R:38
    return tx, ty


def diffT(bed_x, bed_y, ctx=None):
    """diffT score between two TAD calls (R/DiffT.R:19-50)."""
    ctx = ctx or get_context()
    tx, ty = _difft_labels(bed_x, bed_y)
    return ctx.difft_batch(tx[None, :], ty[None, :])[0]


def diffT_batch(labels_x, labels_y, ctx=None):
    """Many comparisons at once on padded label vectors ([npairs, L] int32 each)."""
    ctx = ctx or get_context()
    return ctx.difft_batch(labels_x, labels_y)


def random_bed(bed, bad_columns=None, rng=None):
    """Random partition with the same number of TADs (R/DiffT.R:61-73).  Uses numpy's RNG, so
    draws differ from R's sample(); the distribution is the same."""
    rows = _bed_rows(bed)
    rng = rng or np.random.default_rng()
    start, end = int(rows[0, 0]), int(rows[-1, 1])
    size = end - start + 1
    bins = np.arange(start, end + 1)
    if bad_columns is not None:
        bins = np.delete(bins, np.asarray(bad_columns, dtype=np.int64) - 1)
    borders = np.sort(rng.choice(bins[1:], size=rows.shape[0] - 1, replace=False))
    return np.stack([np.concatenate(([start], borders - 1)), np.concatenate((borders - 2, [start + size - 1]))], axis=1)


def _bad_positions(bad_columns):
    return None if bad_columns is None else np.asarray(bad_columns, dtype=np.int64).astype(np.int32)


def _beds_from_borders(rows, borders):
    """data.frame(start = c(start, borders - 1), end = c(borders - 2, start + size - 1)) (R/DiffT.R:70-72)."""
    start, end = int(rows[0, 0]), int(rows[-1, 1])
    b = borders.astype(np.int64) + start
    n = b.shape[0]
    return np.stack([np.concatenate((np.full((n, 1), start), b - 1), axis=1),
                     np.concatenate((b - 2, np.full((n, 1), end)), axis=1)], axis=2)


def random_bed_batch(bed, n, bad_columns=None, seed=0, ctx=None):
    """n draws of random_bed(bed, bad_columns) (R/DiffT.R:61-73) generated on the GPU: [n, T, 2] (start, end)."""
    ctx = ctx or get_context()
    rows = _bed_rows(bed)
    size = int(rows[-1, 1] - rows[0, 0] + 1)
    res = ctx.difft_null(np.ones(size, np.int32), rows.shape[0], n, bad_positions=_bad_positions(bad_columns), seed=seed,
                         want_curves=False)
    return _beds_from_borders(rows, res["borders"])


def diffT_null(bed_x, bed_y=None, nperm=1000, bad_columns=None, seed=0, ctx=None):
    """The diffT null distribution: diffT(bed_x, random_bed(bed_y, bad_columns)) for nperm random partitions
    (R/DiffT.R:19-50 and :61-73), partitions drawn and scored on the GPU.  bed_y defaults to bed_x (random
    partitions with the observed call's own extent and TAD count).  Returns an object with `curves` [nperm, L],
    `totals` [nperm] (un-normalised total score) and `beds` [nperm, T, 2]."""
    ctx = ctx or get_context()
    bx = _bed_rows(bed_x)
    by = bx if bed_y is None else _bed_rows(bed_y)
    if bx.shape[0] != by.shape[0]:
        raise ValueError("Both calls must have the same number of TADs.")       # R/DiffT.R:20
    sx, sy, ex, ey = int(bx[0, 0]), int(by[0, 0]), int(bx[-1, 1]), int(by[-1, 1])
    tx = bin_index(bx, ex - sx + 1)
    tx = np.concatenate((np.ones(max(0, sx - sy), np.int32), tx, np.full(max(0, ey - ex), tx.max(), np.int32)))
    res = ctx.difft_null(tx, by.shape[0], nperm, pad_left=max(0, sy - sx), pad_right=max(0, ex - ey),
                         bad_positions=_bad_positions(bad_columns), seed=seed)
    out = _Obj()
    out.curves, out.totals, out.beds = res["curves"], res["totals"], _beds_from_borders(by, res["borders"])
    return out
