"""Several independent TADpole() calls in flight on the GPUs of one box.

The reference processes one chromosome per call; genome-wide use loops over chromosomes (and the foreach workers of
R/TADpole.R:103-104 only parallelise inside one call).  On a B200 a single 2 000-bin call keeps most of the 148 SMs
idle, so independent calls overlap almost perfectly when each has its own context (own stream, own device buffers).
The overlap is the library's job (tp_call_batch, csrc/group.cu): library-owned host threads keep `streams` calls in
flight per device, over every device of the context, and also build the per-level start / end tables; the caller --
one Python thread here, one R thread behind .Call -- just waits.  Results are the same objects, in the same order, as
calling TADpole() on each matrix in turn.

TADpole_genome() starts from what Hi-C pipelines write for a whole genome: one pixel list with global bin ids (HiC-Pro
*.matrix, cooler dump -t pixels) and its bin table.  The pixels are split by chromosome on the GPU (tp_genome_ingest),
and each chromosome's dense matrix exists only in HBM, only while its call runs (tp_call_genome).
"""
from __future__ import annotations

import os

import numpy as np

from . import _lib
from .api import (NOSPLIT_MESSAGE, Tadpole, _arm_object, _merging_arms, _messages_bad, _messages_optimal, _messages_split,
                  message, read_matrix)
from .hclust import Dendro

__all__ = ["ContextPool", "TADpole_batch", "GenomePixels", "TADpole_genome", "read_bins"]


class ContextPool:
    """A context whose batch calls keep `streams` calls in flight per device (the pool of per-call contexts lives in the
    library and is reused from batch to batch).  device: one index or a list of devices."""

    def __init__(self, device=0, streams=4):
        self.device = device
        self.streams = int(streams)
        self.ctx = _lib.Context(device)

    def close(self):
        self.ctx.close()


def _tadpole_from_batch_item(res, centromere_fix=False):
    """The object and the messages TADpole() gives for one item of a batch; a centromere_search item
    (call_batch(centromere_search=True)) as TADpole(centromere_search=True, centromere_fix=centromere_fix) gives it."""
    bad = res["bad"]
    _messages_bad(bad)
    if "split" in res:
        _messages_split(res["centromere"], res["split"])
    if res.get("split"):
        tp = Tadpole()
        for arm in ("p", "q"):
            a = res[arm]
            tp[arm] = _arm_object(arm, a, (a["keep"] + 1).astype(np.int32), {str(k): t for k, t in a["tables"].items()},
                                  centromere_fix)
        tp.merging_arms = _merging_arms(res["p"]["labels"], res["q"]["labels"], res["centromere"].size)
        return tp
    _messages_optimal(res)
    tp = Tadpole()
    tp.n_pcs = res["n_pcs"]
    tp.optimal_n_clusters = res["n_clusters"]
    tp.dendro = Dendro(res["seqdist"], labels=(np.flatnonzero(~bad) + 1).astype(np.int32))
    tp.clusters = {str(k): t for k, t in res["tables"].items()}
    tp.scores = res["scores"]
    return tp                          # no device handle: the per-call contexts are reused by the next call


def _failed_item(err):
    """What TADpole(centromere_search=True) says and raises for a matrix whose batch item failed: load_mat's messages when
    the filter ran, then the ValueError of an unsplit matrix (quirk Q4) or the library's error."""
    if getattr(err, "split", -1) >= 0:
        _messages_bad(err.bad)
        _messages_split(err.centromere, err.split)
    return ValueError(NOSPLIT_MESSAGE) if err.code == _lib.TP_ERR_NOSPLIT else err


def TADpole_batch(mat_files, max_pcs=200, min_clusters=2, bad_frac=0.01, centromere_search=False, pool=None,
                  device=0, streams=4, ctx=None, centromere_fix=False):
    """TADpole() on every matrix of `mat_files` (paths or arrays), `streams` calls in flight per GPU.  centromere_search
    (and centromere_fix, see TADpole()): every matrix is split at its centromere and both arms are called in the library's
    workers; the objects and messages are TADpole(centromere_search=True)'s, and the first matrix TADpole() would fail on
    raises its exception."""
    own = pool is None and ctx is None
    if ctx is None:
        pool = pool or ContextPool(device, streams)
        ctx, streams = pool.ctx, pool.streams
    try:
        mats = [read_matrix(m, ctx) for m in mat_files]
        res = ctx.call_batch(mats, max_pcs=max_pcs, min_clusters=min_clusters, bad_frac=bad_frac, inflight=streams,
                             centromere_search=centromere_search, centromere_fix=centromere_fix)
        if centromere_search:
            out = []
            for r in res:                   # messages in input order, up to the first matrix that fails
                if isinstance(r, Exception):
                    raise _failed_item(r)
                out.append(_tadpole_from_batch_item(r, centromere_fix))
            return out
        for r in res:
            if isinstance(r, Exception):
                raise r
        return [_tadpole_from_batch_item(r) for r in res]
    finally:
        if own:
            pool.close()


# ---- genome-wide input ----------------------------------------------------------------------------------------------

def _is_int(text):
    return text.strip().lstrip("+-").isdigit()


def _runs(names):
    """Chromosome names and bins per chromosome from the chromosome of every bin, in id order."""
    out = []
    for nm in names:
        nm = str(nm)
        if out and out[-1][0] == nm:
            out[-1][1] += 1
        else:
            out.append([nm, 1])
    return _checked([(nm, n) for nm, n in out])


def _checked(pairs):
    seen = set()
    for nm, n in pairs:
        if nm in seen:
            raise ValueError(f"chromosome {nm!r} reappears after another chromosome: the bins of a chromosome must be "
                             "contiguous in the bin table")
        if int(n) < 1:
            raise ValueError(f"chromosome {nm!r} has {n} bins")
        seen.add(nm)
    return [nm for nm, _ in pairs], np.array([int(n) for _, n in pairs], dtype=np.int32)


def read_bins(bins):
    """(chromosome names, bins per chromosome) of a bin table.  bins: the path of a bin table whose rows are the bins in
    id order and whose first column is the chromosome (HiC-Pro *_abs.bed; `cooler dump -t bins`, with or without its
    header line); a table whose first column is the chromosome of each bin (a pandas DataFrame, a 2-D array, or a 1-D
    sequence of names); or a list of (name, n_bins).  A chromosome that reappears after another one is a ValueError."""
    if isinstance(bins, (str, os.PathLike)):
        names = []
        with open(bins) as fh:
            for k, line in enumerate(fh):
                f = line.split()
                if not f:
                    continue
                if k == 0 and (f[0] == "chrom" or (len(f) >= 2 and not _is_int(f[1]))):
                    continue                                            # a header line
                names.append(f[0])
        return _runs(names)
    if hasattr(bins, "iloc"):
        return _runs(bins.iloc[:, 0].tolist())
    if isinstance(bins, (list, tuple)) and bins and isinstance(bins[0], (list, tuple)) and len(bins[0]) == 2 \
            and not isinstance(bins[0][1], str):
        return _checked([(str(nm), int(n)) for nm, n in bins])
    arr = np.asarray(bins, dtype=object)
    return _runs(arr[:, 0].tolist() if arr.ndim == 2 else arr.tolist())


class GenomePixels:
    """The contacts of a whole genome as one pixel list with global bin ids, the layout Hi-C pipelines write:
    GenomePixels(bin1, bin2, count, bins=..., index_base=0) from arrays, or GenomePixels(path=..., bins=..., index_base=1,
    sep="\\t") for a three-column text file (HiC-Pro *.matrix: 1-based; `cooler dump -t pixels`: 0-based, header line
    allowed).  bins: see read_bins.  Only the upper triangle of each chromosome counts; trans pixels are dropped."""

    def __init__(self, bin1=None, bin2=None, count=None, bins=None, index_base=None, path=None, sep="\t"):
        if bins is None:
            raise ValueError("GenomePixels needs the bin table (bins=)")
        if path is None and (bin1 is None or bin2 is None or count is None):
            raise ValueError("GenomePixels needs bin1, bin2 and count, or a path")
        self.names, self.chrom_bins = read_bins(bins)
        self.bin1, self.bin2, self.count, self.path, self.sep = bin1, bin2, count, path, sep
        self.index_base = int((1 if path is not None else 0) if index_base is None else index_base)

    def _ingest(self, ctx):
        return ctx.genome_ingest(self.chrom_bins, self.bin1, self.bin2, self.count, self.index_base, self.path, self.sep)


class GenomeResult(dict):
    """{chromosome name: Tadpole}; .failed {name: message of the library}; .stats dict(cis={name: pixels}, trans=,
    below=)."""
    failed: dict
    stats: dict


def TADpole_genome(pixels, chroms=None, max_pcs=200, min_clusters=2, bad_frac=0.01, ctx=None, device=0, streams=4,
                   centromere_search=False, centromere_fix=False):
    """TADpole() on every chromosome of a genome-wide pixel list (GenomePixels), `streams` calls in flight per GPU.
    Each chromosome's Tadpole is the one TADpole() returns for that chromosome's dense matrix (with centromere_search /
    centromere_fix as TADpole() takes them: p, q and merging_arms; a chromosome that does not split fails with
    TADpole()'s message unless centromere_fix).  Returns a GenomeResult in bin-table order, or in `chroms` order when
    chroms (a list of names) is given."""
    index = {nm: c for c, nm in enumerate(pixels.names)}
    sel = list(pixels.names) if chroms is None else [str(c) for c in chroms]
    unknown = [c for c in sel if c not in index]
    if unknown:
        raise ValueError(f"unknown chromosome(s) {unknown}: not in the bin table")
    own = ctx is None
    ctx = ctx or _lib.Context(device)
    try:
        g = pixels._ingest(ctx)
        try:
            cis, trans, below = g.stats()
            res = ctx.call_genome(g, [index[c] for c in sel], max_pcs=max_pcs, min_clusters=min_clusters, bad_frac=bad_frac,
                                  inflight=streams, centromere_search=centromere_search, centromere_fix=centromere_fix)
        finally:
            g.close()
    finally:
        if own:
            ctx.close()
    out = GenomeResult()
    out.failed = {}
    out.stats = dict(cis={nm: int(k) for nm, k in zip(pixels.names, cis)}, trans=trans, below=below)
    for nm, r in zip(sel, res):
        message(f"Processing chromosome {nm}")
        if isinstance(r, Exception):
            out.failed[nm] = NOSPLIT_MESSAGE if r.code == _lib.TP_ERR_NOSPLIT else str(r)
            continue
        out[nm] = _tadpole_from_batch_item(r, centromere_fix)
    return out
