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
and each chromosome's dense matrix exists only in HBM, only while its call runs (tp_call_genome).  GenomePairs starts one
step earlier, from the read-pair files themselves (4DN .pairs, HiC-Pro *.allValidPairs, Juicer merged_nodups.txt), binned
at any bin size on the GPU (tp_genome_ingest_pairs_file).
"""
from __future__ import annotations

import math
import os

import numpy as np

from . import _lib
from .api import (NOSPLIT_MESSAGE, ResidentArm, Tadpole, _Obj, _arm_object, _bed_rows, _difft_labels, _merging_arms,
                  _messages_bad, _messages_optimal, _messages_split, get_context, message, read_matrix)
from .hclust import Dendro

__all__ = ["ContextPool", "TADpole_batch", "GenomePixels", "GenomePairs", "LoadedGenome", "TADpole_genome", "read_bins",
           "read_chromsizes", "diffT_genome", "equal_depth"]


class ContextPool:
    """A context whose batch calls keep `streams` calls in flight per device (the pool of per-call contexts lives in the
    library and is reused from batch to batch).  device: one index or a list of devices."""

    def __init__(self, device=0, streams=4):
        self.device = device
        self.streams = int(streams)
        self.ctx = _lib.Context(device)

    def close(self):
        self.ctx.close()


def _handle(obj, resident, **kw):
    """Attach the device handle of item `resident` = (ResidentBatch, item) to obj."""
    object.__getattribute__(obj, "__dict__")["_handle"] = dict(batch=resident[0], item=resident[1], **kw)


def _tadpole_from_batch_item(res, centromere_fix=False, resident=None):
    """The object and the messages TADpole() gives for one item of a batch; a centromere_search item
    (call_batch(centromere_search=True)) as TADpole(centromere_search=True, centromere_fix=centromere_fix) gives it.
    resident: (ResidentBatch, item index) of a batch run with resident=True, which the object (and its arms) then keep
    as their device handle."""
    bad = res["bad"]
    _messages_bad(bad)
    if "split" in res:
        _messages_split(res["centromere"], res["split"])
    if res.get("split"):
        tp = Tadpole()
        for part, arm in enumerate(("p", "q")):
            a = res[arm]
            names = (a["keep"] + 1).astype(np.int32)
            tp[arm] = _arm_object(arm, a, names, {str(k): t for k, t in a["tables"].items()}, centromere_fix,
                                  ResidentArm if resident else _Obj)
            if resident:
                _handle(tp[arm], resident, part=part, nf=int(a["nf"]), names=names)
        tp.merging_arms = _merging_arms(res["p"]["labels"], res["q"]["labels"], res["centromere"].size)
        if resident:
            _handle(tp, resident, part=-1, centromere_fix=centromere_fix)
        return tp
    _messages_optimal(res)
    tp = Tadpole()
    names = (np.flatnonzero(~bad) + 1).astype(np.int32)
    tp.n_pcs = res["n_pcs"]
    tp.optimal_n_clusters = res["n_clusters"]
    tp.dendro = Dendro(res["seqdist"], labels=names)
    tp.clusters = {str(k): t for k, t in res["tables"].items()}
    tp.scores = res["scores"]
    if resident:
        _handle(tp, resident, part=-1, nf=int(names.size), names=names, centromere_fix=centromere_fix)
    # without resident no device handle: the per-call contexts are reused by the next call
    return tp


def _failed_item(err):
    """What TADpole(centromere_search=True) says and raises for a matrix whose batch item failed: load_mat's messages when
    the filter ran, then the ValueError of an unsplit matrix (quirk Q4) or the library's error."""
    if getattr(err, "split", -1) >= 0:
        _messages_bad(err.bad)
        _messages_split(err.centromere, err.split)
    return ValueError(NOSPLIT_MESSAGE) if err.code == _lib.TP_ERR_NOSPLIT else err


def TADpole_batch(mat_files, max_pcs=200, min_clusters=2, bad_frac=0.01, centromere_search=False, pool=None,
                  device=0, streams=4, ctx=None, centromere_fix=False, resident=False):
    """TADpole() on every matrix of `mat_files` (paths or arrays), `streams` calls in flight per GPU.  centromere_search
    (and centromere_fix, see TADpole()): every matrix is split at its centromere and both arms are called in the library's
    workers; the objects and messages are TADpole(centromere_search=True)'s, and the first matrix TADpole() would fail on
    raises its exception.
    resident: every object keeps its PC scores and all its candidates' dendrograms in HBM (16 bytes per good bin and PC
    computed), so recall() and dendro_for() work on it (and dendro_for() on its arms) as on TADpole()'s objects; that
    memory is released with the last object.  Recalls run on the given pool or ctx, or else on a context made for each
    recall: a context this function makes for the call is closed when it returns, as without resident."""
    own = pool is None and ctx is None
    if ctx is None:
        pool = pool or ContextPool(device, streams)
        ctx, streams = pool.ctx, pool.streams
    try:
        mats = [read_matrix(m, ctx) for m in mat_files]
        res = ctx.call_batch(mats, max_pcs=max_pcs, min_clusters=min_clusters, bad_frac=bad_frac, inflight=streams,
                             centromere_search=centromere_search, centromere_fix=centromere_fix, resident=resident)
        res, store = res if resident else (res, None)
        if own and store is not None:
            store.detach()
        handle = lambda i: (store, i) if resident else None
        if centromere_search:
            out = []
            for i, r in enumerate(res):     # messages in input order, up to the first matrix that fails
                if isinstance(r, Exception):
                    raise _failed_item(r)
                out.append(_tadpole_from_batch_item(r, centromere_fix, handle(i)))
            return out
        for r in res:
            if isinstance(r, Exception):
                raise r
        return [_tadpole_from_batch_item(r, False, handle(i)) for i, r in enumerate(res)]
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

    def load(self, ctx=None, device=0):
        """Ingest the pixels once and keep them on the GPU: a LoadedGenome, which TADpole_genome takes in place of the
        pixels and which can be subsampled (downsample, equal_depth).  Without ctx, a context on `device` is made and
        closed with the last LoadedGenome that uses it."""
        ref = _CtxRef(ctx or _lib.Context(device), ctx is None)
        try:
            return LoadedGenome(self._ingest(ref.ctx), self.names, ref)
        except BaseException:
            ref.release()
            raise


def read_chromsizes(chromsizes, first_path=None):
    """[(name, length in bp)] of a chromosome table: the path of a two-column chrom.sizes file, a list of (name, length),
    a dict {name: length}, or None for the '#chromsize: <name> <length>' header lines at the top of `first_path` (the 4DN
    pairs header; a file without them is a ValueError).  Names must be unique, non-empty and free of whitespace, lengths
    whole numbers >= 1."""
    if chromsizes is None:
        table = []
        with open(first_path, "rb") as fh:
            for raw in fh:
                if not raw.startswith(b"#"):
                    break
                if raw.startswith(b"#chromsize:"):
                    f = raw[len(b"#chromsize:"):].split()
                    if len(f) != 2:
                        raise ValueError(f"{first_path}: malformed header line {raw.decode(errors='replace').strip()!r}")
                    table.append((f[0].decode(), f[1].decode()))
        if not table:
            raise ValueError(f"{first_path} has no '#chromsize:' header lines: give the chromosome table (chromsizes=)")
    elif isinstance(chromsizes, (str, os.PathLike)):
        table = []
        with open(chromsizes) as fh:
            for line in fh:
                f = line.split()
                if not f:
                    continue
                if len(f) < 2:
                    raise ValueError(f"{chromsizes}: a chrom.sizes line needs a name and a length: {line.strip()!r}")
                table.append((f[0], f[1]))
    elif isinstance(chromsizes, dict):
        table = list(chromsizes.items())
    else:
        table = [tuple(x) for x in chromsizes]
    out, seen = [], set()
    for item in table:
        if len(item) != 2:
            raise ValueError(f"a chromosome table entry is (name, length), not {item!r}")
        nm, ln = item
        nm = str(nm)
        if not nm or any(ch.isspace() for ch in nm):
            raise ValueError(f"chromosome name {nm!r} is empty or contains whitespace")
        if nm in seen:
            raise ValueError(f"chromosome {nm!r} appears twice in the chromosome table")
        seen.add(nm)
        try:
            n = int(ln)
        except (TypeError, ValueError, OverflowError):
            n = None
        if n is None or isinstance(ln, bool) or n < 1 or (isinstance(ln, float) and ln != n):
            raise ValueError(f"chromosome {nm!r} has length {ln!r}: a whole number >= 1 is needed")
        out.append((nm, n))
    if not out:
        raise ValueError("the chromosome table is empty")
    return out


class GenomePairs:
    """The contacts of a whole genome as the read-pair files a Hi-C pipeline writes, binned at `binsize` bp on the GPU:
    a drop-in for GenomePixels (names, chrom_bins, load(), TADpole_genome()).  Several files are pooled at read level
    (replicates), and the result is the same in any file order.  Plain text only (gzip input is refused).

    paths: one path or a list.  chromsizes: see read_chromsizes (None: the '#chromsize:' header of the first file).
    Chromosome c gets ceil(length / binsize) bins, and position p falls in bin (p - index_base) // binsize.
    columns: the 0-based columns of (chrom1, pos1, chrom2, pos2):
      4DN pairs (readID chrom1 pos1 chrom2 pos2 ...):                  (1, 2, 3, 4)
      HiC-Pro validPairs (readID chr1 pos1 strand1 chr2 pos2 ...):     (1, 2, 4, 5)
      Juicer merged_nodups (str1 chr1 pos1 frag1 str2 chr2 pos2 ...):  (1, 2, 5, 6)
    index_base: 1 (the 4DN definition of positions) or 0.  Lines starting with '#' and blank lines are skipped; a pair on a
    chromosome outside the table is unplaced and a pair between two chromosomes is trans: both are counted and dropped
    (LoadedGenome.pair_counts).  DESIGN S0f has the whole spec."""

    def __init__(self, paths, chromsizes=None, binsize=None, columns=(1, 2, 3, 4), index_base=1):
        paths = [paths] if isinstance(paths, (str, os.PathLike)) else list(paths)
        if not paths or not all(isinstance(p, (str, os.PathLike)) for p in paths):
            raise ValueError("GenomePairs needs one or more file paths")
        if binsize is None or isinstance(binsize, bool) or not isinstance(binsize, (int, np.integer)) or binsize < 1:
            raise ValueError(f"binsize must be an integer >= 1 (bp), not {binsize!r}")
        cols = tuple(columns) if isinstance(columns, (list, tuple, np.ndarray)) else ()
        if len(cols) != 4 or not all(isinstance(c, (int, np.integer)) and not isinstance(c, bool) and 0 <= c <= 63
                                     for c in cols) or len(set(int(c) for c in cols)) != 4:
            raise ValueError(f"columns must be four different 0-based column indices in 0..63, not {columns!r}")
        if isinstance(index_base, bool) or index_base not in (0, 1):
            raise ValueError(f"index_base must be 0 or 1, not {index_base!r}")
        self.paths = [os.fspath(p) for p in paths]
        self.chromsizes = read_chromsizes(chromsizes, self.paths[0])
        self.binsize, self.columns, self.index_base = int(binsize), tuple(int(c) for c in cols), int(index_base)
        nb = [(ln - 1) // self.binsize + 1 for _, ln in self.chromsizes]
        if sum(nb) >= 2 ** 31 - 1:
            raise ValueError(f"{self.binsize} bp bins give {sum(nb)} bins in all; at most 2^31 - 2 are supported")
        self.names = [nm for nm, _ in self.chromsizes]
        self.chrom_bins = np.array(nb, dtype=np.int32)

    def _load(self, ctx):
        return ctx.genome_ingest_pairs(self.paths, self.names, [ln for _, ln in self.chromsizes], self.binsize,
                                       self.columns, self.index_base)

    def _ingest(self, ctx):
        return self._load(ctx)[0]

    def load(self, ctx=None, device=0):
        """Read, bin and merge the pairs once and keep the cells on the GPU: a LoadedGenome with binsize and pair_counts
        (dict(lines, cis, trans, unplaced)).  Without ctx, a context on `device` is made and closed with the last
        LoadedGenome that uses it."""
        ref = _CtxRef(ctx or _lib.Context(device), ctx is None)
        try:
            g, counts = self._load(ref.ctx)
            return LoadedGenome(g, self.names, ref, binsize=self.binsize, pair_counts=counts)
        except BaseException:
            ref.release()
            raise


class _CtxRef:
    """The context of one or more LoadedGenomes; a context made for them is closed when the last one is closed."""

    def __init__(self, ctx, own):
        self.ctx, self.own, self.users = ctx, own, 0

    def acquire(self):
        self.users += 1
        return self

    def release(self):
        self.users -= 1
        if self.users <= 0 and self.own:
            self.ctx.close()


class LoadedGenome:
    """A genome-wide pixel list held on the GPU, one bucket of cis pixels per chromosome (GenomePixels.load,
    GenomePairs.load, or a subsample or coarsening of another LoadedGenome).  names / chrom_bins: the bin table's
    chromosomes and their bins.  factor: the bin size as a multiple of the ingested file's (1 after load(), multiplied by
    each coarsen(), kept by downsample()); bin b (1-based) of a chromosome of n_fine ingested bins covers the ingested bins
    factor * (b - 1) + 1 .. min(factor * b, n_fine).  binsize: the bin size in bp (None for a pixel-file load; multiplied
    by coarsen(), kept by downsample()).  pair_counts: dict(lines, cis, trans, unplaced) of the files a GenomePairs load
    read, else None.  TADpole_genome takes it wherever it takes GenomePixels, and does not free it.  Close it (or use it
    as a context manager) to release its device memory."""

    def __init__(self, genome, names, ref, factor=1, binsize=None, pair_counts=None):
        self._g, self.names, self.chrom_bins = genome, list(names), np.asarray(genome.chrom_bins, dtype=np.int32)
        self.factor, self.binsize, self.pair_counts = factor, binsize, pair_counts
        self._ref = ref.acquire()
        self.ctx = ref.ctx

    def depth(self):
        """{chromosome: cis contacts}: the sum of the integer counts of its pixels"""
        return {nm: int(x) for nm, x in zip(self.names, self._g.depth())}

    @property
    def total_depth(self):
        return sum(self.depth().values())

    def downsample(self, contacts=None, fraction=None, seed=0):
        """A new LoadedGenome holding a uniform random subset of exactly `contacts` of this genome's cis contacts, or of
        floor(fraction * total_depth) of them: the counts stay raw integers, the matrix a library with that many reads
        would give.  The draw is a function of the merged pixels, seed and contacts only (DESIGN S0d), on the GPU that
        holds this genome.  Both genomes stay valid and either may be closed first."""
        if (contacts is None) == (fraction is None):
            raise ValueError("downsample needs exactly one of contacts and fraction")
        total = self.total_depth
        if fraction is not None:
            f = float(fraction)
            if not 0.0 <= f <= 1.0:
                raise ValueError(f"fraction must be in [0, 1], not {fraction}")
            contacts = math.floor(f * total)                 # in double precision, as R's floor(fraction * total)
        contacts = int(contacts)
        if not 0 <= contacts <= total:
            raise ValueError(f"contacts must be in 0..{total} (the genome's cis contacts), not {contacts}")
        return LoadedGenome(self._g.downsample(contacts, int(seed) % 2 ** 64), self.names, self._ref, self.factor,
                            self.binsize)

    def coarsen(self, factor):
        """A new LoadedGenome at `factor` times this genome's bin size, on the GPU that holds it (DESIGN S0e): chromosome c
        gets ceil(chrom_bins[c] / factor) bins (the last one narrower when factor does not divide it), and coarse cell
        (I, J) holds the sum of the counts of the cells (i, j) with i // factor = I and j // factor = J (a NaN count adds
        0; cells that sum to 0 are left out).  Integer counts add exactly.  Both genomes stay valid and either may be
        closed first."""
        if isinstance(factor, bool) or not isinstance(factor, (int, np.integer, float, np.floating)):
            raise ValueError(f"factor must be an integer >= 1, not {factor!r}")
        if isinstance(factor, (float, np.floating)) and not float(factor).is_integer():
            raise ValueError(f"factor must be an integer >= 1, not {factor!r}")
        f = int(factor)
        if not 1 <= f <= 2 ** 31 - 1:
            raise ValueError(f"factor must be an integer in 1..2^31-1, not {factor!r}")
        if self._g is None:
            raise ValueError("the LoadedGenome has been closed")
        return LoadedGenome(self._g.coarsen(f), self.names, self._ref, self.factor * f,
                            None if self.binsize is None else self.binsize * f)

    def pixels(self, chrom):
        """(i, j, count) of chromosome `chrom` (a name): chromosome-local 0-based bins, sorted by (i, j)"""
        if chrom not in self.names:
            raise ValueError(f"unknown chromosome {chrom!r}: not in the bin table")
        i, j, v = self._g.pixels(self.names.index(chrom))
        o = np.lexsort((j, i))
        return i[o], j[o], v[o]

    def stats(self):
        return self._g.stats()

    def close(self):
        if self._g is not None:
            self._g.close()
            self._g = None
            self._ref.release()

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def equal_depth(*genomes, seed=0):
    """The LoadedGenomes at the same cis depth: every genome deeper than the shallowest is subsampled to the shallowest's
    total (genome s with seed + s), the others are returned as they are.  Returns the list, in argument order."""
    totals = [g.total_depth for g in genomes]
    low = min(totals)
    return [g.downsample(contacts=low, seed=(int(seed) + s) % 2 ** 64) if t > low else g
            for s, (g, t) in enumerate(zip(genomes, totals))]


class GenomeResult(dict):
    """{chromosome name: Tadpole}; .failed {name: message of the library}; .stats dict(cis={name: pixels}, trans=,
    below=)."""
    failed: dict
    stats: dict

    def recall(self, max_pcs=200, min_clusters=2, chroms=None, streams=4):
        """TADpole_genome() again with another max_pcs (<= the one computed) / min_clusters, from the PC scores resident
        for every chromosome (TADpole_genome(resident=True)): only the n_pcs sweep and the selection run, all selected
        chromosomes in one library call.  chroms: names (default every chromosome of this result).  Returns a
        GenomeResult with the same messages, .stats, and .failed = the earlier failures plus this recall's."""
        names = list(self) if chroms is None else [str(c) for c in chroms]
        missing = [c for c in names if c not in self]
        if missing:
            raise ValueError(f"chromosome(s) {missing} are not in this result")
        handles = [self[nm]._resident() for nm in names]
        stores = {id(h["batch"]): h["batch"] for h in handles}
        if len(stores) > 1:
            raise ValueError("the chromosomes come from different genome calls: recall them separately")
        out = GenomeResult()
        out.failed = dict(self.failed)
        out.stats = self.stats
        if not names:
            return out
        res, store = handles[0]["batch"].recall([h["item"] for h in handles], max_pcs=max_pcs, min_clusters=min_clusters,
                                                inflight=streams)
        for i, (nm, h, r) in enumerate(zip(names, handles, res)):
            message(f"Processing chromosome {nm}")
            if isinstance(r, Exception):
                out.failed[nm] = str(r)
                continue
            out[nm] = _tadpole_from_batch_item(r, h["centromere_fix"], (store, i))
        return out


def TADpole_genome(pixels, chroms=None, max_pcs=200, min_clusters=2, bad_frac=0.01, ctx=None, device=0, streams=4,
                   centromere_search=False, centromere_fix=False, resident=False):
    """TADpole() on every chromosome of a genome-wide pixel list (GenomePixels, GenomePairs, or a LoadedGenome: then with
    ctx=None the call runs on the context the genome was loaded on, and the genome stays loaded), `streams` calls in
    flight per GPU.
    Each chromosome's Tadpole is the one TADpole() returns for that chromosome's dense matrix (with centromere_search /
    centromere_fix as TADpole() takes them: p, q and merging_arms; a chromosome that does not split fails with
    TADpole()'s message unless centromere_fix).  Returns a GenomeResult in bin-table order, or in `chroms` order when
    chroms (a list of names) is given.
    resident: as TADpole_batch's (recalls run on ctx when it is given, else on a context made for each recall); the
    result then also has recall() over all its chromosomes at once."""
    index = {nm: c for c, nm in enumerate(pixels.names)}
    sel = list(pixels.names) if chroms is None else [str(c) for c in chroms]
    unknown = [c for c in sel if c not in index]
    if unknown:
        raise ValueError(f"unknown chromosome(s) {unknown}: not in the bin table")
    loaded = isinstance(pixels, LoadedGenome)
    if loaded and pixels._g is None:
        raise ValueError("the LoadedGenome has been closed")
    if loaded and ctx is None:
        ctx = pixels.ctx
    own = ctx is None
    ctx = ctx or _lib.Context(device)
    try:
        g = pixels._g if loaded else pixels._ingest(ctx)
        try:
            cis, trans, below = g.stats()
            res = ctx.call_genome(g, [index[c] for c in sel], max_pcs=max_pcs, min_clusters=min_clusters, bad_frac=bad_frac,
                                  inflight=streams, centromere_search=centromere_search, centromere_fix=centromere_fix,
                                  resident=resident)
        finally:
            if not loaded:
                g.close()
    finally:
        if own:
            ctx.close()
    res, store = res if resident else (res, None)
    if own and store is not None:
        store.detach()
    out = GenomeResult()
    out.failed = {}
    out.stats = dict(cis={nm: int(k) for nm, k in zip(pixels.names, cis)}, trans=trans, below=below)
    for i, (nm, r) in enumerate(zip(sel, res)):
        message(f"Processing chromosome {nm}")
        if isinstance(r, Exception):
            out.failed[nm] = NOSPLIT_MESSAGE if r.code == _lib.TP_ERR_NOSPLIT else str(r)
            continue
        out[nm] = _tadpole_from_batch_item(r, centromere_fix, (store, i) if resident else None)
    return out


# ---- comparing two genome-wide calls ---------------------------------------------------------------------------------

def _field(obj, name):
    if isinstance(obj, dict):
        return obj.get(name)
    return getattr(obj, name, None)


def _difft_genome_problems(control, case, levels=None):
    """The problems of diffT_genome (one per chromosome and level compared) and the `skipped` dict.  Each problem is a
    dict: chrom, level, x / y (the control's and the case's start / end tables), tx / ty (padded labels, as diffT pads
    them), pad_left / pad_right / ntads (of y within the common extent) and bad (1-based positions within y's start:end
    of the case's filtered bins there).  Host bookkeeping only."""
    skipped = {}
    failed_x, failed_y = getattr(control, "failed", None) or {}, getattr(case, "failed", None) or {}
    problems = []
    for chrom, tx_obj in control.items():
        if chrom not in case:
            skipped[chrom] = (f"failed in case: {failed_y[chrom]}" if chrom in failed_y else "missing from case")
            continue
        ty_obj = case[chrom]
        if _field(tx_obj, "clusters") is None or _field(ty_obj, "clusters") is None:
            skipped[chrom] = "centromere_search result: comparing the arms is not supported"
            continue
        cx = {int(k): v for k, v in _field(tx_obj, "clusters").items()}
        cy = {int(k): v for k, v in _field(ty_obj, "clusters").items()}
        if levels is None:
            ks = sorted(set(cx) & set(cy))
        else:
            ks = []
            for k in sorted({int(k) for k in levels}):
                if k not in cx or k not in cy:
                    skipped[(chrom, k)] = f"level {k} is not scored in {'control' if k not in cx else 'case'}"
                else:
                    ks.append(k)
        dendro = _field(ty_obj, "dendro")
        kept = np.asarray(_field(dendro, "labels"), dtype=np.int64)
        for k in ks:
            bx, by = _bed_rows(cx[k]), _bed_rows(cy[k])
            if bx.shape[0] != by.shape[0]:
                skipped[(chrom, k)] = "Both calls must have the same number of TADs."      # R/DiffT.R:20
                continue
            tx, ty = _difft_labels(bx, by)
            sx, sy, ex, ey = int(bx[0, 0]), int(by[0, 0]), int(bx[-1, 1]), int(by[-1, 1])
            span = np.arange(sy, ey + 1)
            bad = (span[~np.isin(span, kept)] - sy + 1).astype(np.int32)
            problems.append(dict(chrom=chrom, level=k, x=bx, y=by, tx=tx, ty=ty, pad_left=max(0, sy - sx),
                                 pad_right=max(0, ex - ey), ntads=int(by.shape[0]), bad=bad))
    for chrom in case:
        if chrom not in control:
            skipped[chrom] = (f"failed in control: {failed_x[chrom]}" if chrom in failed_x else "missing from control")
    for chrom, msg in failed_x.items():
        if chrom not in control and chrom not in skipped:
            skipped[chrom] = f"failed in control: {msg}"
    for chrom, msg in failed_y.items():
        if chrom not in case and chrom not in control and chrom not in skipped:
            skipped[chrom] = f"failed in case: {msg}"
    return problems, skipped


def _population(pr):
    """Candidate border positions of a problem's random partitions (tp_difft_null's count)."""
    size = int(pr["ty"].size) - pr["pad_left"] - pr["pad_right"]
    bad = np.unique(pr["bad"][(pr["bad"] >= 1) & (pr["bad"] <= size)])
    return max(size - bad.size - 1, 0)


def diffT_genome(control, case, levels=None, nperm=1000, seed=0, ctx=None):
    """diffT (R/DiffT.R:19-50) between two genome-wide calls, level by level, each comparison with its own null
    distribution; every comparison and every random partition is computed in one call to the library.

    control, case: GenomeResults of TADpole_genome (or {chromosome: Tadpole} mappings).  One problem per chromosome
    present in both as a whole-chromosome object (in control's order) and per level k scored in both (or listed in
    `levels`), ascending: diffT(control[chrom].clusters[k], case[chrom].clusters[k]), and diffT against nperm random
    partitions of the case's extent with its TAD count, as diffT_null(x, y, bad_columns=...) draws them.  The bad columns
    of the null are the case's filtered bins inside its table's extent, as positions within start:end
    (bin - start + 1): the reference's random_bed takes positions, so the chromosome's own bad_columns would be
    misplaced whenever the table does not start at bin 1.  Problem p (0-based, in this order) draws with seed + p.

    Returns an object of parallel lists / arrays, one entry per compared problem: chrom, level, total (observed,
    un-normalised), p_value = (1 + #{null totals <= total}) / (nperm + 1), curves (observed normalised curves),
    null_totals [nproblems, nperm] and seed (per problem); and skipped: {chromosome or (chromosome, level): reason}.
    p_value (the share of random partitions at least as close to the control as the case is) is not in the reference."""
    ctx = ctx or get_context()
    problems, skipped = _difft_genome_problems(control, case, levels)
    nperm = int(nperm)
    out = _Obj(chrom=[], level=np.zeros(0, np.int64), total=np.zeros(0), p_value=np.zeros(0), curves=[],
               null_totals=np.zeros((0, nperm)), seed=[], skipped=skipped)
    if not problems:
        return out
    lens = np.array([pr["tx"].size for pr in problems], dtype=np.int64)
    off = np.concatenate(([0], np.cumsum(lens)))
    nbad = np.array([pr["bad"].size for pr in problems], dtype=np.int64)
    res = ctx.difft_multi(off, np.concatenate([pr["tx"] for pr in problems]), np.concatenate([pr["ty"] for pr in problems]),
                          [pr["pad_left"] for pr in problems], [pr["pad_right"] for pr in problems],
                          [pr["ntads"] for pr in problems], np.concatenate(([0], np.cumsum(nbad))),
                          np.concatenate([pr["bad"] for pr in problems]), seed=seed, nperm=nperm)
    keep = []
    for p, pr in enumerate(problems):
        if res["status"][p] != _lib.TP_OK:
            skipped[(pr["chrom"], pr["level"])] = (
                f"the library refused it: random_bed cannot draw {pr['ntads'] - 1} borders from {_population(pr)} "
                "candidate bins (sample() errors here, R/DiffT.R:69)")
            continue
        keep.append(p)
    keep = np.array(keep, dtype=np.int64)
    null = res["null_totals"][keep]
    total = res["totals"][keep]
    out.chrom = [problems[p]["chrom"] for p in keep]
    out.level = np.array([problems[p]["level"] for p in keep], dtype=np.int64)
    out.total = total
    out.p_value = (1 + (null <= total[:, None]).sum(axis=1)) / (nperm + 1)
    out.curves = [res["curves"][off[p]:off[p + 1]] for p in keep]
    out.null_totals = null
    out.seed = [(int(seed) + int(p)) % 2 ** 64 for p in keep]
    return out
