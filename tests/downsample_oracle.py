"""Reference of equal-depth subsampling (tadpole_b200/csrc/downsample.cu, DESIGN S0d), read by read: the checker the
subsampling tests compare the GPU with.  Plain numpy on top of the oracle's genome split (oracle/genome_oracle.py:
split_genome_pixels) and its Philox4x32-10 (oracle/tadpole_oracle.py: philox4x32)."""
from __future__ import annotations

import numpy as np

from oracle.genome_oracle import split_genome_pixels
from oracle.tadpole_oracle import philox4x32


def merged_cells(chrom_bins, bin1, bin2, count):
    """The cells (c, i, j, C) of a genome-wide pixel list (global 0-based bins): every cis pixel on or above the diagonal,
    pixels naming the same cell added up, cells of count 0 dropped, sorted by (c, i, j).  A count that is not an integer
    in [0, 2^32), or a merged cell of 2^32 reads or more, is a ValueError."""
    per, _, _ = split_genome_pixels(bin1, bin2, count, chrom_bins)
    cs, is_, js, ns = [], [], [], []
    for c, (i, j, v) in enumerate(per):
        bad = ~((v >= 0) & (v < 2.0 ** 32) & (v == np.floor(v)))
        if bad.any():
            k = int(np.flatnonzero(bad)[0])
            raise ValueError(f"chromosome {c}, bins ({i[k]}, {j[k]}): count {float(v[k])!r} is not an integer in [0, 2^32)")
        cells = {}
        for a, b, n in zip(i.tolist(), j.tolist(), v.astype(np.int64).tolist()):
            cells[(a, b)] = cells.get((a, b), 0) + n
        for (a, b), n in sorted(cells.items()):
            if n >= 2 ** 32:
                raise ValueError(f"chromosome {c}, bins ({a}, {b}): the cell adds up to 2^32 reads or more")
            if n:
                cs.append(c); is_.append(a); js.append(b); ns.append(n)
    return (np.array(cs, dtype=np.int64), np.array(is_, dtype=np.int64), np.array(js, dtype=np.int64),
            np.array(ns, dtype=np.int64))


def downsample(chrom_bins, bin1, bin2, count, contacts, seed):
    """The subsample of `contacts` reads of tp_genome_downsample (csrc/downsample.cu, DESIGN S0d), read by read: cell
    (c, i, j) of count C holds the reads (c, i, j, r), r < C; key(read) = the first 64 bits of Philox4x32-10 on counter
    (r, i, j, 0xD5000000 | c) with key words (seed mod 2^32, seed >> 32); the reads with the `contacts` smallest
    (key, c, i, j, r) are kept.  Returns [(i, j, kept) of each chromosome, sorted by (i, j), cells keeping no read
    dropped]."""
    seed = int(seed) % 2 ** 64
    c, i, j, n = merged_cells(chrom_bins, bin1, bin2, count)
    total = int(n.sum())
    if not 0 <= contacts <= total:
        raise ValueError(f"{contacts} contacts asked for, but the genome holds {total}")
    cell = np.repeat(np.arange(n.size), n)
    first = np.concatenate(([0], np.cumsum(n)[:-1])).astype(np.int64)
    r = np.arange(total, dtype=np.int64) - first[cell]
    x0, x1, _, _ = philox4x32(r, i[cell], j[cell], np.int64(0xD5000000) | c[cell], seed & 0xFFFFFFFF, seed >> 32)
    key = (x0 << np.uint64(32)) | x1
    # the reads are listed in (c, i, j, r) order already: a stable sort on the key orders them by (key, c, i, j, r)
    take = np.argsort(key, kind="stable")[:contacts]
    kept = np.bincount(cell[take], minlength=n.size)
    out = []
    for ch in range(len(chrom_bins)):
        m = (c == ch) & (kept > 0)
        out.append((i[m], j[m], kept[m].astype(np.float64)))
    return out
