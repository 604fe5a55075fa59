"""Reference of coarsening (tadpole_b200/csrc/coarsen.cu, DESIGN S0e): the checker the coarsening tests compare the GPU
with.  coarsen_pixels restates the spec one pixel at a time on top of the oracle's genome split
(oracle/genome_oracle.py: split_genome_pixels); coarsen_pixels_np is a vectorised restatement for genome-sized inputs,
held equal to the loop by the CPU tests."""
from __future__ import annotations

import numpy as np

from oracle.genome_oracle import split_genome_pixels


def coarse_bins(chrom_bins, factor):
    """ceil(n_c / factor) bins per chromosome"""
    return [-(-int(n) // int(factor)) for n in chrom_bins]


def coarsen_pixels(chrom_bins, bin1, bin2, count, factor, index_base=0):
    """tp_genome_coarsen on a genome-wide pixel list (global bins), one pixel at a time: every cis pixel (c, i, j, v) on
    or above the diagonal adds v (0 when v is NaN) to coarse cell (c, i // factor, j // factor); cells whose sum is 0 are
    dropped.  Sums are Python floats added in input order (exact for integer counts below 2^53).  Returns
    ([(I, J, count) of each chromosome, sorted by (I, J)], trans, below)."""
    per, trans, below = split_genome_pixels(bin1, bin2, count, chrom_bins, index_base)
    out = []
    for i, j, v in per:
        cells = {}
        for a, b, x in zip(i.tolist(), j.tolist(), v.tolist()):
            key = (a // factor, b // factor)
            cells[key] = cells.get(key, 0.0) + (0.0 if x != x else x)
        kept = sorted((k, s) for k, s in cells.items() if s != 0.0)
        out.append((np.array([k[0] for k, _ in kept], dtype=np.int64), np.array([k[1] for k, _ in kept], dtype=np.int64),
                    np.array([s for _, s in kept], dtype=np.float64)))
    return out, trans, below


def coarsen_pixels_np(chrom_bins, bin1, bin2, count, factor, index_base=0):
    """The same as coarsen_pixels, vectorised (np.unique on the cell keys, np.add.at): for integer counts below 2^53 it
    gives the same bits; fractional sums may round differently."""
    sizes = np.asarray(chrom_bins, dtype=np.int64)
    starts = np.concatenate(([0], np.cumsum(sizes)))
    x = np.asarray(bin1, dtype=np.int64) - index_base
    y = np.asarray(bin2, dtype=np.int64) - index_base
    v = np.asarray(count, dtype=np.float64)
    total = int(starts[-1])
    bad = (x < 0) | (y < 0) | (x >= total) | (y >= total)
    if bad.any():
        raise ValueError(f"entry {int(np.flatnonzero(bad)[0]) + 1} is outside the {total} bins of the bin table")
    cx = np.searchsorted(starts, x, side="right") - 1
    cy = np.searchsorted(starts, y, side="right") - 1
    tr = cx != cy
    bl = ~tr & (x > y)
    cis = ~tr & ~bl
    c, i, j, v = cx[cis], x[cis] - starts[cx[cis]], y[cis] - starts[cx[cis]], np.where(np.isnan(v[cis]), 0.0, v[cis])
    cb = np.array(coarse_bins(sizes, factor), dtype=np.int64)
    cstarts = np.concatenate(([0], np.cumsum(cb)))
    key = ((cstarts[c] + i // factor) << 31) | (cstarts[c] + j // factor)
    uk, inv = np.unique(key, return_inverse=True)
    s = np.zeros(uk.size)
    np.add.at(s, inv, v)
    keep = s != 0.0
    uk, s = uk[keep], s[keep]
    gi, gj = uk >> 31, uk & 0x7FFFFFFF
    ch = np.searchsorted(cstarts, gi, side="right") - 1
    out = []
    for k in range(sizes.size):
        m = ch == k                                          # np.unique sorted the keys: (I, J) order per chromosome
        out.append((gi[m] - cstarts[k], gj[m] - cstarts[k], s[m]))
    return out, int(tr.sum()), int(bl.sum())
