"""Genome-wide pixel lists: the checker of the route kernel of the genome-wide input (tadpole_b200/csrc/ingest.cu, S0c).

A plain numpy restatement, one pixel at a time; tadpole_oracle.coo_to_dense then gives the dense matrix of each
chromosome from its local pixels."""
from __future__ import annotations

import numpy as np


def split_genome_pixels(bin1, bin2, count, chrom_bins, index_base=0):
    """A genome-wide pixel list (global bin ids; chromosome c holds chrom_bins[c] consecutive bins, the first one
    index_base) split by chromosome, one pixel at a time: a pixel whose bins lie on two chromosomes is trans, one with
    bin1 > bin2 on one chromosome is below the diagonal; both are dropped and counted.  A bin outside the table is an
    error.  Returns ([(i, j, count) local pixels of each chromosome, in input order], trans, below)."""
    starts = np.concatenate(([0], np.cumsum(np.asarray(chrom_bins, dtype=np.int64))))
    total = int(starts[-1])
    out = [([], [], []) for _ in range(len(chrom_bins))]
    trans = below = 0
    for e, (a, b, v) in enumerate(zip(np.asarray(bin1).tolist(), np.asarray(bin2).tolist(),
                                      np.asarray(count, dtype=float).tolist())):
        x, y = a - index_base, b - index_base
        if not (0 <= x < total and 0 <= y < total):
            raise ValueError(f"entry {e + 1} is outside the {total} bins of the bin table")
        cx = int(np.searchsorted(starts, x, side="right")) - 1
        cy = int(np.searchsorted(starts, y, side="right")) - 1
        if cx != cy:
            trans += 1
        elif x > y:
            below += 1
        else:
            for lst, val in zip(out[cx], (x - starts[cx], y - starts[cx], v)):
                lst.append(val)
    return [(np.array(i, dtype=np.int64), np.array(j, dtype=np.int64), np.array(v, dtype=np.float64)) for i, j, v in out], \
        trans, below
