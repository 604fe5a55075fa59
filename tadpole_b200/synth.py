"""Synthetic Hi-C matrices and TAD partitions (SURVEY.md section 8(d)).

The reference ships no runnable example matrix (its README names
inst/extdata/raw_chr18_300_500_30kb.tsv, which is absent from the checkout), so every
configuration of BASELINE.json is run on matrices from this generator:

    lambda_ij = A * (|i-j|+1)^(-alpha) * prod_levels boost_l^[i,j in the same block at level l]
    M_ij      ~ Poisson(lambda_ij), drawn for the upper triangle and mirrored

with nested block TADs, a few bins zeroed entirely (zero diagonal => bad columns,
reference R/TADpole.R:36) and, optionally, one contiguous zeroed run that plays the
centromere (R/TADpole.R:58-64).  Everything is seeded and pure numpy.
"""
from __future__ import annotations

import numpy as np

__all__ = ["synth_hic", "synth_hic_gpu", "synth_genome_pixels", "synth_partition_pairs", "write_tsv"]


def _random_blocks(rng, n, mean_len):
    """Block id per bin; block lengths uniform in [mean/2, 3*mean/2]."""
    ids = np.empty(n, dtype=np.int64)
    pos, b = 0, 0
    lo, hi = max(1, int(mean_len // 2)), max(2, int(round(mean_len * 1.5)))
    while pos < n:
        ln = int(rng.integers(lo, hi + 1))
        ids[pos:pos + ln] = b
        pos += ln
        b += 1
    return ids


def synth_hic(n, seed=1, amp=200.0, alpha=1.0, levels=((None, 1.5), (40, 3.0), (10, 6.0)),
              zero_frac=0.005, centromere=False, centromere_frac=0.03, dtype=np.float64):
    """Return an n x n symmetric count matrix (float64, C order).

    levels: (mean block length, boost); None for the length means n/5 ("compartments").
    zero_frac: fraction of bins zeroed entirely (they become bad columns).
    centromere: zero one contiguous run of ~centromere_frac*n bins near the middle.
    """
    rng = np.random.default_rng(seed)
    idx = np.arange(n)
    lam = np.empty((n, n), dtype=np.float32)
    # build row blocks to bound temporary memory at large n
    blocks = []
    for mean_len, boost in levels:
        ml = n / 5.0 if mean_len is None else float(mean_len)
        blocks.append((_random_blocks(rng, n, ml), np.float32(boost)))
    step = max(1, min(n, (1 << 24) // max(n, 1)))
    for r0 in range(0, n, step):
        r1 = min(n, r0 + step)
        d = np.abs(idx[r0:r1, None] - idx[None, :]).astype(np.float32) + 1.0
        l = np.float32(amp) * d ** np.float32(-alpha)
        for ids, boost in blocks:
            same = ids[r0:r1, None] == ids[None, :]
            l = np.where(same, l * boost, l)
        lam[r0:r1] = l
    mat = np.zeros((n, n), dtype=dtype)
    for r0 in range(0, n, step):
        r1 = min(n, r0 + step)
        mat[r0:r1] = rng.poisson(lam[r0:r1]).astype(dtype)
    del lam
    # symmetrise from the upper triangle (what forceSymmetric(uplo='U') will do anyway)
    iu = np.triu_indices(n, 1)
    mat[(iu[1], iu[0])] = mat[iu]
    nz = int(round(zero_frac * n))
    if nz:
        z = rng.choice(n, size=nz, replace=False)
        mat[z, :] = 0.0
        mat[:, z] = 0.0
    if centromere:
        ln = max(2, int(round(centromere_frac * n)))
        c0 = n // 2 - ln // 2 + int(rng.integers(-n // 50 - 1, n // 50 + 2))
        c0 = min(max(c0, 2), n - ln - 2)
        mat[c0:c0 + ln, :] = 0.0
        mat[:, c0:c0 + ln] = 0.0
    return mat


def synth_hic_gpu(n, seed=1, device=0, centromere=False, centromere_frac=0.03, zero_frac=0.005):
    """The same lambda structure drawn on the GPU with torch.poisson (numpy's generator needs ~26 s at 25 000 bins): for
    the chromosome-sized configurations of bench.py and the GPU tests.  The block structure comes from numpy's seeded
    generator, the Poisson draws from torch's (same seed + same GPU model = same matrix on every rank; callers that need
    that compare a checksum).  Returns an n x n float64 CUDA tensor (symmetric integer counts)."""
    import torch
    rng = np.random.default_rng(seed)
    dev = torch.device("cuda", device)
    idx = torch.arange(n, device=dev)
    blocks = [(torch.from_numpy(_random_blocks(rng, n, n / 5.0 if ml is None else float(ml))).to(dev), bo)
              for ml, bo in ((None, 1.5), (40, 3.0), (10, 6.0))]
    g = torch.Generator(device=dev)
    g.manual_seed(seed)
    mat = torch.empty((n, n), dtype=torch.float64, device=dev)
    step = max(1, (1 << 26) // n)
    for r0 in range(0, n, step):
        r1 = min(n, r0 + step)
        lam = 200.0 / ((idx[r0:r1, None] - idx[None, :]).abs().float() + 1.0)
        for ids, bo in blocks:
            lam = torch.where(ids[r0:r1, None] == ids[None, :], lam * bo, lam)
        mat[r0:r1] = torch.poisson(lam, generator=g).double()
        del lam
    for r0 in range(0, n, step):            # lower := upper^T, in row blocks (no second n x n temporary)
        r1 = min(n, r0 + step)
        blk = mat[:, r0:r1].T.contiguous()                    # blk[i, j] = mat[j, r0 + i]
        cols = torch.arange(n, device=dev)[None, :]
        rows = torch.arange(r0, r1, device=dev)[:, None]
        mat[r0:r1] = torch.where(cols < rows, blk, mat[r0:r1])
        del blk
    z = torch.from_numpy(rng.choice(n, size=int(round(zero_frac * n)), replace=False)).to(dev)
    mat[z, :] = 0.0
    mat[:, z] = 0.0
    if centromere:
        ln = max(2, int(round(centromere_frac * n)))
        c0 = n // 2 - ln // 2 + int(rng.integers(-n // 50 - 1, n // 50 + 2))
        c0 = min(max(c0, 2), n - ln - 2)
        mat[c0:c0 + ln, :] = 0.0
        mat[:, c0:c0 + ln] = 0.0
    return mat


def synth_genome_pixels(sizes, seed=1, trans_per_chrom=100, centromere=None):
    """A seeded genome-wide pixel list, as HiC-Pro or cooler write one: chromosome c has sizes[c] bins and its contacts
    are synth_hic(sizes[c], seed + c) (any size, 1 included); its non-zero upper-triangle cells become pixels with global
    0-based bin ids, and trans_per_chrom pixels per chromosome join one of its bins to a bin of another chromosome.  The
    pixels are shuffled.  centromere: indices of the chromosomes (of 2 bins or more) drawn with
    synth_hic(..., centromere=True); the others, and the random stream, are the same as without it.  Returns (names,
    (bin1, bin2, count), mats): names "chr1", ...; bin1 <= bin2 int32, count float64; mats[c] the symmetric matrix of
    chromosome c, whose upper triangle its cis pixels are."""
    rng = np.random.default_rng(seed)
    sizes = [int(n) for n in sizes]
    cen = set() if centromere is None else {int(c) for c in centromere}
    starts = np.concatenate(([0], np.cumsum(sizes)))
    b1, b2, v, mats = [], [], [], []
    for c, n in enumerate(sizes):
        m = synth_hic(n, seed=seed + c, centromere=c in cen) if n >= 2 else np.full((n, n), float(rng.integers(1, 9)))
        mats.append(m)
        i, j = np.triu_indices(n)
        sel = m[i, j] != 0
        b1.append(i[sel] + starts[c]); b2.append(j[sel] + starts[c]); v.append(m[i, j][sel])
        if len(sizes) > 1 and trans_per_chrom:
            x = rng.integers(0, n, trans_per_chrom) + starts[c]
            other = rng.integers(0, len(sizes) - 1, trans_per_chrom)
            other += other >= c                                          # any chromosome but c
            y = starts[other] + (rng.random(trans_per_chrom) * np.asarray(sizes)[other]).astype(np.int64)
            b1.append(np.minimum(x, y)); b2.append(np.maximum(x, y))
            v.append(rng.integers(1, 5, trans_per_chrom).astype(np.float64))
    b1, b2, v = np.concatenate(b1), np.concatenate(b2), np.concatenate(v)
    perm = rng.permutation(b1.size)
    names = [f"chr{c + 1}" for c in range(len(sizes))]
    return names, (b1[perm].astype(np.int32), b2[perm].astype(np.int32), v[perm].astype(np.float64)), mats


def synth_partition_pairs(npairs, length, ntads, seed=1, zero_frac=0.01):
    """Label vectors for diffT batches (BASELINE.json config 5).

    Returns (labels_x, labels_y), each int32 [npairs, length]: contiguous partitions of
    `length` bins into `ntads` TADs labelled 1..ntads (equal count within a pair, as
    R/DiffT.R:20 requires), with ~zero_frac of bins relabelled 0 (uncovered / bad bins).
    """
    rng = np.random.default_rng(seed)
    out = []
    for _ in range(2):
        lab = np.empty((npairs, length), dtype=np.int32)
        for p in range(npairs):
            cuts = np.sort(rng.choice(np.arange(1, length), size=ntads - 1, replace=False))
            edges = np.concatenate(([0], cuts, [length]))
            lab[p] = np.repeat(np.arange(1, ntads + 1, dtype=np.int32), np.diff(edges))
            nz = int(round(zero_frac * length))
            if nz:
                # interior bins only: the first/last bin define the BED extent
                lab[p, rng.choice(np.arange(1, length - 1), size=nz, replace=False)] = 0
        out.append(lab)
    return out[0], out[1]


def write_tsv(path, mat):
    """Header-less tab-separated matrix, the format read at R/TADpole.R:17."""
    np.savetxt(path, mat, fmt="%.17g", delimiter="\t")
