// genome_util.cuh -- helpers of the handle -> handle transforms of a tp_genome (downsample.cu S0d, coarsen.cu S0e): the
// chromosome of a bucket entry or of a global bin, the hash of a cell key, the context member that holds a handle, the
// grid of the grid-stride kernels and the owner guard of a handle being built.
#pragma once
#include "common.cuh"

#define DS_THREADS 256                       // threads per CTA of the grid-stride kernels

// largest c in [0, nchrom) with offs[c] <= e (the chromosome whose bucket holds entry e)
__device__ __forceinline__ int ds_chrom_of_entry(const unsigned long long *__restrict__ offs, int nchrom, unsigned long long e) {
    int lo = 0, hi = nchrom - 1;
    while (lo < hi) {
        const int mid = (lo + hi + 1) >> 1;
        if (__ldg(offs + mid) <= e) lo = mid; else hi = mid - 1;
    }
    return lo;
}
__device__ __forceinline__ int ds_chrom_of_bin(const int *__restrict__ starts, int nchrom, int x) {
    int lo = 0, hi = nchrom - 1;
    while (lo < hi) {
        const int mid = (lo + hi + 1) >> 1;
        if (__ldg(starts + mid) <= x) lo = mid; else hi = mid - 1;
    }
    return lo;
}

__device__ __forceinline__ unsigned long long ds_hash(unsigned long long key) {
    key ^= key >> 33; key *= 0xff51afd7ed558ccdULL; key ^= key >> 33; key *= 0xc4ceb9fe1a85ec53ULL; key ^= key >> 33;
    return key;
}

// the member of ctx on the device that holds g (multi-device contexts: any of their devices), or an error
static inline int ds_member(tp_ctx *ctx, const tp_genome *g, const char *who, tp_ctx **out) {
    for (int r = 0; r < tp_group_size(ctx); r++) {
        tp_ctx *m = tp_group_member(ctx, r);
        if (m && m->device == g->device) { *out = m; return TP_OK; }
    }
    tp_set_error("%s: the handle is on device %d, which is not a device of the context", who, g->device);
    return TP_ERR_ARG;
}

static inline unsigned ds_grid(const tp_ctx *c, unsigned long long work) {
    const unsigned long long want = (work + DS_THREADS - 1) / DS_THREADS, cap = (unsigned long long)c->sm_count * 16;
    return (unsigned)(want < 1 ? 1 : want < cap ? want : cap);
}

struct GenomeOwnerDs { tp_genome *g = nullptr; ~GenomeOwnerDs() { if (g) tp_genome_free(g); } };
