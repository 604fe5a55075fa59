// genome_util.cuh -- helpers of the kernels that build a tp_genome from a cell table or another handle (downsample.cu S0d,
// coarsen.cu S0e, pairs.cu S0f): the chromosome of a bucket entry or of a global bin, the hash of a cell key, the walks
// of an open-addressing cell table that write the buckets, the context member that holds a handle, the grid of the
// grid-stride kernels and the owner guard of a handle being built.
#pragma once
#include "common.cuh"

#define DS_THREADS 256                       // threads per CTA of the grid-stride kernels
#define CS_EMPTY 0xffffffffffffffffULL       // the key of an empty slot of a cell table
#define CS_FULL 0xffffffffu

typedef unsigned long long u64;

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

// ---- a cell table -> buckets: slot s holds key ((S_c + I) << 31) | (S_c + J) (S_c the first global bin of chromosome c)
// and the cell's count; an empty slot's key is CS_EMPTY.  cs_count_kernel gives the stored cells per chromosome, the host
// scans them into the offsets, and cs_scatter_kernel writes (count, I, J) through per-chromosome cursors.  static: each
// translation unit that includes this header gets its own copy of the kernels.

// the chromosome of table slot s when it holds a cell to store (a sum that is not exactly 0), else -1
__device__ __forceinline__ int cs_slot_chrom(const u64 *__restrict__ tkeys, const double *__restrict__ tval, u64 cap, u64 s,
                                             const int *__restrict__ cstarts, int nchrom, u64 *key, double *v) {
    if (s >= cap) return -1;
    *key = tkeys[s];
    if (*key == CS_EMPTY) return -1;
    *v = tval[s];
    if (*v == 0.0) return -1;
    return ds_chrom_of_bin(cstarts, nchrom, (int)(*key >> 31));
}

// stored cells per chromosome
static __global__ void __launch_bounds__(DS_THREADS)
cs_count_kernel(const u64 *__restrict__ tkeys, const double *__restrict__ tval, u64 cap, const int *__restrict__ cstarts,
                int nchrom, u64 *__restrict__ hist) {
    const u64 stride = (u64)gridDim.x * DS_THREADS;
    for (u64 base = (u64)blockIdx.x * DS_THREADS; base < cap; base += stride) {
        u64 key = 0;
        double v = 0.0;
        const int c = cs_slot_chrom(tkeys, tval, cap, base + threadIdx.x, cstarts, nchrom, &key, &v);
        const unsigned grp = __match_any_sync(CS_FULL, c);
        if (c >= 0 && (threadIdx.x & 31) == __ffs(grp) - 1) atomicAdd(hist + c, (u64)__popc(grp));
    }
}

// the new buckets
static __global__ void __launch_bounds__(DS_THREADS)
cs_scatter_kernel(const u64 *__restrict__ tkeys, const double *__restrict__ tval, u64 cap, const int *__restrict__ cstarts,
                  int nchrom, u64 *__restrict__ cursor, double *__restrict__ ov, int *__restrict__ oi, int *__restrict__ oj) {
    const u64 stride = (u64)gridDim.x * DS_THREADS;
    const int lane = threadIdx.x & 31;
    for (u64 base = (u64)blockIdx.x * DS_THREADS; base < cap; base += stride) {
        u64 key = 0;
        double v = 0.0;
        const int c = cs_slot_chrom(tkeys, tval, cap, base + threadIdx.x, cstarts, nchrom, &key, &v);
        const unsigned grp = __match_any_sync(CS_FULL, c);
        const int leader = __ffs(grp) - 1;
        u64 pos = 0;
        if (c >= 0 && lane == leader) pos = atomicAdd(cursor + c, (u64)__popc(grp));
        pos = __shfl_sync(CS_FULL, pos, leader) + (u64)__popc(grp & ((1u << lane) - 1));
        if (c >= 0) {
            const int s0 = __ldg(cstarts + c);
            ov[pos] = v; oi[pos] = (int)(key >> 31) - s0; oj[pos] = (int)(key & 0x7fffffffULL) - s0;
        }
    }
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

// ingest.cu: a handle with chrom_bins[nchrom] bins per chromosome and no buckets yet; TP_ERR_ARG naming `who` when
// nchrom is outside 1..2^20, a chromosome has < 1 bin, the total is >= 2^31 - 1 or index_base is not 0 or 1
int genome_new(const int32_t *chrom_bins, int nchrom, int index_base, const char *who, tp_genome **out);
