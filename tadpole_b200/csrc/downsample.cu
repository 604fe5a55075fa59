// downsample.cu -- equal-depth subsampling of genome-wide pixels (S0d): a uniform subset of exactly N of the cis reads of
// a tp_genome, drawn on the device that holds it, returned as a new tp_genome of raw integer counts.
//
// A cell is (c, i, j): chromosome c in bin-table order, chromosome-local bins i <= j.  Its count C is the sum of every
// bucket entry naming it (duplicates merge, as the dense build adds them) and it holds the reads (c, i, j, r), r < C.
//   key(read) = first 64 bits of Philox4x32-10(counter = (r, i, j, 0xD5000000 | c), key = seed)
// and the subsample of N contacts keeps the N reads with the smallest (key, c, i, j, r).  That is a uniform N-subset of
// the reads (the multivariate hypergeometric draw), and it depends on the merged cells, the seed and N only: not on the
// order of the bucket (decided by atomics in genome_bucket_kernel) nor on how a cell is split into duplicates.
//   1. ds_insert_kernel: every entry is checked (an integer in [0, 2^32): the lowest offending entry by atomicMin) and
//      added into an open-addressing table in HBM on (global i, global j); counts add with u64 atomics, so the merge is
//      exact in any order.  ds_compact_kernel lists the U cells with C > 0 (and the smallest key of a cell >= 2^32).
//   2. ds_scan_*: exclusive u64 scan of C = each cell's first read; T = total reads.
//   3. radix select of the N-th smallest key, 12-bit digits, 6 passes: no key is stored, every pass regenerates all T.
//      A CTA walks contiguous tiles of 4096 reads: a warp-wide 32-ary search finds the tile's first and last cell, the
//      tile's cell starts go to shared memory, and each thread walks 16 consecutive reads -- a cell of 10^7 reads spans
//      many CTAs.  ds_pick_kernel picks the digit on the device: the host is out of the pass loop.
//   4. ds_count_kernel: reads with key < K add to their cell; reads with key == K (almost always the N-th alone) go to a
//      small buffer and ds_ties_kernel keeps the first N - #below of them in (c, i, j, r) order.
//   5. cells that keep reads go into a new tp_genome through the per-chromosome histogram and cursor scatter of
//      genome_bucket (ingest.cu).
// All arithmetic is integer: the result is the same bits on every run.  Cost: (passes + 1) x T Philox evaluations plus
// three passes over the cells (N = 0 and N = T skip the select); memory: 16 bytes per table slot (2 slots per bucket
// entry, rounded up to a power of two) + 28 bytes per cell, the table released before the output is built.
#include <algorithm>
#include "genome_util.cuh"
#include "philox.cuh"

#define DS_ITEMS 16
#define DS_TILE (DS_THREADS * DS_ITEMS)      // reads per tile of the select passes; cells per tile of the scan
#define DS_DIGIT 12
#define DS_BINS (1 << DS_DIGIT)
#define DS_EMPTY 0xffffffffffffffffULL
#define DS_EQ_CAP 4096                       // reads whose key equals the threshold that are kept track of
#define DS_CHROM_TAG 0xD5000000u             // counter word 3 = tag | chromosome: a stream apart from diffT's (0x7ad)

typedef unsigned long long u64;

// status words of one call: [0] lowest entry that is no integer in [0, 2^32) [1] smallest key of a merged cell >= 2^32
// [2] cells listed [3] reads tied with the threshold  [4] selection prefix [5] reads still needed at the prefix
enum { DS_BAD = 0, DS_BIG, DS_NCELL, DS_NEQ, DS_PREFIX, DS_NEED, DS_NSTATUS = 8 };

__device__ __forceinline__ bool ds_is_count(double v) { return v >= 0.0 && v < 4294967296.0 && v == floor(v); }

// exclusive scan of one u64 per thread over the CTA; *total = the sum
__device__ __forceinline__ u64 ds_block_scan(u64 v, u64 *s_warp, u64 *total) {
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    u64 inc = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const u64 t = __shfl_up_sync(0xffffffffu, inc, o);
        if (lane >= o) inc += t;
    }
    __syncthreads();
    if (lane == 31) s_warp[wid] = inc;
    __syncthreads();
    u64 base = 0, tot = 0;
#pragma unroll
    for (int w = 0; w < DS_THREADS / 32; w++) {
        const u64 x = s_warp[w];
        if (w < wid) base += x;
        tot += x;
    }
    *total = tot;
    return base + inc - v;
}

// ---- depth: exact cis reads per chromosome ----------------------------------------------------------------------------
__global__ void __launch_bounds__(DS_THREADS)
ds_depth_kernel(const double *__restrict__ cnt, u64 m, const u64 *__restrict__ offs, int nchrom, u64 *__restrict__ depth,
                u64 *__restrict__ status) {
    const u64 stride = (u64)gridDim.x * DS_THREADS;
    for (u64 base = (u64)blockIdx.x * DS_THREADS; base < m; base += stride) {
        const u64 e = base + threadIdx.x;
        int c = -1;
        u64 v = 0;
        if (e < m) {
            const double x = cnt[e];
            if (ds_is_count(x)) { c = ds_chrom_of_entry(offs, nchrom, e); v = (u64)x; }
            else atomicMin(status + DS_BAD, e);
        }
        const unsigned grp = __match_any_sync(0xffffffffu, c);
        if (grp == 0xffffffffu) {                    // the usual case: 32 entries of one bucket
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
            if (threadIdx.x % 32 == 0 && c >= 0 && v) atomicAdd(depth + c, v);
        } else if (c >= 0 && v) {
            atomicAdd(depth + c, v);
        }
    }
}

// ---- 1. merge ---------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(DS_THREADS)
ds_insert_kernel(const double *__restrict__ cnt, const int *__restrict__ bi, const int *__restrict__ bj, u64 m,
                 const u64 *__restrict__ offs, const int *__restrict__ starts, int nchrom, u64 *__restrict__ tkeys,
                 u64 *__restrict__ tcnt, u64 mask, u64 *__restrict__ status) {
    const u64 stride = (u64)gridDim.x * DS_THREADS;
    for (u64 e = (u64)blockIdx.x * DS_THREADS + threadIdx.x; e < m; e += stride) {
        const double x = cnt[e];
        if (!ds_is_count(x)) { atomicMin(status + DS_BAD, e); continue; }
        if (x == 0.0) continue;                      // no reads
        const int c = ds_chrom_of_entry(offs, nchrom, e), s0 = __ldg(starts + c);
        const u64 key = ((u64)(unsigned)(s0 + bi[e]) << 31) | (u64)(unsigned)(s0 + bj[e]);
        u64 s = ds_hash(key) & mask;
        while (true) {
            u64 k = tkeys[s];
            if (k == DS_EMPTY) k = atomicCAS(tkeys + s, DS_EMPTY, key);
            if (k == DS_EMPTY || k == key) { atomicAdd(tcnt + s, (u64)x); break; }
            s = (s + 1) & mask;
        }
    }
}

// every occupied slot -> one cell (c, i, j, C); a merged count of 2^32 or more is an error
__global__ void __launch_bounds__(DS_THREADS)
ds_compact_kernel(const u64 *__restrict__ tkeys, const u64 *__restrict__ tcnt, u64 cap, const int *__restrict__ starts,
                  int nchrom, int *__restrict__ cc, int *__restrict__ ci, int *__restrict__ cj, unsigned *__restrict__ ccnt,
                  u64 *__restrict__ status) {
    const u64 stride = (u64)gridDim.x * DS_THREADS;
    const int lane = threadIdx.x & 31;
    for (u64 base = (u64)blockIdx.x * DS_THREADS; base < cap; base += stride) {
        const u64 s = base + threadIdx.x;
        const u64 key = s < cap ? tkeys[s] : DS_EMPTY;
        bool ok = key != DS_EMPTY;
        u64 n = 0;
        if (ok) {
            n = tcnt[s];
            if (n >= (1ULL << 32)) { atomicMin(status + DS_BIG, key); ok = false; }
        }
        const unsigned b = __ballot_sync(0xffffffffu, ok);
        u64 pos = 0;
        if (lane == 0 && b) pos = atomicAdd(status + DS_NCELL, (u64)__popc(b));
        pos = __shfl_sync(0xffffffffu, pos, 0) + __popc(b & ((1u << lane) - 1));
        if (ok) {
            const int gi = (int)(key >> 31), gj = (int)(key & 0x7fffffffULL), c = ds_chrom_of_bin(starts, nchrom, gi);
            const int s0 = __ldg(starts + c);
            cc[pos] = c; ci[pos] = gi - s0; cj[pos] = gj - s0; ccnt[pos] = (unsigned)n;
        }
    }
}

// ---- 2. first read of every cell ---------------------------------------------------------------------------------------
__global__ void __launch_bounds__(DS_THREADS)
ds_scan_tiles_kernel(const unsigned *__restrict__ ccnt, u64 U, u64 *__restrict__ tile_sum) {
    __shared__ u64 s_warp[DS_THREADS / 32];
    const u64 b0 = (u64)blockIdx.x * DS_TILE + (u64)threadIdx.x * DS_ITEMS;
    u64 v = 0;
#pragma unroll
    for (int q = 0; q < DS_ITEMS; q++) if (b0 + q < U) v += ccnt[b0 + q];
    u64 tot;
    ds_block_scan(v, s_warp, &tot);
    if (threadIdx.x == 0) tile_sum[blockIdx.x] = tot;
}

// exclusive scan of the tile sums in place (one CTA); *total_out = T
__global__ void __launch_bounds__(DS_THREADS)
ds_scan_top_kernel(u64 *__restrict__ tile_sum, u64 ntiles, u64 *__restrict__ total_out) {
    __shared__ u64 s_warp[DS_THREADS / 32];
    u64 carry = 0;
    for (u64 b0 = 0; b0 < ntiles; b0 += DS_THREADS) {
        const u64 b = b0 + threadIdx.x;
        const u64 v = b < ntiles ? tile_sum[b] : 0;
        u64 tot;
        const u64 ex = ds_block_scan(v, s_warp, &tot);
        if (b < ntiles) tile_sum[b] = carry + ex;
        carry += tot;
    }
    if (threadIdx.x == 0) *total_out = carry;
}

__global__ void __launch_bounds__(DS_THREADS)
ds_scan_apply_kernel(const unsigned *__restrict__ ccnt, u64 U, const u64 *__restrict__ tile_base, u64 *__restrict__ off) {
    __shared__ u64 s_warp[DS_THREADS / 32];
    const u64 b0 = (u64)blockIdx.x * DS_TILE + (u64)threadIdx.x * DS_ITEMS;
    unsigned c[DS_ITEMS];
    u64 v = 0;
#pragma unroll
    for (int q = 0; q < DS_ITEMS; q++) { c[q] = b0 + q < U ? ccnt[b0 + q] : 0u; v += c[q]; }
    u64 tot;
    u64 run = tile_base[blockIdx.x] + ds_block_scan(v, s_warp, &tot);
#pragma unroll
    for (int q = 0; q < DS_ITEMS; q++) if (b0 + q < U) { off[b0 + q] = run; run += c[q]; }
}

// ---- 3./4. walking the reads ----------------------------------------------------------------------------------------------
// largest c in [0, U) with off[c] <= x (off[0] = 0 <= x); every lane of the warp calls it and gets the answer
__device__ __forceinline__ u64 ds_warp_cell_of(const u64 *__restrict__ off, u64 U, u64 x) {
    const int lane = threadIdx.x & 31;
    u64 lo = 0, hi = U;                                  // off[lo] <= x, and hi == U or off[hi] > x
    while (hi - lo > 32) {
        const u64 step = (hi - lo + 31) / 32, p = lo + (u64)lane * step;
        const unsigned b = __ballot_sync(0xffffffffu, p < hi && off[p] <= x);
        const u64 nlo = lo + (u64)(31 - __clz((int)b)) * step;
        hi = nlo + step < hi ? nlo + step : hi;
        lo = nlo;
    }
    const unsigned b = __ballot_sync(0xffffffffu, lo + lane < hi && off[lo + lane] <= x);
    return lo + (u64)(31 - __clz((int)b));
}

struct DsCells {
    const int *c, *i, *j;
    const unsigned *cnt;
    const u64 *off;      // U + 1 entries: off[U] = T
    u64 U, T;
    u64 seed;
};

struct DsTile {
    unsigned rel[DS_TILE];       // cell starts relative to the tile (0 for the cell the tile starts in)
    u64 cell0, cell1;            // first and last cell of the tile
};

// Load tile t into shared memory, then f(cell, key, read index within the cell) for this thread's DS_ITEMS consecutive
// reads, and flush(cell) each time the thread leaves a cell and at its end.
template <class F, class G>
__device__ __forceinline__ void ds_tile_reads(const DsCells &C, u64 t, DsTile &s, F f, G flush) {
    const u64 t0 = t * DS_TILE, t1 = t0 + DS_TILE < C.T ? t0 + DS_TILE : C.T;
    const int wid = threadIdx.x >> 5;
    __syncthreads();                                     // the previous tile's cells are no longer read
    if (wid < 2) {
        const u64 cell = ds_warp_cell_of(C.off, C.U, wid == 0 ? t0 : t1 - 1);
        if ((threadIdx.x & 31) == 0) {
            if (wid == 0) s.cell0 = cell;
            else s.cell1 = cell;
        }
    }
    __syncthreads();
    const u64 cell0 = s.cell0;
    const int ncell = (int)(s.cell1 - cell0) + 1;        // every cell holds a read: at most DS_TILE
    for (int k = threadIdx.x; k < ncell; k += DS_THREADS) {
        const u64 o = C.off[cell0 + k];
        s.rel[k] = o <= t0 ? 0u : (unsigned)(o - t0);
    }
    __syncthreads();
    const unsigned r0 = threadIdx.x * DS_ITEMS;
    if (t0 + r0 >= t1) return;
    int lo = 0, hi = ncell - 1;                          // the cell of this thread's first read
    while (lo < hi) {
        const int mid = (lo + hi + 1) >> 1;
        if (s.rel[mid] <= r0) lo = mid; else hi = mid - 1;
    }
    int k = -1;
    unsigned ci = 0, cj = 0, ctag = 0;
    u64 cbeg = 0;
    const int nr = (int)(t1 - t0 - r0 < DS_ITEMS ? t1 - t0 - r0 : DS_ITEMS);
    for (int q = 0; q < nr; q++) {
        const unsigned rr = r0 + q;
        int kk = k < 0 ? lo : k;
        while (kk + 1 < ncell && s.rel[kk + 1] <= rr) kk++;
        if (kk != k) {
            if (k >= 0) flush(cell0 + k);
            k = kk;
            const u64 cell = cell0 + k;
            ci = (unsigned)C.i[cell]; cj = (unsigned)C.j[cell]; ctag = DS_CHROM_TAG | (unsigned)C.c[cell];
            cbeg = C.off[cell];
        }
        const unsigned r = (unsigned)(t0 + rr - cbeg);
        f(cell0 + k, philox4x32_key64(r, ci, cj, ctag, C.seed), r);
    }
    if (k >= 0) flush(cell0 + k);
}

// digit histogram of the keys that share the prefix found so far: bits [shift, shift + width) of every key whose bits
// above shift + width equal the prefix's
__global__ void __launch_bounds__(DS_THREADS)
ds_hist_kernel(DsCells C, int shift, int width, const u64 *__restrict__ status, u64 *__restrict__ ghist) {
    __shared__ DsTile s;
    __shared__ unsigned s_hist[DS_BINS];
    for (int b = threadIdx.x; b < DS_BINS; b += DS_THREADS) s_hist[b] = 0;
    const u64 prefix = status[DS_PREFIX];
    const int top = shift + width;
    const unsigned dmask = (1u << width) - 1u;
    const u64 ntiles = (C.T + DS_TILE - 1) / DS_TILE;
    for (u64 t = blockIdx.x; t < ntiles; t += gridDim.x)
        ds_tile_reads(C, t, s, [&](u64, u64 key, unsigned) {
            if (top >= 64 || (key >> top) == (prefix >> top)) atomicAdd(s_hist + ((unsigned)(key >> shift) & dmask), 1u);
        }, [](u64) {});
    __syncthreads();
    for (int b = threadIdx.x; b <= (int)dmask; b += DS_THREADS)
        if (s_hist[b]) atomicAdd(ghist + b, (u64)s_hist[b]);
}

// the digit in which the need-th smallest key of the prefix falls: prefix |= digit << shift, need -= keys below it
__global__ void __launch_bounds__(DS_THREADS)
ds_pick_kernel(const u64 *__restrict__ ghist, int shift, int width, u64 *__restrict__ status) {
    __shared__ u64 s_warp[DS_THREADS / 32];
    const int nb = 1 << width, per = nb >= DS_THREADS ? nb / DS_THREADS : 1;
    const int b0 = threadIdx.x * per, b1 = b0 + per < nb ? b0 + per : nb;
    const u64 need = status[DS_NEED];
    u64 v = 0;
    for (int b = b0; b < b1; b++) v += ghist[b];
    u64 tot;
    u64 cum = ds_block_scan(v, s_warp, &tot);
    if (cum < need && need <= cum + v) {
        for (int b = b0; b < b1; b++) {
            const u64 h = ghist[b];
            if (cum + h >= need) {
                status[DS_PREFIX] |= (u64)b << shift;
                status[DS_NEED] = need - cum;
                break;
            }
            cum += h;
        }
    }
}

// kept[cell] = reads of the cell with key < K; the reads with key == K are listed
__global__ void __launch_bounds__(DS_THREADS)
ds_count_kernel(DsCells C, u64 *__restrict__ status, unsigned *__restrict__ kept, u64 *__restrict__ eq_cell,
                unsigned *__restrict__ eq_r) {
    __shared__ DsTile s;
    const u64 K = status[DS_PREFIX];
    const u64 ntiles = (C.T + DS_TILE - 1) / DS_TILE;
    unsigned run = 0;
    for (u64 t = blockIdx.x; t < ntiles; t += gridDim.x)
        ds_tile_reads(C, t, s, [&](u64 cell, u64 key, unsigned r) {
            if (key < K) run++;
            else if (key == K) {
                const u64 q = atomicAdd(status + DS_NEQ, 1ULL);
                if (q < DS_EQ_CAP) { eq_cell[q] = cell; eq_r[q] = r; }
            }
        }, [&](u64 cell) {
            if (run) atomicAdd(kept + cell, run);
            run = 0;
        });
}

// the first `need` of the tied reads in (c, i, j, r) order are kept (one thread: there is almost always one tied read)
__global__ void ds_ties_kernel(DsCells C, const u64 *__restrict__ status, unsigned *__restrict__ kept,
                               u64 *__restrict__ eq_cell, unsigned *__restrict__ eq_r) {
    const u64 neq = status[DS_NEQ] < DS_EQ_CAP ? status[DS_NEQ] : DS_EQ_CAP;
    for (u64 n = status[DS_NEED]; n > 0; n--) {
        u64 best = DS_EMPTY;
        for (u64 q = 0; q < neq; q++) {
            if (eq_cell[q] == DS_EMPTY) continue;
            if (best == DS_EMPTY) { best = q; continue; }
            const u64 a = eq_cell[q], b = eq_cell[best];
            const int ca = C.c[a], cb = C.c[b], ia = C.i[a], ib = C.i[b], ja = C.j[a], jb = C.j[b];
            if (ca != cb ? ca < cb : ia != ib ? ia < ib : ja != jb ? ja < jb : eq_r[q] < eq_r[best]) best = q;
        }
        if (best == DS_EMPTY) return;
        kept[eq_cell[best]] += 1u;
        eq_cell[best] = DS_EMPTY;
    }
}

// ---- 5. the new buckets -----------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(DS_THREADS)
ds_out_hist_kernel(const int *__restrict__ cc, const unsigned *__restrict__ kept, u64 U, u64 *__restrict__ hist) {
    const u64 stride = (u64)gridDim.x * DS_THREADS;
    for (u64 base = (u64)blockIdx.x * DS_THREADS; base < U; base += stride) {
        const u64 u = base + threadIdx.x;
        const int c = u < U && kept[u] ? cc[u] : -1;
        const unsigned grp = __match_any_sync(0xffffffffu, c);
        if (c >= 0 && (threadIdx.x & 31) == __ffs(grp) - 1) atomicAdd(hist + c, (u64)__popc(grp));
    }
}

__global__ void __launch_bounds__(DS_THREADS)
ds_out_scatter_kernel(const int *__restrict__ cc, const int *__restrict__ ci, const int *__restrict__ cj,
                      const unsigned *__restrict__ kept, u64 U, u64 *__restrict__ cursor, double *__restrict__ ov,
                      int *__restrict__ oi, int *__restrict__ oj) {
    const u64 stride = (u64)gridDim.x * DS_THREADS;
    const int lane = threadIdx.x & 31;
    for (u64 base = (u64)blockIdx.x * DS_THREADS; base < U; base += stride) {
        const u64 u = base + threadIdx.x;
        const unsigned n = u < U ? kept[u] : 0u;
        const int c = n ? cc[u] : -1;
        const unsigned grp = __match_any_sync(0xffffffffu, c);
        const int leader = __ffs(grp) - 1;
        u64 pos = 0;
        if (c >= 0 && lane == leader) pos = atomicAdd(cursor + c, (u64)__popc(grp));
        pos = __shfl_sync(0xffffffffu, pos, leader) + (u64)__popc(grp & ((1u << lane) - 1));
        if (c >= 0) { ov[pos] = (double)n; oi[pos] = ci[u]; oj[pos] = cj[u]; }
    }
}

// ---- host side ------------------------------------------------------------------------------------------------------------
struct DsBufs {
    DevBuf aux, table, cells, kept, out_tmp;
    ~DsBufs() { aux.release(); table.release(); cells.release(); kept.release(); out_tmp.release(); }
};

// "chromosome c, bins (i, j)" of bucket entry e, and its count, read back for an error message
static int ds_entry(tp_ctx *m, const tp_genome *g, u64 e, int *c, int *i, int *j, double *v) {
    const u64 ncis = g->offs.back();
    const double *pv = g->px.as<double>();
    const int *pi = (const int *)(pv + ncis), *pj = pi + ncis;
    TP_CUDA(cudaMemcpyAsync(v, pv + e, 8, cudaMemcpyDeviceToHost, m->stream));
    TP_CUDA(cudaMemcpyAsync(i, pi + e, 4, cudaMemcpyDeviceToHost, m->stream));
    TP_CUDA(cudaMemcpyAsync(j, pj + e, 4, cudaMemcpyDeviceToHost, m->stream));
    TP_CUDA(tp_stream_sync(m));
    *c = (int)(std::upper_bound(g->offs.begin(), g->offs.end() - 1, e) - g->offs.begin()) - 1;
    return TP_OK;
}

static int ds_bad_entry(tp_ctx *m, const tp_genome *g, u64 e, const char *who) {
    int c = 0, i = 0, j = 0;
    double v = 0;
    TP_TRY(ds_entry(m, g, e, &c, &i, &j, &v));
    tp_set_error("%s: chromosome %d (0-based), bins (%d, %d) (0-based, chromosome-local): count %.17g is not an integer in "
                 "[0, 2^32); only read counts can be subsampled", who, c, i, j, v);
    return TP_ERR_ARG;
}

extern "C" int tp_genome_depth(tp_ctx *ctx, const tp_genome *g, unsigned long long *reads_out) {
    TP_ARG(ctx && g && reads_out, "tp_genome_depth: null argument");
    tp_ctx *m = nullptr;
    TP_TRY(ds_member(ctx, g, "tp_genome_depth", &m));
    TP_CUDA(cudaSetDevice(m->device));
    const int nchrom = (int)g->bins.size();
    const u64 ncis = g->offs.back();
    DevBuf aux;
    struct Rel { DevBuf &b; ~Rel() { b.release(); } } rel{aux};
    TP_TRY(aux.reserve((size_t)DS_NSTATUS * 8 + (size_t)nchrom * 8 + ((size_t)nchrom + 1) * 8));
    u64 *status = aux.as<u64>(), *depth = status + DS_NSTATUS, *doffs = depth + nchrom;
    TP_CUDA(cudaMemsetAsync(status, 0xff, 8, m->stream));
    TP_CUDA(cudaMemsetAsync(depth, 0, (size_t)nchrom * 8, m->stream));
    TP_CUDA(cudaMemcpyAsync(doffs, g->offs.data(), ((size_t)nchrom + 1) * 8, cudaMemcpyHostToDevice, m->stream));
    if (ncis) {
        ds_depth_kernel<<<ds_grid(m, ncis), DS_THREADS, 0, m->stream>>>(g->px.as<double>(), ncis, doffs, nchrom, depth, status);
        m->launches += 1;
        TP_CUDA(cudaGetLastError());
    }
    u64 bad = 0;
    TP_CUDA(cudaMemcpyAsync(&bad, status + DS_BAD, 8, cudaMemcpyDeviceToHost, m->stream));
    TP_CUDA(cudaMemcpyAsync(reads_out, depth, (size_t)nchrom * 8, cudaMemcpyDeviceToHost, m->stream));
    TP_CUDA(tp_stream_sync(m));
    if (bad != DS_EMPTY) return ds_bad_entry(m, g, bad, "tp_genome_depth");
    return TP_OK;
}

extern "C" int tp_genome_downsample(tp_ctx *ctx, const tp_genome *src, unsigned long long contacts,
                                    unsigned long long seed, tp_genome **out) {
    TP_ARG(ctx && src && out, "tp_genome_downsample: null argument");
    const char *who = "tp_genome_downsample";
    tp_ctx *m = nullptr;
    TP_TRY(ds_member(ctx, src, who, &m));
    TP_CUDA(cudaSetDevice(m->device));
    cudaStream_t st = m->stream;
    const int nchrom = (int)src->bins.size();
    const u64 ncis = src->offs.back();
    std::vector<int> starts((size_t)nchrom + 1, 0);
    for (int c = 0; c < nchrom; c++) starts[c + 1] = starts[c] + src->bins[c];

    DsBufs B;
    // status words, selection histogram, tied reads, bucket offsets, bin starts, output histogram and cursors
    const size_t aux_bytes = (size_t)DS_NSTATUS * 8 + (size_t)DS_BINS * 8 + (size_t)DS_EQ_CAP * 12 + ((size_t)nchrom + 1) * 8 +
                             ((size_t)nchrom + 1) * 4 + (size_t)nchrom * 16 + 64;
    TP_TRY(B.aux.reserve(aux_bytes));
    u64 *status = B.aux.as<u64>(), *ghist = status + DS_NSTATUS, *eq_cell = ghist + DS_BINS, *doffs = eq_cell + DS_EQ_CAP;
    u64 *ohist = doffs + nchrom + 1, *cursor = ohist + nchrom;
    unsigned *eq_r = (unsigned *)(cursor + nchrom);
    int *dstarts = (int *)(eq_r + DS_EQ_CAP);
    const u64 init[DS_NSTATUS] = {DS_EMPTY, DS_EMPTY, 0, 0, 0, 0, 0, 0};
    TP_CUDA(cudaMemcpyAsync(status, init, sizeof(init), cudaMemcpyHostToDevice, st));
    TP_CUDA(cudaMemcpyAsync(doffs, src->offs.data(), ((size_t)nchrom + 1) * 8, cudaMemcpyHostToDevice, st));
    TP_CUDA(cudaMemcpyAsync(dstarts, starts.data(), ((size_t)nchrom + 1) * 4, cudaMemcpyHostToDevice, st));
    TP_CUDA(cudaMemsetAsync(ohist, 0, (size_t)nchrom * 8, st));

    // 1. merge
    u64 cap = 1024;
    while (cap < 2 * ncis) cap <<= 1;
    TP_TRY(device_room(m, 16.0 * (double)cap + 28.0 * (double)ncis, 0, who, "the cell table and the cells"));
    TP_TRY(B.table.reserve((size_t)cap * 16));
    u64 *tkeys = B.table.as<u64>(), *tcnt = tkeys + cap;
    TP_CUDA(cudaMemsetAsync(tkeys, 0xff, (size_t)cap * 8, st));
    TP_CUDA(cudaMemsetAsync(tcnt, 0, (size_t)cap * 8, st));
    TP_TRY(B.cells.reserve((size_t)ncis * 24 + 64));
    int *cc = B.cells.as<int>(), *ci = cc + ncis, *cj = ci + ncis;
    unsigned *ccnt = (unsigned *)(cj + ncis);
    u64 *off = (u64 *)(((uintptr_t)(ccnt + ncis) + 15) & ~(uintptr_t)15);     // U + 1 entries
    if (ncis) {
        const double *pv = src->px.as<double>();
        const int *pi = (const int *)(pv + ncis), *pj = pi + ncis;
        ds_insert_kernel<<<ds_grid(m, ncis), DS_THREADS, 0, st>>>(pv, pi, pj, ncis, doffs, dstarts, nchrom, tkeys, tcnt, cap - 1,
                                                                 status);
        ds_compact_kernel<<<ds_grid(m, cap), DS_THREADS, 0, st>>>(tkeys, tcnt, cap, dstarts, nchrom, cc, ci, cj, ccnt, status);
        m->launches += 2;
        TP_CUDA(cudaGetLastError());
    }
    u64 hs[DS_NSTATUS];
    TP_CUDA(cudaMemcpyAsync(hs, status, sizeof(hs), cudaMemcpyDeviceToHost, st));
    TP_CUDA(tp_stream_sync(m));
    if (hs[DS_BAD] != DS_EMPTY) return ds_bad_entry(m, src, hs[DS_BAD], who);
    if (hs[DS_BIG] != DS_EMPTY) {
        const int gi = (int)(hs[DS_BIG] >> 31), gj = (int)(hs[DS_BIG] & 0x7fffffffULL);
        const int c = (int)(std::upper_bound(starts.begin(), starts.end() - 1, gi) - starts.begin()) - 1;
        tp_set_error("%s: chromosome %d (0-based), bins (%d, %d) (0-based, chromosome-local): the entries naming this cell add "
                     "up to 2^32 reads or more", who, c, gi - starts[c], gj - starts[c]);
        return TP_ERR_ARG;
    }
    B.table.release();
    const u64 U = hs[DS_NCELL];

    // 2. first read of every cell
    const u64 ntiles = (U + DS_TILE - 1) / DS_TILE;
    u64 T = 0;
    if (U) {
        TP_TRY(B.out_tmp.reserve((size_t)ntiles * 8));
        u64 *tile_sum = B.out_tmp.as<u64>();
        ds_scan_tiles_kernel<<<(unsigned)ntiles, DS_THREADS, 0, st>>>(ccnt, U, tile_sum);
        ds_scan_top_kernel<<<1, DS_THREADS, 0, st>>>(tile_sum, ntiles, off + U);
        ds_scan_apply_kernel<<<(unsigned)ntiles, DS_THREADS, 0, st>>>(ccnt, U, tile_sum, off);
        m->launches += 3;
        TP_CUDA(cudaGetLastError());
        TP_CUDA(cudaMemcpyAsync(&T, off + U, 8, cudaMemcpyDeviceToHost, st));
        TP_CUDA(tp_stream_sync(m));
    }
    if (contacts > T) {
        tp_set_error("%s: %llu contacts asked for, but the genome holds %llu cis contacts", who, contacts, T);
        return TP_ERR_ARG;
    }

    // 3./4. kept reads per cell
    const unsigned *kept = ccnt;                          // contacts == T: every read
    if (contacts < T && contacts > 0) {
        TP_TRY(B.kept.reserve((size_t)U * 4));
        unsigned *kk = B.kept.as<unsigned>();
        TP_CUDA(cudaMemsetAsync(kk, 0, (size_t)U * 4, st));
        const u64 need = contacts;
        TP_CUDA(cudaMemcpyAsync(status + DS_NEED, &need, 8, cudaMemcpyHostToDevice, st));
        DsCells C{cc, ci, cj, ccnt, off, U, T, seed};
        const u64 rtiles = (T + DS_TILE - 1) / DS_TILE;
        u64 grid = (u64)m->sm_count * 8;
        const u64 min_grid = (rtiles + (1ULL << 19) - 1) >> 19;       // at most 2^31 reads per CTA: u32 shared counters
        if (grid < min_grid) grid = min_grid;
        if (grid > rtiles) grid = rtiles;
        for (int top = 64; top > 0; top -= DS_DIGIT) {
            const int width = top < DS_DIGIT ? top : DS_DIGIT, shift = top - width;
            TP_CUDA(cudaMemsetAsync(ghist, 0, (size_t)DS_BINS * 8, st));
            ds_hist_kernel<<<(unsigned)grid, DS_THREADS, 0, st>>>(C, shift, width, status, ghist);
            ds_pick_kernel<<<1, DS_THREADS, 0, st>>>(ghist, shift, width, status);
            m->launches += 2;
        }
        ds_count_kernel<<<(unsigned)grid, DS_THREADS, 0, st>>>(C, status, kk, eq_cell, eq_r);
        ds_ties_kernel<<<1, 1, 0, st>>>(C, status, kk, eq_cell, eq_r);
        m->launches += 2;
        TP_CUDA(cudaGetLastError());
        kept = kk;
    }

    // 5. the new buckets
    GenomeOwnerDs own;
    own.g = new tp_genome();
    own.g->device = src->device;
    own.g->bins = src->bins;
    own.g->trans = src->trans;
    own.g->below = src->below;
    std::vector<u64> h((size_t)nchrom, 0);
    if (contacts > 0) {
        ds_out_hist_kernel<<<ds_grid(m, U), DS_THREADS, 0, st>>>(cc, kept, U, ohist);
        m->launches += 1;
        TP_CUDA(cudaGetLastError());
        TP_CUDA(cudaMemcpyAsync(h.data(), ohist, (size_t)nchrom * 8, cudaMemcpyDeviceToHost, st));
    }
    TP_CUDA(cudaMemcpyAsync(hs, status, sizeof(hs), cudaMemcpyDeviceToHost, st));
    TP_CUDA(tp_stream_sync(m));
    if (hs[DS_NEQ] > DS_EQ_CAP) {                      // 2^64 keys: practically never more than a handful tie
        tp_set_error("%s: %llu reads share the threshold key; at most %d are supported", who, hs[DS_NEQ], DS_EQ_CAP);
        return TP_ERR_ARG;
    }
    own.g->offs.assign((size_t)nchrom + 1, 0);
    for (int c = 0; c < nchrom; c++) own.g->offs[c + 1] = own.g->offs[c] + h[c];
    const u64 nout = own.g->offs[nchrom];
    TP_TRY(device_room(m, 16.0 * (double)nout, 0, who, "the buckets of the subsample"));
    TP_TRY(own.g->px.reserve((size_t)nout * 16 + 16));
    if (nout) {
        double *ov = own.g->px.as<double>();
        int *oi = (int *)(ov + nout), *oj = oi + nout;
        TP_CUDA(cudaMemcpyAsync(cursor, own.g->offs.data(), (size_t)nchrom * 8, cudaMemcpyHostToDevice, st));
        ds_out_scatter_kernel<<<ds_grid(m, U), DS_THREADS, 0, st>>>(cc, ci, cj, kept, U, cursor, ov, oi, oj);
        m->launches += 1;
        TP_CUDA(cudaGetLastError());
    }
    TP_CUDA(tp_stream_sync(m));
    *out = own.g;
    own.g = nullptr;
    return TP_OK;
}

extern "C" int tp_genome_pixels(tp_ctx *ctx, const tp_genome *g, int chrom, int32_t *i_out, int32_t *j_out,
                                double *count_out) {
    TP_ARG(ctx && g && i_out && j_out && count_out, "tp_genome_pixels: null argument");
    TP_ARG(chrom >= 0 && chrom < (int)g->bins.size(), "tp_genome_pixels: chromosome index out of range");
    tp_ctx *m = nullptr;
    TP_TRY(ds_member(ctx, g, "tp_genome_pixels", &m));
    TP_CUDA(cudaSetDevice(m->device));
    const u64 ncis = g->offs.back(), o = g->offs[(size_t)chrom], n = g->offs[(size_t)chrom + 1] - o;
    if (!n) return TP_OK;
    const double *pv = g->px.as<double>();
    const int *pi = (const int *)(pv + ncis), *pj = pi + ncis;
    TP_CUDA(cudaMemcpyAsync(count_out, pv + o, n * 8, cudaMemcpyDeviceToHost, m->stream));
    TP_CUDA(cudaMemcpyAsync(i_out, pi + o, n * 4, cudaMemcpyDeviceToHost, m->stream));
    TP_CUDA(cudaMemcpyAsync(j_out, pj + o, n * 4, cudaMemcpyDeviceToHost, m->stream));
    TP_CUDA(tp_stream_sync(m));
    return TP_OK;
}
