// difft.cu -- stage 6: diffT (reference R/DiffT.R:41-49) on padded per-bin TAD labels.
//
// The reference, for every bin b, builds two length-L logical vectors
//     x = tad_x[b] != tad_x | tad_x[b] == 0 ,   y = likewise for tad_y
// and scores sum(xor(x, y)): O(L^2) per pair.  With SX(b) = {j : tad_x[j] == tad_x[b] != 0} (empty
// for an uncovered bin) and SY(b) likewise, xor(x, y) is TRUE exactly on the symmetric
// difference of SX and SY, so
//     score[b] = |SX| + |SY| - 2 |SX & SY| = cnt_x[lx] + cnt_y[ly] - 2 joint[lx, ly]
// which needs only three label histograms: O(L) per pair and HBM-bound (16 L bytes per pair).
// One CTA per pair; the histograms live in one shared-memory hash table (keys tagged x-only /
// y-only / joint), filled with warp-aggregated atomics because consecutive bins share labels.
// All arithmetic is integer until the final division, so results are bit-identical to R.
#include <algorithm>
#include "common.cuh"
#include "philox.cuh"

#define DT_THREADS 256
#define DT_EMPTY 0xffffffffffffffffULL

__device__ __forceinline__ unsigned dt_hash(unsigned long long key) {
    key ^= key >> 33; key *= 0xff51afd7ed558ccdULL; key ^= key >> 33;
    return (unsigned)key;
}

__device__ __forceinline__ bool dt_add(unsigned long long *keys, int *vals, unsigned mask,
                                       unsigned long long key, int cnt) {
    unsigned s = dt_hash(key) & mask;
    for (unsigned probe = 0; probe <= mask; probe++) {
        unsigned long long old = keys[s];
        if (old != key) {
            if (old != DT_EMPTY) { s = (s + 1) & mask; continue; }
            old = atomicCAS(&keys[s], DT_EMPTY, key);
            if (old != DT_EMPTY && old != key) { s = (s + 1) & mask; continue; }
        }
        atomicAdd(&vals[s], cnt);
        return true;
    }
    return false;
}

__device__ __forceinline__ int dt_get(const unsigned long long *keys, const int *vals, unsigned mask,
                                      unsigned long long key) {
    unsigned s = dt_hash(key) & mask;
    for (unsigned probe = 0; probe <= mask; probe++) {
        unsigned long long old = keys[s];
        if (old == key) return vals[s];
        if (old == DT_EMPTY) return 0;
        s = (s + 1) & mask;
    }
    return 0;
}

// add `key` once per distinct value in the warp, with the number of lanes holding it
__device__ __forceinline__ bool dt_add_aggregated(unsigned long long *keys, int *vals, unsigned mask,
                                                  unsigned long long key, bool active) {
    unsigned amask = __ballot_sync(0xffffffffu, active);
    bool ok = true;
    if (active) {
        unsigned peers = __match_any_sync(amask, key);
        if ((int)(threadIdx.x & 31) == __ffs(peers) - 1) ok = dt_add(keys, vals, mask, key, __popc(peers));
    }
    return ok;
}

__device__ __forceinline__ long long dt_score(const unsigned long long *keys, const int *vals, unsigned mask,
                                              int lx, int ly) {
    long long s = 0;
    if (lx != 0) s += dt_get(keys, vals, mask, ((unsigned long long)(unsigned)(lx + 1) << 32));
    if (ly != 0) s += dt_get(keys, vals, mask, (unsigned long long)(unsigned)(ly + 1));
    if (lx != 0 && ly != 0)
        s -= 2LL * dt_get(keys, vals, mask, ((unsigned long long)(unsigned)(lx + 1) << 32) | (unsigned)(ly + 1));
    return s;
}

// GLOBAL_TABLE = false: table in shared memory; a pair whose labels do not fit is appended to
// `overflow` (count in overflow[0]) and left for a second launch with GLOBAL_TABLE = true, where
// `pair_list` names the pairs and each CTA owns `slots` entries of a global table.
// poff (ragged pairs, tp_difft_multi): pair p has length poff[p+1] - poff[p] and its labels, curve and those of x at
// poff[p]; Lfixed and xstride are then unused.  Otherwise every pair has length Lfixed, its labels and curve at
// pair * Lfixed, its x labels at pair * xstride.
template <bool GLOBAL_TABLE>
__global__ void __launch_bounds__(DT_THREADS)
difft_kernel(const int *__restrict__ labx, size_t xstride, const int *__restrict__ laby, int Lfixed, int npairs,
             double *__restrict__ out, double *__restrict__ totals, unsigned slots,
             unsigned long long *__restrict__ gkeys, int *__restrict__ gvals,
             const int *__restrict__ pair_list, int *__restrict__ overflow, const long long *__restrict__ poff) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    unsigned long long *keys = GLOBAL_TABLE ? gkeys + (size_t)blockIdx.x * slots : (unsigned long long *)smem_raw;
    int *vals = GLOBAL_TABLE ? gvals + (size_t)blockIdx.x * slots : (int *)(keys + slots);
    const unsigned mask = slots - 1;
    __shared__ long long s_warp[DT_THREADS / 32];
    __shared__ long long s_carry;
    __shared__ long long s_total;
    __shared__ int s_overflow;
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;

    for (int pi = blockIdx.x; pi < npairs; pi += gridDim.x) {
        const int pair = pair_list ? pair_list[pi] : pi;
        const size_t base = poff ? (size_t)poff[pair] : (size_t)pair * Lfixed;
        const int L = poff ? (int)(poff[pair + 1] - poff[pair]) : Lfixed;
        const int *lx = labx + (poff ? base : (size_t)pair * xstride), *ly = laby + base;
        double *o = out ? out + base : nullptr;
        {
            for (unsigned s = tid; s <= mask; s += DT_THREADS) { keys[s] = DT_EMPTY; vals[s] = 0; }
            if (tid == 0) { s_overflow = 0; s_total = 0; s_carry = 0; }
            __syncthreads();
            // pass 1: histograms
            bool ok = true;
            for (int b0 = 0; b0 < L; b0 += DT_THREADS) {
                const int b = b0 + tid;
                const bool act = b < L;
                const int x = act ? lx[b] : 0, y = act ? ly[b] : 0;
                ok &= dt_add_aggregated(keys, vals, mask, ((unsigned long long)(unsigned)(x + 1) << 32), act && x != 0);
                ok &= dt_add_aggregated(keys, vals, mask, (unsigned long long)(unsigned)(y + 1), act && y != 0);
                ok &= dt_add_aggregated(keys, vals, mask,
                                        ((unsigned long long)(unsigned)(x + 1) << 32) | (unsigned)(y + 1),
                                        act && x != 0 && y != 0);
            }
            if (!ok) s_overflow = 1;
            __syncthreads();
            if (s_overflow) {           // table too small for this pair: leave it to the second launch
                if (tid == 0 && overflow) overflow[1 + atomicAdd(&overflow[0], 1)] = pair;
                __syncthreads();
                continue;
            }
        }
        // total = sum over bins of score = sum over joint keys of count * score(key), plus the bins
        // with a zero label on one side; simplest exact form: one more pass over the bins.
        long long part = 0;
        for (int b = tid; b < L; b += DT_THREADS) part += dt_score(keys, vals, mask, lx[b], ly[b]);
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) part += __shfl_xor_sync(0xffffffffu, part, off);
        if (lane == 0) atomicAdd((unsigned long long *)&s_total, (unsigned long long)part);
        __syncthreads();
        const long long total = s_total;
        const double dtotal = (double)total;
        if (totals && tid == 0) totals[pair] = dtotal;
        if (!o) { __syncthreads(); continue; }
        // pass 2: per-bin score, inclusive scan, normalise
        for (int b0 = 0; b0 < L; b0 += DT_THREADS) {
            const int b = b0 + tid;
            long long v = (b < L) ? dt_score(keys, vals, mask, lx[b], ly[b]) : 0;
#pragma unroll
            for (int off = 1; off < 32; off <<= 1) {
                long long u = __shfl_up_sync(0xffffffffu, v, off);
                if (lane >= off) v += u;
            }
            if (lane == 31) s_warp[wid] = v;
            __syncthreads();
            long long base = s_carry;
            for (int w = 0; w < wid; w++) base += s_warp[w];
            v += base;
            if (b < L) o[b] = (total != 0) ? (double)v / dtotal : (double)v;
            __syncthreads();
            if (tid == DT_THREADS - 1) s_carry = v;
            __syncthreads();
        }
        __syncthreads();
    }
}

// device pointers in, device pointers out; dout (npairs x L) and dtotals (npairs) may each be null; xstride = L for
// per-pair x labels, 0 when every pair is scored against the same x.  dpoff: ragged pairs (see difft_kernel), L is then
// the longest of them
static int difft_device(tp_ctx *ctx, const int *dx, size_t xstride, const int *dy, int L, int npairs, double *dout,
                        double *dtotals, const long long *dpoff = nullptr) {
    cudaStream_t st = ctx->stream;
    const unsigned smem_slots = 4096;                       // 48 KB: 4 CTAs per SM
    const size_t smem = (size_t)smem_slots * 12;
    int grid = npairs < ctx->sm_count * 4 ? npairs : ctx->sm_count * 4;
    TP_TRY(ctx->dhash.reserve((size_t)(npairs + 1) * sizeof(int)));
    int *d_over = ctx->dhash.as<int>();
    TP_CUDA(cudaMemsetAsync(d_over, 0, sizeof(int), st));
    TP_CUDA(tp_optin_smem(difft_kernel<false>, ctx));
    TP_MARK(ctx, EV_DIFFT0);
    tp_prof_begin(ctx, PC_DIFFT);
    difft_kernel<false><<<grid, DT_THREADS, smem, st>>>(dx, xstride, dy, L, npairs, dout, dtotals, smem_slots, nullptr,
                                                       nullptr, nullptr, d_over, dpoff);
    tp_prof_end(ctx);
    ctx->launches += 1;
    TP_CUDA(cudaGetLastError());
    int nover = 0;
    TP_CUDA(cudaMemcpyAsync(&nover, d_over, sizeof(int), cudaMemcpyDeviceToHost, st));
    TP_CUDA(tp_stream_sync(ctx));
    if (nover > 0) {
        // pairs with more distinct labels than the shared table holds: global tables, <= 3L keys
        unsigned gslots = 1024;
        while (gslots < 6u * (unsigned)L) gslots <<= 1;
        int grid2 = nover < 64 ? nover : 64;
        TP_TRY(ctx->lhash.reserve((size_t)grid2 * gslots * 12));
        unsigned long long *gkeys = ctx->lhash.as<unsigned long long>();
        int *gvals = (int *)(gkeys + (size_t)grid2 * gslots);
        difft_kernel<true><<<grid2, DT_THREADS, 0, st>>>(dx, xstride, dy, L, nover, dout, dtotals, gslots, gkeys, gvals,
                                                        d_over + 1, nullptr, dpoff);
        ctx->launches += 1;
        TP_CUDA(cudaGetLastError());
    }
    TP_MARK(ctx, EV_DIFFT1);
    return TP_OK;
}

int tp_difft_batch(tp_ctx *ctx, const int32_t *labels_x, const int32_t *labels_y, int L, int npairs,
                   int on_device, double *out) {
    TP_ARG(ctx && labels_x && labels_y && out, "tp_difft_batch: null argument");
    TP_ARG(L >= 1 && npairs >= 0, "tp_difft_batch: bad sizes");
    if (npairs == 0) return TP_OK;
    TP_CUDA(cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->stream;
    const size_t nl = (size_t)npairs * L;
    const int *dx = labels_x, *dy = labels_y;
    double *dout = out;
    if (!on_device) {
        TP_TRY(ctx->lx.reserve(nl * sizeof(int)));
        TP_TRY(ctx->ly.reserve(nl * sizeof(int)));
        TP_TRY(ctx->dout.reserve(nl * sizeof(double)));
        TP_CUDA(cudaMemcpyAsync(ctx->lx.p, labels_x, nl * sizeof(int), cudaMemcpyHostToDevice, st));
        TP_CUDA(cudaMemcpyAsync(ctx->ly.p, labels_y, nl * sizeof(int), cudaMemcpyHostToDevice, st));
        dx = ctx->lx.as<int>(); dy = ctx->ly.as<int>(); dout = ctx->dout.as<double>();
    }
    TP_TRY(difft_device(ctx, dx, (size_t)L, dy, L, npairs, dout, nullptr));
    if (!on_device) TP_CUDA(cudaMemcpyAsync(out, dout, nl * sizeof(double), cudaMemcpyDeviceToHost, st));
    TP_CUDA(tp_stream_sync(ctx));
    return TP_OK;
}

// ---- diffT null distribution: random_bed (R/DiffT.R:61-73) on the device ----------------------------------------
//
//   bins    <- (start:end)[-bad_columns]                 positions that may carry a border
//   borders <- sort(sample(bins[-1], nrow(bed) - 1))     T - 1 of them, without replacement, never the first one
//   start   =  c(start, borders - 1) ; end = c(borders - 2, start + size - 1)
//
// so TAD t covers [border_{t-1} - 1, border_t - 2] and, through bin_index (later rows overwrite earlier ones,
// R/DiffT.R:1-9), the label of the bin at 0-based offset o from `start` is 1 + #{borders <= start + o + 1}.
// One CTA per permutation.  A uniformly random (T-1)-subset of the M candidate positions = the T-1 candidates with
// the smallest of M independent random keys: key(p) = first 64 bits of Philox4x32-10(counter = (p, perm, 0, 0x7ad),
// key = seed), ties by position.  The (T-1)-th smallest key is found by an 8-pass radix select (256-bin shared
// histograms, keys regenerated on the fly -- nothing is stored or sorted), then one scan over the positions writes
// the sorted borders and the label vector.  R's Mersenne-Twister stream cannot be reproduced, so draws differ from
// R's sample(); the distribution (uniform subsets) is the same, and the oracle restates this generator exactly.
__host__ __device__ __forceinline__ unsigned long long philox_key64(unsigned c0, unsigned c1, unsigned long long seed) {
    return philox4x32_key64(c0, c1, 0u, 0x7adu, seed);
}

#define RP_THREADS 256
// The (nborders)-th smallest key of the allowed positions (radix select, most significant byte first: after pass b the
// top (b + 1) bytes of the threshold key are known) -> *thr, and how many keys equal to it are taken -> *need_eq (the
// lowest positions first).  Every thread of the CTA calls it; hist[256], s_prefix and s_need are shared scratch.
__device__ __forceinline__ void rp_threshold(const unsigned char *__restrict__ allowed, int size, int nborders,
                                             unsigned long long seed, unsigned pc, int *hist, unsigned long long *s_prefix,
                                             int *s_need, unsigned long long *thr, int *need_eq) {
    const int tid = threadIdx.x;
    if (tid == 0) { *s_prefix = 0ULL; *s_need = nborders; }
    __syncthreads();
    for (int byte = 7; byte >= 0 && nborders > 0; byte--) {
        hist[tid] = 0;
        __syncthreads();
        const unsigned long long prefix = *s_prefix;
        const int sh = byte * 8;
        for (int p = tid; p < size; p += RP_THREADS) {
            if (!allowed[p]) continue;
            const unsigned long long k = philox_key64((unsigned)p, pc, seed);
            if (byte == 7 || (k >> (sh + 8)) == (prefix >> (sh + 8))) atomicAdd(&hist[(unsigned)(k >> sh) & 255u], 1);
        }
        __syncthreads();
        if (tid == 0) {
            int need = *s_need, b = 0;
            while (b < 255 && hist[b] < need) { need -= hist[b]; b++; }
            *s_need = need;                                  // how many of the keys sharing the new prefix are wanted
            *s_prefix = prefix | ((unsigned long long)b << sh);
        }
        __syncthreads();
    }
    *thr = *s_prefix;
    *need_eq = *s_need;
}

// allowed[size]: 1 = the position may carry a border (not a bad column, not the first kept bin)
__global__ void __launch_bounds__(RP_THREADS)
random_partition_kernel(const unsigned char *__restrict__ allowed, int size, int nborders, unsigned long long seed,
                        int perm0, int pad_left, int pad_right, int *__restrict__ labels, int *__restrict__ borders) {
    __shared__ int hist[256];
    __shared__ unsigned long long s_prefix;
    __shared__ int s_need;
    __shared__ int s_warp[RP_THREADS / 32][2];
    __shared__ int s_carry[2];
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    const int perm = blockIdx.x;
    const unsigned pc = (unsigned)(perm0 + perm);
    const int L = pad_left + size + pad_right;
    int *lab = labels + (size_t)perm * L;
    int *bor = borders ? borders + (size_t)perm * nborders : nullptr;
    unsigned long long thr;
    int need_eq;
    rp_threshold(allowed, size, nborders, seed, pc, hist, &s_prefix, &s_need, &thr, &need_eq);
    if (tid == 0) { s_carry[0] = 0; s_carry[1] = 0; }
    __syncthreads();
    // one pass over the positions in order: selected flags -> running count -> borders and labels.
    // label(o) = 1 + #{selected positions <= o + 1}, so the count is needed one position ahead.
    for (int p0 = 0; p0 < size + 1; p0 += RP_THREADS) {
        const int p = p0 + tid;                              // position whose flag this thread evaluates
        int lt = 0, eq = 0;
        if (p < size && nborders > 0 && allowed[p]) {
            const unsigned long long k = philox_key64((unsigned)p, pc, seed);
            lt = k < thr; eq = k == thr;
        }
        int ilt = lt, ieq = eq;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int a = __shfl_up_sync(0xffffffffu, ilt, o), b = __shfl_up_sync(0xffffffffu, ieq, o);
            if (lane >= o) { ilt += a; ieq += b; }
        }
        if (lane == 31) { s_warp[wid][0] = ilt; s_warp[wid][1] = ieq; }
        __syncthreads();
        int blt = s_carry[0], beq = s_carry[1];
        for (int w = 0; w < wid; w++) { blt += s_warp[w][0]; beq += s_warp[w][1]; }
        ilt += blt; ieq += beq;                              // inclusive counts up to p over the whole permutation
        const int eq_taken_incl = ieq < need_eq ? ieq : need_eq;
        const int sel = lt || (eq && ieq <= need_eq);
        const int cnt_incl = ilt + eq_taken_incl;            // selected positions <= p
        if (sel && bor) bor[cnt_incl - 1] = p;               // offset of the border bin from `start`
        if (p >= 1 && p <= size) lab[pad_left + p - 1] = 1 + cnt_incl;       // bin at offset p - 1 sees borders <= p
        __syncthreads();
        if (tid == RP_THREADS - 1) { s_carry[0] = ilt; s_carry[1] = ieq; }
        __syncthreads();
    }
    for (int i = tid; i < pad_left; i += RP_THREADS) lab[i] = 1;                          // R/DiffT.R:31,34
    for (int i = tid; i < pad_right; i += RP_THREADS) lab[pad_left + size + i] = nborders + 1;   // max(tad) = T
}

int tp_difft_null(tp_ctx *ctx, const int32_t *labels_x, int L, int pad_left, int pad_right, int ntads,
                  const int32_t *bad_positions, int nbad, unsigned long long seed, int nperm,
                  int32_t *borders_out, int32_t *labels_out, double *curves_out, double *totals_out) {
    TP_ARG(ctx && labels_x, "tp_difft_null: null argument");
    TP_ARG(L >= 1 && pad_left >= 0 && pad_right >= 0 && pad_left + pad_right < L, "tp_difft_null: bad extent");
    TP_ARG(ntads >= 1 && nperm >= 0 && nbad >= 0 && (nbad == 0 || bad_positions), "tp_difft_null: bad sizes");
    if (nperm == 0) return TP_OK;
    const int size = L - pad_left - pad_right;
    // (start:end)[-bad_columns] then bins[-1]: positions that may carry a border
    std::vector<unsigned char> allowed((size_t)size, 1);
    for (int i = 0; i < nbad; i++) {
        const int p = bad_positions[i];
        TP_ARG(p != 0, "tp_difft_null: bad_columns are 1-based positions");
        if (p >= 1 && p <= size) allowed[p - 1] = 0;           // out-of-range negative subscripts are ignored by R
    }
    int m = 0, first = -1;
    for (int p = 0; p < size; p++) if (allowed[p]) { if (first < 0) first = p; m++; }
    if (first >= 0) { allowed[first] = 0; m--; }
    if (ntads - 1 > m) {
        tp_set_error("tp_difft_null: cannot take a sample larger than the population (%d borders from %d bins; "
                     "sample() errors here, R/DiffT.R:69)", ntads - 1, m);
        return TP_ERR_ARG;
    }
    TP_CUDA(cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->stream;
    const size_t nl = (size_t)nperm * L;
    const int nb = ntads - 1;
    TP_TRY(ctx->lx.reserve((size_t)L * sizeof(int) + (size_t)size + 64));
    TP_TRY(ctx->ly.reserve(nl * sizeof(int) + (size_t)nperm * (nb + 1) * sizeof(int)));
    if (curves_out) TP_TRY(ctx->dout.reserve(nl * sizeof(double)));
    TP_TRY(ctx->qtmp.reserve((size_t)(nperm + 4) * sizeof(double)));
    int *dx = ctx->lx.as<int>();
    unsigned char *dallowed = (unsigned char *)(dx + L);
    int *dy = ctx->ly.as<int>();
    int *dbor = dy + nl;
    double *dtot = ctx->qtmp.as<double>();
    TP_CUDA(cudaMemcpyAsync(dx, labels_x, (size_t)L * sizeof(int), cudaMemcpyHostToDevice, st));
    TP_CUDA(cudaMemcpyAsync(dallowed, allowed.data(), (size_t)size, cudaMemcpyHostToDevice, st));
    tp_prof_begin(ctx, PC_DIFFT);
    random_partition_kernel<<<nperm, RP_THREADS, 0, st>>>(dallowed, size, nb, seed, 0, pad_left, pad_right, dy, dbor);
    tp_prof_end(ctx);
    TP_CUDA(cudaGetLastError());
    ctx->launches += 1;
    TP_TRY(difft_device(ctx, dx, 0, dy, L, nperm, curves_out ? ctx->dout.as<double>() : nullptr, dtot));
    if (borders_out && nb > 0) TP_CUDA(cudaMemcpyAsync(borders_out, dbor, (size_t)nperm * nb * sizeof(int), cudaMemcpyDeviceToHost, st));
    if (labels_out) TP_CUDA(cudaMemcpyAsync(labels_out, dy, nl * sizeof(int), cudaMemcpyDeviceToHost, st));
    if (curves_out) TP_CUDA(cudaMemcpyAsync(curves_out, ctx->dout.p, nl * sizeof(double), cudaMemcpyDeviceToHost, st));
    if (totals_out) TP_CUDA(cudaMemcpyAsync(totals_out, dtot, (size_t)nperm * sizeof(double), cudaMemcpyDeviceToHost, st));
    TP_CUDA(tp_stream_sync(ctx));
    return TP_OK;
}

// ---- tp_difft_multi: many diffT comparisons of different lengths, each with its own null distribution ---------------
//
// Observed pairs: difft_kernel over ragged pairs (poff), with the same shared-table / global-table overflow split.
// Null draws: one CTA per (problem, permutation) draws the partition exactly as random_partition_kernel does and scores
// it in the same CTA; only the total leaves the CTA.  With J the joint histogram of the (x, y) labels and cx / cy those
// of x / y over non-zero labels, the sum of the per-bin scores |SX| + |SY| - 2 |SX & SY| is
//     total = sum_t cx_t^2 + sum_u cy_u^2 - 2 sum_{t,u} J_tu^2 .
// sum cx^2 depends on x alone (host, once per problem).  A random partition's labels are non-decreasing over the padded
// extent, so y TAD u is one interval [s_u, s_u+1) whose ends follow from the sorted borders, kept in shared memory:
// sum cy^2 is one pass over the borders.  For J, the host lists the bins with a non-zero x label ordered by (label, bin)
// (xorder); in that order every non-zero J_tu is one run of equal (x label, y label), whatever the layout of x
// (overwritten rows, quirk Q11, included), and a run of n entries adds 1 + 3 + ... + (2n - 1) = n^2.  The y label of a
// bin is a binary search in the borders.  Integer arithmetic throughout: the totals are those of tp_difft_null.
struct DmProb {
    long long off;                  // labels of the problem in labx (and its observed curve in the curves)
    long long aoff;                 // allowed[size] flags in the allowed bytes
    long long xoff;                 // xorder[nnzx] in the xorder array
    long long cx2;                  // sum over non-zero x labels of their count squared
    unsigned long long seed;
    int L, pad_left, size, nb, nnzx, pad_;
};

__device__ __forceinline__ int dm_ylab(const int *bor, int nb, int pad_left, int size, int b) {
    if (b < pad_left) return 0;
    if (b >= pad_left + size) return nb;
    const int q = b - pad_left + 1;                          // bin at offset o sees the borders <= o + 1
    int lo = 0, hi = nb;
    while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        if (bor[mid] <= q) lo = mid + 1; else hi = mid;
    }
    return lo;
}

// gbor: null = borders in dynamic shared memory (bor_cap ints); else each CTA owns bor_cap ints of it
__global__ void __launch_bounds__(RP_THREADS)
difft_null_multi_kernel(const DmProb *__restrict__ probs, const int *__restrict__ run, long long nwork, int nperm,
                        const int *__restrict__ labx, const unsigned char *__restrict__ allowed_all,
                        const int *__restrict__ xorder_all, int *__restrict__ gbor, int bor_cap,
                        double *__restrict__ null_totals) {
    extern __shared__ __align__(16) int s_bor[];
    __shared__ int hist[256];
    __shared__ unsigned long long s_prefix;
    __shared__ int s_need;
    __shared__ int s_warp[RP_THREADS / 32][2];
    __shared__ int s_carry[2];
    __shared__ int s_gstart;
    __shared__ long long s_part[RP_THREADS / 32];
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    int *bor = gbor ? gbor + (size_t)blockIdx.x * bor_cap : s_bor;
    for (long long w = blockIdx.x; w < nwork; w += gridDim.x) {
        const int pi = run[w / nperm];
        const int perm = (int)(w % nperm);
        const DmProb P = probs[pi];
        const unsigned char *allowed = allowed_all + P.aoff;
        unsigned long long thr;
        int need_eq;
        rp_threshold(allowed, P.size, P.nb, P.seed, (unsigned)perm, hist, &s_prefix, &s_need, &thr, &need_eq);
        if (tid == 0) { s_carry[0] = 0; s_carry[1] = 0; s_gstart = 0; }
        __syncthreads();
        // the sorted borders, selected exactly as random_partition_kernel selects them
        for (int p0 = 0; p0 < P.size && P.nb > 0; p0 += RP_THREADS) {
            const int p = p0 + tid;
            int lt = 0, eq = 0;
            if (p < P.size && allowed[p]) {
                const unsigned long long k = philox_key64((unsigned)p, (unsigned)perm, P.seed);
                lt = k < thr; eq = k == thr;
            }
            int ilt = lt, ieq = eq;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const int a = __shfl_up_sync(0xffffffffu, ilt, o), b = __shfl_up_sync(0xffffffffu, ieq, o);
                if (lane >= o) { ilt += a; ieq += b; }
            }
            if (lane == 31) { s_warp[wid][0] = ilt; s_warp[wid][1] = ieq; }
            __syncthreads();
            int blt = s_carry[0], beq = s_carry[1];
            for (int v = 0; v < wid; v++) { blt += s_warp[v][0]; beq += s_warp[v][1]; }
            ilt += blt; ieq += beq;
            const int eq_taken_incl = ieq < need_eq ? ieq : need_eq;
            if (lt || (eq && ieq <= need_eq)) bor[ilt + eq_taken_incl - 1] = p;
            __syncthreads();
            if (tid == RP_THREADS - 1) { s_carry[0] = ilt; s_carry[1] = ieq; }
            __syncthreads();
        }
        // sum_u cy_u^2: y TAD u covers [s_u, s_u+1), s_0 = 0, s_u = pad_left + bor[u - 1] - 1, s_nb+1 = L
        long long acc = 0;
        for (int u = tid; u <= P.nb; u += RP_THREADS) {
            const long long a = u == 0 ? 0 : (long long)P.pad_left + bor[u - 1] - 1;
            const long long b = u == P.nb ? (long long)P.L : (long long)P.pad_left + bor[u] - 1;
            acc += (b - a) * (b - a);
        }
        // -2 sum J^2 over runs of equal (x label, y label) in xorder; the start of the run of entry i is a max-scan
        const int *lx = labx + P.off, *xo = xorder_all + P.xoff;
        for (int i0 = 0; i0 < P.nnzx; i0 += RP_THREADS) {
            const int i = i0 + tid;
            int start = -1;
            if (i < P.nnzx) {
                const int b = xo[i];
                if (i == 0) start = 0;
                else {
                    const int bp = xo[i - 1];
                    if (lx[b] != lx[bp] || dm_ylab(bor, P.nb, P.pad_left, P.size, b) != dm_ylab(bor, P.nb, P.pad_left, P.size, bp))
                        start = i;
                }
            }
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const int a = __shfl_up_sync(0xffffffffu, start, o);
                if (lane >= o && a > start) start = a;
            }
            if (lane == 31) s_warp[wid][0] = start;
            __syncthreads();
            int m = s_gstart;
            for (int v = 0; v < wid; v++) m = max(m, s_warp[v][0]);
            m = max(m, start);
            if (i < P.nnzx) acc -= 2LL * (2LL * (i - m) + 1);
            __syncthreads();
            if (tid == RP_THREADS - 1) s_gstart = m;
            __syncthreads();
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
        if (lane == 0) s_part[wid] = acc;
        __syncthreads();
        if (tid == 0) {
            long long total = P.cx2;
            for (int v = 0; v < RP_THREADS / 32; v++) total += s_part[v];
            null_totals[(size_t)pi * nperm + perm] = (double)total;
        }
        __syncthreads();
    }
}

static size_t dm_align(size_t x) { return (x + 15) & ~(size_t)15; }

int tp_difft_multi(tp_ctx *ctx, int nprob, const int64_t *off, const int32_t *labels_x, const int32_t *labels_y,
                   const int32_t *pad_left, const int32_t *pad_right, const int32_t *ntads, const int64_t *bad_off,
                   const int32_t *bad_positions, unsigned long long seed, int nperm, double *curves_out,
                   double *totals_out, double *null_totals_out, int *status_out) {
    TP_ARG(ctx && nprob >= 0 && nperm >= 0, "tp_difft_multi: bad sizes");
    if (nprob == 0) return TP_OK;
    TP_ARG(off && labels_x && labels_y && pad_left && pad_right && ntads && bad_off, "tp_difft_multi: null argument");
    TP_ARG(off[0] == 0 && bad_off[0] == 0, "tp_difft_multi: offsets must start at 0");
    int Lmax = 0;
    for (int p = 0; p < nprob; p++) {
        const long long L = off[p + 1] - off[p];
        TP_ARG(L >= 1 && L <= 0x7fffffffLL, "tp_difft_multi: every problem needs 1 <= L_p < 2^31 (offsets monotone)");
        TP_ARG(pad_left[p] >= 0 && pad_right[p] >= 0 && (long long)pad_left[p] + pad_right[p] < L,
               "tp_difft_multi: bad extent");
        TP_ARG(ntads[p] >= 1 && bad_off[p + 1] >= bad_off[p], "tp_difft_multi: bad sizes");
        if (L > Lmax) Lmax = (int)L;
    }
    const long long nbad_all = bad_off[nprob];
    TP_ARG(nbad_all == 0 || bad_positions, "tp_difft_multi: null bad_positions");
    for (long long i = 0; i < nbad_all; i++) TP_ARG(bad_positions[i] != 0, "tp_difft_multi: bad_columns are 1-based positions");
    const long long sumL = off[nprob];

    // host side, per problem: allowed flags and refusals exactly as tp_difft_null; xorder and sum cx^2 of x
    std::vector<DmProb> probs((size_t)nprob);
    std::vector<int> run, xorder, cnt;
    std::vector<unsigned char> allowed;
    std::vector<std::pair<int, int>> srt;
    int bor_cap = 1, nrefused = 0;
    for (int p = 0; p < nprob; p++) {
        DmProb &P = probs[p];
        P.off = off[p];
        P.L = (int)(off[p + 1] - off[p]);
        P.pad_left = pad_left[p];
        P.size = P.L - pad_left[p] - pad_right[p];
        P.nb = ntads[p] - 1;
        P.seed = seed + (unsigned long long)p;
        P.aoff = (long long)allowed.size();
        allowed.resize(allowed.size() + (size_t)P.size, 1);
        unsigned char *al = allowed.data() + P.aoff;
        for (long long i = bad_off[p]; i < bad_off[p + 1]; i++) {
            const int q = bad_positions[i];
            if (q >= 1 && q <= P.size) al[q - 1] = 0;
        }
        int m = 0, first = -1;
        for (int q = 0; q < P.size; q++) if (al[q]) { if (first < 0) first = q; m++; }
        if (first >= 0) { al[first] = 0; m--; }
        const int ok = P.nb <= m;
        if (status_out) status_out[p] = ok ? TP_OK : TP_ERR_ARG;
        if (!ok) {
            if (nrefused++ == 0)
                tp_set_error("tp_difft_multi: problem %d: cannot take a sample larger than the population (%d borders from "
                             "%d bins; sample() errors here, R/DiffT.R:69)", p, P.nb, m);
            allowed.resize((size_t)P.aoff);
            P.size = 0; P.nnzx = 0; P.xoff = (long long)xorder.size(); P.cx2 = 0;
            continue;
        }
        run.push_back(p);
        if (P.nb > bor_cap) bor_cap = P.nb;
        // bins with a non-zero x label ordered by (label, bin): a counting sort when the labels span a short range
        const int32_t *x = labels_x + off[p];
        int lo = 0x7fffffff, hi = -0x7fffffff - 1, nnz = 0;
        for (int b = 0; b < P.L; b++) if (x[b] != 0) { lo = x[b] < lo ? x[b] : lo; hi = x[b] > hi ? x[b] : hi; nnz++; }
        P.xoff = (long long)xorder.size();
        P.nnzx = nnz;
        P.cx2 = 0;
        xorder.resize(xorder.size() + (size_t)nnz);
        int *xo = xorder.data() + P.xoff;
        if (nnz == 0) continue;
        if ((long long)hi - lo <= 4LL * P.L + 16) {
            cnt.assign((size_t)(hi - lo) + 2, 0);
            for (int b = 0; b < P.L; b++) if (x[b] != 0) cnt[(size_t)(x[b] - lo) + 1]++;
            for (size_t v = 1; v < cnt.size(); v++) { P.cx2 += (long long)cnt[v] * cnt[v]; cnt[v] += cnt[v - 1]; }
            for (int b = 0; b < P.L; b++) if (x[b] != 0) xo[cnt[(size_t)(x[b] - lo)]++] = b;
        } else {
            srt.clear();
            for (int b = 0; b < P.L; b++) if (x[b] != 0) srt.emplace_back(x[b], b);
            std::sort(srt.begin(), srt.end());
            long long c = 0;
            for (int i = 0; i < nnz; i++) {
                xo[i] = srt[i].second;
                c++;
                if (i + 1 == nnz || srt[i + 1].first != srt[i].first) { P.cx2 += c * c; c = 0; }
            }
        }
    }
    const int nrun = (int)run.size();

    // one upload: problem table | run list | offsets | x labels | y labels | xorder | allowed flags
    size_t o_probs = 0, o_run = dm_align(o_probs + probs.size() * sizeof(DmProb));
    size_t o_off = dm_align(o_run + (size_t)nrun * sizeof(int));
    size_t o_lx = dm_align(o_off + (size_t)(nprob + 1) * sizeof(long long));
    size_t o_ly = dm_align(o_lx + (size_t)sumL * sizeof(int));
    size_t o_xo = dm_align(o_ly + (size_t)sumL * sizeof(int));
    size_t o_al = dm_align(o_xo + xorder.size() * sizeof(int));
    const size_t nblob = dm_align(o_al + allowed.size());
    std::vector<unsigned char> blob(nblob);
    memcpy(blob.data() + o_probs, probs.data(), probs.size() * sizeof(DmProb));
    if (nrun) memcpy(blob.data() + o_run, run.data(), (size_t)nrun * sizeof(int));
    memcpy(blob.data() + o_off, off, (size_t)(nprob + 1) * sizeof(long long));
    memcpy(blob.data() + o_lx, labels_x, (size_t)sumL * sizeof(int));
    memcpy(blob.data() + o_ly, labels_y, (size_t)sumL * sizeof(int));
    if (!xorder.empty()) memcpy(blob.data() + o_xo, xorder.data(), xorder.size() * sizeof(int));
    if (!allowed.empty()) memcpy(blob.data() + o_al, allowed.data(), allowed.size());

    TP_CUDA(cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->stream;
    const size_t nnull = (size_t)nprob * nperm;
    TP_TRY(ctx->lx.reserve(nblob));
    TP_TRY(ctx->qtmp.reserve(((size_t)nprob + nnull + 4) * sizeof(double)));
    if (curves_out) TP_TRY(ctx->dout.reserve((size_t)sumL * sizeof(double)));
    unsigned char *dblob = ctx->lx.as<unsigned char>();
    double *dtot = ctx->qtmp.as<double>(), *dnull = dtot + nprob;
    double *dcurves = curves_out ? ctx->dout.as<double>() : nullptr;
    TP_CUDA(cudaMemcpyAsync(dblob, blob.data(), nblob, cudaMemcpyHostToDevice, st));
    const int *dlx = (const int *)(dblob + o_lx);
    TP_TRY(difft_device(ctx, dlx, 0, (const int *)(dblob + o_ly), Lmax, nprob, dcurves, dtot,
                        (const long long *)(dblob + o_off)));
    const long long nwork = (long long)nrun * nperm;
    if (nwork > 0) {
        // borders in shared memory when the largest border count fits beside the kernel's static shared memory
        size_t smem = (size_t)bor_cap * sizeof(int);
        int *gbor = nullptr;
        long long grid = (long long)ctx->sm_count * 8;
        if (smem + 8192 > (size_t)ctx->max_smem_optin) {
            grid = (long long)ctx->sm_count * 4;
            if (grid > nwork) grid = nwork;
            TP_TRY(ctx->ly.reserve((size_t)grid * bor_cap * sizeof(int)));
            gbor = ctx->ly.as<int>();
            smem = 0;
        } else {
            TP_CUDA(tp_optin_smem(difft_null_multi_kernel, ctx));
        }
        if (grid > nwork) grid = nwork;
        tp_prof_begin(ctx, PC_DIFFT);
        difft_null_multi_kernel<<<(unsigned)grid, RP_THREADS, smem, st>>>(
            (const DmProb *)(dblob + o_probs), (const int *)(dblob + o_run), nwork, nperm, dlx,
            (const unsigned char *)(dblob + o_al), (const int *)(dblob + o_xo), gbor, bor_cap, dnull);
        tp_prof_end(ctx);
        ctx->launches += 1;
        TP_CUDA(cudaGetLastError());
    }
    if (curves_out) TP_CUDA(cudaMemcpyAsync(curves_out, dcurves, (size_t)sumL * sizeof(double), cudaMemcpyDeviceToHost, st));
    if (totals_out) TP_CUDA(cudaMemcpyAsync(totals_out, dtot, (size_t)nprob * sizeof(double), cudaMemcpyDeviceToHost, st));
    if (null_totals_out && nnull)
        TP_CUDA(cudaMemcpyAsync(null_totals_out, dnull, nnull * sizeof(double), cudaMemcpyDeviceToHost, st));
    TP_CUDA(tp_stream_sync(ctx));
    if (null_totals_out && nrefused) {
        for (int p = 0, r = 0; p < nprob; p++) {
            if (r < nrun && run[r] == p) { r++; continue; }
            for (int i = 0; i < nperm; i++) null_totals_out[(size_t)p * nperm + i] = NAN;
        }
    }
    return TP_OK;
}
