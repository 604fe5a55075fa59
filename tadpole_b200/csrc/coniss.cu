// coniss.cu -- stages 4 and 5: the find_params sweep (reference R/TADpole.R:104-123).
//
// Per candidate number of PCs i the reference builds dist(pcs[,1:i]) (O(n^2 i)) and runs
// rioja::chclust(method="coniss") on it.  CONISS on Euclidean data is Ward clustering restricted
// to ADJACENT clusters; every cluster is a contiguous interval of bins, so a cluster sum is a
// difference of two rows of a column-wise prefix sum P of the score matrix, and the same P
// (n+1 x k, L2 resident) serves every candidate: candidate i reads the first i columns.
//
//   dSS(A,B) = nA nB / (nA + nB) * sum_c (sumA_c / nA - sumB_c / nB)^2
//
// One warp owns one candidate.  The per-boundary dSS array lives in shared memory under a 32-ary
// min tree (block minima of 32 entries, two levels), so one merge step costs: descend the tree
// (ballots), two dot products over i columns (L2 loads + shuffle reduce), and re-reduce at most
// three leaf blocks.  Ties resolve to the lowest boundary index at every level, which is the
// reference's strict '<' scan.  The loop is serial in n by nature (SURVEY.md 7.3-2).
#include "common.cuh"

#define INF_D (__longlong_as_double(0x7ff0000000000000LL))

// boundary links live in shared memory when they fit, otherwise in global memory read through L2
template <bool SMEM, typename T> __device__ __forceinline__ int ld_link(const T *p) { return SMEM ? (int)*p : (int)__ldcg(p); }
template <bool SMEM, typename T> __device__ __forceinline__ void st_link(T *p, int v) { if (SMEM) *p = (T)v; else __stcg(p, (T)v); }

// ------------------------------------------------------------------------------------------
// prefix sums: P[0] = 0, P[r+1] = P[r] + scores[r]  (per column);  Qp[r+1] = Qp[r] + |scores[r]|^2
// ------------------------------------------------------------------------------------------
__global__ void rownorm2_kernel(const double *__restrict__ s, int n, int k, int ldk, double *__restrict__ out) {
    int w = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (w >= n) return;
    double a = 0.0;
    for (int c = lane; c < k; c += 32) { double v = s[(size_t)w * ldk + c]; a += v * v; }
    a = warp_sum(a);
    if (lane == 0) out[w] = a;
}

// Blocked scan over the bins: rows are cut into chunks of PF_CHUNK; (1) every (chunk, column) sums its rows, (2) every
// (chunk, column) adds up the sums of the chunks before it and writes its rows' prefixes.  Two launches of Nf / 128 x k / 64
// CTAs instead of one thread per column walking all Nf rows (0.40 ms at 2000 bins, ~5 ms at 25 000: the dependent adds of one
// thread); the order of the additions is fixed by the chunking, so every rank and every run gets the same bits.
// Column ldk is the squared row norms (rn2 -> Qp); columns k..ldk-1 are padding (zero).
#define PF_CHUNK 128
__global__ void __launch_bounds__(64)
prefix_sums_kernel(const double *__restrict__ s, const double *__restrict__ rn2, int n, int k, int ldk,
                   double *__restrict__ csum) {
    const int c = blockIdx.y * 64 + threadIdx.x, ch = blockIdx.x;
    if (c > ldk) return;
    const int r0 = ch * PF_CHUNK, r1 = min(n, r0 + PF_CHUNK);
    double a0 = 0.0, a1 = 0.0;
    if (c < k) {
        int r = r0;
        for (; r + 1 < r1; r += 2) { a0 += s[(size_t)r * ldk + c]; a1 += s[(size_t)(r + 1) * ldk + c]; }
        if (r < r1) a0 += s[(size_t)r * ldk + c];
    } else if (c == ldk) {
        int r = r0;
        for (; r + 1 < r1; r += 2) { a0 += rn2[r]; a1 += rn2[r + 1]; }
        if (r < r1) a0 += rn2[r];
    }
    csum[(size_t)ch * (ldk + 1) + c] = a0 + a1;
}
__global__ void __launch_bounds__(64)
prefix_write_kernel(const double *__restrict__ s, const double *__restrict__ rn2, const double *__restrict__ csum, int n, int k,
                    int ldk, double *__restrict__ P, double *__restrict__ Qp) {
    const int c = blockIdx.y * 64 + threadIdx.x, ch = blockIdx.x;
    if (c > ldk) return;
    const int r0 = ch * PF_CHUNK, r1 = min(n, r0 + PF_CHUNK);
    double acc = 0.0;
    for (int q = 0; q < ch; q++) acc += csum[(size_t)q * (ldk + 1) + c];
    if (c < k) {
        if (ch == 0) P[c] = 0.0;
        for (int r = r0; r < r1; r++) { acc += s[(size_t)r * ldk + c]; P[(size_t)(r + 1) * ldk + c] = acc; }
    } else if (c < ldk) {
        if (ch == 0) P[c] = 0.0;
        for (int r = r0; r < r1; r++) P[(size_t)(r + 1) * ldk + c] = 0.0;
    } else {
        if (ch == 0) Qp[0] = 0.0;
        for (int r = r0; r < r1; r++) { acc += rn2[r]; Qp[r + 1] = acc; }
    }
}

// d0[c][j] = 1/2 sum_{c' <= c} (x_j[c'] - x_{j+1}[c'])^2 : the initial adjacent-pair dSS of every
// candidate is a running sum over columns, so all k candidates are initialised in O(n k).
__global__ void d0_kernel(const double *__restrict__ s, int n, int k, int ldk, double *__restrict__ d0, int ldd) {
    int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= n - 1) return;
    const double *a = s + (size_t)j * ldk, *b = a + ldk;
    double acc = 0.0;
    for (int c = 0; c < k; c++) {
        double t = a[c] - b[c];
        acc += 0.5 * t * t;
        d0[(size_t)c * ldd + j] = acc;
    }
}

// ------------------------------------------------------------------------------------------
// the merge loop
// ------------------------------------------------------------------------------------------
// shared memory through explicit 32-bit shared-window addresses: the merge loop is one warp's
// dependent chain, so every instruction of address arithmetic the compiler would add for generic
// pointers is latency on the critical path
__device__ __forceinline__ double lds_f64(unsigned a) { double v; asm volatile("ld.shared.f64 %0, [%1];" : "=d"(v) : "r"(a) : "memory"); return v; }
__device__ __forceinline__ void sts_f64(unsigned a, double v) { asm volatile("st.shared.f64 [%0], %1;" ::"r"(a), "d"(v) : "memory"); }
__device__ __forceinline__ int lds_u16(unsigned a) { unsigned short v; asm volatile("ld.shared.u16 %0, [%1];" : "=h"(v) : "r"(a) : "memory"); return v; }
__device__ __forceinline__ void sts_u16(unsigned a, int v) { asm volatile("st.shared.u16 [%0], %1;" ::"r"(a), "h"((unsigned short)v) : "memory"); }
__device__ __forceinline__ unsigned lds_u32(unsigned a) { unsigned v; asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(a) : "memory"); return v; }
__device__ __forceinline__ void sts_u32(unsigned a, unsigned v) { asm volatile("st.shared.u32 [%0], %1;" ::"r"(a), "r"(v) : "memory"); }
__device__ __forceinline__ int lds_s32(unsigned a) { int v; asm volatile("ld.shared.s32 %0, [%1];" : "=r"(v) : "r"(a) : "memory"); return v; }
__device__ __forceinline__ void sts_s32(unsigned a, int v) { asm volatile("st.shared.s32 [%0], %1;" ::"r"(a), "r"(v) : "memory"); }
// the dSS leaf array in global memory (DSS_GLOBAL), through L2 only: one lane writes what the whole warp reads next
__device__ __forceinline__ double ldcg_f64(const double *p) { double v; asm volatile("ld.global.cg.f64 %0, [%1];" : "=d"(v) : "l"(p) : "memory"); return v; }
__device__ __forceinline__ void stcg_f64(double *p, double v) { asm volatile("st.global.cg.f64 [%0], %1;" ::"l"(p), "d"(v) : "memory"); }

template <typename LinkT, bool SMEM> struct Links {
    unsigned sp, sn;          // shared addresses (SMEM)
    LinkT *gp, *gn;           // global pointers (!SMEM)
    __device__ __forceinline__ int prv(int j) const {
        if (SMEM) return sizeof(LinkT) == 2 ? lds_u16(sp + 2 * j) : lds_s32(sp + 4 * j);
        return (int)__ldcg(gp + j);
    }
    __device__ __forceinline__ int nxt(int j) const {
        if (SMEM) return sizeof(LinkT) == 2 ? lds_u16(sn + 2 * j) : lds_s32(sn + 4 * j);
        return (int)__ldcg(gn + j);
    }
    __device__ __forceinline__ void set_prv(int j, int v) const {
        if (SMEM) { if (sizeof(LinkT) == 2) sts_u16(sp + 2 * j, v); else sts_s32(sp + 4 * j, v); }
        else __stcg(gp + j, (LinkT)v);
    }
    __device__ __forceinline__ void set_nxt(int j, int v) const {
        if (SMEM) { if (sizeof(LinkT) == 2) sts_u16(sn + 2 * j, v); else sts_s32(sn + 4 * j, v); }
        else __stcg(gn + j, (LinkT)v);
    }
};

#define CS_CHUNK 8     // 8 x 32 = 256 score columns loaded per batch
#define TIE_REL 1e-11  // increases this close (relative) to the minimum are tied: the lowest index is merged
#define TIE_ABS 1e-24  // ... or this close in units of the total squared norm of the scores (exact-zero ties)

// INV_SMEM: a table of 1/m, m = 0..n, sits in shared memory (cluster sizes are integers), replacing
// the five FP64 divisions of a merge step by loads
// One warp per candidate, WPC = blockDim.x / 32 candidates per CTA (per-candidate shared memory `cand_smem` bytes each, the
// reciprocal table shared by the CTA after them).  Packing several candidates into one CTA keeps the sweep on few SMs:
// 200 one-warp CTAs would be spread over all 148 SMs, and their 25-40 KB of shared memory each would keep the
// ~200 KB CTAs of the tcgen05 kernels of OTHER calls in flight on the same GPU off every SM for the whole sweep.
// TRACE: cycles of one merge step by phase, summed over the merge loop of the first candidate of the list (the widest),
// written to trace[0..5] = find, links, P rows + dot products, shuffle reduce + scale, write back + level-1 re-reduce,
// level-2 re-reduce; trace[6] = steps (TADPOLE_SWEEP_TRACE; profiles/r02_coniss_merge_step.md)
// DSS_GLOBAL: the leaf level of the dSS array (n1 doubles) stays in the candidate's own row of d0 in global memory, read
// and written through L2; only the two min-tree levels and the live-boundary bitmap are in shared memory (~19 KB at 50k
// bins instead of ~400 KB).  The leaf block of the minimum is loaded once by the find step and kept in registers, the
// blocks of the two neighbours are loaded beside the P rows of the dot products, and the re-reductions patch those
// registers with the values written back: the same operations on the same values as the shared-memory path, so the same
// bits, for one more L2 round trip per merge step.
template <typename LinkT, bool LINKS_SMEM, bool INV_SMEM, bool TRACE, bool DSS_GLOBAL>
__global__ void __launch_bounds__(256)
coniss_sweep_kernel(const double *__restrict__ P, int ldk, int n,
                    const double *__restrict__ d0, int ldd,
                    const int *__restrict__ cand_list, int ncand, unsigned cand_smem,
                    double *__restrict__ seqdist, int4 *__restrict__ merges,
                    LinkT *__restrict__ glinks, const double *__restrict__ qtot, long long *__restrict__ trace) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, wpc = blockDim.x >> 5;
    const int slot = blockIdx.x * wpc + warp;
    const int n1 = n - 1;
    const int n1p = (n1 + 31) & ~31;
    const int B1 = n1p >> 5;
    const int B1p = (B1 + 31) & ~31;
    const int B2 = B1p >> 5;
    const int B2p = (B2 + 31) & ~31;

    const unsigned sbase0 = (unsigned)__cvta_generic_to_shared(smem_raw);
    const unsigned sinv = sbase0 + (unsigned)wpc * cand_smem;      // inv[n + 1] when INV_SMEM, shared by the CTA
    if (INV_SMEM) {
        for (int m = threadIdx.x; m <= n; m += blockDim.x) sts_f64(sinv + 8u * m, m ? 1.0 / (double)m : 0.0);
        __syncthreads();
    }
    if (slot >= ncand) return;
    const int cand = cand_list[slot];
    const int ncol = cand + 1;
    const unsigned sbase = sbase0 + (unsigned)warp * cand_smem;
    const unsigned sd = sbase;                       // d[n1p] (not DSS_GLOBAL)
    const unsigned sm1 = DSS_GLOBAL ? sbase : sd + 8u * n1p;      // m1[B1p]
    const unsigned sm2 = sm1 + 8u * B1p;             // m2[B2p]
    // Neighbours of a boundary (previous / next boundary still alive).  LINKS_SMEM: two link arrays in shared memory, two
    // dependent loads per merge.  Otherwise (the arrays do not fit beside the dSS array: above ~18k bins; or they would push
    // the reciprocal table out): one BIT per boundary in shared memory, 32 x smaller; the previous / next set bit is found
    // by the warp together (one word per lane covers 1024 boundaries per step).  The links used to go to global memory
    // here: two dependent L2 round trips, 1100 of the 3800 cycles of a merge step at 25k bins (profiles/r02_coniss_merge_step.md).
    Links<LinkT, true> lk;
    lk.sp = lk.sn = 0; lk.gp = lk.gn = nullptr;
    const unsigned sbits = sm2 + 8u * B2p;
    const int W = (n1 + 31) >> 5;
    if (LINKS_SMEM) { lk.sp = sbits; lk.sn = lk.sp + (unsigned)sizeof(LinkT) * n1; }
    // one word per lane: the word of j (only its bits below / above j) and the 31 words before / after it, 1024 boundaries
    // per step; a second step only when a cluster is longer than that (the last few dozen merges of a chromosome)
    auto bm_prev = [&](int j) -> int {             // largest live boundary below j, or -1 (warp-collective, uniform j)
        for (int w0 = j >> 5; w0 >= 0; w0 -= 32) {
            const int wi = w0 - lane;
            unsigned v = wi >= 0 ? lds_u32(sbits + 4u * wi) : 0u;
            if (wi == (j >> 5)) v &= (1u << (j & 31)) - 1u;
            const unsigned bal = __ballot_sync(0xffffffffu, v != 0u);
            if (bal) {
                const int src = __ffs(bal) - 1;
                return ((w0 - src) << 5) + 31 - __clz(__shfl_sync(0xffffffffu, v, src));
            }
        }
        return -1;
    };
    auto bm_next = [&](int j) -> int {             // smallest live boundary above j, or n1
        for (int w0 = j >> 5; w0 < W; w0 += 32) {
            const int wi = w0 + lane;
            unsigned v = wi < W ? lds_u32(sbits + 4u * wi) : 0u;
            if (wi == (j >> 5)) v &= ~((2u << (j & 31)) - 1u);
            const unsigned bal = __ballot_sync(0xffffffffu, v != 0u);
            if (bal) {
                const int src = __ffs(bal) - 1;
                return ((w0 + src) << 5) + __ffs(__shfl_sync(0xffffffffu, v, src)) - 1;
            }
        }
        return n1;
    };
    const double *d0row = d0 + (size_t)cand * ldd;
    double *seq = seqdist + (size_t)cand * ldd;
    int4 *mrg = merges + (size_t)cand * ldd;
    // DSS_GLOBAL: this candidate's row of d0 (written by d0_kernel of this sweep, read by nobody else) becomes its leaf
    // array; entries n1..n1p-1 are not stored: a load there reads +inf, as the padding of the shared array does
    double *const gd = const_cast<double *>(d0row);
    auto ld_leaf = [&](int b) -> double { const int q = (b << 5) + lane; return q < n1 ? ldcg_f64(gd + q) : INF_D; };

    if (!DSS_GLOBAL)
        for (int j = lane; j < n1p; j += 32) sts_f64(sd + 8u * j, (j < n1) ? d0row[j] : INF_D);
    if (LINKS_SMEM) {
        for (int j = lane; j < n1; j += 32) { lk.set_prv(j, j); lk.set_nxt(j, j + 1); }   // prv holds index+1, 0 = none
    } else {
        for (int w = lane; w < W; w += 32)
            sts_u32(sbits + 4u * w, (w << 5) + 32 <= n1 ? 0xffffffffu : ((1u << (n1 - (w << 5))) - 1u));
    }
    for (int b = lane; b < B1p; b += 32) sts_f64(sm1 + 8u * b, INF_D);
    for (int b = lane; b < B2p; b += 32) sts_f64(sm2 + 8u * b, INF_D);
    __syncwarp();
    if (DSS_GLOBAL) {
        // eight leaf blocks per L2 round trip
        for (int b0 = 0; b0 < B1; b0 += 8) {
            double x[8];
#pragma unroll
            for (int u = 0; u < 8; u++) x[u] = b0 + u < B1 ? ld_leaf(b0 + u) : INF_D;
#pragma unroll
            for (int u = 0; u < 8; u++) {
                const double v = warp_min_nonneg(x[u]);
                if (lane == 0 && b0 + u < B1) sts_f64(sm1 + 8u * (b0 + u), v);
            }
        }
    } else {
        for (int b = 0; b < B1; b++) {
            double v = warp_min_nonneg(lds_f64(sd + 8u * ((b << 5) + lane)));
            if (lane == 0) sts_f64(sm1 + 8u * b, v);
        }
    }
    __syncwarp();
    for (int b = 0; b < B2; b++) {
        double v = warp_min_nonneg(lds_f64(sm1 + 8u * ((b << 5) + lane)));
        if (lane == 0) sts_f64(sm2 + 8u * b, v);
    }
    __syncwarp();

    auto inv_of = [&](int m) -> double { return INV_SMEM ? lds_f64(sinv + 8u * m) : 1.0 / (double)m; };
    const double tie_abs = TIE_ABS * __ldg(qtot);       // qtot: sum of the squared norms of all score rows
    const double *Plane = P + lane;
    double total = 0.0;
    long long tr_acc[6] = {0, 0, 0, 0, 0, 0}, tr_t = 0;
#define CS_TR(ph) do { if (TRACE) { const long long t_ = clock64(); tr_acc[ph] += t_ - tr_t; tr_t = t_; } } while (0)
    for (int t = 0; t < n1; t++) {
        if (TRACE) tr_t = clock64();
        // ---- find the minimum; among increases equal to it, the lowest index ---------------------------
        // The reference's scan keeps the first of EQUAL increases (strict '<').  Equal means equal in exact arithmetic:
        // bins with identical score rows (zero-variance bins all map to one row of the correlation matrix, quirk Q9) give
        // families of exactly tied increases, which Lance-Williams arithmetic on the distance matrix reproduces bit for bit
        // while differences of prefix sums taken at different offsets differ in their last bits.  So an increase within
        // TIE_REL (relative, two orders above the rounding of this kernel's arithmetic) + tie_abs (for exact zeros: identical
        // adjacent rows) of the minimum counts as tied.  Two increases that close without being structurally equal are
        // ordered by rounding noise in the reference too.
        double mn;
        int b2 = 0;
        if (B2p == 32) {
            const double v = lds_f64(sm2 + 8u * lane);
            mn = warp_min_nonneg(v);
            const double thr = fma(mn, TIE_REL, mn) + tie_abs;
            b2 = __ffs(__ballot_sync(0xffffffffu, v <= thr)) - 1;
        } else {
            double v = INF_D;
            for (int q = lane; q < B2p; q += 32) v = fmin(v, lds_f64(sm2 + 8u * q));
            mn = warp_min_nonneg(v);
            const double thr = fma(mn, TIE_REL, mn) + tie_abs;
            for (int q0 = 0; q0 < B2p; q0 += 32) {
                unsigned bal = __ballot_sync(0xffffffffu, lds_f64(sm2 + 8u * (q0 + lane)) <= thr);
                if (bal) { b2 = q0 + __ffs(bal) - 1; break; }
            }
        }
        const double thr = fma(mn, TIE_REL, mn) + tie_abs;
        const unsigned bal1 = __ballot_sync(0xffffffffu, lds_f64(sm1 + 8u * ((b2 << 5) + lane)) <= thr);
        const int b1 = (b2 << 5) + __ffs(bal1) - 1;
        const double leaf = DSS_GLOBAL ? ld_leaf(b1) : lds_f64(sd + 8u * ((b1 << 5) + lane));
        const unsigned bal0 = __ballot_sync(0xffffffffu, leaf <= thr);
        const int j = (b1 << 5) + __ffs(bal0) - 1;
        mn = __shfl_sync(0xffffffffu, leaf, j & 31);          // the increase of the boundary that is merged

        CS_TR(0);
        // ---- neighbours ---------------------------------------------------------------------
        int pj, nj, ppj, nnj;                    // previous / next live boundary (-1 / n1: none) and theirs
        if (LINKS_SMEM) {
            pj = lk.prv(j) - 1; nj = lk.nxt(j);
            ppj = pj >= 0 ? lk.prv(pj) - 1 : -1;
            nnj = nj < n1 ? lk.nxt(nj) : n1;
        } else {
            pj = bm_prev(j); nj = bm_next(j);
            ppj = pj >= 0 ? bm_prev(pj) : -1;
            nnj = nj < n1 ? bm_next(nj) : n1;
        }
        const bool hasL = pj >= 0, hasR = nj < n1;
        // P rows: LL = [a, b), C = [b, c), RR = [c, e)
        const int a = ppj + 1, b = pj + 1, c = nj + 1, e = nnj + 1;
        const double *Pa = Plane + (size_t)a * ldk, *Pb = Plane + (size_t)b * ldk;
        const double *Pc = Plane + (size_t)c * ldk, *Pe = Plane + (size_t)e * ldk;
        const int cC = c - b, cLL = b - a, cRR = e - c;
        const double iC = inv_of(cC), iLL = inv_of(cLL), iRR = inv_of(cRR);
        // DSS_GLOBAL: the leaf blocks of the neighbours, when not the one in registers, in flight with the P rows
        double xk1 = 0.0, xk2 = 0.0;
        if (DSS_GLOBAL) {
            const int q0 = j >> 5, q1 = hasL ? (pj >> 5) : q0, q2 = hasR ? (nj >> 5) : q0;
            if (q1 != q0) xk1 = ld_leaf(q1);
            if (q2 != q0 && q2 != q1) xk2 = ld_leaf(q2);
        }
        double accL = 0.0, accR = 0.0;
        if (TRACE) { asm volatile("" ::"d"(iC), "d"(iLL), "d"(iRR)); CS_TR(1); }
        for (int c0 = 0; c0 < ncol; c0 += 32 * CS_CHUNK) {
            double va[CS_CHUNK], vb[CS_CHUNK], vc[CS_CHUNK], ve[CS_CHUNK];
            // all loads of the batch first: one L2 round trip per step instead of one per 32 columns
#pragma unroll
            for (int u = 0; u < CS_CHUNK; u++) {
                const int col = c0 + 32 * u;
                if (col >= ncol) break;
                const bool ok = col + lane < ncol;
                vb[u] = ok ? __ldg(Pb + col) : 0.0;
                vc[u] = ok ? __ldg(Pc + col) : 0.0;
                va[u] = (ok && hasL) ? __ldg(Pa + col) : 0.0;
                ve[u] = (ok && hasR) ? __ldg(Pe + col) : 0.0;
            }
#pragma unroll
            for (int u = 0; u < CS_CHUNK; u++) {
                if (c0 + 32 * u >= ncol) break;
                const double mC = (vc[u] - vb[u]) * iC;
                const double tL = hasL ? (vb[u] - va[u]) * iLL - mC : 0.0;
                const double tR = hasR ? mC - (ve[u] - vc[u]) * iRR : 0.0;
                accL = fma(tL, tL, accL);
                accR = fma(tR, tR, accR);
            }
        }
        if (TRACE) { asm volatile("" ::"d"(accL), "d"(accR)); CS_TR(2); }
        total += mn;
        if (lane == 0) {
            seq[j] = total;
            mrg[t] = make_int4(j, pj, nj, 0);
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            accL += __shfl_xor_sync(0xffffffffu, accL, o);
            accR += __shfl_xor_sync(0xffffffffu, accR, o);
        }
        // n_a n_b / (n_a + n_b): integer product (exact), then the table reciprocal
        accL *= (double)cLL * (double)cC * inv_of(cLL + cC);
        accR *= (double)cC * (double)cRR * inv_of(cC + cRR);

        if (TRACE) { asm volatile("" ::"d"(accL), "d"(accR)); CS_TR(3); }
        // ---- write back: boundary j dies, its neighbours get new increases ---------------
        if (lane == 0) {
            auto st_d = [&](int q, double v) { if (DSS_GLOBAL) stcg_f64(gd + q, v); else sts_f64(sd + 8u * q, v); };
            st_d(j, INF_D);
            if (hasL) { st_d(pj, accL); if (LINKS_SMEM) lk.set_nxt(pj, nj); }
            if (hasR) { st_d(nj, accR); if (LINKS_SMEM) lk.set_prv(nj, pj + 1); }
            if (!LINKS_SMEM) sts_u32(sbits + 4u * (j >> 5), lds_u32(sbits + 4u * (j >> 5)) & ~(1u << (j & 31)));
        }
        __syncwarp();
        const int k0 = j >> 5;
        const int k1 = hasL ? (pj >> 5) : k0;
        const int k2 = hasR ? (nj >> 5) : k0;
        // independent re-reductions issued back to back (ILP), then stored
        double x0, x1, x2;
        if (DSS_GLOBAL) {
            // the blocks as loaded, with this step's write-back applied (accL / accR are the same on every lane: the
            // butterfly adds the same two values on both lanes of each pair)
            auto patch = [&](double x, int blk) -> double {
                const int q = (blk << 5) + lane;
                if (q == j) x = INF_D;
                if (hasL && q == pj) x = accL;
                if (hasR && q == nj) x = accR;
                return x;
            };
            x0 = patch(leaf, k0);
            x1 = k1 != k0 ? patch(xk1, k1) : x0;
            x2 = k2 == k0 ? x0 : (k2 == k1 ? x1 : patch(xk2, k2));
        } else {
            x0 = lds_f64(sd + 8u * ((k0 << 5) + lane));
            x1 = lds_f64(sd + 8u * ((k1 << 5) + lane));
            x2 = lds_f64(sd + 8u * ((k2 << 5) + lane));
        }
        const double r0 = warp_min_nonneg(x0);
        const double r1 = (k1 != k0) ? warp_min_nonneg(x1) : r0;
        const double r2 = (k2 != k0) ? warp_min_nonneg(x2) : r0;
        if (lane == 0) {
            sts_f64(sm1 + 8u * k0, r0);
            if (k1 != k0) sts_f64(sm1 + 8u * k1, r1);
            if (k2 != k0) sts_f64(sm1 + 8u * k2, r2);
        }
        __syncwarp();
        CS_TR(4);
        const int g0 = k0 >> 5, g1 = k1 >> 5, g2 = k2 >> 5;
        const double y0 = warp_min_nonneg(lds_f64(sm1 + 8u * ((g0 << 5) + lane)));
        if (lane == 0) sts_f64(sm2 + 8u * g0, y0);
        if (g1 != g0) {
            const double y1 = warp_min_nonneg(lds_f64(sm1 + 8u * ((g1 << 5) + lane)));
            if (lane == 0) sts_f64(sm2 + 8u * g1, y1);
        }
        if (g2 != g0 && g2 != g1) {
            const double y2 = warp_min_nonneg(lds_f64(sm1 + 8u * ((g2 << 5) + lane)));
            if (lane == 0) sts_f64(sm2 + 8u * g2, y2);
        }
        __syncwarp();
        CS_TR(5);
    }
    if (TRACE && slot == 0 && lane == 0) {
        for (int p = 0; p < 6; p++) trace[p] = tr_acc[p];
        trace[6] = n1;
        trace[7] = ncol;
    }
#undef CS_TR
}

// ------------------------------------------------------------------------------------------
// stage 5: rioja::bstick + first-TRUE-run rule + fpc::calinhara per level (R/TADpole.R:111-120)
// ------------------------------------------------------------------------------------------
#define CH_WARPS 4
__global__ void __launch_bounds__(32 * CH_WARPS)
ch_kernel(const double *__restrict__ P, const double *__restrict__ Qp, int ldk, int n, int k,
          const double *__restrict__ seqdist, const int4 *__restrict__ merges, int ldd,
          const int *__restrict__ cand_list, int min_clusters,
          double *__restrict__ bs_scratch, int *__restrict__ ncl_out,
          double *__restrict__ chs, int ld_chs) {
    // One CTA of CH_WARPS warps per candidate.  What is serial in the reference's arithmetic stays serial on one thread, in
    // the reference's order (the cumulative sum of the broken stick, the running within-cluster dispersion); what feeds
    // those chains is computed by all warps first: the quotients tot / m, and the dispersion each level undoes.
    extern __shared__ double s_dl[];                  // s_dl[lev]: decrease of W when level lev undoes its merge
    __shared__ int s_ncl;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int cand = cand_list[blockIdx.x];
    const int n1 = n - 1;                 // nobj = number of merges = length(height)
    const double *seq = seqdist + (size_t)cand * ldd;
    const int4 *mrg = merges + (size_t)cand * ldd;
    double *bs = bs_scratch + (size_t)blockIdx.x * ldd;
    double *out = chs + (size_t)cand * ld_chs;

    for (int l = tid; l < ld_chs; l += blockDim.x) out[l] = __longlong_as_double(0x7ff8000000000000LL);

    // height[t] = cumulative dispersion after merge t; tot = height[n1-1]
    const double tot = seq[mrg[n1 - 1].x];
    // vegan::bstick.default(nobj, tot) = rev(cumsum(tot / nobj:1) / nobj): the quotients in parallel, then the cumulative
    // sum from m = nobj down to 1 on one thread, so that it rounds exactly as R's cumsum does, then the division by nobj.
    const double dn = (double)n1;
    for (int m = 1 + tid; m <= n1; m += blockDim.x) bs[m - 1] = tot / (double)m;
    __syncthreads();
    if (tid == 0) {
        double c = 0.0;
        for (int m = n1; m >= 1; m--) { c += bs[m - 1]; bs[m - 1] = c; }
    }
    __syncthreads();
    for (int m = 1 + tid; m <= n1; m += blockDim.x) bs[m - 1] = bs[m - 1] / dn;
    __syncthreads();
    // dispersion_j = |disp[j+1] - disp[j]|, disp = rev(height), j = 1..n1-1;  flag_j = dispersion_j > bs_j
    if (warp == 0) {
        int first = -1, runlen = 0;
        bool done = false;
        for (int j0 = 1; j0 <= n1 - 1 && !done; j0 += 32) {
            const int j = j0 + lane;
            bool f = false;
            if (j <= n1 - 1) {
                const double hi = seq[mrg[n1 - j].x];        // disp[j]   = height[n1 - j]
                const double lo = seq[mrg[n1 - j - 1].x];    // disp[j+1] = height[n1 - j - 1]
                f = fabs(lo - hi) > bs[j - 1];
            }
            unsigned bal = __ballot_sync(0xffffffffu, f);
            unsigned valid = (j0 + 31 <= n1 - 1) ? 0xffffffffu : ((1u << (n1 - j0)) - 1u);
            if (first < 0) {
                if (bal) {
                    int sft = __ffs(bal) - 1;
                    first = j0 + sft;
                    unsigned rest = (~bal & valid) >> sft;      // first FALSE at or after sft
                    if (rest) { runlen = __ffs(rest) - 1; done = true; }
                    else if (valid != 0xffffffffu) { runlen = (n1 - 1) - first + 1; done = true; }
                    else runlen = 32 - sft;
                }
            } else {
                unsigned nb = ~bal & valid;
                if (nb) { runlen += __ffs(nb) - 1; done = true; }
                else if (valid != 0xffffffffu) { runlen += n1 - j0; done = true; }
                else runlen += 32;
            }
        }
        if (lane == 0) { s_ncl = (first < 0) ? -1 : runlen; ncl_out[cand] = s_ncl; }
    }
    __syncthreads();
    const int ncl = s_ncl;
    if (ncl < 1) return;

    // Calinski-Harabasz on all k columns; level lev is reached by undoing the last lev - 1 merges, in MERGE-STEP order.
    // cutree (tp_assemble*, and R's .find.groups) ranks the boundaries by (height, index) instead; the two orders differ only
    // among merges whose heights are equal as doubles, i.e. whose increases vanish against the running total -- W, and
    // with it every CH value, is the same to rounding whichever of those merges is undone first, and the tables the
    // caller gets come from the (height, index) order.  The merge undone by
    // level lev lowers W by n_a n_b / (n_a + n_b) |c_a - c_b|^2: one warp per level (only levels the caller's row holds)
    const int nlev = min(ncl, ld_chs);
    for (int lev = 2 + warp; lev <= nlev; lev += CH_WARPS) {
        const int4 mg = mrg[n1 - (lev - 1)];
        const int a = mg.y + 1, b = mg.x + 1, c = mg.z + 1;   // A = [a, b), B = [b, c) in P rows
        const double nA = (double)(b - a), nB = (double)(c - b);
        const double iA = 1.0 / nA, iB = 1.0 / nB;
        const double *Pa = P + (size_t)a * ldk, *Pb = P + (size_t)b * ldk, *Pc = P + (size_t)c * ldk;
        double acc = 0.0;
        for (int col = lane; col < k; col += 32) {
            const double pb = Pb[col];
            const double tt = (pb - Pa[col]) * iA - (Pc[col] - pb) * iB;
            acc += tt * tt;
        }
        acc = warp_sum(acc);
        if (lane == 0) s_dl[lev] = acc * (nA * nB / (nA + nB));
    }
    double ssq = 0.0;
    if (warp == 0) {
        for (int c = lane; c < k; c += 32) { double v = P[(size_t)n * ldk + c]; ssq += v * v; }
        ssq = warp_sum(ssq);
    }
    __syncthreads();
    if (tid == 0) {
        const double trS = Qp[n] - ssq / (double)n;
        double W = trS;
        const int mc = min(min_clusters, ncl);
        const double dN = (double)n;
        if (mc <= 1 && ld_chs > 0) out[0] = (dN - 1.0) * (trS - W) / (0.0 * W);
        for (int lev = 2; lev <= nlev; lev++) {
            W -= s_dl[lev];
            if (lev >= mc) out[lev - 1] = (dN - (double)lev) * (trS - W) / ((double)(lev - 1) * W);
        }
    }
}

// ------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------
static int build_cand_list(int k, int begin, int stride, std::vector<int> &out) {
    out.clear();
    for (int c = begin; c < k; c += stride) out.push_back(c);
    // heaviest (most columns) first
    for (size_t i = 0, j = out.size(); i + 1 < j; i++, j--) std::swap(out[i], out[j - 1]);
    return (int)out.size();
}

int tp_sweep_device(tp_ctx *ctx, int min_clusters, int cand_begin, int cand_stride, int *ncand_out) {
    TP_ARG(ctx->have_scores, "tp_sweep: no PC scores in the context (run tp_pca or tp_set_scores)");
    TP_ARG(cand_stride >= 1 && cand_begin >= 0, "tp_sweep: bad candidate range");
    TP_ARG(min_clusters >= 1, "tp_sweep: min_clusters must be >= 1");
    const int n = ctx->nf, k = ctx->k, ldk = ctx->ldk;
    TP_ARG(n >= 3, "tp_sweep: need at least 3 bins");
    const int n1 = n - 1;
    const int ldd = round_up(n1, 8);
    std::vector<int> cands;
    const int ncand = build_cand_list(k, cand_begin, cand_stride, cands);
    *ncand_out = ncand;
    cudaStream_t st = ctx->stream;
    if (ncand == 0) {          // a rank of a sharded sweep with more ranks than candidates: nothing to run, rows stay empty
        TP_TRY(ctx->ncl.reserve((size_t)(2 * k + 8) * sizeof(int)));
        TP_CUDA(cudaMemsetAsync(ctx->ncl.p, 0, k * sizeof(int), st));
        TP_TRY(ctx->seqdist.reserve((size_t)k * ldd * sizeof(double)));
        TP_TRY(ctx->order.reserve((size_t)k * ldd * sizeof(int4)));
        TP_MARK(ctx, EV_SWEEP0);
        TP_MARK(ctx, EV_SWEEP1);
        ctx->have_sweep = true;
        return TP_OK;
    }

    TP_TRY(ctx->P.reserve((size_t)(n + 1) * ldk * sizeof(double)));
    TP_TRY(ctx->Qp.reserve((size_t)(n + 2) * sizeof(double) * 2));
    TP_TRY(ctx->d0.reserve((size_t)k * ldd * sizeof(double)));
    TP_TRY(ctx->seqdist.reserve((size_t)k * ldd * sizeof(double)));
    TP_TRY(ctx->order.reserve((size_t)k * ldd * sizeof(int4)));
    TP_TRY(ctx->ncl.reserve((size_t)(2 * k + 8) * sizeof(int)));
    TP_TRY(ctx->bsbuf.reserve((size_t)ncand * ldd * sizeof(double)));
    int *d_cands = ctx->ncl.as<int>() + k;
    TP_CUDA(cudaMemcpyAsync(d_cands, cands.data(), ncand * sizeof(int), cudaMemcpyHostToDevice, st));
    TP_CUDA(cudaMemsetAsync(ctx->ncl.p, 0, k * sizeof(int), st));

    double *rn2 = ctx->Qp.as<double>() + (n + 2);
    TP_MARK(ctx, EV_SWEEP0);
    rownorm2_kernel<<<(n * 32 + 255) / 256, 256, 0, st>>>(ctx->scores.as<double>(), n, k, ldk, rn2);
    {
        const int nch = (n + PF_CHUNK - 1) / PF_CHUNK;
        TP_TRY(ctx->harm.reserve((size_t)nch * (ldk + 1) * sizeof(double)));
        const dim3 pg(nch, (ldk + 1 + 63) / 64);
        prefix_sums_kernel<<<pg, 64, 0, st>>>(ctx->scores.as<double>(), rn2, n, k, ldk, ctx->harm.as<double>());
        prefix_write_kernel<<<pg, 64, 0, st>>>(ctx->scores.as<double>(), rn2, ctx->harm.as<double>(), n, k, ldk,
                                               ctx->P.as<double>(), ctx->Qp.as<double>());
    }
    d0_kernel<<<(n1 + 127) / 128, 128, 0, st>>>(ctx->scores.as<double>(), n, k, ldk, ctx->d0.as<double>(), ldd);
    ctx->launches += 4;

    // shared memory plan: per candidate the dSS array with its min tree (+ the boundary links when they fit); several
    // candidates per CTA (one warp each) sharing one reciprocal table while that fits.  When the dSS array does not fit
    // (above ~27 700 bins) its leaf level goes to global memory (DSS_GLOBAL) and only the tree and the bitmap stay.
    const int n1p = round_up(n1, 32), B1p = round_up(n1p / 32, 32), B2p = round_up(B1p / 32, 32);
    const size_t base = (size_t)(n1p + B1p + B2p) * sizeof(double);
    const size_t tree = (size_t)(B1p + B2p) * sizeof(double);
    const bool small_links = n <= 65535;
    const size_t link_bytes = round_up((int)((size_t)2 * n1 * (small_links ? 2 : 4)), 8);
    const size_t bitmap_bytes = (size_t)round_up(((n1 + 31) / 32) * 4, 16);
    const size_t inv_bytes = (size_t)(n + 1) * sizeof(double);
    const size_t limit = (size_t)ctx->max_smem_optin;
    const char *e_dss = getenv("TADPOLE_SWEEP_DSS");             // "global": the global leaf array at any size (tests)
    const bool dss_global = base + bitmap_bytes > limit || (e_dss && e_dss[0] == 'g');
    // link arrays while they fit (two dependent loads: ~90 cycles per merge against ~400 for the bitmap searches), else the
    // bitmap (32 x smaller: above ~18k bins; always beside a global leaf array)
    const char *force = getenv("TADPOLE_SWEEP_LINKS");           // "bitmap" / "array": experiments
    bool links_smem = base + link_bytes <= limit;
    if (force && force[0] == 'b') links_smem = false;
    if (force && force[0] == 'a' && base + link_bytes <= limit) links_smem = true;
    if (dss_global) links_smem = false;
    const size_t cand_smem = round_up((int)(links_smem ? base + link_bytes : (dss_global ? tree : base) + bitmap_bytes), 16);
    TP_ARG(cand_smem <= limit, "tp_sweep: matrix too large for the shared-memory min tree of the dSS array (n > ~600k bins)");
    // the reciprocal table goes to shared memory while at least two candidates still fit beside it (never beside a global
    // leaf array: that only runs where the table would not fit either)
    bool inv_smem = !dss_global && 2 * cand_smem + inv_bytes <= limit;
    const char *e_inv = getenv("TADPOLE_SWEEP_INV"), *e_wpc = getenv("TADPOLE_SWEEP_WPC");       // experiments
    if (e_inv && e_inv[0] == 'g') inv_smem = false;
    int wpc = (int)((limit - (inv_smem ? inv_bytes : 0)) / cand_smem);
    const int wpc_cap = e_wpc && atoi(e_wpc) > 0 ? atoi(e_wpc) : 4;
    wpc = wpc < 1 ? 1 : (wpc > wpc_cap ? wpc_cap : wpc);      // one warp per SM sub-partition: 8 slowed each merge chain by 19 %
    // (not more warps than needed to give every SM-sized group of candidates a CTA: a lone call still wants them spread)
    while (wpc > 1 && (ncand + wpc - 1) / wpc < 16) wpc--;
    const size_t smem = (size_t)wpc * cand_smem + (inv_smem ? inv_bytes : 0);
    const int nblocks = (ncand + wpc - 1) / wpc;
    void *glinks = nullptr;
    long long *trace = nullptr;
    DevBuf trbuf;
    if (getenv("TADPOLE_SWEEP_TRACE")) { TP_TRY(trbuf.reserve(8 * sizeof(long long))); trace = trbuf.as<long long>(); }
#define LAUNCH_SWEEP2(LT, LS, IS, TR, DG)                                                                 \
    do {                                                                                                  \
        TP_CUDA(tp_optin_smem(coniss_sweep_kernel<LT, LS, IS, TR, DG>, ctx)); \
        tp_prof_begin(ctx, PC_SWEEP);                                                                     \
        coniss_sweep_kernel<LT, LS, IS, TR, DG><<<nblocks, 32 * wpc, smem, st>>>(ctx->P.as<double>(), ldk, n, ctx->d0.as<double>(), ldd, \
                                                                 d_cands, ncand, (unsigned)cand_smem, ctx->seqdist.as<double>(), \
                                                                 ctx->order.as<int4>(), (LT *)glinks, ctx->Qp.as<double>() + n, trace); \
        tp_prof_end(ctx);                                                                                 \
    } while (0)
#define LAUNCH_SWEEP(LT, LS, IS, DG) do { if (trace) LAUNCH_SWEEP2(LT, LS, IS, true, DG); else LAUNCH_SWEEP2(LT, LS, IS, false, DG); } while (0)
    if (dss_global) {
        LAUNCH_SWEEP(unsigned short, false, false, true);
    } else if (links_smem) {
        if (small_links) { if (inv_smem) LAUNCH_SWEEP(unsigned short, true, true, false); else LAUNCH_SWEEP(unsigned short, true, false, false); }
        else { if (inv_smem) LAUNCH_SWEEP(int, true, true, false); else LAUNCH_SWEEP(int, true, false, false); }
    } else {
        if (inv_smem) LAUNCH_SWEEP(unsigned short, false, true, false); else LAUNCH_SWEEP(unsigned short, false, false, false);
    }
#undef LAUNCH_SWEEP2
#undef LAUNCH_SWEEP
    ctx->launches += 1;
    TP_CUDA(cudaGetLastError());
    TP_MARK(ctx, EV_SWEEP1);
    if (trace) {
        long long h[8];
        TP_CUDA(cudaStreamSynchronize(st));
        TP_CUDA(cudaMemcpy(h, trace, sizeof(h), cudaMemcpyDeviceToHost));
        static const char *ph[6] = {"find", "links", "p_rows_dot", "reduce_scale", "writeback_l1", "l2"};
        fprintf(stderr, "[sweep trace] n=%d cols=%lld wpc=%d links_smem=%d inv_smem=%d dss_global=%d cycles per merge step:", n, h[7], wpc,
                (int)links_smem, (int)inv_smem, (int)dss_global);
        for (int p = 0; p < 6; p++) fprintf(stderr, " %s %.0f", ph[p], (double)h[p] / (double)h[6]);
        fprintf(stderr, "\n");
        trbuf.release();
    }
    ctx->have_sweep = true;
    (void)min_clusters;
    return TP_OK;
}

int tp_ch_device(tp_ctx *ctx, int min_clusters, int ncand, int ld_chs) {
    const int n = ctx->nf, k = ctx->k, ldk = ctx->ldk;
    const int ldd = round_up(n - 1, 8);
    cudaStream_t st = ctx->stream;
    TP_TRY(ctx->chs.reserve((size_t)k * ld_chs * sizeof(double)));
    ctx->ld_chs = ld_chs;
    int *d_cands = ctx->ncl.as<int>() + k;
    // rows of candidates that are not run must read as NaN too
    TP_CUDA(cudaMemsetAsync(ctx->chs.p, 0xff, (size_t)k * ld_chs * sizeof(double), st));
    if (ncand == 0) { TP_MARK(ctx, EV_CH1); return TP_OK; }
    tp_prof_begin(ctx, PC_CH);
    ch_kernel<<<ncand, 32 * CH_WARPS, (size_t)(ld_chs + 2) * sizeof(double), st>>>(ctx->P.as<double>(), ctx->Qp.as<double>(), ldk, n, k,
                                    ctx->seqdist.as<double>(), ctx->order.as<int4>(), ldd, d_cands, min_clusters,
                                    ctx->bsbuf.as<double>(), ctx->ncl.as<int>(), ctx->chs.as<double>(), ld_chs);
    tp_prof_end(ctx);
    ctx->launches += 1;
    TP_CUDA(cudaGetLastError());
    TP_MARK(ctx, EV_CH1);
    return TP_OK;
}
