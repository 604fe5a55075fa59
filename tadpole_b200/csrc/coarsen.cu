// coarsen.cu -- a genome at a multiple of its bin size (S0e): tp_genome_coarsen sums the cells of a tp_genome into cells
// `factor` times wider, on the device that holds it, and returns them as a new tp_genome.
//
// Coarse chromosome c has ceil(n_c / factor) bins; bucket entry (c, i, j, v) goes to coarse cell (c, i / factor,
// j / factor) (integer division keeps I <= J).  A NaN count adds 0 (the reference's NA -> 0 at the fine resolution), a
// coarse cell's count is the sum of its entries', and a cell whose sum is exactly 0 is not stored.
//   1. cs_insert_kernel: every entry is added into an open-addressing table in HBM on the coarse key
//      ((S_c + I) << 31) | (S_c + J), S_c the first coarse bin of c, with CAS and native FP64 atomicAdd.  (Adding up the
//      runs of one cell in the warp first, with __shfl_down_sync, measured no faster on sorted input: DESIGN S0e.)
//   2. cs_count_kernel (genome_util.cuh): the stored cells of each chromosome (warp-aggregated atomics); the host scans
//      them into offsets.
//   3. cs_scatter_kernel (genome_util.cuh): (count, I, J) of every stored cell into its chromosome's bucket through
//      per-chromosome cursors.
// Integer counts whose cell sums of |count| stay below 2^53 add exactly, so the result is the same bits in any order;
// otherwise the rounding order is unspecified (as in coo_scatter_kernel).  Memory: 16 bytes per table slot (2 slots per
// bucket entry, rounded up to a power of two), and 16 bytes per output cell while the buckets are written; the table is
// released before the call returns.
#include "genome_util.cuh"

// ---- 1. merge ---------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(DS_THREADS)
cs_insert_kernel(const double *__restrict__ cnt, const int *__restrict__ bi, const int *__restrict__ bj, u64 m,
                 const u64 *__restrict__ offs, const int *__restrict__ cstarts, int nchrom, int factor,
                 u64 *__restrict__ tkeys, double *__restrict__ tval, u64 mask) {
    const u64 stride = (u64)gridDim.x * DS_THREADS;
    for (u64 e = (u64)blockIdx.x * DS_THREADS + threadIdx.x; e < m; e += stride) {
        const double v = cnt[e];
        if (v != v || v == 0.0) continue;                         // NaN adds 0; so does 0
        const int c = ds_chrom_of_entry(offs, nchrom, e), s0 = __ldg(cstarts + c);
        const u64 key = ((u64)(unsigned)(s0 + bi[e] / factor) << 31) | (u64)(unsigned)(s0 + bj[e] / factor);
        u64 s = ds_hash(key) & mask;
        while (true) {
            u64 k = tkeys[s];
            if (k == CS_EMPTY) k = atomicCAS(tkeys + s, CS_EMPTY, key);
            if (k == CS_EMPTY || k == key) { atomicAdd(tval + s, v); break; }
            s = (s + 1) & mask;
        }
    }
}

// ---- host side ------------------------------------------------------------------------------------------------------------
struct CsBufs {
    DevBuf aux, table;
    ~CsBufs() { aux.release(); table.release(); }
};

extern "C" int tp_genome_coarsen(tp_ctx *ctx, const tp_genome *src, int factor, tp_genome **out) {
    TP_ARG(ctx && src && out, "tp_genome_coarsen: null argument");
    TP_ARG(factor >= 1, "tp_genome_coarsen: factor must be >= 1");
    const char *who = "tp_genome_coarsen";
    tp_ctx *m = nullptr;
    TP_TRY(ds_member(ctx, src, who, &m));
    TP_CUDA(cudaSetDevice(m->device));
    cudaStream_t st = m->stream;
    const int nchrom = (int)src->bins.size();
    const u64 ncis = src->offs.back();

    GenomeOwnerDs own;
    own.g = new tp_genome();
    own.g->device = src->device;
    own.g->trans = src->trans;
    own.g->below = src->below;
    own.g->bins.resize((size_t)nchrom);
    std::vector<int> cstarts((size_t)nchrom + 1, 0);
    for (int c = 0; c < nchrom; c++) {
        own.g->bins[c] = (int)(((long long)src->bins[c] + factor - 1) / factor);
        cstarts[c + 1] = cstarts[c] + own.g->bins[c];
    }

    CsBufs B;
    // bucket offsets, output histogram and cursors, coarse bin starts
    TP_TRY(B.aux.reserve(((size_t)nchrom + 1) * 8 + (size_t)nchrom * 16 + ((size_t)nchrom + 1) * 4));
    u64 *doffs = B.aux.as<u64>(), *hist = doffs + nchrom + 1, *cursor = hist + nchrom;
    int *dstarts = (int *)(cursor + nchrom);
    TP_CUDA(cudaMemcpyAsync(doffs, src->offs.data(), ((size_t)nchrom + 1) * 8, cudaMemcpyHostToDevice, st));
    TP_CUDA(cudaMemcpyAsync(dstarts, cstarts.data(), ((size_t)nchrom + 1) * 4, cudaMemcpyHostToDevice, st));
    TP_CUDA(cudaMemsetAsync(hist, 0, (size_t)nchrom * 8, st));

    // 1. merge
    u64 cap = 1024;
    while (cap < 2 * ncis) cap <<= 1;
    TP_TRY(device_room(m, 16.0 * (double)cap, 0, who, "the cell table"));
    TP_TRY(B.table.reserve((size_t)cap * 16));
    u64 *tkeys = B.table.as<u64>();
    double *tval = (double *)(tkeys + cap);
    TP_CUDA(cudaMemsetAsync(tkeys, 0xff, (size_t)cap * 8, st));
    TP_CUDA(cudaMemsetAsync(tval, 0, (size_t)cap * 8, st));
    if (ncis) {
        const double *pv = src->px.as<double>();
        const int *pi = (const int *)(pv + ncis), *pj = pi + ncis;
        cs_insert_kernel<<<ds_grid(m, ncis), DS_THREADS, 0, st>>>(pv, pi, pj, ncis, doffs, dstarts, nchrom, factor, tkeys, tval,
                                                                 cap - 1);
        m->launches += 1;
    }

    // 2. stored cells per chromosome
    cs_count_kernel<<<ds_grid(m, cap), DS_THREADS, 0, st>>>(tkeys, tval, cap, dstarts, nchrom, hist);
    m->launches += 1;
    TP_CUDA(cudaGetLastError());
    std::vector<u64> h((size_t)nchrom, 0);
    TP_CUDA(cudaMemcpyAsync(h.data(), hist, (size_t)nchrom * 8, cudaMemcpyDeviceToHost, st));
    TP_CUDA(tp_stream_sync(m));
    own.g->offs.assign((size_t)nchrom + 1, 0);
    for (int c = 0; c < nchrom; c++) own.g->offs[c + 1] = own.g->offs[c] + h[c];
    const u64 nout = own.g->offs[nchrom];

    // 3. the new buckets
    TP_TRY(device_room(m, 16.0 * (double)nout, 0, who, "the buckets of the coarse genome"));
    TP_TRY(own.g->px.reserve((size_t)nout * 16 + 16));
    if (nout) {
        double *ov = own.g->px.as<double>();
        int *oi = (int *)(ov + nout), *oj = oi + nout;
        TP_CUDA(cudaMemcpyAsync(cursor, own.g->offs.data(), (size_t)nchrom * 8, cudaMemcpyHostToDevice, st));
        cs_scatter_kernel<<<ds_grid(m, cap), DS_THREADS, 0, st>>>(tkeys, tval, cap, dstarts, nchrom, cursor, ov, oi, oj);
        m->launches += 1;
        TP_CUDA(cudaGetLastError());
    }
    TP_CUDA(tp_stream_sync(m));
    B.table.release();
    *out = own.g;
    own.g = nullptr;
    return TP_OK;
}
