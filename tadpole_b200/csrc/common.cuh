// common.cuh -- context, error plumbing and small device helpers shared by every translation unit.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>
#include <math.h>
#include <string>
#include <vector>
#include <functional>
#include "../../include/tadpole_b200.h"

void tp_set_error(const char *fmt, ...);

#define TP_CUDA(call)                                                                     \
    do {                                                                                  \
        cudaError_t e_ = (call);                                                          \
        if (e_ != cudaSuccess) {                                                          \
            tp_set_error("%s:%d: %s -> %s", __FILE__, __LINE__, #call, cudaGetErrorString(e_)); \
            return TP_ERR_CUDA;                                                           \
        }                                                                                 \
    } while (0)

#define TP_TRY(call)                   \
    do {                               \
        int rc_ = (call);              \
        if (rc_ != TP_OK) return rc_;  \
    } while (0)

#define TP_ARG(cond, msg)                               \
    do {                                                \
        if (!(cond)) {                                  \
            tp_set_error("%s (%s)", msg, #cond);        \
            return TP_ERR_ARG;                          \
        }                                               \
    } while (0)

// grow-only device buffer
struct DevBuf {
    void *p = nullptr;
    size_t cap = 0;
    int reserve(size_t bytes) {
        if (bytes <= cap) return TP_OK;
        // cudaFree waits for the device; with several devices driven by one process (multi-device contexts, group.cu) that
        // wait must not happen inside the runtime call, where it could hold up another thread's launch of the collective
        // this device is waiting for: drain the device first, then free
        if (p) { cudaDeviceSynchronize(); cudaFree(p); }
        p = nullptr; cap = 0;
        size_t want = bytes + (bytes >> 3);
        cudaError_t e = cudaMalloc(&p, want);
        if (e != cudaSuccess) {
            e = cudaMalloc(&p, bytes);
            want = bytes;
        }
        if (e != cudaSuccess) {
            (void)cudaGetLastError();   // clear the sticky-free error state
            tp_set_error("cudaMalloc(%zu) failed: %s", bytes, cudaGetErrorString(e));
            return TP_ERR_NOMEM;
        }
        cap = want;
        return TP_OK;
    }
    void release() { if (p) cudaFree(p); p = nullptr; cap = 0; }
    template <class T> T *as() const { return (T *)p; }
};

enum { EV_FILTER0 = 0, EV_FILTER1, EV_COMPACT0, EV_COMPACT1, EV_CORR0, EV_CORR1, EV_PCA0, EV_PCA1,
       EV_SWEEP0, EV_SWEEP1, EV_CH1, EV_TOTAL0, EV_TOTAL1, EV_DIFFT0, EV_DIFFT1, EV_INGEST0, EV_INGEST1, EV_COUNT };

static inline int round_up(int x, int m) { return (x + m - 1) / m * m; }

#define TP_COMM_SLOTS 4
struct TpCommSlot { void *handle = nullptr; int rank = 0, nranks = 1; };

struct TpGroup;
struct TpPool;

struct tp_ctx {
    // multi-device context (group.cu): every member points to the group; the member with group_rank 0 is the handle the
    // caller holds.  One host thread per member device runs the members' calls (the members are the "ranks" of comm.cu).
    TpGroup *group = nullptr;
    int group_rank = 0;
    TpPool *pool = nullptr;        // contexts of tp_call_batch, owned by the context the batch was first run on
    long long generation = 0;      // bumped whenever the resident matrix / scores / sweep state are replaced

    int device = 0;
    int sm_count = 148;
    int max_smem_optin = 0;
    cudaStream_t stream = nullptr;
    cudaEvent_t ev[EV_COUNT] = {};
    bool ev_set[EV_COUNT] = {};
    long long launches = 0;

    // communicators (comm.cu): slot 0 is conventionally the whole job, others sub-groups (chromosome arms);
    // comm_cur = -1: no collective (single GPU, or replicated / independent work)
    TpCommSlot comm[TP_COMM_SLOTS];
    int comm_cur = -1;
    bool comm_grouped = false;   // between tp_comm_group_begin / end
    int last_sweep_ranks = 1;    // ranks the candidates of the last sweep were dealt out over (owner of candidate c: c % ranks)
    int dist_min_n = 4096;       // matrices smaller than this are not row-sharded over the ranks (only the candidate sweep is)
    int igemm_min_n = 1024;      // integer-count matrices at least this large take the tcgen05 int8 Gram path (0 = never)
    int iop_min_n = 1024;        // smallest nf whose early subspace-iteration rounds use the sliced int8 operator (0 = never)
    int sync_blocking = 0;       // 1: the host waits for the stream on a blocking-sync event (the thread sleeps) instead of
                                 // cudaStreamSynchronize (which spins on a core): for hosts with more waiting threads than cores
    cudaEvent_t sync_ev = nullptr;
    int shard_sym = 1;           // several ranks: symmetric products computed once per block pair (SymShard); 0 = full-width row blocks
    int mgram_min_n = 1024;      // smallest nf whose M = Xc Xc^T is formed by the sliced int8 Gram (needs the sliced operator; 0 = FP64 DMMA)
    int iop_final_min_n = 1024;  // below this nf the later rounds use the FP64 DMMA operator whatever iop_final says (measured at N = 2000, 8 calls in flight: 224 -> 264 calls/s with the sliced operator)
    int iop_final = 8;           // operator of the later rounds where the sliced one is in use: 8 digit planes, or 0 = FP64 DMMA
    int io_bn32 = -1;            // operator applications on 32-column tiles: -1 = when 64-column tiles would not fill the SMs, 0 / 1 = never / always
    double iop_switch = 1e-3;    // relative residual below which the 8-plane (or FP64 DMMA) operator takes over (the first iteration always starts with 5 planes)

    // tunables
    int pca_block = 0;
    double pca_tol = 1e-12;
    int pca_maxit = 16;
    int pca_inner = 4;
    int jacobi_direct_max = 512;
    int level_cap = 256;

    // input side (ingest.cu): text of the matrix file, row-end offsets, fields left to the host, pinned staging
    DevBuf itext, icounts, irows, islow, icoo;   // icoo: (count, bin1, bin2) triplets of a sparse input
    void *ipin[2] = {nullptr, nullptr};
    cudaEvent_t ipin_ev[2] = {nullptr, nullptr};
    // pageable host matrices (filter.cu, upload_upper): lanes of pinned staging filled by helper threads
    struct UploadLane { cudaStream_t st = nullptr; void *pin[2] = {nullptr, nullptr}; cudaEvent_t ev[2] = {nullptr, nullptr}; cudaEvent_t done = nullptr; };
    std::vector<UploadLane> lanes;
    int upload_lanes = 4;                // tunable: 0 = always the driver's own staging
    int ingested_n = 0;                  // > 0: raw_own holds a matrix parsed on the device (row-major n x n)
    double ingest_stats[4] = {};         // wall ms (read + upload + parse), parse kernels ms, text bytes, host-converted fields

    // stage 1 state
    DevBuf raw_own;              // uploaded copy of the caller's matrix (when it came from the host)
    // batch pool (group.cu): the NEXT call's host matrix is uploaded on a second stream under this call's compute
    // (tp_stage_input); tp_filter adopts it when it is handed the same host pointer
    DevBuf raw_next;
    cudaStream_t copy_stream = nullptr;
    cudaEvent_t staged_ev = nullptr;
    const double *staged_mat = nullptr;
    int staged_n = 0, staged_colmajor = 0;
    std::function<void()> after_filter, after_pca;      // hooks of the batch worker inside tp_call
    const double *raw = nullptr; // device pointer to the N x N input (raw_own.p or caller's)
    int n = 0;
    int colmajor = 0;
    DevBuf rowmean, ranks, flags, qtmp, keep;
    // filtered matrix / correlation (nf x ldx row-major, ldx multiple of 8)
    int nf = 0, ldx = 0;
    DevBuf ioA, ioB, ioscale;            // digit planes / scales of the sliced int8 operator of stage 3 (igemm.cu)
    int io_n = 0;
    bool io_cmax_clean = false;          // the column-maximum scratch of the sliced operator is zero (io_colmax_kernel leaves it so)
    DevBuf X, C, colstat, islices;      // islices: int8 digit planes of X for the tcgen05 integer Gram (igemm.cu)
    bool have_X = false, have_C = false;
    // PCA
    int k = 0, ldk = 0;          // scores: nf x ldk row-major; the sweep uses the first k columns
    int k_full = 0;              // PCs computed by the last tp_pca (tp_recall may lower k below it)
    DevBuf scores, M, Y0, Y1, Y2, W, G, T, Q, Jw, Jv, Jt, small1, small2, part, resid;
    // sticky status words of the small dense kernels, read back at the solver's own sync points:
    // [0] Cholesky met a non-positive pivot  [1] eigensolver did not converge  [2] eigensolver sweeps (sum)
    DevBuf status;
    bool have_scores = false;
    // sweep
    DevBuf P, Qp, d0, seqdist, order, ncl, chs, bsbuf, links, harm;
    int ld_chs = 0;
    int last_maxlev = 0;         // levels (columns) of the score matrix of the last sweep
    std::vector<double> sweep_scores;   // that score matrix on the host: k x last_maxlev row-major, NaN where unscored
    bool have_sweep = false;
    // diffT
    DevBuf lx, ly, dout, dhash, lhash;
    // pinned staging for small read-backs
    void *pin = nullptr;
    size_t pin_cap = 0;
    int *pin_flags = nullptr;    // 64 pinned bytes for the status words

    double timing[10] = {};
    long lowprec_applications = 0;     // operator applications of the last tp_pca done by the sliced int8 operator

    // per-kernel-class profiling (tp_ctx_profile)
    bool prof = false;
    std::vector<cudaEvent_t> prof_ev;      // pool, pairs
    std::vector<int> prof_cls;             // class of pair i
    size_t prof_used = 0;                  // events used
    double prof_gemm_flop = 0.0;           // algorithmic flops of the GEMM launches profiled
    double prof_imma_ops = 0.0;            // executed int8 multiply-add operations (2 per MAC) of the tcgen05 launches profiled
};

enum { PC_ROWMEAN = 0, PC_COMPACT, PC_GEMM, PC_JACOBI, PC_SWEEP, PC_CH, PC_DIFFT, PC_SPARE, PC_CHOL, PC_IGEMM, PC_COMM, PC_SPARE3, PC_ISLICE, PC_SPARE4, PC_SPARE5, PC_SPARE6, PC_COUNT };   // 16 slots
void tp_prof_begin(tp_ctx *ctx, int cls);
void tp_prof_end(tp_ctx *ctx);

// Opt-in limit of dynamic shared memory of a kernel: ALWAYS the most the device allows (minus the kernel's static shared
// memory), never the size of the launch at hand.  The attribute is per function and process-wide, and several host threads
// (tp_call_batch, the member threads of a multi-device context) launch the same kernel with different sizes: "set my
// size, then launch" raced with another thread setting a smaller size in between (cudaErrorInvalidValue at the launch).
// Set once per kernel and device.
cudaError_t tp_optin_smem_fn(const void *kernel, const tp_ctx *ctx);      // api.cu: once per (kernel, device)
template <class K> static inline cudaError_t tp_optin_smem(K kernel, const tp_ctx *ctx) {
    return tp_optin_smem_fn((const void *)kernel, ctx);
}
int tp_pin_reserve(tp_ctx *ctx, size_t bytes);
// wait for everything queued on the context stream (spinning or sleeping, see sync_blocking)
cudaError_t tp_stream_sync(tp_ctx *ctx);

// ---- multi-GPU (comm.cu) ----
static inline int tp_nranks(const tp_ctx *ctx) { return ctx->comm_cur < 0 ? 1 : ctx->comm[ctx->comm_cur].nranks; }
static inline int tp_rank(const tp_ctx *ctx) { return ctx->comm_cur < 0 ? 0 : ctx->comm[ctx->comm_cur].rank; }
// rows of an n-row matrix owned by this rank when the matrix is row-sharded: equal chunks of `rpr` rows
// (a multiple of 64), the last ones possibly short or empty.  Buffers that are all-gathered in place are
// allocated with nranks * rpr rows.
struct TpRows { int rpr, r0, r1, padded; };
static inline TpRows tp_rows(const tp_ctx *ctx, int n) {
    const int R = tp_nranks(ctx), rank = tp_rank(ctx);
    TpRows t;
    t.rpr = round_up((n + R - 1) / R, 64);
    t.r0 = rank * t.rpr < n ? rank * t.rpr : n;
    t.r1 = t.r0 + t.rpr < n ? t.r0 + t.rpr : n;
    t.padded = R * t.rpr;
    return t;
}
static inline bool tp_row_sharded(const tp_ctx *ctx, int n) { return tp_nranks(ctx) > 1 && n >= ctx->dist_min_n; }

// Symmetric n x n products (Gram matrices) over R row-block owners.  Every off-diagonal pair of blocks (a, c) is computed
// ONCE, by the owner of the block row that sees the other block within half a ring ((c - a) mod R < R / 2); the two
// blocks half a ring apart (even R) share theirs along the anti-diagonal of local indices; inside its own diagonal block
// a rank computes the tiles on and above the diagonal and mirrors them on store.  After the all-gather of the row blocks
// every rank holds every computed element and fills the rest by a local transpose (tp_mirror_fill): no extra exchange,
// each rank does 1 / R of the symmetric work, and every element is the same bits whoever computed it.
// R == 1 is the plain symmetric launch.
struct SymShard { int R, rpr; };
// does the owner of row i compute element (i, j)?  (inside a diagonal block: the upper triangle; mirrored on store)
__host__ __device__ inline bool ss_need(int i, int j, SymShard s) {
    const int a = i / s.rpr, c = j / s.rpr;
    int d = c - a; if (d < 0) d += s.R;
    if (d == 0) return j >= i;
    if (2 * d < s.R) return true;
    if (2 * d > s.R) return false;
    const int li = i - a * s.rpr, lj = j - c * s.rpr;
    return a < c ? li + lj < s.rpr : li + lj >= s.rpr;
}
// any needed element in rows [r_lo, r_hi] x columns [c_lo, c_hi]?  (rows within one row block, columns within one column
// block: rpr is a multiple of 64 and tiles are 64 columns wide)
__host__ __device__ inline bool ss_tile_needed(int r_lo, int r_hi, int c_lo, int c_hi, SymShard s) {
    const int a = r_lo / s.rpr, c = c_lo / s.rpr;
    int d = c - a; if (d < 0) d += s.R;
    if (d == 0) return c_hi >= r_lo;
    if (2 * d < s.R) return true;
    if (2 * d > s.R) return false;
    return a < c ? (r_lo - a * s.rpr) + (c_lo - c * s.rpr) < s.rpr : (r_hi - a * s.rpr) + (c_hi - c * s.rpr) >= s.rpr;
}
// D[i][j] = D[j][i] wherever the owner of row i did not compute (i, j); every rank, on its gathered copy
int tp_mirror_fill(tp_ctx *ctx, double *D, int n, int ld, SymShard s);
int tp_comm_allgather(tp_ctx *ctx, double *buf, size_t chunk);          // in place, chunk doubles per rank
int tp_comm_allreduce_sum(tp_ctx *ctx, void *buf, size_t count, int is_double);
int tp_comm_bcast(tp_ctx *ctx, double *buf, size_t count, int root);
int tp_comm_destroy_all(tp_ctx *ctx);
int tp_comm_bcast_bytes(tp_ctx *ctx, void *buf, size_t bytes, int root);            // in place
int tp_comm_group_begin(tp_ctx *ctx);                                               // ncclGroupStart / End around several
int tp_comm_group_end(tp_ctx *ctx);                                                 // collectives of one rank
int tp_comm_init_all(tp_ctx **members, int nmembers, int slot);                     // ncclCommInitAll over the members' devices
// ---- multi-device contexts (group.cu) ----
// true when `ctx` is the handle of a multi-device context and the caller is not one of its own rank threads: the entry
// point then runs itself once per member device (tp_group_run) instead of on this context alone
bool tp_group_dispatch(const tp_ctx *ctx);
// fn(member, rank) on every member concurrently (rank 0 on the calling thread); first failure wins, its message becomes
// the calling thread's tp_last_error()
int tp_group_run(tp_ctx *ctx, const std::function<int(tp_ctx *, int)> &fn);
int tp_group_size(const tp_ctx *ctx);
tp_ctx *tp_group_member(const tp_ctx *ctx, int rank);
void tp_group_destroy(tp_ctx *leader);
void tp_pool_destroy(tp_ctx *ctx);
// ---- genome-wide pixels (ingest.cu, S0c): every cis pixel in its chromosome's bucket, on one device ----
struct tp_genome {
    int device = 0;
    std::vector<int> bins;                        // bins per chromosome, file order
    std::vector<unsigned long long> offs;         // bucket c = cis pixels [offs[c], offs[c + 1])
    unsigned long long trans = 0, below = 0;
    DevBuf px;                                    // count[ncis] (double), then i[ncis], j[ncis] (int, chromosome-local)
};
// the dense n_c x n_c row-major matrix of chromosome `chrom` into c->raw_own, on c's stream (a bucket held by another device
// is first copied into c->icoo); *out = c->raw_own
int tp_genome_dense(tp_ctx *c, const tp_genome *g, int chrom, double **out);
int tp_upload_range(tp_ctx *ctx, void *dst, const void *src, size_t bytes, cudaStream_t st);   // filter.cu: pageable -> lanes
int tp_stage_input(tp_ctx *ctx, const double *mat, int n, int colmajor);   // filter.cu: upload under the running call
int tp_flags_reset(tp_ctx *ctx);                 // zero the status words (stream ordered)
int tp_flags_read(tp_ctx *ctx, int out[4]);      // copy them to the host (synchronises the stream)
int tp_flags_enqueue(tp_ctx *ctx);               // async copy into ctx->pin_flags; valid after the next stream sync
// record a timing event on the context stream
#define TP_MARK(ctx, id)                                              \
    do {                                                              \
        TP_CUDA(cudaEventRecord((ctx)->ev[id], (ctx)->stream));       \
        (ctx)->ev_set[id] = true;                                     \
    } while (0)

// ---- device helpers ------------------------------------------------------------------------
#ifdef __CUDACC__
__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
// min over the warp of non-negative doubles (or +inf); IEEE bit patterns of non-negative doubles
// order like unsigned integers, so two 32-bit REDUX ops do it.
__device__ __forceinline__ double warp_min_nonneg(double v) {
    unsigned hi = (unsigned)__double2hiint(v);
    unsigned mh = __reduce_min_sync(0xffffffffu, hi);
    unsigned lo = (hi == mh) ? (unsigned)__double2loint(v) : 0xffffffffu;
    unsigned ml = __reduce_min_sync(0xffffffffu, lo);
    return __hiloint2double((int)mh, (int)ml);
}
__device__ __forceinline__ double nan_to_zero(double x) { return x == x ? x : 0.0; }
#endif
