// api.cu -- context management, one-shot pipeline, host-side reductions and result assembly.
#include "common.cuh"
#include "gemm.cuh"
#include <stdarg.h>
#include <algorithm>
#include <mutex>
#include <numeric>
#include <unordered_map>

int tp_sweep_device(tp_ctx *ctx, int min_clusters, int cand_begin, int cand_stride, int *ncand_out);
int tp_ch_device(tp_ctx *ctx, int min_clusters, int ncand, int ld_chs);

static thread_local char g_err[1024] = "";

void tp_set_error(const char *fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

extern "C" const char *tp_last_error(void) { return g_err; }
extern "C" int tp_version(void) { return 109; }

int tp_pin_reserve(tp_ctx *ctx, size_t bytes) {
    if (bytes <= ctx->pin_cap) return TP_OK;
    if (ctx->pin) cudaFreeHost(ctx->pin);
    ctx->pin = nullptr; ctx->pin_cap = 0;
    TP_CUDA(cudaMallocHost(&ctx->pin, bytes));
    ctx->pin_cap = bytes;
    return TP_OK;
}

cudaError_t tp_optin_smem_fn(const void *kernel, const tp_ctx *ctx) {
    static std::mutex mu;
    static std::unordered_map<const void *, unsigned> done;          // kernel -> devices it has been set on
    const unsigned bit = 1u << (ctx->device & 31);
    std::lock_guard<std::mutex> lock(mu);
    unsigned &mask = done[kernel];
    if (mask & bit) return cudaSuccess;
    cudaFuncAttributes a;
    cudaError_t e = cudaFuncGetAttributes(&a, kernel);
    if (e != cudaSuccess) return e;
    e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, ctx->max_smem_optin - (int)a.sharedSizeBytes);
    if (e == cudaSuccess) mask |= bit;
    return e;
}

int tp_flags_reset(tp_ctx *ctx) {
    TP_TRY(ctx->status.reserve(64));
    TP_CUDA(cudaMemsetAsync(ctx->status.p, 0, 64, ctx->stream));
    return TP_OK;
}
int tp_flags_enqueue(tp_ctx *ctx) {
    TP_TRY(ctx->status.reserve(64));
    if (!ctx->pin_flags) TP_CUDA(cudaMallocHost((void **)&ctx->pin_flags, 64));
    TP_CUDA(cudaMemcpyAsync(ctx->pin_flags, ctx->status.p, 4 * sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
    return TP_OK;
}
int tp_flags_read(tp_ctx *ctx, int out[4]) {
    TP_TRY(tp_flags_enqueue(ctx));
    TP_CUDA(tp_stream_sync(ctx));
    for (int i = 0; i < 4; i++) out[i] = ctx->pin_flags[i];
    return TP_OK;
}

extern "C" int tp_ctx_set(tp_ctx *ctx, const char *key, double value);
extern "C" int tp_ctx_destroy(tp_ctx *ctx);

cudaError_t tp_stream_sync(tp_ctx *ctx) {
    if (!ctx->sync_blocking || !ctx->sync_ev) return cudaStreamSynchronize(ctx->stream);
    cudaError_t e = cudaEventRecord(ctx->sync_ev, ctx->stream);
    if (e != cudaSuccess) return e;
    return cudaEventSynchronize(ctx->sync_ev);
}

extern "C" int tp_ctx_create(int device, tp_ctx **out) {
    TP_ARG(out, "tp_ctx_create: null output pointer");
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0) {
        tp_set_error("tp_ctx_create: no CUDA device available (%s); this library has no CPU fallback",
                     e == cudaSuccess ? "device count is 0" : cudaGetErrorString(e));
        return TP_ERR_CUDA;
    }
    TP_ARG(device >= 0 && device < ndev, "tp_ctx_create: device index out of range");
    TP_CUDA(cudaSetDevice(device));
    cudaDeviceProp prop;
    TP_CUDA(cudaGetDeviceProperties(&prop, device));
    if (prop.major < 10) {
        tp_set_error("tp_ctx_create: device %d is sm_%d%d; this library is built for sm_100a (B200) only",
                     device, prop.major, prop.minor);
        return TP_ERR_CUDA;
    }
    tp_ctx *ctx = new tp_ctx();
    ctx->device = device;
    ctx->sm_count = prop.multiProcessorCount;
    ctx->max_smem_optin = (int)prop.sharedMemPerBlockOptin;
    TP_CUDA(cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking));
    for (int i = 0; i < EV_COUNT; i++) TP_CUDA(cudaEventCreate(&ctx->ev[i]));
    TP_CUDA(cudaEventCreateWithFlags(&ctx->sync_ev, cudaEventBlockingSync | cudaEventDisableTiming));
    TP_TRY(tp_pin_reserve(ctx, 1 << 16));
    TP_TRY(tp_flags_reset(ctx));
    // TADPOLE_TUNE="key=value,key=value": tp_ctx_set applied to every new context (for hosts that do not expose the
    // tunables, e.g. the R functions, and for experiments); an unknown key is an error, not ignored
    if (const char *tune = getenv("TADPOLE_TUNE")) {
        std::string t(tune);
        size_t pos = 0;
        while (pos < t.size()) {
            size_t end = t.find(',', pos);
            if (end == std::string::npos) end = t.size();
            const std::string item = t.substr(pos, end - pos);
            pos = end + 1;
            if (item.empty()) continue;
            const size_t eq = item.find('=');
            char *endp = nullptr;
            const double v = eq == std::string::npos ? 0.0 : strtod(item.c_str() + eq + 1, &endp);
            if (eq == std::string::npos || eq == 0 || endp == item.c_str() + eq + 1 || *endp) {
                tp_set_error("tp_ctx_create: TADPOLE_TUNE item '%s' is not key=number", item.c_str());
                tp_ctx_destroy(ctx);
                return TP_ERR_ARG;
            }
            if (tp_ctx_set(ctx, item.substr(0, eq).c_str(), v) != TP_OK) { tp_ctx_destroy(ctx); return TP_ERR_ARG; }
        }
    }
    *out = ctx;
    return TP_OK;
}

extern "C" int tp_ctx_destroy(tp_ctx *ctx) {
    if (!ctx) return TP_OK;
    tp_pool_destroy(ctx);
    tp_group_destroy(ctx);           // a multi-device handle takes its member contexts and their threads with it
    cudaSetDevice(ctx->device);
    tp_stream_sync(ctx);
    DevBuf *bufs[] = {&ctx->raw_own, &ctx->rowmean, &ctx->ranks, &ctx->flags, &ctx->qtmp, &ctx->keep, &ctx->X, &ctx->C,
                      &ctx->colstat, &ctx->scores, &ctx->M, &ctx->Y0, &ctx->Y1, &ctx->Y2, &ctx->W, &ctx->G, &ctx->T,
                      &ctx->Q, &ctx->Jw, &ctx->Jv, &ctx->Jt, &ctx->small1, &ctx->small2, &ctx->part, &ctx->resid,
                      &ctx->P, &ctx->Qp, &ctx->d0, &ctx->seqdist, &ctx->order, &ctx->ncl, &ctx->chs, &ctx->bsbuf,
                      &ctx->links, &ctx->harm, &ctx->status, &ctx->islices, &ctx->ioA, &ctx->ioB, &ctx->ioscale, &ctx->lx, &ctx->ly, &ctx->dout, &ctx->dhash, &ctx->lhash,
                      &ctx->itext, &ctx->icounts, &ctx->irows, &ctx->islow, &ctx->icoo, &ctx->raw_next};
    for (DevBuf *b : bufs) b->release();
    tp_comm_destroy_all(ctx);
    for (int i = 0; i < EV_COUNT; i++) if (ctx->ev[i]) cudaEventDestroy(ctx->ev[i]);
    for (cudaEvent_t e : ctx->prof_ev) cudaEventDestroy(e);
    if (ctx->sync_ev) cudaEventDestroy(ctx->sync_ev);
    if (ctx->staged_ev) cudaEventDestroy(ctx->staged_ev);
    for (tp_ctx::UploadLane &ln : ctx->lanes) {
        if (ln.st) { cudaStreamSynchronize(ln.st); cudaStreamDestroy(ln.st); }
        if (ln.done) cudaEventDestroy(ln.done);
        for (int b = 0; b < 2; b++) { if (ln.pin[b]) cudaFreeHost(ln.pin[b]); if (ln.ev[b]) cudaEventDestroy(ln.ev[b]); }
    }
    if (ctx->copy_stream) { cudaStreamSynchronize(ctx->copy_stream); cudaStreamDestroy(ctx->copy_stream); }
    for (int b = 0; b < 2; b++) {
        if (ctx->ipin[b]) cudaFreeHost(ctx->ipin[b]);
        if (ctx->ipin_ev[b]) cudaEventDestroy(ctx->ipin_ev[b]);
    }
    if (ctx->pin) cudaFreeHost(ctx->pin);
    if (ctx->pin_flags) cudaFreeHost(ctx->pin_flags);
    if (ctx->stream) cudaStreamDestroy(ctx->stream);
    delete ctx;
    return TP_OK;
}

extern "C" int tp_ctx_sync(tp_ctx *ctx) {
    TP_ARG(ctx, "tp_ctx_sync: null context");
    for (int r = tp_group_size(ctx) - 1; r >= 0; r--) {
        tp_ctx *m = tp_group_member(ctx, r);
        TP_CUDA(cudaSetDevice(m->device));
        TP_CUDA(tp_stream_sync(m));
    }
    return TP_OK;
}

extern "C" void *tp_ctx_stream(tp_ctx *ctx) { return ctx ? (void *)ctx->stream : nullptr; }
extern "C" long long tp_ctx_launches(tp_ctx *ctx) { return ctx ? ctx->launches : 0; }

extern "C" int tp_ctx_set(tp_ctx *ctx, const char *key, double value) {
    TP_ARG(ctx && key, "tp_ctx_set: null argument");
    if (tp_group_dispatch(ctx)) {     // host-side fields only: no need for the member threads
        for (int r = 1; r < tp_group_size(ctx); r++) {
            tp_ctx *m = tp_group_member(ctx, r);
            TpGroup *g = m->group;
            m->group = nullptr;
            const int rc = tp_ctx_set(m, key, value);
            m->group = g;
            TP_TRY(rc);
        }
    }
    std::string k(key);
    if (k == "pca_block") ctx->pca_block = (int)value;
    else if (k == "pca_tol") ctx->pca_tol = value;
    else if (k == "pca_maxit") ctx->pca_maxit = (int)value;
    else if (k == "pca_inner") ctx->pca_inner = (int)value < 1 ? 1 : (int)value;
    else if (k == "jacobi_direct_max") ctx->jacobi_direct_max = (int)value;
    else if (k == "level_cap") ctx->level_cap = (int)value;
    else if (k == "dist_min_n") ctx->dist_min_n = (int)value;
    else if (k == "igemm_min_n") ctx->igemm_min_n = (int)value;
    else if (k == "iop_min_n") ctx->iop_min_n = (int)value;
    else if (k == "mgram_min_n") ctx->mgram_min_n = (int)value;
    else if (k == "shard_sym") ctx->shard_sym = (int)value != 0;
    else if (k == "sync_blocking") ctx->sync_blocking = (int)value != 0;
    else if (k == "upload_lanes") ctx->upload_lanes = (int)value < 0 ? 0 : ((int)value > 16 ? 16 : (int)value);
    else if (k == "iop_switch") ctx->iop_switch = value;
    else if (k == "io_bn32") ctx->io_bn32 = (int)value;
    else if (k == "batch_resident") ctx->batch_resident = (int)value != 0;
    else if (k == "iop_final") ctx->iop_final = ((int)value == 8) ? 8 : 0;
    else if (k == "iop_final_min_n") ctx->iop_final_min_n = (int)value;
    else { tp_set_error("tp_ctx_set: unknown key '%s'", key); return TP_ERR_ARG; }
    return TP_OK;
}

extern "C" int tp_ctx_get(tp_ctx *ctx, const char *key, double *value_out) {
    TP_ARG(ctx && key && value_out, "tp_ctx_get: null argument");
    const std::string k(key);
    double v;
    if (k == "pca_block") v = ctx->pca_block;
    else if (k == "pca_tol") v = ctx->pca_tol;
    else if (k == "pca_maxit") v = ctx->pca_maxit;
    else if (k == "pca_inner") v = ctx->pca_inner;
    else if (k == "jacobi_direct_max") v = ctx->jacobi_direct_max;
    else if (k == "level_cap") v = ctx->level_cap;
    else if (k == "dist_min_n") v = ctx->dist_min_n;
    else if (k == "igemm_min_n") v = ctx->igemm_min_n;
    else if (k == "iop_min_n") v = ctx->iop_min_n;
    else if (k == "mgram_min_n") v = ctx->mgram_min_n;
    else if (k == "shard_sym") v = ctx->shard_sym;
    else if (k == "sync_blocking") v = ctx->sync_blocking;
    else if (k == "upload_lanes") v = ctx->upload_lanes;
    else if (k == "iop_switch") v = ctx->iop_switch;
    else if (k == "io_bn32") v = ctx->io_bn32;
    else if (k == "batch_resident") v = ctx->batch_resident;
    else if (k == "iop_final") v = ctx->iop_final;
    else if (k == "iop_final_min_n") v = ctx->iop_final_min_n;
    else { tp_set_error("tp_ctx_get: unknown key '%s'", key); return TP_ERR_ARG; }
    *value_out = v;
    return TP_OK;
}

static double ev_ms(tp_ctx *ctx, int a, int b) {
    if (!ctx->ev_set[a] || !ctx->ev_set[b]) return 0.0;
    float ms = 0.f;
    if (cudaEventElapsedTime(&ms, ctx->ev[a], ctx->ev[b]) != cudaSuccess) { (void)cudaGetLastError(); return 0.0; }
    return ms;
}

extern "C" int tp_ctx_timings(tp_ctx *ctx, double *out10) {
    TP_ARG(ctx && out10, "tp_ctx_timings: null argument");
    TP_CUDA(tp_stream_sync(ctx));
    out10[0] = ev_ms(ctx, EV_FILTER0, EV_FILTER1);
    out10[1] = ev_ms(ctx, EV_COMPACT0, EV_COMPACT1);
    out10[2] = ev_ms(ctx, EV_CORR0, EV_CORR1);
    out10[3] = ev_ms(ctx, EV_PCA0, EV_PCA1);
    out10[4] = ev_ms(ctx, EV_SWEEP0, EV_SWEEP1);
    out10[5] = ev_ms(ctx, EV_SWEEP1, EV_CH1);
    out10[6] = ev_ms(ctx, EV_TOTAL0, EV_TOTAL1);
    out10[7] = ctx->timing[7]; out10[8] = ctx->timing[8]; out10[9] = ctx->timing[9];
    return TP_OK;
}

void tp_prof_begin(tp_ctx *ctx, int cls) {
    if (!ctx->prof) return;
    if (ctx->prof_used + 2 > ctx->prof_ev.size()) {
        for (int i = 0; i < 512; i++) { cudaEvent_t e; cudaEventCreate(&e); ctx->prof_ev.push_back(e); }
    }
    ctx->prof_cls.resize(ctx->prof_ev.size() / 2);
    ctx->prof_cls[ctx->prof_used / 2] = cls;
    cudaEventRecord(ctx->prof_ev[ctx->prof_used], ctx->stream);
}
void tp_prof_end(tp_ctx *ctx) {
    if (!ctx->prof) return;
    cudaEventRecord(ctx->prof_ev[ctx->prof_used + 1], ctx->stream);
    ctx->prof_used += 2;
}

extern "C" int tp_ctx_profile(tp_ctx *ctx, int enable, double *ms_out16, long long *count_out16) {
    TP_ARG(ctx, "tp_ctx_profile: null context");
    TP_CUDA(tp_stream_sync(ctx));
    if (ms_out16 || count_out16) {
        double ms[PC_COUNT] = {};
        long long cnt[PC_COUNT] = {};
        for (size_t i = 0; i + 1 < ctx->prof_used; i += 2) {
            float t = 0.f;
            if (cudaEventElapsedTime(&t, ctx->prof_ev[i], ctx->prof_ev[i + 1]) == cudaSuccess) {
                ms[ctx->prof_cls[i / 2]] += t;
                cnt[ctx->prof_cls[i / 2]]++;
            } else (void)cudaGetLastError();
        }
        ms[PC_SPARE] = ctx->prof_gemm_flop * 1e-9;   // slot 7: GFLOP of the profiled GEMM launches
        ms[PC_SPARE3] = ctx->prof_imma_ops * 1e-9;   // slot 11: executed int8 GOP of the profiled tcgen05 launches
        for (int c = 0; c < PC_COUNT; c++) { if (ms_out16) ms_out16[c] = ms[c]; if (count_out16) count_out16[c] = cnt[c]; }
    }
    if (enable == 1) { ctx->prof = true; ctx->prof_used = 0; ctx->prof_gemm_flop = 0.0; ctx->prof_imma_ops = 0.0; }
    else if (enable == 0) ctx->prof = false;
    return TP_OK;
}

// ---- test hooks for the b x b kernels of stage 3 ---------------------------------------------------
int tp_chol_inv(tp_ctx *ctx, double *G, double *Linv, int b, int ld, int *bad_out);
int tp_chol_factor(tp_ctx *ctx, double *G, int b, int ld);
int tp_jacobi(tp_ctx *ctx, double *A, int b, int ld, double *w, double *Vs, int lds, int ncols_out, int *sweeps_out,
              double tol, double predict = 0.0);

extern "C" int tp_test_cholinv(tp_ctx *ctx, const double *g, int b, int factor_only, double *l_out, double *linv_out,
                               int *bad_out) {
    TP_ARG(ctx && g && b >= 1 && l_out, "tp_test_cholinv: bad arguments");
    TP_CUDA(cudaSetDevice(ctx->device));
    const int ld = round_up(b, 8);
    const size_t bytes = (size_t)b * ld * sizeof(double);
    TP_TRY(ctx->G.reserve(bytes)); TP_TRY(ctx->small1.reserve(bytes));
    TP_CUDA(cudaMemsetAsync(ctx->G.p, 0, bytes, ctx->stream));
    TP_CUDA(cudaMemsetAsync(ctx->small1.p, 0, bytes, ctx->stream));
    TP_CUDA(cudaMemcpy2DAsync(ctx->G.p, (size_t)ld * sizeof(double), g, (size_t)b * sizeof(double),
                              (size_t)b * sizeof(double), b, cudaMemcpyHostToDevice, ctx->stream));
    int bad = 0;
    if (factor_only) TP_TRY(tp_chol_factor(ctx, ctx->G.as<double>(), b, ld));
    else TP_TRY(tp_chol_inv(ctx, ctx->G.as<double>(), ctx->small1.as<double>(), b, ld, &bad));
    if (bad_out) *bad_out = bad;
    TP_CUDA(cudaMemcpy2DAsync(l_out, (size_t)b * sizeof(double), ctx->G.p, (size_t)ld * sizeof(double),
                              (size_t)b * sizeof(double), b, cudaMemcpyDeviceToHost, ctx->stream));
    if (linv_out && !factor_only)
        TP_CUDA(cudaMemcpy2DAsync(linv_out, (size_t)b * sizeof(double), ctx->small1.p, (size_t)ld * sizeof(double),
                                  (size_t)b * sizeof(double), b, cudaMemcpyDeviceToHost, ctx->stream));
    TP_CUDA(tp_stream_sync(ctx));
    return TP_OK;
}

extern "C" int tp_test_eig(tp_ctx *ctx, const double *t, int b, double tol, double *w_out, double *v_out,
                           int *sweeps_out) {
    TP_ARG(ctx && t && b >= 1 && w_out && v_out, "tp_test_eig: bad arguments");
    TP_CUDA(cudaSetDevice(ctx->device));
    const int ld = round_up(b, 8);
    const size_t bytes = (size_t)b * ld * sizeof(double);
    TP_TRY(ctx->T.reserve(bytes)); TP_TRY(ctx->Jv.reserve(bytes)); TP_TRY(ctx->Jw.reserve((size_t)4 * b * sizeof(double)));
    TP_CUDA(cudaMemsetAsync(ctx->T.p, 0, bytes, ctx->stream));
    TP_CUDA(cudaMemsetAsync(ctx->Jv.p, 0, bytes, ctx->stream));
    TP_CUDA(cudaMemcpy2DAsync(ctx->T.p, (size_t)ld * sizeof(double), t, (size_t)b * sizeof(double),
                              (size_t)b * sizeof(double), b, cudaMemcpyHostToDevice, ctx->stream));
    int sweeps = 0;
    TP_TRY(tp_jacobi(ctx, ctx->T.as<double>(), b, ld, ctx->Jw.as<double>(), ctx->Jv.as<double>(), ld, b, &sweeps, tol));
    if (sweeps_out) *sweeps_out = sweeps;
    TP_CUDA(cudaMemcpyAsync(w_out, ctx->Jw.p, (size_t)b * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    TP_CUDA(cudaMemcpy2DAsync(v_out, (size_t)b * sizeof(double), ctx->Jv.p, (size_t)ld * sizeof(double),
                              (size_t)b * sizeof(double), b, cudaMemcpyDeviceToHost, ctx->stream));
    TP_CUDA(tp_stream_sync(ctx));
    return TP_OK;
}

int tp_igram(tp_ctx *ctx, const double *X, int n, int ld, double *C, int ldc, const double *mean, const double *sd,
             int raw, int *used_out, int row_begin, int row_end, SymShard ss);

// Gram matrix X X^T of a symmetric n x n matrix of integer counts through the tcgen05 int8 path (host in / out,
// row-major); *used_out = 0 when the input is not integer-valued (gram_out untouched)
extern "C" int tp_test_igram(tp_ctx *ctx, const double *x, int n, double *gram_out, int *used_out) {
    TP_ARG(ctx && x && n >= 1 && gram_out && used_out, "tp_test_igram: bad arguments");
    TP_CUDA(cudaSetDevice(ctx->device));
    const int ld = round_up(n, 8);
    const size_t bytes = (size_t)n * ld * sizeof(double);
    TP_TRY(ctx->X.reserve(bytes)); TP_TRY(ctx->C.reserve(bytes));
    TP_CUDA(cudaMemsetAsync(ctx->X.p, 0, bytes, ctx->stream));
    TP_CUDA(cudaMemcpy2DAsync(ctx->X.p, (size_t)ld * sizeof(double), x, (size_t)n * sizeof(double),
                              (size_t)n * sizeof(double), n, cudaMemcpyHostToDevice, ctx->stream));
    ctx->have_X = ctx->have_C = false;
    TP_TRY(tp_igram(ctx, ctx->X.as<double>(), n, ld, ctx->C.as<double>(), ld, nullptr, nullptr, 1, used_out, 0, n,
                    SymShard{1, 1 << 30}));
    if (*used_out)
        TP_CUDA(cudaMemcpy2DAsync(gram_out, (size_t)n * sizeof(double), ctx->C.p, (size_t)ld * sizeof(double),
                                  (size_t)n * sizeof(double), n, cudaMemcpyDeviceToHost, ctx->stream));
    TP_CUDA(tp_stream_sync(ctx));
    return TP_OK;
}

int tp_igram_sliced(tp_ctx *ctx, const double *A, int n, int ld, double *M, int ldm, int row_begin, int row_end,
                    int sym, SymShard ss);

// A A^T of a general n x n FP64 matrix through the sliced int8 Gram that forms M = Xc Xc^T in tp_pca (host in / out,
// row-major); rows [row_begin, row_end) of the result are written, the others left as they are in gram_out
extern "C" int tp_test_mgram(tp_ctx *ctx, const double *a, int n, int row_begin, int row_end, double *gram_out) {
    TP_ARG(ctx && a && n >= 1 && gram_out && 0 <= row_begin && row_begin <= row_end && row_end <= n, "tp_test_mgram: bad arguments");
    TP_CUDA(cudaSetDevice(ctx->device));
    const int ld = round_up(n, 8);
    const size_t bytes = (size_t)n * ld * sizeof(double);
    TP_TRY(ctx->C.reserve(bytes)); TP_TRY(ctx->M.reserve(bytes));
    TP_CUDA(cudaMemsetAsync(ctx->C.p, 0, bytes, ctx->stream));
    TP_CUDA(cudaMemcpy2DAsync(ctx->C.p, (size_t)ld * sizeof(double), a, (size_t)n * sizeof(double),
                              (size_t)n * sizeof(double), n, cudaMemcpyHostToDevice, ctx->stream));
    TP_CUDA(cudaMemcpy2DAsync(ctx->M.p, (size_t)ld * sizeof(double), gram_out, (size_t)n * sizeof(double),
                              (size_t)n * sizeof(double), n, cudaMemcpyHostToDevice, ctx->stream));
    ctx->have_C = ctx->have_scores = ctx->have_sweep = false;
    TP_TRY(tp_igram_sliced(ctx, ctx->C.as<double>(), n, ld, ctx->M.as<double>(), ld, row_begin, row_end,
                           row_begin == 0 && row_end == n, SymShard{1, 1 << 30}));
    TP_CUDA(cudaMemcpy2DAsync(gram_out, (size_t)n * sizeof(double), ctx->M.p, (size_t)ld * sizeof(double),
                              (size_t)n * sizeof(double), n, cudaMemcpyDeviceToHost, ctx->stream));
    TP_CUDA(tp_stream_sync(ctx));
    return TP_OK;
}

// host-only views of the SymShard rule the kernels use (no GPU needed): element predicate and tile predicate
extern "C" int tp_test_ss_need(int i, int j, int nranks, int rpr) { return ss_need(i, j, SymShard{nranks, rpr}) ? 1 : 0; }
extern "C" int tp_test_ss_tile(int r_lo, int r_hi, int c_lo, int c_hi, int nranks, int rpr) {
    return ss_tile_needed(r_lo, r_hi, c_lo, c_hi, SymShard{nranks, rpr}) ? 1 : 0;
}

// The symmetric products as `nranks` ranks of a sharded call would compute them (SymShard, common.cuh), emulated on this one
// GPU: every emulated rank's launch writes its row block of one matrix pre-filled with `fill` (standing for the stale
// contents of the other ranks' blocks before the all-gather), then tp_mirror_fill.  kind 0: exact integer Gram of a symmetric
// count matrix (ig_gram_kernel, raw); kind 1: sliced FP64 Gram a a^T (io_gemm_kernel<8>).  The result must equal the
// one-GPU launch bit for bit.
extern "C" int tp_test_symshard(tp_ctx *ctx, const double *a, int n, int nranks, int kind, double fill, double *gram_out) {
    TP_ARG(ctx && a && n >= 1 && nranks >= 1 && gram_out && (kind == 0 || kind == 1), "tp_test_symshard: bad arguments");
    TP_CUDA(cudaSetDevice(ctx->device));
    const int ld = round_up(n, 8);
    const size_t bytes = (size_t)n * ld * sizeof(double);
    DevBuf &in = kind == 0 ? ctx->X : ctx->C, &out = kind == 0 ? ctx->C : ctx->M;
    TP_TRY(in.reserve(bytes)); TP_TRY(out.reserve(bytes));
    TP_CUDA(cudaMemsetAsync(in.p, 0, bytes, ctx->stream));
    TP_CUDA(cudaMemcpy2DAsync(in.p, (size_t)ld * sizeof(double), a, (size_t)n * sizeof(double),
                              (size_t)n * sizeof(double), n, cudaMemcpyHostToDevice, ctx->stream));
    std::vector<double> f((size_t)n * ld, fill);
    TP_CUDA(cudaMemcpyAsync(out.p, f.data(), bytes, cudaMemcpyHostToDevice, ctx->stream));
    TP_CUDA(tp_stream_sync(ctx));
    ctx->have_X = ctx->have_C = ctx->have_scores = ctx->have_sweep = false;
    const SymShard ss{nranks, round_up((n + nranks - 1) / nranks, 64)};
    for (int r = 0; r < nranks; r++) {
        const int r0 = std::min(r * ss.rpr, n), r1 = std::min(r0 + ss.rpr, n);
        if (kind == 0) {
            int used = 0;
            TP_TRY(tp_igram(ctx, in.as<double>(), n, ld, out.as<double>(), ld, nullptr, nullptr, 1, &used, r0, r1, ss));
            TP_ARG(used, "tp_test_symshard: kind 0 needs integer counts below 2^20");
        } else {
            TP_TRY(tp_igram_sliced(ctx, in.as<double>(), n, ld, out.as<double>(), ld, r0, r1, 1, ss));
        }
    }
    TP_TRY(tp_mirror_fill(ctx, out.as<double>(), n, ld, ss));
    TP_CUDA(cudaMemcpy2DAsync(gram_out, (size_t)n * sizeof(double), out.p, (size_t)ld * sizeof(double),
                              (size_t)n * sizeof(double), n, cudaMemcpyDeviceToHost, ctx->stream));
    TP_CUDA(tp_stream_sync(ctx));
    return TP_OK;
}

// ---- test hooks of the two matrix-product engines of stages 2 and 3 ---------------------------------------------------
// Operands live in buffers of their own (no pipeline buffer or have_* flag of the context changes).  A host matrix of
// rows x cols goes up with its leading dimension rounded up to 8 and the padding columns set to NaN (all bits one), so a
// kernel that reads past the logical edge shows it in its result.
struct TestBufs {
    DevBuf b[5];
    ~TestBufs() { for (DevBuf &x : b) x.release(); }
};

static int upload_nan_padded(tp_ctx *ctx, DevBuf &buf, size_t off, const double *h, int rows, int cols, int ld) {
    double *d = buf.as<double>() + off;
    TP_CUDA(cudaMemsetAsync(d, 0xff, (size_t)rows * ld * sizeof(double), ctx->stream));
    TP_CUDA(cudaMemcpy2DAsync(d, (size_t)ld * sizeof(double), h, (size_t)cols * sizeof(double), (size_t)cols * sizeof(double),
                              rows, cudaMemcpyHostToDevice, ctx->stream));
    return TP_OK;
}

// One tp_gemm: D = alpha A B + beta E1 + gamma E2, or the EPI_CORR epilogue when mean != NULL (mean / sd hold
// max(epi_row0 + M, N) entries).  A is M x K row-major (a_kc) or K x M; B is N x K (b_kc) or K x N; E1 / E2 (may be NULL)
// are M x N.  D_inout (M x ldd, ldd >= N) goes up whole and comes back whole.  TADPOLE_GEMM_CFG = 10 / 11 / 12 forces the
// 32x64 / 64x64 / 128x128 tiles.
extern "C" int tp_test_gemm(tp_ctx *ctx, int M, int N, int K, const double *A, int a_kc, const double *B, int b_kc,
                            double alpha, const double *E1, double beta, const double *E2, double gamma, int sym, int splitk,
                            const double *mean, const double *sd, double nrows, int epi_row0, int ldd, double *D_inout) {
    TP_ARG(ctx && M >= 1 && N >= 1 && K >= 1 && A && B && ldd >= N && D_inout && (!mean || (sd && epi_row0 >= 0)),
           "tp_test_gemm: bad arguments");
    TP_CUDA(cudaSetDevice(ctx->device));
    const int ar = a_kc ? M : K, ac = a_kc ? K : M, br = b_kc ? N : K, bc = b_kc ? K : N;
    const int lda = round_up(ac, 8), ldb = round_up(bc, 8), lde = round_up(N, 8);
    const int nv = std::max(epi_row0 + M, N);
    TestBufs t;
    TP_TRY(t.b[0].reserve((size_t)ar * lda * sizeof(double)));
    TP_TRY(t.b[1].reserve((size_t)br * ldb * sizeof(double)));
    TP_TRY(t.b[2].reserve((size_t)2 * M * lde * sizeof(double)));
    TP_TRY(t.b[3].reserve((size_t)M * ldd * sizeof(double)));
    TP_TRY(t.b[4].reserve((size_t)2 * nv * sizeof(double)));
    TP_TRY(upload_nan_padded(ctx, t.b[0], 0, A, ar, ac, lda));
    TP_TRY(upload_nan_padded(ctx, t.b[1], 0, B, br, bc, ldb));
    if (E1) TP_TRY(upload_nan_padded(ctx, t.b[2], 0, E1, M, N, lde));
    if (E2) TP_TRY(upload_nan_padded(ctx, t.b[2], (size_t)M * lde, E2, M, N, lde));
    TP_CUDA(cudaMemcpyAsync(t.b[3].p, D_inout, (size_t)M * ldd * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
    GemmArgs g;
    g.A = t.b[0].as<double>(); g.lda = lda; g.a_kc = a_kc ? 1 : 0;
    g.B = t.b[1].as<double>(); g.ldb = ldb; g.b_kc = b_kc ? 1 : 0;
    g.D = t.b[3].as<double>(); g.ldd = ldd;
    g.M = M; g.N = N; g.K = K;
    g.alpha = alpha; g.beta = beta; g.gamma = gamma;
    if (E1) { g.E1 = t.b[2].as<double>(); g.lde1 = lde; }
    if (E2) { g.E2 = t.b[2].as<double>() + (size_t)M * lde; g.lde2 = lde; }
    g.sym = sym ? 1 : 0; g.splitk = splitk;
    if (mean) {
        double *st = t.b[4].as<double>();
        TP_CUDA(cudaMemcpyAsync(st, mean, (size_t)nv * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
        TP_CUDA(cudaMemcpyAsync(st + nv, sd, (size_t)nv * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
        g.epi = EPI_CORR; g.mean = st; g.sd = st + nv; g.nrows = nrows; g.epi_row0 = epi_row0;
    }
    TP_TRY(tp_gemm(ctx, g));
    TP_CUDA(cudaMemcpyAsync(D_inout, t.b[3].p, (size_t)M * ldd * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    TP_CUDA(tp_stream_sync(ctx));
    return TP_OK;
}

int tp_iop_prepare(tp_ctx *ctx, const double *S, int n, int ld);
int tp_iop_apply(tp_ctx *ctx, const double *Yin, int b, int ldy, double *D, int ldd, double alpha, const double *E1,
                 int lde1, double beta, const double *E2, int lde2, double gamma, int row_begin, int row_end, int np);

// tp_iop_prepare of the symmetric n x n operator S once, then `napps` tp_iop_apply in order on this context:
// D_a[rows] = alpha S[rows, :] Y_a + beta E1_a[rows] + gamma E2_a[rows], rows = [row_begin, row_end), block width bs[a]
// (<= 1024), np = 5 or 8 digit planes.  Ys, E1, E2 (may be NULL) and D_inout hold the n x bs[a] blocks back to back.
// Rows of D outside the range keep their values; a write into the padding columns of a D block is reported as an error.
// Tile width: the context's "io_bn32".
extern "C" int tp_test_iop(tp_ctx *ctx, const double *S, int n, int napps, const int *bs, const double *Ys, int np,
                           int row_begin, int row_end, double alpha, const double *E1, double beta, const double *E2,
                           double gamma, double *D_inout) {
    TP_ARG(ctx && S && n >= 1 && napps >= 1 && bs && Ys && D_inout && 0 <= row_begin && row_begin < row_end && row_end <= n,
           "tp_test_iop: bad arguments");
    TP_CUDA(cudaSetDevice(ctx->device));
    size_t tot = 0;
    for (int a = 0; a < napps; a++) {
        TP_ARG(bs[a] >= 1 && bs[a] <= 1024, "tp_test_iop: block widths 1..1024");
        tot += (size_t)n * round_up(bs[a], 8);
    }
    const int lds = round_up(n, 8);
    TestBufs t;
    TP_TRY(t.b[0].reserve((size_t)n * lds * sizeof(double)));
    for (int i = 1; i < 5; i++) TP_TRY(t.b[i].reserve(tot * sizeof(double)));
    TP_TRY(upload_nan_padded(ctx, t.b[0], 0, S, n, n, lds));
    size_t ho = 0, dof = 0;                 // host / device offsets of block a
    for (int a = 0; a < napps; a++) {
        const int b = bs[a], ld = round_up(b, 8);
        TP_TRY(upload_nan_padded(ctx, t.b[1], dof, Ys + ho, n, b, ld));
        if (E1) TP_TRY(upload_nan_padded(ctx, t.b[2], dof, E1 + ho, n, b, ld));
        if (E2) TP_TRY(upload_nan_padded(ctx, t.b[3], dof, E2 + ho, n, b, ld));
        TP_TRY(upload_nan_padded(ctx, t.b[4], dof, D_inout + ho, n, b, ld));
        ho += (size_t)n * b; dof += (size_t)n * ld;
    }
    TP_TRY(tp_iop_prepare(ctx, t.b[0].as<double>(), n, lds));
    ho = dof = 0;
    for (int a = 0; a < napps; a++) {
        const int b = bs[a], ld = round_up(b, 8);
        TP_TRY(tp_iop_apply(ctx, t.b[1].as<double>() + dof, b, ld, t.b[4].as<double>() + dof, ld, alpha,
                            E1 ? t.b[2].as<double>() + dof : nullptr, ld, beta, E2 ? t.b[3].as<double>() + dof : nullptr, ld,
                            gamma, row_begin, row_end, np));
        dof += (size_t)n * ld;
    }
    std::vector<double> h(tot);
    TP_CUDA(cudaMemcpyAsync(h.data(), t.b[4].p, tot * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    TP_CUDA(tp_stream_sync(ctx));
    ho = dof = 0;
    for (int a = 0; a < napps; a++) {
        const int b = bs[a], ld = round_up(b, 8);
        for (int r = 0; r < n; r++) {
            memcpy(D_inout + ho + (size_t)r * b, h.data() + dof + (size_t)r * ld, (size_t)b * sizeof(double));
            for (int c = b; c < ld; c++) {
                unsigned long long bits;
                memcpy(&bits, h.data() + dof + (size_t)r * ld + c, sizeof(bits));
                if (bits != ~0ull) {
                    tp_set_error("tp_test_iop: application %d wrote D[%d][%d], a padding column of its block", a, r, c);
                    return TP_ERR_CUDA;
                }
            }
        }
        ho += (size_t)n * b; dof += (size_t)n * ld;
    }
    return TP_OK;
}

// ---- set / get hooks ----------------------------------------------------------------------------
static int upload_square(tp_ctx *ctx, DevBuf &buf, const double *h, int n, int ld) {
    TP_TRY(buf.reserve((size_t)n * ld * sizeof(double)));
    TP_CUDA(cudaMemsetAsync(buf.p, 0, (size_t)n * ld * sizeof(double), ctx->stream));
    TP_CUDA(cudaMemcpy2DAsync(buf.p, (size_t)ld * sizeof(double), h, (size_t)n * sizeof(double),
                              (size_t)n * sizeof(double), n, cudaMemcpyHostToDevice, ctx->stream));
    TP_CUDA(tp_stream_sync(ctx));
    return TP_OK;
}
static int download(tp_ctx *ctx, const DevBuf &buf, double *h, int rows, int cols, int ld) {
    TP_CUDA(cudaMemcpy2DAsync(h, (size_t)cols * sizeof(double), buf.p, (size_t)ld * sizeof(double),
                              (size_t)cols * sizeof(double), rows, cudaMemcpyDeviceToHost, ctx->stream));
    TP_CUDA(tp_stream_sync(ctx));
    return TP_OK;
}

extern "C" int tp_set_filtered(tp_ctx *ctx, const double *x, int nf) {
    TP_ARG(ctx && x && nf >= 2, "tp_set_filtered: bad arguments");
    if (tp_group_dispatch(ctx)) return tp_group_run(ctx, [&](tp_ctx *gc, int) -> int { return tp_set_filtered(gc, x, nf); });
    TP_CUDA(cudaSetDevice(ctx->device));
    ctx->generation++;
    ctx->nf = nf; ctx->ldx = round_up(nf, 8);
    TP_TRY(upload_square(ctx, ctx->X, x, nf, ctx->ldx));
    ctx->have_X = true; ctx->have_C = ctx->have_scores = ctx->have_sweep = false;
    return TP_OK;
}
extern "C" int tp_get_filtered(tp_ctx *ctx, double *x_out) {
    TP_ARG(ctx && x_out && ctx->have_X, "tp_get_filtered: no filtered matrix");
    return download(ctx, ctx->X, x_out, ctx->nf, ctx->nf, ctx->ldx);
}
extern "C" int tp_set_correlation(tp_ctx *ctx, const double *cor, int nf) {
    TP_ARG(ctx && cor && nf >= 2, "tp_set_correlation: bad arguments");
    if (tp_group_dispatch(ctx)) return tp_group_run(ctx, [&](tp_ctx *gc, int) -> int { return tp_set_correlation(gc, cor, nf); });
    TP_CUDA(cudaSetDevice(ctx->device));
    ctx->generation++;
    ctx->nf = nf; ctx->ldx = round_up(nf, 8);
    TP_TRY(upload_square(ctx, ctx->C, cor, nf, ctx->ldx));
    ctx->have_C = true; ctx->have_scores = ctx->have_sweep = false;
    return TP_OK;
}
extern "C" int tp_get_correlation(tp_ctx *ctx, double *cor_out) {
    TP_ARG(ctx && cor_out && ctx->have_C, "tp_get_correlation: no correlation matrix (tp_pca consumes it)");
    return download(ctx, ctx->C, cor_out, ctx->nf, ctx->nf, ctx->ldx);
}
extern "C" int tp_set_scores(tp_ctx *ctx, const double *scores, int nf, int k) {
    TP_ARG(ctx && scores && nf >= 3 && k >= 1 && k <= nf, "tp_set_scores: bad arguments");
    if (tp_group_dispatch(ctx)) return tp_group_run(ctx, [&](tp_ctx *gc, int) -> int { return tp_set_scores(gc, scores, nf, k); });
    TP_CUDA(cudaSetDevice(ctx->device));
    ctx->generation++;
    ctx->nf = nf; ctx->k = ctx->k_full = k; ctx->ldk = round_up(k, 8);
    TP_TRY(ctx->scores.reserve((size_t)nf * ctx->ldk * sizeof(double)));
    TP_CUDA(cudaMemsetAsync(ctx->scores.p, 0, (size_t)nf * ctx->ldk * sizeof(double), ctx->stream));
    TP_CUDA(cudaMemcpy2DAsync(ctx->scores.p, (size_t)ctx->ldk * sizeof(double), scores, (size_t)k * sizeof(double),
                              (size_t)k * sizeof(double), nf, cudaMemcpyHostToDevice, ctx->stream));
    TP_CUDA(tp_stream_sync(ctx));
    ctx->have_scores = true; ctx->have_sweep = false;
    return TP_OK;
}
extern "C" int tp_get_scores(tp_ctx *ctx, double *scores_out) {
    TP_ARG(ctx && scores_out && ctx->have_scores, "tp_get_scores: no scores");
    return download(ctx, ctx->scores, scores_out, ctx->nf, ctx->k, ctx->ldk);
}

// ---- stages 4 + 5 ---------------------------------------------------------------------------------
// rows of candidates this rank did not run become 0 so that the sum over ranks is the union (NaN + 0 = NaN)
__global__ void zero_foreign_rows_kernel(double *chs, int *ncl, int k, int ld, int begin, int stride) {
    const size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= (size_t)k * ld) return;
    const int c = (int)(idx / ld);
    if (c < begin || (c - begin) % stride != 0) {
        chs[idx] = 0.0;
        if (idx % ld == 0) ncl[c] = 0;       // (a second, wider pass finds the sums of the first one here)
    }
}

// collective == true: the candidates are dealt out rank-interleaved over the current communicator (cost grows with
// the number of PCs) and the level counts / CH rows are combined on every rank; cand_begin / cand_stride are ignored
static int sweep_impl(tp_ctx *ctx, int min_clusters, int cand_begin, int cand_stride,
                      int *n_cluster_out, int *maxlev_out, bool collective = false) {
    int ncand = 0;
    collective = collective && tp_nranks(ctx) > 1;
    if (collective) { cand_begin = tp_rank(ctx); cand_stride = tp_nranks(ctx); }    // (a rank may end up with no candidate)
    ctx->generation++;
    ctx->last_sweep_ranks = collective ? tp_nranks(ctx) : 1;
    // a sweep that runs no candidate or fails leaves no width or scores of an earlier sweep readable
    ctx->last_maxlev = 0;
    ctx->sweep_scores.clear();
    if (maxlev_out) *maxlev_out = 0;
    TP_TRY(tp_sweep_device(ctx, min_clusters, cand_begin, cand_stride, &ncand));
    const int k = ctx->k;
    if (ncand == 0 && !collective) {
        if (n_cluster_out) std::fill(n_cluster_out, n_cluster_out + k, 0);
        return TP_OK;
    }
    int ld = ctx->level_cap > 8 ? ctx->level_cap : 8;
    TP_TRY(tp_pin_reserve(ctx, (size_t)k * sizeof(int) + 64));
    int *h_ncl = (int *)ctx->pin;
    int maxlev = 0;
    for (int pass = 0; pass < 2; pass++) {
        TP_TRY(tp_ch_device(ctx, min_clusters, ncand, ld));
        if (collective) {
            zero_foreign_rows_kernel<<<(unsigned)(((size_t)k * ld + 255) / 256), 256, 0, ctx->stream>>>(
                ctx->chs.as<double>(), ctx->ncl.as<int>(), k, ld, cand_begin, cand_stride);
            ctx->launches += 1;
            TP_TRY(tp_comm_allreduce_sum(ctx, ctx->ncl.p, (size_t)k, 0));
            TP_TRY(tp_comm_allreduce_sum(ctx, ctx->chs.p, (size_t)k * ld, 1));
        }
        TP_CUDA(cudaMemcpyAsync(h_ncl, ctx->ncl.p, (size_t)k * sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
        TP_CUDA(tp_stream_sync(ctx));
        maxlev = 0;
        for (int c = 0; c < k; c++) {
            if (h_ncl[c] < 0) {
                tp_set_error("candidate %d PCs: no broken-stick level is significant (the reference fails here too: "
                             "n_cluster is NA at R/TADpole.R:113)", c + 1);
                return TP_ERR_NOLEVEL;
            }
            maxlev = std::max(maxlev, h_ncl[c]);
        }
        if (maxlev <= ld) break;
        ld = round_up(maxlev, 8);          // rare: more levels than the cap; redo the cheap CH pass wider
    }
    if (n_cluster_out) memcpy(n_cluster_out, h_ncl, (size_t)k * sizeof(int));
    // the first maxlev columns of every row (in a collective sweep the all-reduced rows, complete on every rank)
    ctx->sweep_scores.resize((size_t)k * maxlev);
    if (maxlev > 0)
        TP_CUDA(cudaMemcpy2DAsync(ctx->sweep_scores.data(), (size_t)maxlev * sizeof(double), ctx->chs.p,
                                  (size_t)ctx->ld_chs * sizeof(double), (size_t)maxlev * sizeof(double), k,
                                  cudaMemcpyDeviceToHost, ctx->stream));
    TP_CUDA(tp_stream_sync(ctx));
    ctx->last_maxlev = maxlev;
    if (maxlev_out) *maxlev_out = maxlev;
    return TP_OK;
}

extern "C" int tp_get_sweep_scores(tp_ctx *ctx, double *scores_out) {
    TP_ARG(ctx && scores_out && ctx->have_sweep, "tp_get_sweep_scores: run tp_sweep / tp_call first");
    std::copy(ctx->sweep_scores.begin(), ctx->sweep_scores.end(), scores_out);
    return TP_OK;
}

extern "C" int tp_sweep(tp_ctx *ctx, int min_clusters, int cand_begin, int cand_stride, int *n_cluster_out,
                        int *maxlev_out) {
    TP_ARG(ctx, "tp_sweep: null context");
    TP_CUDA(cudaSetDevice(ctx->device));
    return sweep_impl(ctx, min_clusters, cand_begin, cand_stride, n_cluster_out, maxlev_out);
}

extern "C" int tp_get_dendro(tp_ctx *ctx, int cand, double *seqdist_out, int *order_out) {
    TP_ARG(ctx && ctx->have_sweep, "tp_get_dendro: run tp_sweep first");
    TP_ARG(cand >= 0 && cand < ctx->k, "tp_get_dendro: candidate out of range");
    const int n1 = ctx->nf - 1, ldd = round_up(n1, 8);
    // after a sweep dealt out over several GPUs the dendrogram lives on the device that ran the candidate
    const int owner = cand % ctx->last_sweep_ranks;
    tp_ctx *src = ctx;
    if (ctx->last_sweep_ranks > 1 && tp_group_dispatch(ctx)) {
        // multi-device context, called by the user (the member threads are idle): read the owner's copy, ordered after
        // whatever is still queued on the owner's stream.  (Inside a grouped call the caller has broadcast what it reads.)
        src = tp_group_member(ctx, owner);
        TP_ARG(src && src->have_sweep && src->nf == ctx->nf && src->k == ctx->k, "tp_get_dendro: the owner device no longer holds this sweep");
    } else if (ctx->last_sweep_ranks > 1 && !ctx->group) {
        // one process per GPU: collective, the owner broadcasts (every rank calls with the same cand)
        TP_ARG(tp_nranks(ctx) == ctx->last_sweep_ranks, "tp_get_dendro: select the communicator the sweep ran over");
        TP_CUDA(cudaSetDevice(ctx->device));
        if (seqdist_out) TP_TRY(tp_comm_bcast(ctx, ctx->seqdist.as<double>() + (size_t)cand * ldd, (size_t)n1, owner));
        if (order_out) TP_TRY(tp_comm_bcast_bytes(ctx, ctx->order.as<int4>() + (size_t)cand * ldd, (size_t)n1 * sizeof(int4), owner));
    }
    TP_CUDA(cudaSetDevice(src->device));
    if (seqdist_out)
        TP_CUDA(cudaMemcpyAsync(seqdist_out, src->seqdist.as<double>() + (size_t)cand * ldd, (size_t)n1 * sizeof(double),
                                cudaMemcpyDeviceToHost, src->stream));
    std::vector<int> tmp;
    if (order_out) {
        tmp.resize((size_t)n1 * 4);
        TP_CUDA(cudaMemcpyAsync(tmp.data(), src->order.as<int4>() + (size_t)cand * ldd, (size_t)n1 * sizeof(int4),
                                cudaMemcpyDeviceToHost, src->stream));
    }
    TP_CUDA(tp_stream_sync(src));
    if (src != ctx) TP_CUDA(cudaSetDevice(ctx->device));
    if (order_out) for (int t = 0; t < n1; t++) order_out[t] = tmp[(size_t)t * 4];
    return TP_OK;
}

// which.max(rowMeans(scores, na.rm = TRUE)); which.max(scores[opt, ])  (R/TADpole.R:134-135)
extern "C" int tp_select(const double *scores, int k, int ld, int maxlev, int *opt_cand, int *opt_level) {
    TP_ARG(scores && opt_cand && opt_level && k >= 1 && maxlev >= 1 && ld >= maxlev, "tp_select: bad arguments");
    int best = -1;
    long double bestv = 0;
    for (int r = 0; r < k; r++) {
        long double s = 0;   // R accumulates rowMeans in long double
        int cnt = 0;
        for (int c = 0; c < maxlev; c++) {
            const double v = scores[(size_t)r * ld + c];
            if (v == v) { s += v; cnt++; }
        }
        if (!cnt) continue;                       // mean of nothing is NaN: ignored by which.max
        const double m = (double)(s / cnt);
        if (m != m) continue;
        if (best < 0 || m > (double)bestv) { best = r; bestv = m; }
    }
    if (best < 0) { tp_set_error("tp_select: every candidate row is NA"); return TP_ERR_NOLEVEL; }
    int bl = -1;
    double blv = 0;
    for (int c = 0; c < maxlev; c++) {
        const double v = scores[(size_t)best * ld + c];
        if (v == v && (bl < 0 || v > blv)) { bl = c; blv = v; }
    }
    if (bl < 0) { tp_set_error("tp_select: optimal row has no score"); return TP_ERR_NOLEVEL; }
    *opt_cand = best;
    *opt_level = bl;
    return TP_OK;
}

// ---- one-shot -----------------------------------------------------------------------------------------
// stages 4 + 5 and the selection on the context's PC scores (first ctx->k columns)
static int sweep_and_select(tp_ctx *ctx, int min_clusters, int *n_pcs_out, int *n_clusters_out, int *maxlev_out,
                            double *seqdist_out) {
    TP_TRY(sweep_impl(ctx, min_clusters, 0, 1, nullptr, maxlev_out, true));
    const int maxlev = ctx->last_maxlev;
    int oc = 0, ol = 0;
    TP_TRY(tp_select(ctx->sweep_scores.data(), ctx->k, maxlev, maxlev, &oc, &ol));
    if (n_pcs_out) *n_pcs_out = oc + 1;
    if (n_clusters_out) *n_clusters_out = ol + 1;
    // the optimal candidate's dendrogram lives on the rank that ran it: after the broadcast every rank holds the row
    const int n1 = ctx->nf - 1, ldd = round_up(n1, 8);
    double *row = ctx->seqdist.as<double>() + (size_t)oc * ldd;
    if (tp_nranks(ctx) > 1) TP_TRY(tp_comm_bcast(ctx, row, (size_t)n1, oc % tp_nranks(ctx)));
    if (seqdist_out) {
        TP_CUDA(cudaMemcpyAsync(seqdist_out, row, (size_t)n1 * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
        TP_CUDA(tp_stream_sync(ctx));
    }
    TP_MARK(ctx, EV_TOTAL1);
    return TP_OK;
}

static int call_from_compacted(tp_ctx *ctx, int max_pcs, int min_clusters, int *k_out, int *n_pcs_out,
                               int *n_clusters_out, int *maxlev_out, double *seqdist_out) {
    int k = 0;
    TP_TRY(tp_correlation(ctx));
    TP_TRY(tp_pca(ctx, max_pcs, &k));
    if (k_out) *k_out = k;
    if (ctx->after_pca) ctx->after_pca();                // batch worker: the next matrix uploads under the sweep
    return sweep_and_select(ctx, min_clusters, n_pcs_out, n_clusters_out, maxlev_out, seqdist_out);
}

// The PC scores of the last call stay in the context: another (max_pcs, min_clusters) only repeats the n_pcs sweep.
// prcomp(rank. = k') returns the first k' columns of the same decomposition, so the first k' columns of the resident
// scores are what a fresh call with max_pcs = k' computes (R/TADpole.R:366-367; CH on those k' columns, quirk Q2) --
// the same decomposition, not the same bits: that call's subspace iteration runs with a narrower block, whose scores
// differ in the last bits.
extern "C" int tp_recall(tp_ctx *ctx, int max_pcs, int min_clusters, int *k_out, int *n_pcs_out, int *n_clusters_out,
                         int *maxlev_out, double *seqdist_out) {
    TP_ARG(ctx, "tp_recall: null context");
    if (tp_group_dispatch(ctx))
        return tp_group_run(ctx, [&](tp_ctx *gc, int gr) -> int {
            return gr ? tp_recall(gc, max_pcs, min_clusters, nullptr, nullptr, nullptr, nullptr, nullptr)
                      : tp_recall(gc, max_pcs, min_clusters, k_out, n_pcs_out, n_clusters_out, maxlev_out, seqdist_out);
        });
    TP_ARG(ctx->have_scores && ctx->k_full >= 1, "tp_recall: no PC scores in the context (run tp_call / tp_call_arm / tp_pca first)");
    TP_ARG(max_pcs >= 1, "tp_recall: max_pcs must be positive");
    const int want = max_pcs < ctx->nf ? max_pcs : ctx->nf;
    if (want > ctx->k_full) {
        tp_set_error("tp_recall: max_pcs = %d needs %d PCs but the context holds %d; run the call again", max_pcs, want, ctx->k_full);
        return TP_ERR_ARG;
    }
    TP_CUDA(cudaSetDevice(ctx->device));
    TP_MARK(ctx, EV_TOTAL0);
    ctx->k = want;
    ctx->have_sweep = false;
    if (k_out) *k_out = want;
    return sweep_and_select(ctx, min_clusters, n_pcs_out, n_clusters_out, maxlev_out, seqdist_out);
}

extern "C" int tp_call(tp_ctx *ctx, const double *mat, int n, int colmajor, int on_device,
                       int max_pcs, int min_clusters, double bad_frac,
                       uint8_t *bad_out, int *nf_out, int *k_out, int *n_pcs_out, int *n_clusters_out,
                       int *maxlev_out, double *seqdist_out) {
    TP_ARG(ctx && mat && bad_out, "tp_call: null argument");
    if (tp_group_dispatch(ctx))
        return tp_group_run(ctx, [&](tp_ctx *gc, int gr) -> int {
            if (gr == 0)
                return tp_call(gc, mat, n, colmajor, on_device, max_pcs, min_clusters, bad_frac, bad_out, nf_out, k_out, n_pcs_out,
                               n_clusters_out, maxlev_out, seqdist_out);
            std::vector<uint8_t> tmp((size_t)(n > 0 ? n : 1));
            return tp_call(gc, mat, n, colmajor, on_device, max_pcs, min_clusters, bad_frac, tmp.data(), nullptr, nullptr, nullptr,
                           nullptr, nullptr, nullptr);
        });
    TP_CUDA(cudaSetDevice(ctx->device));
    TP_MARK(ctx, EV_TOTAL0);
    const int frc = tp_filter(ctx, mat, n, colmajor, on_device, bad_frac, bad_out, nullptr, nullptr);
    if (ctx->after_filter) ctx->after_filter();          // batch worker: this call's upload is over
    TP_TRY(frc);
    std::vector<int> keep;
    keep.reserve(n);
    for (int i = 0; i < n; i++) if (!bad_out[i]) keep.push_back(i);
    if (nf_out) *nf_out = (int)keep.size();
    TP_ARG(keep.size() >= 3, "tp_call: fewer than 3 good bins left after filtering");
    TP_TRY(tp_compact(ctx, keep.data(), (int)keep.size()));
    return call_from_compacted(ctx, max_pcs, min_clusters, k_out, n_pcs_out, n_clusters_out, maxlev_out, seqdist_out);
}

extern "C" int tp_call_arm(tp_ctx *ctx, const int *keep, int nf, int max_pcs, int min_clusters,
                           int *k_out, int *n_pcs_out, int *n_clusters_out,
                           int *maxlev_out, double *seqdist_out) {
    TP_ARG(ctx && keep, "tp_call_arm: null argument");
    if (tp_group_dispatch(ctx))
        return tp_group_run(ctx, [&](tp_ctx *gc, int gr) -> int {
            return gr ? tp_call_arm(gc, keep, nf, max_pcs, min_clusters, nullptr, nullptr, nullptr, nullptr, nullptr)
                      : tp_call_arm(gc, keep, nf, max_pcs, min_clusters, k_out, n_pcs_out, n_clusters_out, maxlev_out, seqdist_out);
        });
    TP_CUDA(cudaSetDevice(ctx->device));
    TP_MARK(ctx, EV_TOTAL0);
    TP_TRY(tp_compact(ctx, keep, nf));
    return call_from_compacted(ctx, max_pcs, min_clusters, k_out, n_pcs_out, n_clusters_out, maxlev_out, seqdist_out);
}

// ---- result assembly (host integer logic) ------------------------------------------------------------
extern "C" int tp_assemble(const double *seqdist, int nf, int n_clusters, const int *names, const int *bad,
                           int nbad, int *start_out, int *end_out, int *nrows_out, int *labels_out) {
    TP_ARG(seqdist && names && start_out && end_out && nrows_out, "tp_assemble: null argument");
    TP_ARG(nf >= 2 && n_clusters >= 1 && n_clusters <= nf, "tp_assemble: bad sizes");
    const int n1 = nf - 1;
    // stats::cutree(k): undo the k-1 merges that come last in rioja's .find.groups order
    // (ascending value, first index on ties)
    std::vector<int> idx(n1);
    std::iota(idx.begin(), idx.end(), 0);
    const int kb = n_clusters - 1;
    if (kb > 0)
        std::partial_sort(idx.begin(), idx.begin() + kb, idx.end(), [&](int a, int b) {
            return seqdist[a] > seqdist[b] || (seqdist[a] == seqdist[b] && a > b);
        });
    std::vector<char> cut(n1, 0);
    for (int i = 0; i < kb; i++) cut[idx[i]] = 1;
    std::vector<int> good(nf);
    int lab = 1;
    for (int i = 0; i < nf; i++) {
        good[i] = lab;
        if (i < n1 && cut[i]) lab++;
    }
    std::vector<int> fixed;
    if (nbad >= 0) {
        // c(good, bad) ordered by as.numeric(names) (stable): merge two sorted lists, good first on ties
        TP_ARG(nbad == 0 || bad, "tp_assemble: null bad list");
        fixed.reserve((size_t)nf + nbad);
        int i = 0, j = 0;
        while (i < nf || j < nbad) {
            if (j >= nbad || (i < nf && names[i] <= bad[j])) fixed.push_back(good[i++]);
            else { fixed.push_back(0); j++; }
        }
        // fix_values on the run values, left to right
        std::vector<int> vals, lens;
        for (size_t p = 0; p < fixed.size(); p++) {
            if (p == 0 || fixed[p] != fixed[p - 1]) { vals.push_back(fixed[p]); lens.push_back(1); }
            else lens.back()++;
        }
        for (size_t r = 1; r + 1 < vals.size(); r++)
            if (vals[r] == 0 && vals[r - 1] == vals[r + 1]) vals[r] = vals[r - 1];
        size_t p = 0;
        for (size_t r = 0; r < vals.size(); r++) for (int t = 0; t < lens[r]; t++) fixed[p++] = vals[r];
    } else {
        fixed = good;
    }
    if (labels_out) memcpy(labels_out, fixed.data(), fixed.size() * sizeof(int));
    // rle again -> start / end of the non-zero runs (1-based, inclusive)
    int rows = 0;
    size_t p = 0;
    while (p < fixed.size()) {
        size_t q = p;
        while (q + 1 < fixed.size() && fixed[q + 1] == fixed[p]) q++;
        if (fixed[p] != 0 || nbad < 0) {
            start_out[rows] = (int)p + 1;
            end_out[rows] = (int)q + 1;
            rows++;
        }
        p = q + 1;
    }
    *nrows_out = rows;
    return TP_OK;
}

// All requested levels of one dendrogram at once: the boundaries are ranked once (rioja's .find.groups order), and
// every level re-uses the ranking; same tables as nlev calls of tp_assemble.  levels[nlev] = numbers of clusters;
// offsets_out[nlev + 1] delimits each level's rows in start_out / end_out, which need room for
// sum(levels[i] + max(nbad, 0) + 1) rows.
extern "C" int tp_assemble_levels(const double *seqdist, int nf, const int *levels, int nlev, const int *names,
                                  const int *bad, int nbad, int *start_out, int *end_out, int *offsets_out) {
    TP_ARG(seqdist && levels && names && start_out && end_out && offsets_out && nlev >= 0, "tp_assemble_levels: null argument");
    TP_ARG(nf >= 2, "tp_assemble_levels: bad sizes");
    TP_ARG(nbad <= 0 || bad, "tp_assemble_levels: null bad list");
    const int n1 = nf - 1;
    int kmax = 1;
    for (int l = 0; l < nlev; l++) {
        TP_ARG(levels[l] >= 1 && levels[l] <= nf, "tp_assemble_levels: level out of range");
        kmax = std::max(kmax, levels[l]);
    }
    // idx[0 .. kmax-2] = the boundaries in (seqdist descending, index descending) order: level k cuts the first k - 1 of them
    std::vector<int> idx(n1);
    std::iota(idx.begin(), idx.end(), 0);
    std::partial_sort(idx.begin(), idx.begin() + (kmax - 1), idx.end(), [&](int a, int b) {
        return seqdist[a] > seqdist[b] || (seqdist[a] == seqdist[b] && a > b);
    });
    // positions of the good bins and of the bad bins in the merged order (good first on equal names), once
    const int nb = nbad > 0 ? nbad : 0;
    const int total = nbad >= 0 ? nf + nb : nf;
    std::vector<int> src(total);          // >= 0: index of the good bin, -1: bad bin
    if (nbad >= 0) {
        int i = 0, j = 0, p = 0;
        while (i < nf || j < nb) {
            if (j >= nb || (i < nf && names[i] <= bad[j])) src[p++] = i++;
            else { src[p++] = -1; j++; }
        }
    } else {
        std::iota(src.begin(), src.end(), 0);
    }
    // Labels are non-decreasing along the good bins, so in the merged order a cluster's bins are interleaved only with
    // zeros: fix_values (R/TADpole.R:503-510) absorbs the zero runs INSIDE a cluster (flanked by the same label) and leaves
    // those between two clusters and at the ends, which the rle loop then drops.  A level's table is therefore one row
    // per cluster, from the merged position of its first good bin to that of its last -- one pass over the boundaries
    // instead of materialising the label vector, its run-length encoding and the fixed vector per level.
    std::vector<int> pos(nf);
    for (int p = 0; p < total; p++) if (src[p] >= 0) pos[src[p]] = p;
    // A level of kc clusters has exactly kc rows, so every level's slot is known; the levels are visited in ascending order
    // of kc with the cut boundaries kept sorted by position (one insertion per added cut), which makes a level O(kc)
    // instead of a pass over all bins.
    offsets_out[0] = 0;
    for (int l = 0; l < nlev; l++) offsets_out[l + 1] = offsets_out[l] + levels[l];
    std::vector<int> ord(nlev);
    std::iota(ord.begin(), ord.end(), 0);
    std::stable_sort(ord.begin(), ord.end(), [&](int a, int b) { return levels[a] < levels[b]; });
    std::vector<int> cuts;
    cuts.reserve((size_t)kmax);
    int have = 0;                                   // boundaries of idx[] already in cuts
    for (int o = 0; o < nlev; o++) {
        const int l = ord[o], kc = levels[l];
        for (; have < kc - 1; have++) cuts.insert(std::upper_bound(cuts.begin(), cuts.end(), idx[have]), idx[have]);
        int rows = offsets_out[l], g0 = 0;
        for (int c = 0; c < kc - 1; c++) {            // a cut after good bin cuts[c]
            start_out[rows] = pos[g0] + 1; end_out[rows] = pos[cuts[c]] + 1; rows++;
            g0 = cuts[c] + 1;
        }
        start_out[rows] = pos[g0] + 1; end_out[rows] = pos[n1] + 1;
    }
    return TP_OK;
}
