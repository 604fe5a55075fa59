// group.cu -- what one single-threaded host session (R's .Call) needs to use a whole 8-GPU box:
//
//   * multi-device contexts (tp_ctx_create_multi): ONE process, one library-owned host thread per GPU.  The reference's
//     TADpole() is one call from one R session that spreads over every core (registerDoParallel(detectCores()) + foreach
//     %dopar%, R/TADpole.R:103-104); here the same one call spreads over every GPU handed to the context.  The member
//     contexts are the "ranks" of comm.cu (communicators from ncclCommInitAll), so a grouped call runs exactly the code a
//     torchrun job runs with one process per GPU -- same kernels, same collectives, same bits.
//   * chromosome arms on disjoint halves of the devices at the same time (tp_call_arms, R/TADpole.R:357-374).
//   * batches of independent calls kept in flight by library-owned threads (tp_call_batch): genome-wide use loops over
//     chromosomes, and one 2000-bin call leaves most of a B200 idle.  With centromere_search (the `centromere` argument
//     of tp_call_batch and tp_call_genome) each worker splits its matrix at the centromere and runs both arms one after
//     the other.
//   * small host-side pieces the R wrapper would otherwise do in interpreted loops: the hclust merge matrix of a
//     chclust dendrogram (rioja's .find.groups rule) in O(n log n), and load_mat's centromere split (tp_centromere_split).
//
// The R API never sees threads: every entry point returns when all member devices are done, worker threads never touch
// R (SURVEY.md 8b, "Threading").
#include "common.cuh"
#include <algorithm>
#include <atomic>
#include <condition_variable>
#include <mutex>
#include <numeric>
#include <thread>

static thread_local bool tl_in_group = false;

struct TpGroup {
    std::vector<tp_ctx *> members;
    std::vector<std::thread> threads;
    std::mutex mu, call_mu;
    std::condition_variable cv_job, cv_done;
    const std::function<int(tp_ctx *, int)> *job = nullptr;
    unsigned long long epoch = 0;
    int pending = 0;
    bool quit = false;
    std::vector<int> rc;
    std::vector<std::string> err;
};

struct TpPool {
    std::vector<int> devices;
    std::vector<std::vector<tp_ctx *>> ctxs;     // per device, grown on demand
};

static void group_worker(TpGroup *g, int rank) {
    tl_in_group = true;
    cudaSetDevice(g->members[rank]->device);
    unsigned long long seen = 0;
    for (;;) {
        const std::function<int(tp_ctx *, int)> *job;
        {
            std::unique_lock<std::mutex> lk(g->mu);
            g->cv_job.wait(lk, [&] { return g->quit || g->epoch != seen; });
            if (g->quit) return;
            seen = g->epoch;
            job = g->job;
        }
        const int rc = (*job)(g->members[rank], rank);
        std::string e = rc != TP_OK ? tp_last_error() : "";
        {
            std::lock_guard<std::mutex> lk(g->mu);
            g->rc[rank] = rc;
            g->err[rank] = e;
            if (--g->pending == 0) g->cv_done.notify_all();
        }
    }
}

bool tp_group_dispatch(const tp_ctx *ctx) { return ctx && ctx->group && !tl_in_group; }
int tp_group_size(const tp_ctx *ctx) { return ctx && ctx->group ? (int)ctx->group->members.size() : 1; }
tp_ctx *tp_group_member(const tp_ctx *ctx, int rank) {
    if (!ctx->group) return rank == 0 ? const_cast<tp_ctx *>(ctx) : nullptr;
    return rank >= 0 && rank < (int)ctx->group->members.size() ? ctx->group->members[rank] : nullptr;
}

int tp_group_run(tp_ctx *ctx, const std::function<int(tp_ctx *, int)> &fn) {
    TpGroup *g = ctx->group;
    if (!g) return fn(ctx, 0);
    std::lock_guard<std::mutex> call(g->call_mu);
    const int n = (int)g->members.size();
    {
        std::lock_guard<std::mutex> lk(g->mu);
        g->job = &fn;
        g->epoch++;
        g->pending = n - 1;
        std::fill(g->rc.begin(), g->rc.end(), (int)TP_OK);
    }
    g->cv_job.notify_all();
    const bool was = tl_in_group;
    tl_in_group = true;
    const int rc0 = fn(g->members[0], 0);
    const std::string e0 = rc0 != TP_OK ? tp_last_error() : "";
    tl_in_group = was;
    {
        std::unique_lock<std::mutex> lk(g->mu);
        g->cv_done.wait(lk, [&] { return g->pending == 0; });
    }
    cudaSetDevice(g->members[0]->device);
    if (rc0 != TP_OK) { tp_set_error("%s", e0.c_str()); return rc0; }
    for (int r = 1; r < n; r++)
        if (g->rc[r] != TP_OK) { tp_set_error("device %d (rank %d): %s", g->members[r]->device, r, g->err[r].c_str()); return g->rc[r]; }
    return TP_OK;
}

void tp_group_destroy(tp_ctx *leader) {
    TpGroup *g = leader->group;
    if (!g) return;
    {
        std::lock_guard<std::mutex> lk(g->mu);
        g->quit = true;
    }
    g->cv_job.notify_all();
    for (std::thread &t : g->threads) t.join();
    for (tp_ctx *m : g->members) m->group = nullptr;
    for (size_t r = 1; r < g->members.size(); r++) tp_ctx_destroy(g->members[r]);
    delete g;
}

void tp_pool_destroy(tp_ctx *ctx) {
    if (!ctx->pool) return;
    for (auto &v : ctx->pool->ctxs) for (tp_ctx *c : v) tp_ctx_destroy(c);
    delete ctx->pool;
    ctx->pool = nullptr;
}

extern "C" int tp_ctx_create_multi(const int *devices, int ndev, tp_ctx **out) {
    TP_ARG(devices && out && ndev >= 1, "tp_ctx_create_multi: bad arguments");
    for (int i = 0; i < ndev; i++)
        for (int j = 0; j < i; j++) TP_ARG(devices[i] != devices[j], "tp_ctx_create_multi: a device is listed twice");
    std::vector<tp_ctx *> members;
    auto fail = [&](int rc) {
        const std::string e = tp_last_error();
        for (tp_ctx *m : members) { m->group = nullptr; tp_ctx_destroy(m); }
        tp_set_error("%s", e.c_str());
        return rc;
    };
    for (int i = 0; i < ndev; i++) {
        tp_ctx *c = nullptr;
        const int rc = tp_ctx_create(devices[i], &c);
        if (rc != TP_OK) return fail(rc);
        members.push_back(c);
    }
    if (ndev == 1) { *out = members[0]; return TP_OK; }
    // slot 0: all devices (one call spread over the box); slot 1: the half of the devices that shares a chromosome arm
    int rc = tp_comm_init_all(members.data(), ndev, 0);
    if (rc != TP_OK) return fail(rc);
    const int half = ndev / 2;
    if (half >= 2) { rc = tp_comm_init_all(members.data(), half, 1); if (rc != TP_OK) return fail(rc); }
    if (ndev - half >= 2) { rc = tp_comm_init_all(members.data() + half, ndev - half, 1); if (rc != TP_OK) return fail(rc); }
    TpGroup *g = new TpGroup();
    g->members = members;
    g->rc.assign(ndev, TP_OK);
    g->err.assign(ndev, "");
    for (int i = 0; i < ndev; i++) {
        members[i]->group = g;
        members[i]->group_rank = i;
        members[i]->comm_cur = 0;
    }
    for (int i = 1; i < ndev; i++) g->threads.emplace_back(group_worker, g, i);
    cudaSetDevice(members[0]->device);
    *out = members[0];
    return TP_OK;
}

extern "C" int tp_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) { (void)cudaGetLastError(); return 0; }
    return n;
}

extern "C" int tp_ctx_devices(tp_ctx *ctx, int *devices_out, int cap) {
    TP_ARG(ctx, "tp_ctx_devices: null context");
    const int n = tp_group_size(ctx);
    for (int i = 0; i < n && i < cap && devices_out; i++) devices_out[i] = tp_group_member(ctx, i)->device;
    return n;
}

extern "C" long long tp_ctx_generation(tp_ctx *ctx) { return ctx ? ctx->generation : -1; }

extern "C" int tp_ctx_dims(tp_ctx *ctx, int *n_out, int *nf_out, int *k_out, int *k_full_out, int *maxlev_out) {
    TP_ARG(ctx, "tp_ctx_dims: null context");
    if (n_out) *n_out = ctx->n;
    if (nf_out) *nf_out = ctx->have_X || ctx->have_C || ctx->have_scores ? ctx->nf : 0;
    if (k_out) *k_out = ctx->have_scores ? ctx->k : 0;
    if (k_full_out) *k_full_out = ctx->have_scores ? ctx->k_full : 0;
    if (maxlev_out) *maxlev_out = ctx->have_sweep ? ctx->last_maxlev : 0;
    return TP_OK;
}

// ---- rioja's .find.groups: the hclust merge matrix of a chclust dendrogram ------------------------------------------------
// n1 - 1... for step s = 1..n1: j = which.min(x) (first index on ties); the operands are -(j) / -(j+1) (1-based objects)
// while they are singletons, else the step that last absorbed them.  merge_out: n1 x 2 column-major (R matrix).
extern "C" int tp_find_groups(const double *seqdist, int n1, int *merge_out) {
    TP_ARG(seqdist && merge_out && n1 >= 1, "tp_find_groups: bad arguments");
    std::vector<int> idx(n1), parent(n1 + 1), owner(n1 + 1, 0);
    std::iota(idx.begin(), idx.end(), 0);
    std::iota(parent.begin(), parent.end(), 0);
    std::stable_sort(idx.begin(), idx.end(), [&](int a, int b) { return seqdist[a] < seqdist[b]; });
    auto root = [&](int a) {
        while (parent[a] != a) { parent[a] = parent[parent[a]]; a = parent[a]; }
        return a;
    };
    for (int s = 0; s < n1; s++) {
        const int j = idx[s];
        const int ra = root(j), rb = root(j + 1);
        merge_out[s] = owner[ra] ? owner[ra] : -(j + 1);
        merge_out[s + n1] = owner[rb] ? owner[rb] : -(j + 2);
        parent[rb] = ra;
        owner[ra] = s + 1;
    }
    return TP_OK;
}

// ---- load_mat's centromere split (R/TADpole.R:58-86) on the bad flags ------------------------------------------------
// runs <- split(idx, cumsum(c(1, diff(idx) != 1))); the longest run (which.max: the first one on ties) is the centromere
// cs..ce; no split when it touches either end.  keep_p / keep_q: 0-based original bins of each arm; bad_p / bad_q: the
// arm's bad columns as original 1-based bins, *nbad = -1 when there is none (attr NULL).  The reference drops the q arm's
// rows by the ORIGINAL index of its bad columns used as a position in the arm, ignoring those past the arm's end (quirk
// Q3); fix = 1 drops the bad columns themselves.
extern "C" int tp_centromere_split(const uint8_t *bad, int n, int fix, int *split_out, int *cs_out, int *ce_out, int *keep_p,
                                   int *nkeep_p, int *bad_p, int *nbad_p, int *keep_q, int *nkeep_q, int *bad_q, int *nbad_q) {
    TP_ARG(bad && n >= 0 && split_out && cs_out && ce_out && keep_p && nkeep_p && bad_p && nbad_p && keep_q && nkeep_q && bad_q &&
           nbad_q, "tp_centromere_split: null argument");
    *split_out = *cs_out = *ce_out = *nkeep_p = *nkeep_q = 0;
    *nbad_p = *nbad_q = -1;
    int cs = 0, ce = 0;
    for (int i = 0; i < n;) {
        if (!bad[i]) { i++; continue; }
        int j = i;
        while (j + 1 < n && bad[j + 1]) j++;
        if (cs == 0 || j - i > ce - cs) { cs = i + 1; ce = j + 1; }
        i = j + 1;
    }
    *cs_out = cs;
    *ce_out = ce;
    if (cs == 0 || cs == 1 || ce == n) return TP_OK;
    const int nq = n - ce;
    std::vector<uint8_t> drop_q((size_t)nq, 0);
    int np = 0, bp = 0, bq = 0;
    for (int i = 0; i < cs - 1; i++) {
        if (bad[i]) bad_p[bp++] = i + 1;
        else keep_p[np++] = i;
    }
    for (int i = ce; i < n; i++)
        if (bad[i]) {
            bad_q[bq++] = i + 1;
            const int pos = fix ? i - ce : i;              // 0-based position in the arm of the row that is dropped
            if (pos < nq) drop_q[(size_t)pos] = 1;
        }
    int nk = 0;
    for (int t = 0; t < nq; t++) if (!drop_q[(size_t)t]) keep_q[nk++] = ce + t;
    *split_out = 1;
    *nkeep_p = np;
    *nkeep_q = nk;
    *nbad_p = bp ? bp : -1;
    *nbad_q = bq ? bq : -1;
    return TP_OK;
}

// ---- batches of independent calls ----------------------------------------------------------------------------------------
struct TpBatchItem {
    int rc = TP_OK;
    std::string err;
    int n = 0, nf = 0, k = 0, n_pcs = 0, n_clusters = 0, maxlev = 0;
    std::vector<uint8_t> bad;
    std::vector<double> scores, seqdist;          // scores: k x maxlev row-major, NaN padded
    std::vector<int> levels, offsets, start, end; // per-level start / end tables (R/TADpole.R:470-497)
    double device_ms = 0.0;
    long long launches = 0;
    // centromere_search items (centromere != 0): split = -1 until the bad flags are known, then
    // 0 (processed whole or failed) or 1 (arms[0] = p, arms[1] = q); cs..ce = the longest bad run (1-based, 0 = none)
    int split = -1, cs = 0, ce = 0;
    std::vector<TpBatchItem> arms;
    // an arm: its 0-based original bins, its bad columns (original 1-based; nbad = -1: attr NULL) and the fixed label
    // vector of its optimal level, bad columns re-inserted (R/TADpole.R:411-431)
    std::vector<int> keep, badcols, labels;
    int nbad = -1;
};
struct tp_batch { std::vector<TpBatchItem> items; double device_ms = 0.0; };

// The outputs of a call that has just finished on c, into its batch item: k, maxlev and the score matrix from the context
// (the host copy the sweep made) and the call's device time.  n_pcs, n_clusters, nf and seqdist the call wrote there itself.
static void finish_item(tp_ctx *c, TpBatchItem &it) {
    it.k = c->k;
    it.maxlev = c->last_maxlev;
    it.scores = c->sweep_scores;
    it.seqdist.resize((size_t)it.nf - 1);
    double tm[10];
    if (tp_ctx_timings(c, tm) == TP_OK) it.device_ms = tm[6];
}

// for (k in which(!is.na(scores[n_PCs, ]))) ... the start / end table of every scored level of the optimal candidate of a
// finished item (R/TADpole.R:381-408, 470-497).  names[nf]: original 1-based bin of each kept row; bad[nbad]: the bad
// columns (nbad < 0: attr NULL).
static int level_tables(TpBatchItem &it, const int *names, const int *bad, int nbad) {
    const double *row = it.scores.data() + (size_t)(it.n_pcs - 1) * it.maxlev;
    size_t cap = 0;
    for (int l = 0; l < it.maxlev; l++)
        if (row[l] == row[l]) { it.levels.push_back(l + 1); cap += (size_t)(l + 1) + (size_t)std::max(nbad, 0) + 1; }
    it.offsets.assign(it.levels.size() + 1, 0);
    it.start.assign(cap + 1, 0);
    it.end.assign(cap + 1, 0);
    TP_TRY(tp_assemble_levels(it.seqdist.data(), it.nf, it.levels.data(), (int)it.levels.size(), names, bad, nbad,
                              it.start.data(), it.end.data(), it.offsets.data()));
    it.start.resize((size_t)it.offsets.back());
    it.end.resize((size_t)it.offsets.back());
    return TP_OK;
}

// The result tail of a matrix called whole: finish_item, then (tables) the start / end table of every scored level, with
// the names and bad columns TADpole() packs from the bad flags.
static int finish_whole(tp_ctx *c, TpBatchItem &it, bool tables) {
    finish_item(c, it);
    if (!tables) return TP_OK;
    std::vector<int> names, bad;
    for (int i = 0; i < it.n; i++) (it.bad[(size_t)i] ? bad : names).push_back(i + 1);
    return level_tables(it, names.data(), bad.data(), (int)bad.size());
}

// one chromosome arm on c, after tp_filter: the arm's call (tp_call_arm on its keep list), its tables and its fixed labels
static int arm_one(tp_ctx *c, int max_pcs, int min_clusters, TpBatchItem &a) {
    a.nf = (int)a.keep.size();
    a.seqdist.assign((size_t)(a.nf > 1 ? a.nf - 1 : 1), 0.0);
    TP_TRY(tp_call_arm(c, a.keep.data(), a.nf, max_pcs, min_clusters, nullptr, &a.n_pcs, &a.n_clusters, nullptr,
                       a.seqdist.data()));
    finish_item(c, a);
    std::vector<int> names(a.keep.size());
    for (size_t t = 0; t < names.size(); t++) names[t] = a.keep[t] + 1;
    TP_TRY(level_tables(a, names.data(), a.badcols.data(), a.nbad));
    // the optimal level with the bad columns re-inserted and fix_values applied, for merging_arms
    const int nb = std::max(a.nbad, 0);
    std::vector<int> st((size_t)a.n_clusters + nb + 2), en(st.size());
    int rows = 0;
    a.labels.assign((size_t)a.nf + nb, 0);
    return tp_assemble(a.seqdist.data(), a.nf, a.n_clusters, names.data(), a.badcols.data(), nb, st.data(), en.data(), &rows,
                       a.labels.data());
}

static const char *const NOSPLIT_MSG = "centromere_search=TRUE but load_mat did not split the matrix (no bad columns, or the "
                                       "longest bad stretch touches an end); the reference errors here";

// What every item of a batch call is run with.  centromere: 0 = TADpole(), 1 = centromere_search, 2 = centromere_search
// with centromere_fix.
struct ItemArgs {
    int max_pcs, min_clusters;
    double bad_frac;
    int want_tables, centromere;
};

// One matrix of a batch on c.  centromere = 0: tp_call, then its outputs and (want_tables) its tables.  Otherwise
// TADpole(centromere_search = TRUE) on one matrix (R/TADpole.R:351-442): filter, split at the longest bad stretch, then
// the p arm and the q arm one after the other on c, tables always built.  Unsplit: TP_ERR_NOSPLIT (the reference errors,
// quirk Q4), or with centromere_fix the whole matrix's good bins as TADpole(centromere_fix = TRUE) does.  device_ms of
// a centromere_search item covers the filter and both arms.
static int item_one(tp_ctx *c, const double *mat, int n, int colmajor, int on_device, const ItemArgs &a, TpBatchItem &it) {
    it.n = n;
    const long long launches0 = c->launches;
    struct Count { TpBatchItem &it; tp_ctx *c; long long l0; ~Count() { it.launches = c->launches - l0; } } count{it, c, launches0};
    it.bad.assign((size_t)n, 0);
    TP_ARG(a.max_pcs >= 1, "tp_call_batch: max_pcs must be positive");
    if (!a.centromere) {
        it.seqdist.assign((size_t)(n > 1 ? n - 1 : 1), 0.0);
        TP_TRY(tp_call(c, mat, n, colmajor, on_device, a.max_pcs, a.min_clusters, a.bad_frac, it.bad.data(), &it.nf, nullptr,
                       &it.n_pcs, &it.n_clusters, nullptr, it.seqdist.data()));
        return finish_whole(c, it, a.want_tables);
    }
    struct Events {
        cudaEvent_t e[2] = {nullptr, nullptr};
        ~Events() { for (cudaEvent_t x : e) if (x) cudaEventDestroy(x); }
    } ev;
    TP_CUDA(cudaSetDevice(c->device));
    TP_CUDA(cudaEventCreate(&ev.e[0]));
    TP_CUDA(cudaEventCreate(&ev.e[1]));
    TP_CUDA(cudaEventRecord(ev.e[0], c->stream));
    // tp_call calls the hook itself; here the worker runs tp_filter directly, and the hook releases the first-upload lock
    const int frc = tp_filter(c, mat, n, colmajor, on_device, a.bad_frac, it.bad.data(), nullptr, nullptr);
    if (c->after_filter) c->after_filter();
    TP_TRY(frc);
    std::vector<int> kp((size_t)n), bp((size_t)n), kq((size_t)n), bq((size_t)n);
    int split = 0, nkp = 0, nbp = 0, nkq = 0, nbq = 0;
    TP_TRY(tp_centromere_split(it.bad.data(), n, a.centromere == 2, &split, &it.cs, &it.ce, kp.data(), &nkp, bp.data(), &nbp,
                               kq.data(), &nkq, bq.data(), &nbq));
    it.split = split;
    if (split) {
        // The p arm's after_pca hook may stage the next matrix while the q arm still has to compact from this one.  The
        // staged upload (tp_stage_input) writes raw_next only, on the copy stream; the matrix the arms read is c->raw, which
        // tp_filter pointed at raw_own (after swapping in the previous staged upload), at the caller's device matrix or at
        // the genome worker's dense build in raw_own.  raw_own changes hands only in the next tp_filter, so the q arm reads
        // what the p arm read.
        it.arms.resize(2);
        it.arms[0].keep.assign(kp.begin(), kp.begin() + nkp);
        it.arms[1].keep.assign(kq.begin(), kq.begin() + nkq);
        it.arms[0].nbad = nbp;
        it.arms[1].nbad = nbq;
        if (nbp > 0) it.arms[0].badcols.assign(bp.begin(), bp.begin() + nbp);
        if (nbq > 0) it.arms[1].badcols.assign(bq.begin(), bq.begin() + nbq);
        for (TpBatchItem &arm : it.arms) TP_TRY(arm_one(c, a.max_pcs, a.min_clusters, arm));
    } else {
        if (a.centromere != 2) { tp_set_error("%s", NOSPLIT_MSG); return TP_ERR_NOSPLIT; }
        std::vector<int> keep;
        for (int i = 0; i < n; i++) if (!it.bad[(size_t)i]) keep.push_back(i);
        it.nf = (int)keep.size();
        it.seqdist.assign((size_t)(it.nf > 1 ? it.nf - 1 : 1), 0.0);
        TP_TRY(tp_call_arm(c, keep.data(), it.nf, a.max_pcs, a.min_clusters, nullptr, &it.n_pcs, &it.n_clusters, nullptr,
                           it.seqdist.data()));
        TP_TRY(finish_whole(c, it, true));
    }
    TP_CUDA(cudaEventRecord(ev.e[1], c->stream));
    TP_CUDA(cudaEventSynchronize(ev.e[1]));
    float ms = 0.f;
    TP_CUDA(cudaEventElapsedTime(&ms, ev.e[0], ev.e[1]));
    it.device_ms = ms;
    return TP_OK;
}

// ---- chromosome arms on disjoint halves of the devices (R/TADpole.R:357-374: the arms are independent) --------------
extern "C" int tp_call_arms(tp_ctx *ctx, const int *keep_p, int nf_p, const int *keep_q, int nf_q, int max_pcs, int min_clusters,
                            tp_batch **out) {
    TP_ARG(ctx && keep_p && keep_q && out, "tp_call_arms: null argument");
    const int *keep[2] = {keep_p, keep_q};
    tp_batch *b = new tp_batch();
    b->items.resize(2);
    b->items[0].nf = nf_p;
    b->items[1].nf = nf_q;
    // arm a on context c; only the lead context of the arm reports its outputs
    auto arm = [&](tp_ctx *c, int a, bool lead) -> int {
        TpBatchItem &it = b->items[(size_t)a];
        if (lead) it.seqdist.assign((size_t)(it.nf > 1 ? it.nf - 1 : 1), 0.0);
        TP_TRY(tp_call_arm(c, keep[a], it.nf, max_pcs, min_clusters, nullptr, lead ? &it.n_pcs : nullptr,
                           lead ? &it.n_clusters : nullptr, nullptr, lead ? it.seqdist.data() : nullptr));
        if (lead) finish_item(c, it);
        return TP_OK;
    };
    int rc = TP_OK;
    const int R = tp_group_dispatch(ctx) ? tp_group_size(ctx) : 1;
    if (R >= 2) {
        const int half = R / 2;
        rc = tp_group_run(ctx, [&](tp_ctx *c, int r) -> int {
            const int a = r < half ? 0 : 1;
            const int prev = c->comm_cur;
            c->comm_cur = c->comm[1].handle ? 1 : -1;
            const int e = arm(c, a, r == (a ? half : 0));
            c->comm_cur = prev;
            return e;
        });
    } else {
        for (int a = 0; a < 2 && rc == TP_OK; a++) rc = arm(ctx, a, true);
    }
    if (rc != TP_OK) { delete b; return rc; }
    *out = b;
    return TP_OK;
}

// The worker loop of a batch: up to `inflight` library-owned threads per device of the context, each on its own pool
// context, claim items (in the order order[0..ncalls), or in input order when order is NULL) until none is left.
// one(c, i, it) runs item i on context c.  need: device bytes one call in flight holds.  host_inputs: the items' matrices
// come from host memory; then the first uploads of a device's workers go one after the other, and stage(c, i) starts the
// upload of item i (claimed ahead) under the call that c is running.
static int batch_run(tp_ctx *ctx, int ncalls, double need, int inflight, bool host_inputs, const int *order,
                     const std::function<void(tp_ctx *, int)> &stage, const std::function<int(tp_ctx *, int, TpBatchItem &)> &one,
                     tp_batch **out) {
    if (inflight < 1) inflight = 4;
    if (inflight > 32) inflight = 32;
    const int ndev = tp_group_size(ctx);
    if (!ctx->pool) {
        ctx->pool = new TpPool();
        for (int d = 0; d < ndev; d++) ctx->pool->devices.push_back(tp_group_member(ctx, d)->device);
        ctx->pool->ctxs.resize(ndev);
    }
    TpPool *pool = ctx->pool;
    int per_dev = std::max(1, std::min(inflight, (ncalls + ndev - 1) / ndev));
    {   // do not keep more calls in flight than the device has room for
        for (int d = 0; d < ndev; d++) {
            size_t fr = 0, tot = 0;
            cudaSetDevice(pool->devices[d]);
            if (cudaMemGetInfo(&fr, &tot) != cudaSuccess) { (void)cudaGetLastError(); continue; }
            // memory the pool's contexts on this device already hold counts as available to them
            double have = 0.8 * (double)fr;
            for (tp_ctx *c : pool->ctxs[d])
                for (const DevBuf *bf : {&c->raw_own, &c->raw_next, &c->X, &c->C, &c->M, &c->ioA, &c->ioB, &c->islices, &c->Y0, &c->Y1, &c->Y2, &c->W})
                    have += (double)bf->cap;
            per_dev = std::max(1, std::min(per_dev, (int)(have / need)));
        }
        cudaSetDevice(ctx->device);
    }
    const unsigned hw = std::thread::hardware_concurrency();
    // a waiting host thread spins on a core in cudaStreamSynchronize; with more threads than spare cores they sleep instead
    const bool blocking = hw > 0 && (unsigned)(per_dev * ndev) > hw / 2;
    for (int d = 0; d < ndev; d++)
        while ((int)pool->ctxs[d].size() < per_dev) {
            tp_ctx *c = nullptr;
            TP_TRY(tp_ctx_create(pool->devices[d], &c));
            // the tunables of the handle carry over to the pool
            c->pca_block = ctx->pca_block; c->pca_tol = ctx->pca_tol; c->pca_maxit = ctx->pca_maxit; c->pca_inner = ctx->pca_inner;
            c->jacobi_direct_max = ctx->jacobi_direct_max; c->level_cap = ctx->level_cap; c->igemm_min_n = ctx->igemm_min_n;
            c->iop_min_n = ctx->iop_min_n; c->mgram_min_n = ctx->mgram_min_n; c->iop_final = ctx->iop_final;
            c->iop_final_min_n = ctx->iop_final_min_n; c->iop_switch = ctx->iop_switch;
            pool->ctxs[d].push_back(c);
        }
    for (int d = 0; d < ndev; d++)
        for (tp_ctx *c : pool->ctxs[d]) {
            c->sync_blocking = blocking || ctx->sync_blocking;
            // 32-column tiles of the sliced operator fill an otherwise idle GPU from ONE call (13.7 against 14.2 ms); with
            // several calls in flight the other calls fill it, and the wider tiles' better operand reuse wins
            // (297 against 280 calls/s at 2000 bins, 8 in flight)
            c->io_bn32 = per_dev > 1 ? 0 : ctx->io_bn32;
        }
    tp_batch *b = new tp_batch();
    b->items.resize((size_t)ncalls);
    // device time of the whole batch: one start event per device (its streams are idle: the previous batch was joined), one
    // end event per worker on its own stream after its last call; the batch took max(end - start) over the workers
    std::vector<cudaEvent_t> ev_start((size_t)ndev), ev_end((size_t)ndev * per_dev);
    for (int d = 0; d < ndev; d++) {
        cudaSetDevice(pool->devices[d]);
        cudaEventCreate(&ev_start[d]);
        for (int s2 = 0; s2 < per_dev; s2++) cudaEventCreate(&ev_end[(size_t)d * per_dev + s2]);
        cudaEventRecord(ev_start[d], pool->ctxs[d][0]->stream);
    }
    std::atomic<int> next(0);
    // Host matrices: (1) the first uploads of the workers of one device go one after the other (ticket order), so the
    // first call starts computing after ONE upload instead of after all of them sharing the PCIe link; (2) from then on a
    // worker claims its next matrix while the current call is in the n_pcs sweep and uploads it on its copy stream into the
    // second input buffer (tp_stage_input): the upload leaves the critical path of the call.
    const bool prefetch = host_inputs && !ctx->group && getenv("TADPOLE_BATCH_NOPREFETCH") == nullptr;
    std::vector<std::mutex> first_upload((size_t)ndev);
    auto worker = [&](tp_ctx *c, cudaEvent_t done, int d) {
        cudaSetDevice(c->device);
        int claimed = -1;
        bool holding = false;
        c->after_filter = [&]() { if (holding) { first_upload[(size_t)d].unlock(); holding = false; } };
        c->after_pca = [&]() {
            if (!prefetch || claimed >= 0) return;
            const int j = next.fetch_add(1);
            if (j >= ncalls) return;
            claimed = order ? order[j] : j;
            stage(c, claimed);
        };
        bool first = true;
        for (;;) {
            int i = claimed;
            claimed = -1;
            if (i < 0) {
                const int t = next.fetch_add(1);
                if (t >= ncalls) break;
                i = order ? order[t] : t;
            }
            if (first && host_inputs) { first_upload[(size_t)d].lock(); holding = true; }
            first = false;
            TpBatchItem &it = b->items[(size_t)i];
            it.rc = one(c, i, it);
            if (holding) { first_upload[(size_t)d].unlock(); holding = false; }
            if (it.rc != TP_OK) it.err = tp_last_error();
        }
        c->after_filter = nullptr;
        c->after_pca = nullptr;
        c->staged_mat = nullptr;
        cudaEventRecord(done, c->stream);
    };
    std::vector<std::thread> threads;
    for (int s2 = 0; s2 < per_dev; s2++)
        for (int d = 0; d < ndev; d++)
            if (!(s2 == 0 && d == 0)) threads.emplace_back(worker, pool->ctxs[d][s2], ev_end[(size_t)d * per_dev + s2], d);
    worker(pool->ctxs[0][0], ev_end[0], 0);
    for (std::thread &t : threads) t.join();
    for (int d = 0; d < ndev; d++) {
        cudaSetDevice(pool->devices[d]);
        for (int s2 = 0; s2 < per_dev; s2++) {
            cudaEvent_t e = ev_end[(size_t)d * per_dev + s2];
            float ms = 0.f;
            if (cudaEventSynchronize(e) == cudaSuccess && cudaEventElapsedTime(&ms, ev_start[d], e) == cudaSuccess)
                b->device_ms = std::max(b->device_ms, (double)ms);
            else (void)cudaGetLastError();
            cudaEventDestroy(e);
        }
        cudaEventDestroy(ev_start[d]);
    }
    cudaSetDevice(ctx->device);
    *out = b;
    return TP_OK;
}

extern "C" int tp_call_batch(tp_ctx *ctx, int ncalls, const double *const *mats, const int *n, int colmajor, int on_device,
                             int max_pcs, int min_clusters, double bad_frac, int inflight, int want_tables, int centromere,
                             tp_batch **out) {
    TP_ARG(ctx && mats && n && out && ncalls >= 0 && centromere >= 0 && centromere <= 2, "tp_call_batch: bad arguments");
    TP_ARG(!(on_device && ctx->group), "tp_call_batch: device-resident inputs need a single-device context");
    // every call in flight holds its own working set in HBM (raw + filtered + correlation + M + digit planes + second
    // input buffer + blocks: ~56 bytes per matrix element, 35 GB at 25k bins); an arm is smaller than its chromosome
    size_t nmax = 0;
    for (int i = 0; i < ncalls; i++) nmax = std::max(nmax, (size_t)(n[i] > 0 ? n[i] : 0));
    const double need = 56.0 * (double)nmax * (double)nmax + 64e6;
    auto stage = [&](tp_ctx *c, int j) {
        if (mats[j] && n[j] >= 2) (void)tp_stage_input(c, mats[j], n[j], colmajor);    // a failure leaves the normal upload
    };
    const ItemArgs args{max_pcs, min_clusters, bad_frac, want_tables, centromere};
    auto one = [&](tp_ctx *c, int i, TpBatchItem &it) -> int {
        return mats[i] ? item_one(c, mats[i], n[i], colmajor, on_device, args, it)
                       : (tp_set_error("tp_call_batch: matrix %d is null", i), (int)TP_ERR_ARG);
    };
    return batch_run(ctx, ncalls, need, inflight, !on_device, nullptr, stage, one, out);
}

// ---- genome-wide calls: one per chromosome, each dense matrix built from its bucket in HBM (ingest.cu, S0c) ---------
// The selected chromosomes (checked against the handle), claimed largest first; each worker runs one chromosome's dense
// matrix (device pointer, row-major) on its context.
extern "C" int tp_call_genome(tp_ctx *ctx, const tp_genome *g, const int *chroms, int nsel, int max_pcs, int min_clusters,
                              double bad_frac, int inflight, int want_tables, int centromere, tp_batch **out) {
    TP_ARG(ctx && g && out && nsel >= 0 && (chroms || nsel == 0 || nsel == (int)g->bins.size()) && centromere >= 0 &&
           centromere <= 2, "tp_call_genome: bad arguments");
    TP_ARG(g->device == ctx->device, "tp_call_genome: the handle was ingested on another device than the context's first");
    std::vector<int> sel((size_t)(nsel > 0 ? nsel : 0));
    for (int s = 0; s < nsel; s++) {
        sel[(size_t)s] = chroms ? chroms[s] : s;
        if (sel[(size_t)s] < 0 || sel[(size_t)s] >= (int)g->bins.size()) {
            tp_set_error("tp_call_genome: chromosome index %d is outside 0..%d", sel[(size_t)s], (int)g->bins.size() - 1);
            return TP_ERR_ARG;
        }
    }
    // the cost of a call grows roughly as n^3: the largest chromosomes are claimed first
    std::vector<int> order((size_t)nsel);
    std::iota(order.begin(), order.end(), 0);
    std::stable_sort(order.begin(), order.end(), [&](int a, int b) { return g->bins[(size_t)sel[a]] > g->bins[(size_t)sel[b]]; });
    // per call in flight: the working set of tp_call_batch plus the copy of a bucket held by another device.  The buckets
    // themselves are resident on devices[0] and already missing from its free memory.
    double nmax = 0.0, pmax = 0.0;
    for (int c : sel) {
        nmax = std::max(nmax, (double)g->bins[(size_t)c]);
        pmax = std::max(pmax, (double)(g->offs[(size_t)c + 1] - g->offs[(size_t)c]));
    }
    const double need = 56.0 * nmax * nmax + 16.0 * pmax + 64e6;
    const ItemArgs args{max_pcs, min_clusters, bad_frac, want_tables, centromere};
    auto one = [&](tp_ctx *c, int s, TpBatchItem &it) -> int {
        const int chrom = sel[(size_t)s], n = g->bins[(size_t)chrom];
        it.n = n;
        if (n < 2) {
            it.bad.assign((size_t)n, 0);
            tp_set_error("tp_call_genome: chromosome %d has %d bin; a call needs at least 2", chrom, n);
            return TP_ERR_ARG;
        }
        double *mat = nullptr;
        TP_TRY(tp_genome_dense(c, g, chrom, &mat));
        return item_one(c, mat, n, 0, 1, args, it);
    };
    return batch_run(ctx, nsel, need, inflight, false, order.data(), [](tp_ctx *, int) {}, one, out);
}

extern "C" double tp_batch_device_ms(const tp_batch *b) { return b ? b->device_ms : 0.0; }
extern "C" long long tp_batch_launches(const tp_batch *b) {
    long long s = 0;
    if (b) for (const TpBatchItem &it : b->items) s += it.launches;
    return s;
}
extern "C" int tp_batch_size(const tp_batch *b) { return b ? (int)b->items.size() : 0; }
extern "C" int tp_batch_status(const tp_batch *b, int i) {
    if (!b || i < 0 || i >= (int)b->items.size()) return TP_ERR_ARG;
    return b->items[(size_t)i].rc;
}
extern "C" const char *tp_batch_error(const tp_batch *b, int i) {
    if (!b || i < 0 || i >= (int)b->items.size()) return "tp_batch_error: index out of range";
    return b->items[(size_t)i].err.c_str();
}
// item i of a batch (part -1) or arm `part` (0 = p, 1 = q) of split item i; nullptr when there is no such item or arm
static const TpBatchItem *batch_part(const tp_batch *b, int i, int part) {
    if (!b || i < 0 || i >= (int)b->items.size() || part < -1 || part > 1) return nullptr;
    const TpBatchItem &it = b->items[(size_t)i];
    if (part < 0) return &it;
    return it.rc == TP_OK && it.split == 1 ? &it.arms[(size_t)part] : nullptr;
}
extern "C" int tp_batch_dims(const tp_batch *b, int i, int part, int *n_out, int *nf_out, int *k_out, int *maxlev_out,
                             int *nlevels_out, int *nrows_out, int *nkeep_out, int *nbad_out) {
    const TpBatchItem *it = batch_part(b, i, part);
    TP_ARG(it, part < 0 ? "tp_batch_dims: index out of range"
                          : "tp_batch_dims: no such arm (index out of range, or the item was not split)");
    if (n_out) *n_out = it->n;
    if (nf_out) *nf_out = it->nf;
    if (k_out) *k_out = it->k;
    if (maxlev_out) *maxlev_out = it->maxlev;
    if (nlevels_out) *nlevels_out = (int)it->levels.size();
    if (nrows_out) *nrows_out = (int)it->start.size();
    if (nkeep_out) *nkeep_out = (int)it->keep.size();
    if (nbad_out) *nbad_out = it->nbad;
    return TP_OK;
}
extern "C" int tp_batch_get(const tp_batch *b, int i, int part, uint8_t *bad_out, int *n_pcs_out, int *n_clusters_out,
                            double *scores_out, double *seqdist_out, int *levels_out, int *offsets_out, int *start_out,
                            int *end_out, double *device_ms_out, int *keep_out, int *badcols_out, int *labels_out) {
    const TpBatchItem *it = batch_part(b, i, part);
    TP_ARG(it, part < 0 ? "tp_batch_get: index out of range"
                          : "tp_batch_get: no such arm (index out of range, or the item was not split)");
    if (it->rc != TP_OK) { tp_set_error("%s", it->err.c_str()); return it->rc; }
    if (bad_out) memcpy(bad_out, it->bad.data(), it->bad.size());
    if (n_pcs_out) *n_pcs_out = it->n_pcs;
    if (n_clusters_out) *n_clusters_out = it->n_clusters;
    if (scores_out) memcpy(scores_out, it->scores.data(), it->scores.size() * sizeof(double));
    if (seqdist_out) memcpy(seqdist_out, it->seqdist.data(), it->seqdist.size() * sizeof(double));
    if (levels_out) memcpy(levels_out, it->levels.data(), it->levels.size() * sizeof(int));
    if (offsets_out) memcpy(offsets_out, it->offsets.data(), it->offsets.size() * sizeof(int));
    if (start_out) memcpy(start_out, it->start.data(), it->start.size() * sizeof(int));
    if (end_out) memcpy(end_out, it->end.data(), it->end.size() * sizeof(int));
    if (device_ms_out) *device_ms_out = it->device_ms;
    if (keep_out) memcpy(keep_out, it->keep.data(), it->keep.size() * sizeof(int));
    if (badcols_out) memcpy(badcols_out, it->badcols.data(), it->badcols.size() * sizeof(int));
    if (labels_out) memcpy(labels_out, it->labels.data(), it->labels.size() * sizeof(int));
    return TP_OK;
}
extern "C" int tp_batch_split(const tp_batch *b, int i, int *split_out, int *cs_out, int *ce_out, uint8_t *bad_out) {
    TP_ARG(b && i >= 0 && i < (int)b->items.size(), "tp_batch_split: index out of range");
    const TpBatchItem &it = b->items[(size_t)i];
    if (split_out) *split_out = it.split;
    if (cs_out) *cs_out = it.cs;
    if (ce_out) *ce_out = it.ce;
    if (bad_out && it.split >= 0) memcpy(bad_out, it.bad.data(), it.bad.size());
    return TP_OK;
}
extern "C" int tp_batch_free(tp_batch *b) {
    delete b;
    return TP_OK;
}
