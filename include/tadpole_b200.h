/* tadpole_b200.h -- C ABI of libtadpole_b200 (CUDA sm_100a implementation of the TADpole hot path).
 *
 * The reference (3DGenomes/TADpole) is pure R and has no native interface: the hot path sits
 * behind the exported R functions TADpole() (R/TADpole.R:344), load_mat() (R/TADpole.R:15) and
 * diffT() (R/DiffT.R:19).  These entry points are what an R .Call shim (INTEGRATION.md) or the
 * Python host in tadpole_b200/api.py binds.  Plain pointers and sizes only; no torch types.
 *
 * Conventions
 *   - every function returns 0 (TP_OK) or an error code; tp_last_error() gives the message of the
 *     last failure on the calling thread.
 *   - "host" pointers are ordinary process memory; "dev" pointers are CUDA device pointers on the
 *     context's device.  Functions taking `on_device` accept either.
 *   - matrices handed in by the caller are N x N doubles.  `colmajor` = 1 is R's layout
 *     (element (i,j) at i + j*N), 0 is C / numpy layout (i*N + j).  Only the upper triangle
 *     (i <= j) is ever read, as Matrix::forceSymmetric(uplo='U') does (R/TADpole.R:20).
 *   - bins, candidates and levels are 0-based here; the R shim / Python host add 1.
 *   - internal device state (filtered matrix, correlation, PC scores, per-candidate dendrograms)
 *     lives in the context between calls, so stages can be driven one by one (parity tests) or
 *     all at once (tp_call).
 */
#ifndef TADPOLE_B200_H
#define TADPOLE_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct tp_ctx tp_ctx;

enum {
    TP_OK = 0,
    TP_ERR_ARG = 1,        /* bad argument / call order */
    TP_ERR_CUDA = 2,       /* CUDA runtime failure */
    TP_ERR_NOLEVEL = 3,    /* a candidate has no significant broken-stick level: the reference
                              errors inside the worker here (R/TADpole.R:113-115, n_cluster = NA) */
    TP_ERR_NOCONV = 4,     /* eigensolver did not reach the residual tolerance */
    TP_ERR_NOMEM = 5,
    TP_ERR_NOSPLIT = 6     /* centromere_search: the matrix does not split (no bad columns, or the longest bad stretch
                              touches an end): the reference errors here (quirk Q4) */
};

const char *tp_last_error(void);
int tp_version(void);

/* ---- context --------------------------------------------------------------------------- */
int tp_ctx_create(int device, tp_ctx **out);
/* One context over several GPUs of the box, driven from ONE host thread (R's .Call is single-threaded): the reference's
 * TADpole() is one call that spreads over every core (registerDoParallel(detectCores()) + foreach %dopar%,
 * R/TADpole.R:103-104); a multi-device context spreads the same one call over every device listed.  The library owns one
 * host thread per device and the NCCL communicators between them (ncclCommInitAll); tp_filter / tp_compact /
 * tp_correlation / tp_pca / tp_call / tp_call_arm / tp_call_arms / tp_recall on the returned handle run on all of them and
 * return when all are done, with the results of a single-GPU call (bit-identical).  A host matrix is uploaded once: every
 * device pulls a share of the upper-triangle bands over its own PCIe link and the bands are exchanged over NVLink.
 * ndev = 1 gives a plain context.  Everything else (getters, diffT, ingest) runs on devices[0]. */
int tp_ctx_create_multi(const int *devices, int ndev, tp_ctx **out);
/* CUDA devices visible to the process (0 when there is none or no driver) */
int tp_device_count(void);
/* devices of the context (returns their number; fills at most `cap` entries) */
int tp_ctx_devices(tp_ctx *ctx, int *devices_out, int cap);
/* Counter that changes whenever the state resident in the context (matrix, PC scores, dendrograms) is replaced: a host
 * object that kept a handle on that state compares it before tp_recall / tp_get_dendro. */
long long tp_ctx_generation(tp_ctx *ctx);
/* sizes of the resident state: bins of the input, good bins, PCs in use, PCs computed, levels of the last sweep
 * (0 where that piece is absent); any pointer may be NULL */
int tp_ctx_dims(tp_ctx *ctx, int *n_out, int *nf_out, int *k_out, int *k_full_out, int *maxlev_out);
int tp_ctx_destroy(tp_ctx *ctx);
int tp_ctx_sync(tp_ctx *ctx);
/* cudaStream_t every kernel of this context is launched on (for CUDA-event timing by callers) */
void *tp_ctx_stream(tp_ctx *ctx);
/* number of kernels this context has launched so far */
long long tp_ctx_launches(tp_ctx *ctx);
/* tunables: "pca_block" (subspace width, 0 = auto), "pca_tol" (x1e-16), "pca_maxit",
 * "jacobi_direct_max", "level_cap", "dist_min_n", "igemm_min_n" (smallest nf that takes the tcgen05 int8 Gram path
 * when the counts are integers; 0 = never), "iop_min_n" / "iop_switch" / "iop_final" (sliced int8 operator of the
 * subspace iteration; "iop_final_min_n" = smallest nf whose later rounds stay on the 8-plane sliced operator),
 * "sync_blocking" (1: the host thread sleeps on a blocking-sync event while it waits for the GPU instead of spinning
 * in cudaStreamSynchronize; for hosts that run more calls in flight than they have cores),
 * "shard_sym" (0: ranks of a sharded call compute full-width row blocks of the symmetric products),
 * "mgram_min_n" (smallest nf whose M = Xc Xc^T is formed by the sliced int8 Gram; 0 = FP64 DMMA),
 * "io_bn32" (operator applications on 32-column tiles: -1 auto, 0 never, 1 always),
 * "batch_resident" (1: batch and genome calls keep resident stores for tp_batch_recall, see there; default 0),
 * "upload_lanes" (helper threads that stage a pageable host matrix or pixel array of 64 MB and more through pinned
 * buffers, default 4; 0 = leave pageable memory to the driver's own staging) */
int tp_ctx_set(tp_ctx *ctx, const char *key, double value);
/* the current value of a tp_ctx_set key (TP_ERR_ARG for an unknown key) */
int tp_ctx_get(tp_ctx *ctx, const char *key, double *value_out);
/* The environment variable TADPOLE_TUNE="key=value,key=value" applies tp_ctx_set to every context at creation. */
/* per-stage device milliseconds of the last tp_call / stage call, measured with CUDA events on
 * the context stream: [0] filter [1] compact [2] correlation [3] pca [4] sweep (CONISS) [5] CH
 * [6] total; and counters [7] pca iterations [8] pca operator applications [9] jacobi sweeps */
int tp_ctx_timings(tp_ctx *ctx, double *out10);

/* per-kernel-class device time: when enabled, every launch of the classes below is bracketed by
 * CUDA events on the context stream; reading sums them since the last enable/reset.
 * classes: [0] rowmean (filter) [1] compact [2] dgemm [3] jacobi (b x b eigensolver) [4] coniss_sweep [5] ch
 * [6] difft [8] chol (b x b Cholesky + triangular inverse) [9] igemm (the tcgen05 int8 kernels only) [10] NCCL collectives
 * [12] islice (digit slicing and exponent kernels feeding the tcgen05 kernels; HBM-bound); [13..15] unused;
 * [11] in ms_out16: executed int8 GOP (2 per multiply-add) of the profiled tcgen05 launches;
 * [7] in ms_out16: GFLOP (algorithmic) of the profiled dgemm launches.
 * enable: 1 = start/reset, 0 = stop, -1 = just read. */
int tp_ctx_profile(tp_ctx *ctx, int enable, double *ms_out16, long long *count_out16);

/* ---- multi-GPU: one process per GPU, NCCL bound at run time (single-GPU use never touches it) ------------------
 * The reference shards the n_pcs sweep over forked workers (foreach %dopar%, R/TADpole.R:103-104); here one call can
 * also spread its O(N^3) stages over the GPUs of a node.  tp_comm_unique_id (one rank) -> the 128 bytes travel to the
 * other ranks by any host channel (the Python host uses torch.distributed) -> tp_ctx_comm_init on every rank of the
 * group.  Slots hold several communicators at once (slot 0: the whole job; another slot: the ranks working on one
 * chromosome arm); tp_ctx_comm_select picks the one the following calls are collective over, -1 = none.
 * While a communicator is selected, tp_correlation / tp_pca / tp_call / tp_call_arm must be entered by every rank of
 * it with the same arguments and the same matrix; every rank returns the same results.  Row blocks of the
 * correlation matrix (and of every operator application of the PCA) are computed by their owner and all-gathered
 * when nf >= "dist_min_n" (tp_ctx_set, default 4096); the candidates of the sweep are dealt out rank-interleaved. */
int tp_comm_unique_id(void *id128);
int tp_ctx_comm_init(tp_ctx *ctx, const void *id128, int rank, int nranks, int slot);
int tp_ctx_comm_select(tp_ctx *ctx, int slot);
int tp_ctx_comm_info(tp_ctx *ctx, int *rank_out, int *nranks_out);

/* ---- input side: read.big.matrix(mat_file, type = 'double', sep = '\t') (R/TADpole.R:17) ----------------------
 * A header-less, separator-delimited N x N text matrix (host memory or a file) is uploaded as text and parsed on the
 * device into the context's N x N row-major FP64 matrix; every field is converted exactly (round to nearest even of
 * the decimal value, like strtod).  NA / NaN / empty fields become NaN (zeroed by stage 1, R/TADpole.R:19).  A row
 * whose field count differs from the number of rows is an error.  `sep` is the separator byte ('\t' in the reference).
 * tp_ingested returns the device pointer and N to hand to tp_filter / tp_call with on_device = 1, colmajor = 0; the
 * matrix stays valid until the next tp_ingest_* or the next tp_filter / tp_call from a HOST matrix on this context.
 * tp_get_ingested copies it to the host (n x n doubles, row-major).  tp_ingest_stats: [0] wall ms of the last ingest
 * (read + upload + parse), [1] device ms of the parse kernels, [2] text bytes, [3] fields converted on the host. */
int tp_ingest_tsv(tp_ctx *ctx, const char *text, size_t nbytes, int sep, int *n_out);
int tp_ingest_tsv_file(tp_ctx *ctx, const char *path, int sep, int *n_out);
int tp_ingested(tp_ctx *ctx, const double **dev_out, int *n_out);
int tp_get_ingested(tp_ctx *ctx, double *out);
int tp_ingest_stats(tp_ctx *ctx, double *out4);
/* Sparse input (SURVEY 8(f) row 2): the non-zero pixels of the UPPER triangle as (bin1, bin2, count) triplets, the
 * layout `cooler dump` and HiC-Pro write -- at 25 000 bins a few hundred MB cross PCIe instead of the 2.6 GB upper
 * triangle of the dense matrix.  The dense N x N matrix stage 1 reads is built in HBM (zero fill + one scatter pass) and
 * is handed on exactly like an ingested TSV (tp_ingested, on_device = 1, colmajor = 0).  Pixels below the diagonal are
 * ignored and counted in *below_out (the reference reads the upper triangle only: Matrix::forceSymmetric(uplo = 'U'),
 * R/TADpole.R:20); pixels naming the same cell add up (Matrix::sparseMatrix(i, j, x)); a bin outside [index_base,
 * index_base + n) is an error naming the entry.  tp_ingest_coo: host arrays.  tp_ingest_coo_file: three-column text
 * "bin1 <sep> bin2 <sep> count" parsed on the device (counts through the same exact decimal -> binary64 conversion as
 * matrix fields), a first line that is not such a row is taken as a header; n <= 0: n = largest bin + 1 - index_base. */
int tp_ingest_coo(tp_ctx *ctx, const int32_t *bin1, const int32_t *bin2, const double *count, size_t nnz, int n,
                  int index_base, unsigned long long *below_out);
int tp_ingest_coo_file(tp_ctx *ctx, const char *path, int sep, int n, int index_base, int *n_out,
                       unsigned long long *nnz_out, unsigned long long *below_out);
/* host-only test hook: the field conversion the parse kernel runs; returns 0 (value in *out) or 1 (field is left to
 * the host's strtod); needs no GPU */
int tp_test_parse_field(const char *s, int len, double *out);

/* ---- stage 1: load_mat numeric core (R/TADpole.R:19-22,35-37) ----------------------------- */
/* Uploads (or adopts, when on_device) the N x N matrix, computes rowMeans of the symmetrised
 * matrix, diag == 0, and, when bad_frac != 0, the type-7 quantile threshold; writes the bad flag
 * per bin (host, n bytes), the row means (host, n doubles, may be NULL) and the threshold
 * (may be NULL; NaN when bad_frac == 0).  The matrix stays in the context for tp_compact. */
int tp_filter(tp_ctx *ctx, const double *mat, int n, int colmajor, int on_device, double bad_frac,
              uint8_t *bad_out, double *rowmeans_out, double *thr_out);

/* mat[keep, keep] with NA -> 0 and lower := upper^T (R/TADpole.R:19-20,75-80,88): `keep` (host) lists
 * nf ascending 0-based original bin indices.  Result becomes the context's filtered matrix. */
int tp_compact(tp_ctx *ctx, const int *keep, int nf);

/* test / pipeline hooks: install or read back the context's matrices (row-major n x n, host) */
int tp_set_filtered(tp_ctx *ctx, const double *x, int nf);
int tp_get_filtered(tp_ctx *ctx, double *x_out);

/* ---- stage 2: sparse_cor()$cor + NaN -> 0 (R/TADpole.R:94-100,363,449) -------------------------- */
int tp_correlation(tp_ctx *ctx);
int tp_get_correlation(tp_ctx *ctx, double *cor_out);      /* nf x nf row-major, host */
int tp_set_correlation(tp_ctx *ctx, const double *cor, int nf);

/* ---- stage 3: prcomp(cor, rank. = k)$x (R/TADpole.R:366-367,452-453) ---------------------------- */
/* k = min(max_pcs, nf).  Consumes the context's correlation matrix (it is centred in place). */
int tp_pca(tp_ctx *ctx, int max_pcs, int *k_out);
int tp_get_scores(tp_ctx *ctx, double *scores_out);         /* nf x k row-major, host */
int tp_set_scores(tp_ctx *ctx, const double *scores, int nf, int k);

/* test hooks for the b x b kernels inside tp_pca (host in / out, row-major b x b): Cholesky factor (lower triangle of
 * l_out) and, unless factor_only, L^-1 of a symmetric positive definite g, *bad_out = 1 when it is not; eigenvalues
 * (descending) and eigenvectors (columns of v_out) of a symmetric positive semi-definite t */
int tp_test_cholinv(tp_ctx *ctx, const double *g, int b, int factor_only, double *l_out, double *linv_out, int *bad_out);
int tp_test_eig(tp_ctx *ctx, const double *t, int b, double tol, double *w_out, double *v_out, int *sweeps_out);
/* test hook of the tcgen05 int8 Gram kernel behind tp_correlation: X X^T of a symmetric n x n matrix of integer counts,
 * exact; *used_out = 0 when x is not integer-valued below 2^20 (gram_out untouched) */
int tp_test_igram(tp_ctx *ctx, const double *x, int n, double *gram_out, int *used_out);
/* test hook of the sliced int8 Gram that forms M = Xc Xc^T in tp_pca (8 digit planes per row, FP64 level): rows
 * [row_begin, row_end) of a a^T for a general n x n FP64 matrix a; all rows = the symmetric launch (upper tiles mirrored),
 * a proper row block = what one rank of a sharded call computes.  Rows outside the block keep gram_out's values. */
int tp_test_mgram(tp_ctx *ctx, const double *a, int n, int row_begin, int row_end, double *gram_out);
/* test hook of the symmetric products of a call spread over `nranks` GPUs, emulated on one: each rank's launch computes
 * the block pairs that are its share (every pair once), then the local transpose fills the rest; gram_out starts as `fill`.
 * kind 0: exact Gram of a symmetric integer-count matrix (as tp_test_igram); kind 1: sliced a a^T (as tp_test_mgram).
 * Must equal the one-GPU result bit for bit. */
int tp_test_symshard(tp_ctx *ctx, const double *a, int n, int nranks, int kind, double fill, double *gram_out);
/* host-only: the rule behind it.  Does the owner of row i compute element (i, j) (rows in blocks of rpr per rank)?  Does the
 * 128 x 64 tile rows [r_lo, r_hi] x columns [c_lo, c_hi] hold any such element (i.e. is it launched)? */
int tp_test_ss_need(int i, int j, int nranks, int rpr);
int tp_test_ss_tile(int r_lo, int r_hi, int c_lo, int c_hi, int nranks, int rpr);
/* test hooks of the two matrix-product engines of stages 2 and 3 (host in / out, row-major; operands go up in buffers of
 * their own with their padding columns set to NaN, so a kernel reading past an edge shows it).
 * tp_test_gemm: one FP64 DMMA GEMM, D = alpha A B + beta E1 + gamma E2 (E1 / E2 may be NULL), or, when mean != NULL, the
 * correlation epilogue ((v - nrows mean_i mean_j) / (nrows - 1) / (sd_i sd_j), NaN -> 0, row i = epi_row0 + local row;
 * mean / sd hold max(epi_row0 + M, N) entries).  A: M x K (a_kc) or K x M; B: N x K (b_kc) or K x N; E1 / E2: M x N;
 * sym: only tiles on and above the diagonal are computed and mirrored; splitk > 1: deterministic split-K.  D_inout is
 * M x ldd (ldd >= N) and comes back whole.  The environment variable TADPOLE_GEMM_CFG = 10 / 11 / 12 forces the
 * 32x64 / 64x64 / 128x128 tiles.
 * tp_test_iop: tp_iop_prepare of the symmetric n x n operator S, then napps sliced int8 operator applications in order on
 * this context, D_a[rows] = alpha S[rows, :] Y_a + beta E1_a[rows] + gamma E2_a[rows] with rows [row_begin, row_end),
 * block width bs[a] <= 1024 and np = 5 or 8 digit planes; Ys, E1, E2 (may be NULL) and D_inout hold the n x bs[a] blocks
 * back to back; rows outside the range keep D_inout's values; a write into a padding column of D is an error.  The tile
 * width follows the context's "io_bn32". */
int tp_test_gemm(tp_ctx *ctx, int M, int N, int K, const double *A, int a_kc, const double *B, int b_kc, double alpha,
                 const double *E1, double beta, const double *E2, double gamma, int sym, int splitk, const double *mean,
                 const double *sd, double nrows, int epi_row0, int ldd, double *D_inout);
int tp_test_iop(tp_ctx *ctx, const double *S, int n, int napps, const int *bs, const double *Ys, int np, int row_begin,
                int row_end, double alpha, const double *E1, double beta, const double *E2, double gamma, double *D_inout);

/* ---- stages 4+5: the find_params sweep (R/TADpole.R:104-123) --------------------------------------
 * For candidates i = cand_begin + t*cand_stride < k (0-based: candidate i clusters on the first
 * i+1 score columns): CONISS dendrogram (seqdist), broken-stick level count n_cluster, and the
 * Calinski-Harabasz score of every level min(min_clusters, n_cluster)..n_cluster on ALL k columns.
 * Outputs (host, may be NULL): n_cluster[k] (0 for candidates not run); *maxlev_out = the largest
 * n_cluster, the width of the score matrix (tp_get_sweep_scores). */
int tp_sweep(tp_ctx *ctx, int min_clusters, int cand_begin, int cand_stride,
             int *n_cluster_out, int *maxlev_out);
/* score matrix of the last sweep (tp_sweep, tp_call, tp_call_arm, tp_recall): exactly k x maxlev doubles row-major
 * (row = candidate, column = n_clusters-1), NaN where a level is not scored; k and maxlev as the sweep reported them
 * (or tp_ctx_dims).  A host copy the sweep made: no device work. */
int tp_get_sweep_scores(tp_ctx *ctx, double *scores_out);
/* seqdist (nf-1 doubles) and merge order (nf-1 ints: boundary removed at each step) of one
 * candidate of the last sweep; either pointer may be NULL.  After a sweep that was dealt out over several GPUs the
 * dendrogram lives on the device that ran the candidate: a multi-device context fetches it from there; with one process
 * per GPU the call is collective (every rank calls with the same `cand`, the owner broadcasts). */
int tp_get_dendro(tp_ctx *ctx, int cand, double *seqdist_out, int *order_out);

/* which.max(rowMeans(scores, na.rm=TRUE)) then which.max(scores[opt,]) (R/TADpole.R:134-135);
 * host-side reduction over a k x ld NaN-padded matrix; results 0-based */
int tp_select(const double *scores, int k, int ld, int maxlev, int *opt_cand, int *opt_level);

/* ---- one-shot: filter -> compact -> correlation -> PCA -> sweep -> selection -------------------
 * The non-centromere path of TADpole() (R/TADpole.R:444-468) from an in-memory matrix.
 * bad_out[n]; seqdist_out[nf-1] of the optimal candidate.  nf_out/k_out/maxlev_out report the sizes actually used
 * (k = min(max_pcs, nf)); the k x maxlev score matrix is read afterwards with tp_get_sweep_scores. */
int tp_call(tp_ctx *ctx, const double *mat, int n, int colmajor, int on_device,
            int max_pcs, int min_clusters, double bad_frac,
            uint8_t *bad_out, int *nf_out, int *k_out,
            int *n_pcs_out, int *n_clusters_out,
            int *maxlev_out, double *seqdist_out);
/* same, starting from an explicit keep list (chromosome arms, R/TADpole.R:357-374) on the matrix
 * already held by the context after tp_filter */
int tp_call_arm(tp_ctx *ctx, const int *keep, int nf, int max_pcs, int min_clusters,
                int *k_out, int *n_pcs_out, int *n_clusters_out, int *maxlev_out, double *seqdist_out);

/* Both chromosome arms of a centromere_search call (R/TADpole.R:357-374: the arms are independent from load_mat on), after
 * tp_filter: on a multi-device context the first half of the devices works on p while the second half works on q; on one
 * device p then q.  The results are a tp_batch (below) of two items, p then q, read with tp_batch_dims / tp_batch_get
 * (part = -1) and released with tp_batch_free: n = 0 (no bad flags: the filtering was tp_filter's), nf, k, maxlev, n_pcs,
 * n_clusters, scores, seqdist and device ms as tp_call_arm gives them, no tables. */
typedef struct tp_batch tp_batch;
int tp_call_arms(tp_ctx *ctx, const int *keep_p, int nf_p, const int *keep_q, int nf_q, int max_pcs, int min_clusters,
                 tp_batch **out);

/* ---- batches of independent calls (genome-wide use: one TADpole() per chromosome) -----------------------------------
 * ncalls matrices (mats[i]: n[i] x n[i], host -- or device when on_device, single-device contexts only), same arguments
 * as tp_call.  `inflight` calls per device are kept in flight by library-owned host threads, each on its own context and
 * stream (a lone 2000-bin call leaves most of a B200 idle), over every device of the context; the caller's one thread
 * just waits.  want_tables: also build the start / end table of every scored level of the optimal candidate
 * (R/TADpole.R:470-497) in those threads.
 * centromere: 0 = TADpole() on every matrix.  1 = centromere_search = TRUE (R/TADpole.R:351-442): each worker filters
 * its matrix, splits it (tp_centromere_split, quirk Q3 kept) and runs the p arm, then the q arm, on its own context; the
 * tables of every scored level and the optimal level's fixed labels are built there too, whatever want_tables says.  A
 * matrix that does not split fails as its own item with TP_ERR_NOSPLIT.  2 = the same with centromere_fix: the split
 * repairs quirk Q3, and a matrix that does not split is called whole on its good bins (TADpole(centromere_fix = TRUE)).
 * Results are held by the returned tp_batch, in input order:
 *   tp_batch_status / tp_batch_error  per-call return code and message (a failed call does not stop the others);
 *   tp_batch_split  the split state of a centromere_search item;
 *   tp_batch_dims   sizes to allocate: n, nf, k, maxlev, number of scored levels, total table rows, kept bins, bad
 *                   columns (-1 for NULL);
 *   tp_batch_get    bad[n], n_pcs, n_clusters, scores[k x maxlev] row-major NaN padded, seqdist[nf-1], levels[nlevels],
 *                   offsets[nlevels+1], start/end[nrows] (1-based inclusive), device ms of the call, keep[nkeep] (0-based
 *                   original bins), bad columns[nbad] (original 1-based), labels[nf + max(nbad, 0)] = the optimal level's
 *                   fixed label vector with the bad columns re-inserted (merging_arms joins the two arms'); NULL = skip.
 * The two readers take `part`: -1 = item i itself, 0 / 1 = the p / q arm of item i when it was split (TP_ERR_ARG
 * otherwise).  Kept bins, bad columns and labels exist for arms only; an arm has n = 0.  A split item itself has its bad
 * flags and its device ms (filter and both arms); an unsplit centromere_fix item reads like a whole-matrix item. */
int tp_call_batch(tp_ctx *ctx, int ncalls, const double *const *mats, const int *n, int colmajor, int on_device,
                  int max_pcs, int min_clusters, double bad_frac, int inflight, int want_tables, int centromere,
                  tp_batch **out);
int tp_batch_size(const tp_batch *b);
/* device milliseconds of the whole batch: CUDA events, from the start of the batch to the end of the last call, max over
 * the streams and devices it ran on */
double tp_batch_device_ms(const tp_batch *b);
/* kernels launched by the calls of the batch */
long long tp_batch_launches(const tp_batch *b);
int tp_batch_status(const tp_batch *b, int i);
const char *tp_batch_error(const tp_batch *b, int i);
int tp_batch_dims(const tp_batch *b, int i, int part, int *n_out, int *nf_out, int *k_out, int *maxlev_out,
                  int *nlevels_out, int *nrows_out, int *nkeep_out, int *nbad_out);
int tp_batch_get(const tp_batch *b, int i, int part, uint8_t *bad_out, int *n_pcs_out, int *n_clusters_out,
                 double *scores_out, double *seqdist_out, int *levels_out, int *offsets_out, int *start_out, int *end_out,
                 double *device_ms_out, int *keep_out, int *badcols_out, int *labels_out);
/* item i of a batch, whatever its status: *split_out = 1 when it was split at the centromere, 0 when it was not
 * (processed whole, or failed after the filter), -1 when its bad flags are not known (any item of another
 * batch); cs..ce = the longest bad stretch (1-based, 0 when there is no bad bin); bad_out[n] = the bad flags
 * when split_out >= 0.  Any pointer may be NULL. */
int tp_batch_split(const tp_batch *b, int i, int *split_out, int *cs_out, int *ce_out, uint8_t *bad_out);
int tp_batch_free(tp_batch *b);

/* ---- genome-wide input: one pixel list over every chromosome (HiC-Pro *.matrix, cooler dump -t pixels) --------------
 * The bins are global ids over a bin table: chromosome c holds chrom_bins[c] bins, in file order, the first one starting
 * at id index_base (0 or 1).  tp_genome_ingest takes host arrays; tp_genome_ingest_file a three-column text
 * "bin1 <sep> bin2 <sep> count" parsed on the device as tp_ingest_coo_file parses it (exact decimal conversion, a first
 * line that is not such a row is a header).  On the device every pixel is routed: a bin outside the bin table is an
 * error naming the entry (arrays) or the row (file); a pixel between two chromosomes (trans) and a pixel below the
 * diagonal are counted and dropped; every other (cis) pixel goes into its chromosome's bucket as chromosome-local
 * (i, j, count).  The returned handle holds the buckets on the context's device (devices[0] of a multi-device context),
 * 16 bytes per cis pixel; the input and parse buffers are released.  Device memory needed at the peak: the text, 16 bytes
 * per pixel, 16 bytes per cis pixel; TP_ERR_NOMEM when that does not fit.  1 <= nchrom <= 2^20, every chrom_bins[c] >= 1.
 * The handle is independent of the context's resident state and is released with tp_genome_free (before or after the
 * context).  tp_ingest_stats describes the last genome ingest as it does the other ingests. */
typedef struct tp_genome tp_genome;
int tp_genome_ingest(tp_ctx *ctx, const int32_t *chrom_bins, int nchrom, const int32_t *bin1, const int32_t *bin2,
                     const double *count, size_t nnz, int index_base, tp_genome **out);
int tp_genome_ingest_file(tp_ctx *ctx, const int32_t *chrom_bins, int nchrom, const char *path, int sep, int index_base,
                          tp_genome **out);
/* cis pixels per chromosome (nchrom values), trans pixels, pixels below the diagonal; any pointer may be NULL */
int tp_genome_stats(const tp_genome *g, unsigned long long *cis_out, unsigned long long *trans_out,
                    unsigned long long *below_out);
/* the dense n_c x n_c matrix of chromosome `chrom` (0-based), row-major, upper triangle (pixels naming the same cell add
 * up, the lower triangle is 0), as the calls see it; built on the context's device (it replaces the context's resident
 * matrix) and copied to out */
int tp_genome_matrix(tp_ctx *ctx, const tp_genome *g, int chrom, double *out);
/* TADpole() on every selected chromosome: chroms[nsel] (0-based; NULL = all, in bin-table order).  A tp_batch of nsel
 * items in chroms order: each item is what tp_call_batch gives for that chromosome's dense matrix with the same
 * want_tables and centromere.  The dense matrix of a chromosome is built from its
 * bucket in HBM by the worker that runs its call, and exists only while that call runs; on a multi-device context a
 * worker on another device first copies the bucket over (cudaMemcpyPeerAsync).  Workers claim chromosomes largest first.
 * A chromosome with fewer than 2 bins, or whose call fails, fails as its own item.  The context must be the one the
 * handle was ingested on (or a context whose first device holds it). */
int tp_call_genome(tp_ctx *ctx, const tp_genome *g, const int *chroms, int nsel, int max_pcs, int min_clusters,
                   double bad_frac, int inflight, int want_tables, int centromere, tp_batch **out);
int tp_genome_free(tp_genome *g);

/* ---- equal-depth subsampling: the same genome at fewer reads (DESIGN S0d) ---------------------------------------------
 * A TADpole call depends on sequencing depth (bad bins, the broken-stick level count), so two samples are compared at the
 * same number of cis contacts by subsampling the deeper one.  A cell is (c, i, j): chromosome c, chromosome-local bins
 * i <= j; its count C is the sum of the bucket entries naming it (duplicates merge) and it holds the reads (c, i, j, r),
 * r = 0 .. C-1.  Every count, and every merged cell, must be an integer in [0, 2^32): otherwise TP_ERR_ARG naming the
 * chromosome and bins (fractional counts have no reads to draw).  Only cis contacts count (trans pixels are dropped at
 * ingest).  The handle must be on a device of ctx; the work runs there.
 *
 * tp_genome_depth: reads_out[nchrom] = cis contacts (the sum of the counts) per chromosome. */
int tp_genome_depth(tp_ctx *ctx, const tp_genome *g, unsigned long long *reads_out);
/* A uniform subset of exactly `contacts` of src's reads (<= the total: otherwise TP_ERR_ARG): key(read) = first 64 bits
 * (x0 << 32 | x1) of Philox4x32-10 on counter (r, i, j, 0xD5000000 | c) with key words (seed low 32 bits, seed high 32),
 * and the reads with the `contacts` smallest (key, c, i, j, r) are kept.  *out holds, per chromosome, every cell that
 * keeps a read with its number of kept reads as the count: raw integer counts, exactly the pixels a library with that many
 * reads would give.  The draw is the multivariate hypergeometric one; it depends only on the merged cells, seed and
 * contacts (not on pixel order or duplicate splitting), and is the same bits on every run and device.  *out has src's bin
 * table, device, trans and below counts (tp_genome_stats), and is independent of src: either may be freed first.
 * Device memory: 32 bytes per bucket entry of src (a hash table, rounded up to a power of two) + 28 per merged cell, then
 * 16 per output pixel; TP_ERR_NOMEM when that does not fit. */
int tp_genome_downsample(tp_ctx *ctx, const tp_genome *src, unsigned long long contacts, unsigned long long seed,
                         tp_genome **out);
/* bucket `chrom` (0-based) of g copied to the host: tp_genome_stats gives its length; order unspecified */
int tp_genome_pixels(tp_ctx *ctx, const tp_genome *g, int chrom, int32_t *i_out, int32_t *j_out, double *count_out);

/* ---- coarsening: the same genome at a multiple of its bin size (DESIGN S0e) --------------------------------------------
 * *out = src at `factor` (>= 1) times its bin size.  Coarse chromosome c has ceil(n_c / factor) bins; coarse bin I covers
 * fine bins I*factor .. min((I+1)*factor, n_c) - 1 (the last one is narrower when factor does not divide n_c, as cooler
 * coarsen makes it).  Every bucket entry (c, i, j, v) adds to coarse cell (c, i / factor, j / factor) (integer division:
 * I <= J holds).  A NaN count adds 0 (the reference's NA -> 0 applied at the fine resolution), a cell's count is the sum
 * of its entries' counts, and cells whose sum is exactly 0 are not stored.  When every count is an integer and each
 * cell's sum of |count| is below 2^53 the sums are exact: the same bits in any order, so coarsening by a and then b equals
 * coarsening by a*b, and tp_genome_depth is unchanged.  Otherwise the rounding order is unspecified (as in the dense
 * build); fractional counts are accepted.  factor = 1 gives src with duplicate cells merged.  *out has src's device,
 * trans and below counts (tp_genome_stats), and is independent of src: either may be freed first.  The handle must be on
 * a device of ctx (TP_ERR_ARG otherwise, and for a null argument or factor < 1); the work runs there.
 * Device memory: 16 bytes per table slot (2 per bucket entry of src, rounded up to a power of two), and 16 per output
 * cell while the output is written; the table is released before the call returns.  TP_ERR_NOMEM naming the table or
 * the output buckets when they do not fit. */
int tp_genome_coarsen(tp_ctx *ctx, const tp_genome *src, int factor, tp_genome **out);

/* ---- read pairs: a genome binned at any bin size from the files a Hi-C pipeline writes (DESIGN S0f) -------------------
 * *out = the cis contacts of the plain-text read-pair files paths[npaths] (4DN .pairs, HiC-Pro *.allValidPairs, Juicer
 * merged_nodups.txt), binned at `binsize` (>= 1) bp over the chromosome table names[nchrom] / lengths[nchrom] (bp, table
 * order).  cols = the 0-based columns (each <= 63, all four different) of chrom1, pos1, chrom2, pos2; a position p is
 * index_base-based (0 or 1; the 4DN format is 1-based).  Chromosome c has ceil(lengths[c] / binsize) bins (the last one
 * narrower when binsize does not divide the length) and p falls in bin (p - index_base) / binsize.
 * A line whose first byte is '#' is a comment; a line of only spaces, tabs and '\r' is skipped; every other line is a
 * pair, its fields separated by runs of spaces and tabs (a '\r' before the '\n' is ignored).  A pair naming a chromosome
 * (exact bytes) that is not in the table is unplaced, else a pair on two chromosomes is trans: both are counted and
 * dropped.  A cis pair adds 1 to cell (c, min(b1, b2), max(b1, b2)): a read pair is unordered.
 * TP_ERR_ARG naming the file and the lowest 1-based line number (comment lines count) for: fewer fields than the largest
 * column, a position that is not 1-18 ASCII digits, a position on a chromosome of the table outside index_base ..
 * length - 1 + index_base, a line longer than the device window.  TP_ERR_ARG also for a gzip file (compressed input is
 * not read), a file with no pair lines, and a chromosome table with a duplicate, empty or whitespace-holding name, a
 * length < 1, or 2^31 - 1 or more bins in all.
 * The result is an ordinary handle on ctx's device: every cell with count >= 1, as an exact integer in FP64 (bucket order
 * unspecified).  tp_genome_stats: cis cells per chromosome, trans = trans pairs, below = 0.  counts_out (may be NULL) =
 * {pair lines, cis, trans, unplaced}, pair lines = cis + trans + unplaced.  Several files give what their concatenation
 * gives, in any order (line numbers in errors are per file); nothing depends on the window size or the file order.
 * The files are streamed through device windows of 64 MB (environment variable TADPOLE_PAIRS_WINDOW: another size in
 * bytes): device memory is the window, 8 bytes per line of a window and 16 bytes per slot of the cell table (2 to 4
 * slots per distinct cell), then 16 bytes per cell for the buckets; TP_ERR_NOMEM when the table or the buckets do not
 * fit.  tp_ingest_stats afterwards: [0] wall ms, [1] device ms of the per-window line-end and parse kernels, [2] bytes
 * read, [3] windows. */
int tp_genome_ingest_pairs_file(tp_ctx *ctx, const char *const *paths, int npaths, const char *const *names,
                                const int64_t *lengths, int nchrom, int64_t binsize, const int cols[4], int index_base,
                                unsigned long long counts_out[4], tp_genome **out);

/* The context is a device-resident pipeline handle: after tp_call / tp_call_arm / tp_pca the PC scores stay in HBM, and
 * after a sweep so do all k dendrograms (tp_get_dendro) and the score matrix (tp_get_sweep_scores).  tp_recall repeats
 * only the n_pcs sweep and the selection for another max_pcs (<= the number of PCs computed) and / or min_clusters:
 * prcomp(rank. = k') is the first k' columns of the same decomposition (R/TADpole.R:366-367), so the result equals a
 * fresh tp_call with those arguments; the reference has to repeat load_mat, cor and prcomp for this.
 * Outputs as tp_call_arm. */
int tp_recall(tp_ctx *ctx, int max_pcs, int min_clusters, int *k_out, int *n_pcs_out, int *n_clusters_out,
              int *maxlev_out, double *seqdist_out);

/* ---- the same handle for batches and genome-wide calls ----------------------------------------------------------------
 * With tp_ctx_set(ctx, "batch_resident", 1), tp_call_batch and tp_call_genome on ctx keep a resident store for every
 * item that succeeds and for every arm: the item's PC scores (nf x k_full, in the worker's row-major layout with k_full
 * rounded up to 8 columns) and the seqdist of all k candidates of its sweep (k x (nf - 1), each row padded to a multiple
 * of 8), on the device whose worker ran it.  Cost: 16 bytes per (good bin x PC computed) plus that padding, e.g. about
 * 0.9 GB for a human genome at 10 kb with max_pcs = 200 (arithmetic, not measured).  The store belongs to the returned
 * tp_batch and is released by the last tp_batch_free that refers to it, before or after the context is destroyed.  An
 * item whose store cannot be allocated fails with TP_ERR_NOMEM.  Default 0: no store.
 *
 * tp_batch_recall: tp_recall on each selected part of src -- items[s] with parts[s] = -1 for the item (both arms of a
 * split item) or 0 / 1 for its p / q arm -- run in the worker threads of tp_call_batch (`inflight` per device).  The
 * result is a tp_batch of nsel items read with tp_batch_dims / tp_batch_get / tp_batch_split: item s is what the batch
 * call gives for that part, computed from its resident PC scores (for a selected arm, the arm as item s, part -1).  It
 * equals a fresh call with max_pcs = the source's followed by tp_recall bit for bit (the same sweep and CH kernels on the
 * same scores).  Its items share the source's score stores and hold stores of their own new dendrograms, so a recall can
 * be recalled again.  Errors are per item: max_pcs above the item's k_full is tp_recall's TP_ERR_ARG, no level
 * TP_ERR_NOLEVEL; a part that failed, does not exist or holds no store, or whose store is on a device the context does
 * not have, is TP_ERR_ARG.  The store is installed on another device of the context with cudaMemcpyPeerAsync. */
int tp_batch_recall(tp_ctx *ctx, const tp_batch *src, const int *items, const int *parts, int nsel, int max_pcs,
                    int min_clusters, int inflight, tp_batch **out);
/* the seqdist (nf - 1 doubles) of candidate cand (0-based: cand + 1 PCs) of a resident item or arm */
int tp_batch_dendro(const tp_batch *b, int item, int part, int cand, double *seqdist_out);
/* device bytes of the resident stores a batch refers to, each store counted once (0 without "batch_resident") */
long long tp_batch_resident_bytes(const tp_batch *b);
/* the devices of an item's (or arm's) two stores: its PC scores, and its dendrograms -- the device that ran it.  For an
 * item of tp_batch_recall the two differ when the recall ran on another device than the store it was made from. */
int tp_batch_resident_devices(const tp_batch *b, int item, int part, int *scores_device_out, int *dendro_device_out);

/* ---- stage 6: diffT (R/DiffT.R:41-49) on padded label vectors -------------------------------------
 * labels_x / labels_y: npairs x L int32 row-major (0 = uncovered bin); out: npairs x L doubles =
 * cumulative score, normalised by its last value unless every per-bin score is 0. */
int tp_difft_batch(tp_ctx *ctx, const int32_t *labels_x, const int32_t *labels_y, int L, int npairs,
                   int on_device, double *out);

/* diffT null distribution: random_bed (R/DiffT.R:61-73) drawn nperm times ON THE DEVICE, each random partition scored
 * against the one observed call with diffT (R/DiffT.R:41-49).
 *   labels_x[L]   padded labels of the observed call over the common extent (host), as tp_difft_batch takes them;
 *   the random partitions have `ntads` TADs over the size = L - pad_left - pad_right bins that follow pad_left, and are
 *   padded with label 1 on the left and their largest label on the right (R/DiffT.R:31-36);
 *   bad_positions[nbad]  1-based positions within start:end that cannot carry a border ((start:end)[-bad_columns]);
 *   seed          selects the Philox4x32-10 stream; R's own sample() stream cannot be reproduced, the distribution
 *                 (uniform (ntads-1)-subsets of bins[-1]) is the same.
 * Outputs (host, each may be NULL): borders_out[nperm x (ntads-1)] sorted border bins as offsets from `start`
 * (the BED rows are start = c(start, borders - 1), end = c(borders - 2, end)); labels_out[nperm x L];
 * curves_out[nperm x L] diffT curves; totals_out[nperm] un-normalised totals (last value of cumsum(scores)).
 * Errors as sample() does when ntads - 1 exceeds the number of candidate bins. */
int tp_difft_null(tp_ctx *ctx, const int32_t *labels_x, int L, int pad_left, int pad_right, int ntads,
                  const int32_t *bad_positions, int nbad, unsigned long long seed, int nperm,
                  int32_t *borders_out, int32_t *labels_out, double *curves_out, double *totals_out);

/* nprob diffT comparisons of different lengths, each with its own null distribution, in one call (diffT_genome: one
 * problem per chromosome and level shared by two samples).
 * Problem p: labels_x / labels_y hold its L_p = off[p+1] - off[p] padded labels from off[p] (as tp_difft_batch takes
 * them; off[0] = 0); pad_left[p], pad_right[p], ntads[p] and bad_positions[bad_off[p] .. bad_off[p+1]) (bad_off[0] = 0)
 * describe the random partitions exactly as tp_difft_null takes them; the draws of problem p are tp_difft_null's with
 * seed + p (mod 2^64) and permutations 0 .. nperm-1, scored against labels_x of problem p.
 * Outputs (host, each may be NULL): curves_out[off[nprob]] observed normalised curves, totals_out[nprob] observed
 * un-normalised totals, null_totals_out[nprob x nperm] (row-major) totals of the random partitions, status_out[nprob] =
 * TP_OK, or TP_ERR_ARG for a problem tp_difft_null would refuse ("sample larger than the population"): its null row is
 * NaN, its observed curve and total are still written, and the other problems are unaffected.  Malformed arguments
 * (offsets not increasing, a pad outside the extent, ntads < 1, a bad position 0) fail the whole call.
 * The random label vectors never leave the GPU: one CTA draws and scores each partition.  Launches and host
 * synchronisations do not grow with nprob.  Runs on the context's first device. */
int tp_difft_multi(tp_ctx *ctx, int nprob, const int64_t *off, const int32_t *labels_x, const int32_t *labels_y,
                   const int32_t *pad_left, const int32_t *pad_right, const int32_t *ntads, const int64_t *bad_off,
                   const int32_t *bad_positions, unsigned long long seed, int nperm, double *curves_out,
                   double *totals_out, double *null_totals_out, int *status_out);

/* ---- result assembly (host integer logic, R/TADpole.R:470-497 and fix_values :503-510) ----------
 * Cuts the dendrogram `seqdist` (nf-1) into n_clusters contiguous clusters, re-inserts the bad bins
 * as 0 by original position, absorbs interior 0 runs flanked by the same id, and writes the
 * start/end table (1-based, inclusive) of the non-zero runs.  names[nf] = original 1-based bin of
 * each kept row; bad[nbad] = original 1-based bad bins (may contain names again, quirk Q3);
 * nbad < 0 means "bad_columns attribute is NULL".  start/end need room for n_clusters + nbad + 1
 * rows.  Also returns the fixed label vector when labels_out != NULL (nf + max(nbad,0) ints). */
int tp_assemble(const double *seqdist, int nf, int n_clusters, const int *names, const int *bad,
                int nbad, int *start_out, int *end_out, int *nrows_out, int *labels_out);

/* every requested level of one dendrogram in one call (same tables as nlev calls of tp_assemble): levels[nlev] =
 * numbers of clusters; offsets_out[nlev + 1] delimits each level's rows in start_out / end_out, which need room for
 * sum(levels[i] + max(nbad, 0) + 1) rows */
int tp_assemble_levels(const double *seqdist, int nf, const int *levels, int nlev, const int *names,
                       const int *bad, int nbad, int *start_out, int *end_out, int *offsets_out);

/* rioja's .find.groups (the merge matrix of the chclust / hclust object, R/TADpole.R:108 -> dendro$merge): for step
 * s = 1..n1 the boundary j = which.min(seqdist) (first index on ties) joins the groups of objects j and j+1; an operand is
 * -object while that object is a singleton, else the step that last absorbed it.  merge_out: n1 x 2 ints, column-major
 * (an R matrix).  Host only, O(n log n). */
int tp_find_groups(const double *seqdist, int n1, int *merge_out);

/* load_mat's centromere split (R/TADpole.R:58-86) on the bad flags bad[n]; host only.  The longest run of bad bins (the
 * first one on ties) is the centromere *cs_out..*ce_out (1-based; 0 when there is no bad bin); *split_out = 0 when there
 * is none or it touches either end.  Split: keep_p[*nkeep_p] / keep_q[*nkeep_q] = the arms' kept bins (0-based original
 * indices), bad_p[*nbad_p] / bad_q[*nbad_q] = their bad columns (original 1-based; *nbad = -1 when there is none, the
 * reference's NULL).  fix = 0 keeps quirk Q3: the q arm drops the rows at the ORIGINAL indices of its bad columns used
 * as positions in the arm, ignoring those past its end; fix = 1 drops the bad columns themselves.  Every output array
 * needs room for n ints. */
int tp_centromere_split(const uint8_t *bad, int n, int fix, int *split_out, int *cs_out, int *ce_out, int *keep_p,
                        int *nkeep_p, int *bad_p, int *nbad_p, int *keep_q, int *nkeep_q, int *bad_q, int *nbad_q);

#ifdef __cplusplus
}
#endif
#endif
