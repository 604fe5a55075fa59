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
 * "upload_lanes" (helper threads that stage a pageable host matrix or pixel array of 64 MB and more through pinned
 * buffers, default 4; 0 = leave pageable memory to the driver's own staging) */
int tp_ctx_set(tp_ctx *ctx, const char *key, double value);
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

/* The context is a device-resident pipeline handle: after tp_call / tp_call_arm / tp_pca the PC scores stay in HBM, and
 * after a sweep so do all k dendrograms (tp_get_dendro) and the score matrix (tp_get_sweep_scores).  tp_recall repeats
 * only the n_pcs sweep and the selection for another max_pcs (<= the number of PCs computed) and / or min_clusters:
 * prcomp(rank. = k') is the first k' columns of the same decomposition (R/TADpole.R:366-367), so the result equals a
 * fresh tp_call with those arguments; the reference has to repeat load_mat, cor and prcomp for this.
 * Outputs as tp_call_arm. */
int tp_recall(tp_ctx *ctx, int max_pcs, int min_clusters, int *k_out, int *n_pcs_out, int *n_clusters_out,
              int *maxlev_out, double *seqdist_out);

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
