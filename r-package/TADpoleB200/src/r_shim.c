/* r_shim.c -- the .Call layer between R and libtadpole_b200 (include/tadpole_b200.h).
 *
 * The only translation unit that includes Rinternals.h.  Every entry point converts R objects to plain pointers
 * and sizes, calls the C ABI, and converts back.  Rules (SURVEY.md 8b):
 *   - R owns every host buffer; every SEXP allocated here is PROTECTed until it is reachable from the result;
 *   - error() (a longjmp) is raised only after the core has returned, when no C++ frame is live;
 *   - the core never calls the R API and never keeps a host pointer past the call;
 *   - device memory belongs to the tp_ctx behind an external pointer whose finalizer destroys it.
 * Replaces, in the reference: R/TADpole.R:17 (read.big.matrix), :19-22,35-37 (bad columns), :362-374 / :448-460
 * (cor, prcomp, find_params, final chclust), :470-497 (per-level tables), R/DiffT.R:41-49 (diffT loop) and
 * R/DiffT.R:61-73 (random_bed, batched).
 */
#include <R.h>
#include <Rinternals.h>
#include <R_ext/Rdynload.h>
#include <math.h>
#include <stdint.h>
#include <string.h>
#include "tadpole_b200.h"

static tp_ctx *ctx_of(SEXP p) {
    tp_ctx *c = (tp_ctx *)R_ExternalPtrAddr(p);
    if (!c) error("TADpole: the GPU context has been released");
    return c;
}

static void ctx_finalizer(SEXP p) {
    tp_ctx *c = (tp_ctx *)R_ExternalPtrAddr(p);
    if (c) {
        tp_ctx_destroy(c);
        R_ClearExternalPtr(p);
    }
}

/* devices: one index, or several -> one context over those GPUs driven from this one thread (options(tadpole.gpus=)) */
SEXP C_tp_ctx(SEXP devices) {
    tp_ctx *c = NULL;
    int ndev = length(devices);
    if (ndev < 1) error("TADpole: no device given");
    int *devs = (int *)R_alloc((size_t)ndev, sizeof(int));
    if (ndev == 1) devs[0] = asInteger(devices);
    else for (int i = 0; i < ndev; i++) devs[i] = isReal(devices) ? (int)REAL(devices)[i] : INTEGER(devices)[i];
    if (tp_ctx_create_multi(devs, ndev, &c) != TP_OK) error("%s", tp_last_error());
    SEXP p = PROTECT(R_MakeExternalPtr(c, R_NilValue, R_NilValue));
    R_RegisterCFinalizerEx(p, ctx_finalizer, TRUE);
    UNPROTECT(1);
    return p;
}

/* the counter that changes whenever the state resident in the context is replaced (kept in attr(, 'resident')) */
SEXP C_tp_generation(SEXP ctx) {
    SEXP g = PROTECT(allocVector(REALSXP, 1));
    REAL(g)[0] = (double)tp_ctx_generation(ctx_of(ctx));
    UNPROTECT(1);
    return g;
}

/* stop() unless the context still holds the state the R object was made from */
static void check_generation(tp_ctx *c, SEXP generation) {
    if ((double)tp_ctx_generation(c) != asReal(generation))
        error("TADpole: the GPU context has been used for another matrix since this call; its resident state is gone");
}

/* read.big.matrix(mat_file, type = 'double', sep = '\t') on the device (R/TADpole.R:17): returns N */
SEXP C_tp_ingest(SEXP ctx, SEXP path) {
    int n = 0;
    if (tp_ingest_tsv_file(ctx_of(ctx), CHAR(STRING_ELT(path, 0)), '\t', &n) != TP_OK) error("%s", tp_last_error());
    return ScalarInteger(n);
}

/* Upper-triangle pixels (bin1, bin2, count) -> the dense matrix in HBM (tp_ingest_coo): a Matrix::sparseMatrix, or the
 * columns of a `cooler dump`, without the dense N x N matrix ever existing in R.  Returns c(N, pixels below the
 * diagonal that were ignored). */
SEXP C_tp_ingest_coo(SEXP ctx, SEXP bin1, SEXP bin2, SEXP count, SEXP n, SEXP index_base) {
    if (!isInteger(bin1) || !isInteger(bin2) || !isReal(count) || XLENGTH(bin1) != XLENGTH(bin2) || XLENGTH(bin1) != XLENGTH(count))
        error("TADpole: bin1, bin2 (integer) and count (numeric) of equal length are expected");
    unsigned long long below = 0;
    if (tp_ingest_coo(ctx_of(ctx), INTEGER(bin1), INTEGER(bin2), REAL(count), (size_t)XLENGTH(bin1), asInteger(n),
                      asInteger(index_base), &below) != TP_OK)
        error("%s", tp_last_error());
    SEXP out = PROTECT(allocVector(REALSXP, 2));
    REAL(out)[0] = (double)asInteger(n);
    REAL(out)[1] = (double)below;
    UNPROTECT(1);
    return out;
}

/* the same from a three-column text file "bin1 <tab> bin2 <tab> count" parsed on the device; n <= 0: largest bin + 1.
 * Returns c(N, pixels, pixels below the diagonal). */
SEXP C_tp_ingest_coo_file(SEXP ctx, SEXP path, SEXP n, SEXP index_base) {
    int nn = 0;
    unsigned long long nnz = 0, below = 0;
    if (tp_ingest_coo_file(ctx_of(ctx), CHAR(STRING_ELT(path, 0)), '\t', asInteger(n), asInteger(index_base), &nn, &nnz,
                           &below) != TP_OK)
        error("%s", tp_last_error());
    SEXP out = PROTECT(allocVector(REALSXP, 3));
    REAL(out)[0] = (double)nn;
    REAL(out)[1] = (double)nnz;
    REAL(out)[2] = (double)below;
    UNPROTECT(1);
    return out;
}

/* the ingested matrix as an R matrix (for the plots of load_mat, R/TADpole.R:24-53); symmetric use only needs the
 * upper triangle, so the row-major device matrix is handed back transposed in place of a copy loop */
SEXP C_tp_ingested_matrix(SEXP ctx) {
    const double *dev = NULL;
    int n = 0;
    if (tp_ingested(ctx_of(ctx), &dev, &n) != TP_OK) error("%s", tp_last_error());
    SEXP m = PROTECT(allocMatrix(REALSXP, n, n));
    if (tp_get_ingested(ctx_of(ctx), REAL(m)) != TP_OK) {
        UNPROTECT(1);
        error("%s", tp_last_error());
    }
    /* row-major n x n read as column-major is the transpose: fix it up so that m[i, j] is the file's field (i, j) */
    double *a = REAL(m);
    for (int i = 0; i < n; i++)
        for (int j = i + 1; j < n; j++) {
            double t = a[i + (size_t)j * n];
            a[i + (size_t)j * n] = a[j + (size_t)i * n];
            a[j + (size_t)i * n] = t;
        }
    UNPROTECT(1);
    return m;
}

/* numeric core of load_mat (R/TADpole.R:19-22,35-37): logical vector of bad columns.
 * mat = an R numeric matrix (column-major, host), or NULL to use the matrix ingested by C_tp_ingest. */
SEXP C_tp_filter(SEXP ctx, SEXP mat, SEXP bad_frac) {
    tp_ctx *c = ctx_of(ctx);
    const double *ptr;
    int n, colmajor, on_device;
    if (mat == R_NilValue) {
        if (tp_ingested(c, &ptr, &n) != TP_OK) error("%s", tp_last_error());
        colmajor = 0; on_device = 1;
    } else {
        if (!isReal(mat) || nrows(mat) != ncols(mat)) error("TADpole: a square numeric matrix is expected");
        ptr = REAL(mat); n = nrows(mat); colmajor = 1; on_device = 0;
    }
    SEXP bad = PROTECT(allocVector(LGLSXP, n));
    unsigned char *tmp = (unsigned char *)R_alloc(n, 1);
    int rc = tp_filter(c, ptr, n, colmajor, on_device, asReal(bad_frac), tmp, NULL, NULL);
    if (rc != TP_OK) {
        UNPROTECT(1);
        error("%s", tp_last_error());
    }
    for (int i = 0; i < n; i++) LOGICAL(bad)[i] = tmp[i];
    UNPROTECT(1);
    return bad;
}

/* a row-major k x maxlev score matrix, NaN where a level is not scored -> an R matrix (column-major, NA); unprotected */
static SEXP score_matrix(const double *sc, int k, int maxlev) {
    SEXP scores = allocMatrix(REALSXP, k, maxlev);
    for (int r = 0; r < k; r++)
        for (int l = 0; l < maxlev; l++) {
            double v = sc[(size_t)r * maxlev + l];
            REAL(scores)[r + (size_t)l * k] = ISNAN(v) ? NA_REAL : v;
        }
    return scores;
}

/* list(n_pcs, optimal_n_clusters, seqdist, scores, generation) of one matrix or arm; seq and scores protected by the caller */
static SEXP call_result(tp_ctx *c, int npcs, int ncl, SEXP seq, SEXP scores) {
    SEXP out = PROTECT(allocVector(VECSXP, 5));
    SET_VECTOR_ELT(out, 0, ScalarInteger(npcs));
    SET_VECTOR_ELT(out, 1, ScalarInteger(ncl));
    SET_VECTOR_ELT(out, 2, seq);
    SET_VECTOR_ELT(out, 3, scores);
    SEXP gen = PROTECT(allocVector(REALSXP, 1));
    REAL(gen)[0] = (double)tp_ctx_generation(c);          /* the state this result was read from */
    SET_VECTOR_ELT(out, 4, gen);
    UNPROTECT(2);
    return out;
}

/* the result of tp_call_arm / tp_recall (return code rc), with the score matrix of its sweep */
static SEXP pack_call(tp_ctx *c, int rc, int k, int npcs, int ncl, int maxlev, SEXP seq) {
    if (rc != TP_OK) error("%s", tp_last_error());
    double *sc = (double *)R_alloc((size_t)k * maxlev + 1, sizeof(double));
    if (tp_get_sweep_scores(c, sc) != TP_OK) error("%s", tp_last_error());
    SEXP scores = PROTECT(score_matrix(sc, k, maxlev));
    SEXP out = call_result(c, npcs, ncl, seq, scores);
    UNPROTECT(1);
    return out;
}

/* cor -> prcomp -> find_params -> final chclust for one matrix or one arm (R/TADpole.R:362-374, 448-460);
 * keep = 0-based original indices of the rows load_mat keeps */
SEXP C_tp_call_arm(SEXP ctx, SEXP keep, SEXP max_pcs, SEXP min_clusters) {
    tp_ctx *c = ctx_of(ctx);
    int nf = length(keep), k = 0, npcs = 0, ncl = 0, maxlev = 0;
    if (nf < 3) error("TADpole: fewer than 3 good bins left after filtering");
    SEXP seq = PROTECT(allocVector(REALSXP, nf - 1));
    int rc = tp_call_arm(c, INTEGER(keep), nf, asInteger(max_pcs), asInteger(min_clusters), &k, &npcs, &ncl, &maxlev,
                         REAL(seq));
    SEXP out = pack_call(c, rc, k, npcs, ncl, maxlev, seq);
    UNPROTECT(1);
    return out;
}

/* the sweep again on the resident PC scores with another max_pcs / min_clusters (no reference counterpart).  The sizes
 * come from the context, never from the R object: `generation` proves the object and the context still belong together. */
SEXP C_tp_recall(SEXP ctx, SEXP generation, SEXP max_pcs, SEXP min_clusters) {
    tp_ctx *c = ctx_of(ctx);
    check_generation(c, generation);
    int nf = 0, kfull = 0, k = 0, npcs = 0, ncl = 0, maxlev = 0;
    if (tp_ctx_dims(c, NULL, &nf, NULL, &kfull, NULL) != TP_OK) error("%s", tp_last_error());
    if (nf < 3 || kfull < 1) error("TADpole: the context holds no PC scores");
    if (asInteger(max_pcs) < 1) error("TADpole: max_pcs must be positive");
    SEXP seq = PROTECT(allocVector(REALSXP, nf - 1));
    int rc = tp_recall(c, asInteger(max_pcs), asInteger(min_clusters), &k, &npcs, &ncl, &maxlev, REAL(seq));
    SEXP out = pack_call(c, rc, k, npcs, ncl, maxlev, seq);
    UNPROTECT(1);
    return out;
}

/* seqdist of the candidate that clusters on the first n_pcs PCs (1-based), for CH_map / plot_hierarchy browsing */
SEXP C_tp_dendro(SEXP ctx, SEXP generation, SEXP n_pcs) {
    tp_ctx *c = ctx_of(ctx);
    check_generation(c, generation);
    int nf = 0, k = 0, maxlev = 0;
    if (tp_ctx_dims(c, NULL, &nf, &k, NULL, &maxlev) != TP_OK) error("%s", tp_last_error());
    if (nf < 3 || maxlev < 1) error("TADpole: the context holds no sweep");
    if (asInteger(n_pcs) < 1 || asInteger(n_pcs) > k) error("TADpole: n_pcs must be between 1 and %d", k);
    SEXP seq = PROTECT(allocVector(REALSXP, nf - 1));
    if (tp_get_dendro(c, asInteger(n_pcs) - 1, REAL(seq), NULL) != TP_OK) {
        UNPROTECT(1);
        error("%s", tp_last_error());
    }
    UNPROTECT(1);
    return seq;
}

/* mat[keep, keep] after NA -> 0 and forceSymmetric(uplo = 'U'): the matrix load_mat() returns (R/TADpole.R:85,88-90);
 * keep = 0-based original indices.  Symmetric, so the row-major device copy is also the column-major R matrix. */
SEXP C_tp_get_filtered(SEXP ctx, SEXP keep) {
    tp_ctx *c = ctx_of(ctx);
    int nf = length(keep);
    if (nf < 2) error("TADpole: fewer than 2 good bins left after filtering");
    if (tp_compact(c, INTEGER(keep), nf) != TP_OK) error("%s", tp_last_error());
    SEXP m = PROTECT(allocMatrix(REALSXP, nf, nf));
    if (tp_get_filtered(c, REAL(m)) != TP_OK) {
        UNPROTECT(1);
        error("%s", tp_last_error());
    }
    UNPROTECT(1);
    return m;
}

/* dendro$merge of the chclust object: rioja's .find.groups on seqdist, in C (O(n log n)) */
SEXP C_tp_find_groups(SEXP seqdist) {
    int n1 = length(seqdist);
    SEXP m = PROTECT(allocMatrix(INTSXP, n1, 2));
    if (n1 > 0 && tp_find_groups(REAL(seqdist), n1, INTEGER(m)) != TP_OK) {
        UNPROTECT(1);
        error("%s", tp_last_error());
    }
    UNPROTECT(1);
    return m;
}

/* item i of a tp_batch: list(bad, n_pcs, optimal_n_clusters, seqdist, scores, levels, tables = list of 2-column
 * (start, end) matrices), or the call's error message; unprotected */
static SEXP batch_item(tp_batch *b, int i) {
    if (tp_batch_status(b, i) != TP_OK) {
        SEXP msg = PROTECT(allocVector(STRSXP, 1));
        SET_STRING_ELT(msg, 0, mkChar(tp_batch_error(b, i)));
        UNPROTECT(1);
        return msg;
    }
    int nn, nf, k, maxlev, nlev, nrow;
    tp_batch_dims(b, i, -1, &nn, &nf, &k, &maxlev, &nlev, &nrow, NULL, NULL);
    SEXP bad = PROTECT(allocVector(LGLSXP, nn)), seq = PROTECT(allocVector(REALSXP, nf - 1));
    SEXP levels = PROTECT(allocVector(INTSXP, nlev)), tables = PROTECT(allocVector(VECSXP, nlev));
    unsigned char *tb = (unsigned char *)R_alloc((size_t)nn, 1);
    double *sc = (double *)R_alloc((size_t)k * maxlev + 1, sizeof(double));
    int *off = (int *)R_alloc((size_t)nlev + 1, sizeof(int)), *st = (int *)R_alloc((size_t)nrow + 1, sizeof(int)),
        *en = (int *)R_alloc((size_t)nrow + 1, sizeof(int));
    int npcs = 0, ncl = 0;
    tp_batch_get(b, i, -1, tb, &npcs, &ncl, sc, REAL(seq), INTEGER(levels), off, st, en, NULL, NULL, NULL, NULL);
    for (int j = 0; j < nn; j++) LOGICAL(bad)[j] = tb[j];
    SEXP scores = PROTECT(score_matrix(sc, k, maxlev));
    for (int l = 0; l < nlev; l++) {
        int rows = off[l + 1] - off[l];
        SEXP m = PROTECT(allocMatrix(INTSXP, rows, 2));
        for (int r = 0; r < rows; r++) { INTEGER(m)[r] = st[off[l] + r]; INTEGER(m)[r + rows] = en[off[l] + r]; }
        SET_VECTOR_ELT(tables, l, m);
        UNPROTECT(1);
    }
    SEXP item = PROTECT(allocVector(VECSXP, 7));
    SET_VECTOR_ELT(item, 0, bad);
    SET_VECTOR_ELT(item, 1, ScalarInteger(npcs));
    SET_VECTOR_ELT(item, 2, ScalarInteger(ncl));
    SET_VECTOR_ELT(item, 3, seq);
    SET_VECTOR_ELT(item, 4, scores);
    SET_VECTOR_ELT(item, 5, levels);
    SET_VECTOR_ELT(item, 6, tables);
    UNPROTECT(6);
    return item;
}

/* both arms of a centromere_search call at once (R/TADpole.R:357-374); on a multi-device context the two halves of the
 * devices work on the two arms at the same time.  list(p = <as C_tp_call_arm>, q = ...) */
SEXP C_tp_call_arms(SEXP ctx, SEXP keep_p, SEXP keep_q, SEXP max_pcs, SEXP min_clusters) {
    tp_ctx *c = ctx_of(ctx);
    if (length(keep_p) < 3 || length(keep_q) < 3) error("TADpole: fewer than 3 good bins left in an arm after filtering");
    tp_batch *b = NULL;
    if (tp_call_arms(c, INTEGER(keep_p), length(keep_p), INTEGER(keep_q), length(keep_q), asInteger(max_pcs),
                     asInteger(min_clusters), &b) != TP_OK)
        error("%s", tp_last_error());
    SEXP out = PROTECT(allocVector(VECSXP, 2));
    for (int a = 0; a < 2; a++) {
        SEXP it = PROTECT(batch_item(b, a));
        SET_VECTOR_ELT(out, a, call_result(c, asInteger(VECTOR_ELT(it, 1)), asInteger(VECTOR_ELT(it, 2)), VECTOR_ELT(it, 3),
                                           VECTOR_ELT(it, 4)));
        UNPROTECT(1);
    }
    tp_batch_free(b);
    UNPROTECT(1);
    return out;
}

/* an integer vector of n values plus `add` (NULL when n < 0); unprotected */
static SEXP int_vector(const int *v, int n, int add) {
    if (n < 0) return R_NilValue;
    SEXP x = allocVector(INTSXP, n);
    for (int i = 0; i < n; i++) INTEGER(x)[i] = v[i] + add;
    return x;
}

/* load_mat's centromere split of the bad flags (tp_centromere_split, R/TADpole.R:58-86): list(c(split, cs, ce),
 * p keep, p bad_columns, q keep, q bad_columns) with keep 1-based, bad_columns NULL when empty, the arms NULL when the
 * matrix is not split; fix = the repair of quirk Q3 */
SEXP C_tp_split(SEXP bad, SEXP fix) {
    int n = length(bad);
    uint8_t *b = (uint8_t *)R_alloc((size_t)n + 1, 1);
    for (int i = 0; i < n; i++) b[i] = INTEGER(bad)[i] != 0;
    int *kp = (int *)R_alloc((size_t)n + 1, sizeof(int)), *bp = (int *)R_alloc((size_t)n + 1, sizeof(int));
    int *kq = (int *)R_alloc((size_t)n + 1, sizeof(int)), *bq = (int *)R_alloc((size_t)n + 1, sizeof(int));
    int split = 0, cs = 0, ce = 0, nkp = 0, nbp = 0, nkq = 0, nbq = 0;
    if (tp_centromere_split(b, n, asLogical(fix), &split, &cs, &ce, kp, &nkp, bp, &nbp, kq, &nkq, bq, &nbq) != TP_OK)
        error("%s", tp_last_error());
    SEXP out = PROTECT(allocVector(VECSXP, 5));
    SEXP head = allocVector(INTSXP, 3);
    SET_VECTOR_ELT(out, 0, head);
    INTEGER(head)[0] = split; INTEGER(head)[1] = cs; INTEGER(head)[2] = ce;
    if (split) {
        SET_VECTOR_ELT(out, 1, int_vector(kp, nkp, 1));
        SET_VECTOR_ELT(out, 2, int_vector(bp, nbp, 0));
        SET_VECTOR_ELT(out, 3, int_vector(kq, nkq, 1));
        SET_VECTOR_ELT(out, 4, int_vector(bq, nbq, 0));
    } else {
        for (int i = 1; i < 5; i++) SET_VECTOR_ELT(out, i, R_NilValue);
    }
    UNPROTECT(1);
    return out;
}

/* item i of a batch: a split centromere_search item is list(bad, centromere = cs:ce, p, q), each arm list(n_pcs,
 * optimal_n_clusters, seqdist, scores, keep (1-based), bad_columns (NULL when empty)); any other item as batch_item gives
 * it; unprotected */
static SEXP arms_item(tp_batch *b, int i) {
    int split = -1, cs = 0, ce = 0, nn = 0;
    tp_batch_split(b, i, &split, &cs, &ce, NULL);
    if (tp_batch_status(b, i) != TP_OK || split != 1) return batch_item(b, i);
    tp_batch_dims(b, i, -1, &nn, NULL, NULL, NULL, NULL, NULL, NULL, NULL);
    SEXP item = PROTECT(allocVector(VECSXP, 4));
    SEXP bad = allocVector(LGLSXP, nn);
    SET_VECTOR_ELT(item, 0, bad);
    unsigned char *tb = (unsigned char *)R_alloc((size_t)nn + 1, 1);
    tp_batch_split(b, i, NULL, NULL, NULL, tb);
    for (int j = 0; j < nn; j++) LOGICAL(bad)[j] = tb[j];
    SEXP cen = allocVector(INTSXP, ce - cs + 1);
    SET_VECTOR_ELT(item, 1, cen);
    for (int j = cs; j <= ce; j++) INTEGER(cen)[j - cs] = j;
    for (int a = 0; a < 2; a++) {
        int nk, nf, k, maxlev, nbad, npcs = 0, ncl = 0;
        tp_batch_dims(b, i, a, NULL, &nf, &k, &maxlev, NULL, NULL, &nk, &nbad);
        SEXP arm = PROTECT(allocVector(VECSXP, 6));
        SET_VECTOR_ELT(item, 2 + a, arm);
        UNPROTECT(1);
        SEXP seq = allocVector(REALSXP, nf - 1);
        SET_VECTOR_ELT(arm, 2, seq);
        int *keep = (int *)R_alloc((size_t)nk + 1, sizeof(int)), *bc = (int *)R_alloc((size_t)(nbad > 0 ? nbad : 0) + 1, sizeof(int));
        double *sc = (double *)R_alloc((size_t)k * maxlev + 1, sizeof(double));
        tp_batch_get(b, i, a, NULL, &npcs, &ncl, sc, REAL(seq), NULL, NULL, NULL, NULL, NULL, keep, bc, NULL);
        SET_VECTOR_ELT(arm, 0, ScalarInteger(npcs));
        SET_VECTOR_ELT(arm, 1, ScalarInteger(ncl));
        SET_VECTOR_ELT(arm, 3, score_matrix(sc, k, maxlev));
        SET_VECTOR_ELT(arm, 4, int_vector(keep, nk, 1));
        SET_VECTOR_ELT(arm, 5, int_vector(bc, nbad, 0));
    }
    UNPROTECT(1);
    return item;
}

static void batch_finalizer(SEXP p) {
    tp_batch *b = (tp_batch *)R_ExternalPtrAddr(p);
    if (b) {
        tp_batch_free(b);
        R_ClearExternalPtr(p);
    }
}

/* list(item 0, ..., item n-1) of a batch as arms_item reads them; with `keep` the batch itself follows as element n, an
 * external pointer whose finalizer frees it (its resident stores live as long as an R object refers to it), otherwise
 * the batch is freed here */
static SEXP batch_items(tp_batch *b, int n, int keep) {
    SEXP p = PROTECT(keep ? R_MakeExternalPtr(b, R_NilValue, R_NilValue) : R_NilValue);
    if (keep) R_RegisterCFinalizerEx(p, batch_finalizer, TRUE);
    /* (without keep, an R allocation failure below longjmps past tp_batch_free: the batch, plain host memory, leaks) */
    SEXP out = PROTECT(allocVector(VECSXP, n + (keep ? 1 : 0)));
    for (int i = 0; i < n; i++) SET_VECTOR_ELT(out, i, arms_item(b, i));
    if (keep) SET_VECTOR_ELT(out, n, p);
    else tp_batch_free(b);
    UNPROTECT(2);
    return out;
}

/* is "batch_resident" set on the context (TADpole_batch / TADpole_genome with resident = TRUE)? */
static int resident_on(tp_ctx *c) {
    double v = 0.0;
    return tp_ctx_get(c, "batch_resident", &v) == TP_OK && v != 0.0;
}

/* TADpole() on a list of matrices, `inflight` calls per device kept in flight by the library's own threads over every
 * device of the context (tp_call_batch with `centromere`); this thread only waits.  Per matrix: arms_item, or a character
 * error message. */
static SEXP call_batch(SEXP ctx, SEXP mats, SEXP max_pcs, SEXP min_clusters, SEXP bad_frac, SEXP inflight, int centromere) {
    tp_ctx *c = ctx_of(ctx);
    int nc = length(mats);
    const double **ptr = (const double **)R_alloc((size_t)(nc ? nc : 1), sizeof(double *));
    int *n = (int *)R_alloc((size_t)(nc ? nc : 1), sizeof(int));
    for (int i = 0; i < nc; i++) {
        SEXP m = VECTOR_ELT(mats, i);
        if (!isReal(m) || nrows(m) != ncols(m)) error("TADpole: element %d is not a square numeric matrix", i + 1);
        ptr[i] = REAL(m);
        n[i] = nrows(m);
    }
    tp_batch *b = NULL;
    if (tp_call_batch(c, nc, ptr, n, 1, 0, asInteger(max_pcs), asInteger(min_clusters), asReal(bad_frac), asInteger(inflight),
                      1, centromere, &b) != TP_OK)
        error("%s", tp_last_error());
    return batch_items(b, nc, resident_on(c));
}

/* Per matrix: list(bad, n_pcs, optimal_n_clusters, seqdist, scores, levels, tables = list of 2-column (start, end)
 * matrices), or a character error message; with "batch_resident" set (C_tp_ctx_set) the batch follows as a last
 * element (an external pointer for C_tp_batch_recall / C_tp_batch_dendro).  The same holds for the routines below. */
SEXP C_tp_call_batch(SEXP ctx, SEXP mats, SEXP max_pcs, SEXP min_clusters, SEXP bad_frac, SEXP inflight) {
    return call_batch(ctx, mats, max_pcs, min_clusters, bad_frac, inflight, 0);
}

/* TADpole(centromere_search = TRUE) on a list of matrices: every matrix is split at its centromere and both arms run in
 * the library's workers (a matrix that does not split fails, as the reference's TADpole() does). */
SEXP C_tp_call_batch_arms(SEXP ctx, SEXP mats, SEXP max_pcs, SEXP min_clusters, SEXP bad_frac, SEXP inflight) {
    return call_batch(ctx, mats, max_pcs, min_clusters, bad_frac, inflight, 1);
}

static void genome_finalizer(SEXP p) {
    tp_genome *g = (tp_genome *)R_ExternalPtrAddr(p);
    if (g) {
        tp_genome_free(g);
        R_ClearExternalPtr(p);
    }
}

/* list(handle, cis pixels per chromosome, c(trans, below)) of a freshly ingested genome; the handle is an external
 * pointer whose finalizer releases the buckets, and it keeps the context alive */
static SEXP genome_result(SEXP ctx, tp_genome *g, int nchrom) {
    SEXP p = PROTECT(R_MakeExternalPtr(g, R_NilValue, ctx));
    R_RegisterCFinalizerEx(p, genome_finalizer, TRUE);
    SEXP cis = PROTECT(allocVector(REALSXP, nchrom)), tb = PROTECT(allocVector(REALSXP, 2));
    unsigned long long *tmp = (unsigned long long *)R_alloc((size_t)nchrom, sizeof(unsigned long long)), trans = 0, below = 0;
    tp_genome_stats(g, tmp, &trans, &below);
    for (int i = 0; i < nchrom; i++) REAL(cis)[i] = (double)tmp[i];
    REAL(tb)[0] = (double)trans;
    REAL(tb)[1] = (double)below;
    SEXP out = PROTECT(allocVector(VECSXP, 3));
    SET_VECTOR_ELT(out, 0, p);
    SET_VECTOR_ELT(out, 1, cis);
    SET_VECTOR_ELT(out, 2, tb);
    UNPROTECT(4);
    return out;
}

/* A genome-wide pixel list split by chromosome on the GPU (tp_genome_ingest): chrom_bins = bins per chromosome in
 * bin-table order, the pixels = vectors bin1, bin2 (integer, global ids) and count (numeric).  Returns
 * list(handle, cis pixels per chromosome, c(trans, below)). */
SEXP C_tp_genome(SEXP ctx, SEXP chrom_bins, SEXP bin1, SEXP bin2, SEXP count, SEXP index_base) {
    tp_ctx *c = ctx_of(ctx);
    if (!isInteger(chrom_bins) || length(chrom_bins) < 1) error("TADpole: the bins per chromosome must be an integer vector");
    if (!isInteger(bin1) || !isInteger(bin2) || !isReal(count) || XLENGTH(bin1) != XLENGTH(bin2) || XLENGTH(bin1) != XLENGTH(count))
        error("TADpole: bin1, bin2 (integer) and count (numeric) of equal length are expected");
    tp_genome *g = NULL;
    if (tp_genome_ingest(c, INTEGER(chrom_bins), length(chrom_bins), INTEGER(bin1), INTEGER(bin2), REAL(count),
                         (size_t)XLENGTH(bin1), asInteger(index_base), &g) != TP_OK)
        error("%s", tp_last_error());
    return genome_result(ctx, g, length(chrom_bins));
}

/* the same from a three-column tab-separated pixel file (HiC-Pro *.matrix, cooler dump -t pixels) parsed on the device
 * (tp_genome_ingest_file) */
SEXP C_tp_genome_file(SEXP ctx, SEXP chrom_bins, SEXP path, SEXP index_base) {
    tp_ctx *c = ctx_of(ctx);
    if (!isInteger(chrom_bins) || length(chrom_bins) < 1) error("TADpole: the bins per chromosome must be an integer vector");
    tp_genome *g = NULL;
    if (tp_genome_ingest_file(c, INTEGER(chrom_bins), length(chrom_bins), CHAR(STRING_ELT(path, 0)), '\t', asInteger(index_base),
                              &g) != TP_OK)
        error("%s", tp_last_error());
    return genome_result(ctx, g, length(chrom_bins));
}

static tp_genome *genome_of(SEXP p) {
    tp_genome *g = (tp_genome *)R_ExternalPtrAddr(p);
    if (!g) error("TADpole: the genome pixels have been released");
    return g;
}

static int nchrom_of(SEXP nchrom) {
    const int n = asInteger(nchrom);
    if (n < 1 || n > (1 << 20)) error("TADpole: the number of chromosomes must be in 1..2^20");
    return n;
}

/* a whole number in [0, 2^53] given as an R numeric (contacts, seeds) */
static unsigned long long count_arg(SEXP x, const char *what) {
    const double v = asReal(x);
    if (!(v >= 0 && v <= 9007199254740992.0 && v == floor(v))) error("TADpole: %s must be a whole number >= 0", what);
    return (unsigned long long)v;
}

/* cis contacts per chromosome of a C_tp_genome handle over `nchrom` chromosomes (tp_genome_depth), as doubles */
SEXP C_tp_genome_depth(SEXP ctx, SEXP genome, SEXP nchrom) {
    tp_ctx *c = ctx_of(ctx);
    tp_genome *g = genome_of(genome);
    const int n = nchrom_of(nchrom);
    unsigned long long *tmp = (unsigned long long *)R_alloc((size_t)n, sizeof(unsigned long long));
    if (tp_genome_depth(c, g, tmp) != TP_OK) error("%s", tp_last_error());
    SEXP out = PROTECT(allocVector(REALSXP, n));
    for (int i = 0; i < n; i++) REAL(out)[i] = (double)tmp[i];
    UNPROTECT(1);
    return out;
}

/* a uniform subset of exactly `contacts` of the genome's cis reads drawn with `seed` (tp_genome_downsample): what
 * C_tp_genome returns, for the new buckets */
SEXP C_tp_genome_downsample(SEXP ctx, SEXP genome, SEXP nchrom, SEXP contacts, SEXP seed) {
    tp_ctx *c = ctx_of(ctx);
    tp_genome *g = genome_of(genome);
    const int n = nchrom_of(nchrom);
    const unsigned long long k = count_arg(contacts, "contacts"), sd = count_arg(seed, "seed");
    tp_genome *out = NULL;
    if (tp_genome_downsample(c, g, k, sd, &out) != TP_OK) error("%s", tp_last_error());
    return genome_result(ctx, out, n);
}

/* the genome at `factor` times its bin size (tp_genome_coarsen): what C_tp_genome returns, for the new buckets */
SEXP C_tp_genome_coarsen(SEXP ctx, SEXP genome, SEXP nchrom, SEXP factor) {
    const double f = asReal(factor);
    if (!(f >= 1 && f <= 2147483647.0 && f == floor(f))) error("TADpole: factor must be a whole number >= 1");
    tp_ctx *c = ctx_of(ctx);
    tp_genome *g = genome_of(genome);
    const int n = nchrom_of(nchrom);
    tp_genome *out = NULL;
    if (tp_genome_coarsen(c, g, (int)f, &out) != TP_OK) error("%s", tp_last_error());
    return genome_result(ctx, out, n);
}

/* Read-pair files binned at `binsize` bp on the GPU (tp_genome_ingest_pairs_file): paths and names (character), lengths
 * (numeric, bp), layout = integer c(chrom1, pos1, chrom2, pos2 columns (0-based), index_base).  Returns what C_tp_genome
 * returns, and c(pair lines, cis, trans, unplaced) as a fourth element. */
SEXP C_tp_genome_pairs_file(SEXP ctx, SEXP paths, SEXP names, SEXP lengths, SEXP binsize, SEXP layout) {
    const int np = length(paths), nc = length(names);
    if (np < 1) error("TADpole: at least one pairs file is needed");
    if (nc < 1 || nc > (1 << 20) || !isReal(lengths) || length(lengths) != nc)
        error("TADpole: the chromosome table needs 1..2^20 names and as many numeric lengths");
    for (int c = 0; c < nc; c++) {
        const double v = REAL(lengths)[c];
        if (!(v >= 1 && v <= 9007199254740992.0 && v == floor(v))) error("TADpole: chromosome lengths must be whole numbers >= 1");
    }
    const double b = asReal(binsize);
    if (!(b >= 1 && b <= 9007199254740992.0 && b == floor(b))) error("TADpole: binsize must be a whole number >= 1");
    if (!isInteger(layout) || length(layout) != 5) error("TADpole: layout must be 4 column indices and index_base (integer)");
    tp_ctx *c = ctx_of(ctx);
    const char **pp = (const char **)R_alloc((size_t)np, sizeof(char *)), **nm = (const char **)R_alloc((size_t)nc, sizeof(char *));
    int64_t *len = (int64_t *)R_alloc((size_t)nc, sizeof(int64_t));
    for (int i = 0; i < np; i++) pp[i] = CHAR(STRING_ELT(paths, i));
    for (int i = 0; i < nc; i++) { nm[i] = CHAR(STRING_ELT(names, i)); len[i] = (int64_t)REAL(lengths)[i]; }
    unsigned long long counts[4] = {0, 0, 0, 0};
    tp_genome *g = NULL;
    if (tp_genome_ingest_pairs_file(c, pp, np, nm, len, nc, (int64_t)b, INTEGER(layout), INTEGER(layout)[4], counts, &g) != TP_OK)
        error("%s", tp_last_error());
    SEXP res = PROTECT(genome_result(ctx, g, nc)), cnt = PROTECT(allocVector(REALSXP, 4)), out = PROTECT(allocVector(VECSXP, 4));
    for (int i = 0; i < 4; i++) REAL(cnt)[i] = (double)counts[i];
    for (int i = 0; i < 3; i++) SET_VECTOR_ELT(out, i, VECTOR_ELT(res, i));
    SET_VECTOR_ELT(out, 3, cnt);
    UNPROTECT(3);
    return out;
}

/* bucket `chrom` (0-based) of a genome over `nchrom` chromosomes: list(i, j, count), 0-based local bins, bucket order */
SEXP C_tp_genome_pixels(SEXP ctx, SEXP genome, SEXP chrom, SEXP nchrom) {
    tp_ctx *c = ctx_of(ctx);
    tp_genome *g = genome_of(genome);
    const int n = nchrom_of(nchrom), ch = asInteger(chrom);
    if (ch < 0 || ch >= n) error("TADpole: chromosome index out of range");
    unsigned long long *cis = (unsigned long long *)R_alloc((size_t)n, sizeof(unsigned long long));
    if (tp_genome_stats(g, cis, NULL, NULL) != TP_OK) error("%s", tp_last_error());
    if (cis[ch] > 2147483647ULL) error("TADpole: the bucket holds more than 2^31 - 1 pixels");
    const int m = (int)cis[ch];
    SEXP i = PROTECT(allocVector(INTSXP, m)), j = PROTECT(allocVector(INTSXP, m)), v = PROTECT(allocVector(REALSXP, m));
    if (m > 0 && tp_genome_pixels(c, g, ch, INTEGER(i), INTEGER(j), REAL(v)) != TP_OK) {
        UNPROTECT(3);
        error("%s", tp_last_error());
    }
    SEXP out = PROTECT(allocVector(VECSXP, 3));
    SET_VECTOR_ELT(out, 0, i);
    SET_VECTOR_ELT(out, 1, j);
    SET_VECTOR_ELT(out, 2, v);
    UNPROTECT(4);
    return out;
}

/* TADpole() on the chromosomes `chroms` (0-based) of a C_tp_genome handle, `inflight` calls per device in flight
 * (tp_call_genome with `centromere`).  Per chromosome, in chroms order: arms_item, or a character error message. */
static SEXP call_genome(SEXP ctx, SEXP genome, SEXP chroms, SEXP max_pcs, SEXP min_clusters, SEXP bad_frac, SEXP inflight,
                        int tables, int centromere) {
    tp_ctx *c = ctx_of(ctx);
    tp_genome *g = (tp_genome *)R_ExternalPtrAddr(genome);
    if (!g) error("TADpole: the genome pixels have been released");
    if (!isInteger(chroms)) error("TADpole: chromosome indices must be integers");
    int ns = length(chroms);
    tp_batch *b = NULL;
    if (tp_call_genome(c, g, INTEGER(chroms), ns, asInteger(max_pcs), asInteger(min_clusters), asReal(bad_frac),
                       asInteger(inflight), tables, centromere, &b) != TP_OK)
        error("%s", tp_last_error());
    return batch_items(b, ns, resident_on(c));
}

/* tp_ctx_set(ctx, key, value); returns the key's previous value (so that the R host can restore it) */
SEXP C_tp_ctx_set(SEXP ctx, SEXP key, SEXP value) {
    tp_ctx *c = ctx_of(ctx);
    if (length(key) != 1) error("TADpole: the key must be one string");
    double prev = 0.0;
    if (tp_ctx_get(c, CHAR(STRING_ELT(key, 0)), &prev) != TP_OK || tp_ctx_set(c, CHAR(STRING_ELT(key, 0)), asReal(value)) != TP_OK)
        error("%s", tp_last_error());
    SEXP out = PROTECT(allocVector(REALSXP, 1));
    REAL(out)[0] = prev;
    UNPROTECT(1);
    return out;
}

static tp_batch *batch_of(SEXP p) {
    tp_batch *b = (tp_batch *)R_ExternalPtrAddr(p);
    if (!b) error("TADpole: the resident batch has been released");
    return b;
}

/* tp_batch_recall of items (0-based) / parts (-1 = the item, 0 / 1 = an arm) of a resident batch, 8 recalls in flight per
 * device (TADpole_genome()'s default): per selection what arms_item gives (a character message for a selection that
 * failed), then the new batch as the last element (it shares the source's PC scores and holds its own dendrograms). */
SEXP C_tp_batch_recall(SEXP ctx, SEXP batch, SEXP items, SEXP parts, SEXP max_pcs, SEXP min_clusters) {
    tp_ctx *c = ctx_of(ctx);
    tp_batch *src = batch_of(batch);
    if (!isInteger(items) || !isInteger(parts) || length(items) != length(parts))
        error("TADpole: items and parts must be integer vectors of equal length");
    int ns = length(items);
    tp_batch *b = NULL;
    if (tp_batch_recall(c, src, INTEGER(items), INTEGER(parts), ns, asInteger(max_pcs), asInteger(min_clusters), 8, &b) !=
        TP_OK)
        error("%s", tp_last_error());
    return batch_items(b, ns, 1);
}

/* seqdist of the candidate that clusters on the first n_pcs PCs (1-based) of item (0-based) / part of a resident batch;
 * the buffer is sized from the batch (tp_batch_dims), never from the R object */
SEXP C_tp_batch_dendro(SEXP batch, SEXP item, SEXP part, SEXP n_pcs) {
    tp_batch *b = batch_of(batch);
    int nf = 0, k = 0;
    if (tp_batch_dims(b, asInteger(item), asInteger(part), NULL, &nf, &k, NULL, NULL, NULL, NULL, NULL) != TP_OK)
        error("%s", tp_last_error());
    if (nf < 3) error("TADpole: this item holds no dendrogram");
    if (asInteger(n_pcs) < 1 || asInteger(n_pcs) > k) error("TADpole: n_pcs must be between 1 and %d", k);
    SEXP seq = PROTECT(allocVector(REALSXP, nf - 1));
    int rc = tp_batch_dendro(b, asInteger(item), asInteger(part), asInteger(n_pcs) - 1, REAL(seq));
    UNPROTECT(1);
    if (rc != TP_OK) error("%s", tp_last_error());
    return seq;
}

/* Per chromosome: what C_tp_call_batch gives for its dense matrix (the per-level tables empty unless `tables`). */
SEXP C_tp_call_genome(SEXP ctx, SEXP genome, SEXP chroms, SEXP max_pcs, SEXP min_clusters, SEXP bad_frac, SEXP inflight,
                      SEXP tables) {
    return call_genome(ctx, genome, chroms, max_pcs, min_clusters, bad_frac, inflight, asLogical(tables), 0);
}

/* TADpole(centromere_search = TRUE) on each chromosome.  fix: centromere_fix of the Python host (the repair of quirks Q3
 * and Q4); R's TADpole() has no such flag and passes FALSE. */
SEXP C_tp_call_genome_arms(SEXP ctx, SEXP genome, SEXP chroms, SEXP max_pcs, SEXP min_clusters, SEXP bad_frac, SEXP inflight,
                           SEXP fix) {
    return call_genome(ctx, genome, chroms, max_pcs, min_clusters, bad_frac, inflight, 1, asLogical(fix) ? 2 : 1);
}

/* the cutree / fix_values / rle loop of R/TADpole.R:470-497 for many levels at once: list of 2-column integer
 * matrices (start, end), one per requested level.  bad = integer(0) with nbad_null = TRUE means attr NULL. */
SEXP C_tp_levels(SEXP seqdist, SEXP levels, SEXP names, SEXP bad, SEXP bad_is_null) {
    int nf = length(names), nlev = length(levels);
    int nbad = asLogical(bad_is_null) ? -1 : length(bad);
    size_t cap = 0;
    for (int i = 0; i < nlev; i++) cap += (size_t)INTEGER(levels)[i] + (nbad > 0 ? nbad : 0) + 2;
    int *st = (int *)R_alloc(cap ? cap : 1, sizeof(int)), *en = (int *)R_alloc(cap ? cap : 1, sizeof(int));
    int *off = (int *)R_alloc((size_t)nlev + 1, sizeof(int));
    if (tp_assemble_levels(REAL(seqdist), nf, INTEGER(levels), nlev, INTEGER(names), INTEGER(bad), nbad, st, en, off) != TP_OK)
        error("%s", tp_last_error());
    SEXP out = PROTECT(allocVector(VECSXP, nlev));
    for (int i = 0; i < nlev; i++) {
        int rows = off[i + 1] - off[i];
        SEXP m = PROTECT(allocMatrix(INTSXP, rows, 2));
        for (int r = 0; r < rows; r++) {
            INTEGER(m)[r] = st[off[i] + r];
            INTEGER(m)[r + rows] = en[off[i] + r];
        }
        SET_VECTOR_ELT(out, i, m);
        UNPROTECT(1);
    }
    UNPROTECT(1);
    return out;
}

/* one level: cutree + bad bins re-inserted as 0 + fix_values (R/TADpole.R:411-431): the per-bin label vector */
SEXP C_tp_labels(SEXP seqdist, SEXP n_clusters, SEXP names, SEXP bad, SEXP bad_is_null) {
    int nf = length(names), k = asInteger(n_clusters), nrows_out = 0;
    int nbad = asLogical(bad_is_null) ? -1 : length(bad);
    size_t cap = (size_t)k + (nbad > 0 ? nbad : 0) + 2;
    int *st = (int *)R_alloc(cap, sizeof(int)), *en = (int *)R_alloc(cap, sizeof(int));
    SEXP lab = PROTECT(allocVector(INTSXP, nf + (nbad > 0 ? nbad : 0)));
    if (tp_assemble(REAL(seqdist), nf, k, INTEGER(names), INTEGER(bad), nbad, st, en, &nrows_out, INTEGER(lab)) != TP_OK) {
        UNPROTECT(1);
        error("%s", tp_last_error());
    }
    UNPROTECT(1);
    return lab;
}

/* the loop of diffT (R/DiffT.R:41-49) for npairs padded label vectors of length L (row-major npairs x L) */
SEXP C_tp_difft(SEXP ctx, SEXP lx, SEXP ly, SEXP L, SEXP npairs) {
    size_t n = (size_t)asInteger(L) * asInteger(npairs);
    if ((size_t)length(lx) != n || (size_t)length(ly) != n) error("TADpole: label vectors do not match L x npairs");
    SEXP out = PROTECT(allocVector(REALSXP, n));
    if (tp_difft_batch(ctx_of(ctx), INTEGER(lx), INTEGER(ly), asInteger(L), asInteger(npairs), 0, REAL(out)) != TP_OK) {
        UNPROTECT(1);
        error("%s", tp_last_error());
    }
    UNPROTECT(1);
    return out;
}

/* nperm draws of random_bed (R/DiffT.R:61-73) on the device, each scored against labels_x:
 * list(borders [ (ntads-1) x nperm ], totals [nperm], curves [L x nperm]) -- column per permutation */
SEXP C_tp_difft_null(SEXP ctx, SEXP lx, SEXP pad_left, SEXP pad_right, SEXP ntads, SEXP bad, SEXP seed, SEXP nperm) {
    int L = length(lx), T = asInteger(ntads), P = asInteger(nperm);
    SEXP borders = PROTECT(allocMatrix(INTSXP, T > 1 ? T - 1 : 0, P));
    SEXP totals = PROTECT(allocVector(REALSXP, P));
    SEXP curves = PROTECT(allocMatrix(REALSXP, L, P));
    int rc = tp_difft_null(ctx_of(ctx), INTEGER(lx), L, asInteger(pad_left), asInteger(pad_right), T,
                           length(bad) ? INTEGER(bad) : NULL, length(bad), (unsigned long long)asReal(seed), P,
                           T > 1 ? INTEGER(borders) : NULL, NULL, REAL(curves), REAL(totals));
    if (rc != TP_OK) {
        UNPROTECT(3);
        error("%s", tp_last_error());
    }
    SEXP out = PROTECT(allocVector(VECSXP, 3));
    SET_VECTOR_ELT(out, 0, borders);
    SET_VECTOR_ELT(out, 1, totals);
    SET_VECTOR_ELT(out, 2, curves);
    UNPROTECT(4);
    return out;
}

/* nprob diffT comparisons of different lengths, each with its own null distribution (tp_difft_multi; diffT_genome).
 * off / bad_off: numeric (doubles: R has no 64-bit integers), nprob + 1 offsets into the labels and bad; labels =
 * list(x, y) of integer vectors; problems = integer matrix nprob x 3 (pad_left, pad_right, ntads).  Returns
 * list(curves [off[nprob]], totals [nprob], null_totals [nperm x nprob] -- column per problem, status [nprob]) */
SEXP C_tp_difft_multi(SEXP ctx, SEXP off, SEXP labels, SEXP problems, SEXP bad_off, SEXP bad, SEXP seed, SEXP nperm) {
    int nprob = length(off) - 1, P = asInteger(nperm);
    if (nprob < 0 || length(bad_off) != nprob + 1 || length(problems) != 3 * nprob || length(labels) != 2)
        error("TADpole: off, bad_off, labels and the problem matrix do not describe the same problems");
    SEXP lx = VECTOR_ELT(labels, 0), ly = VECTOR_ELT(labels, 1);
    int64_t *o = (int64_t *)R_alloc((size_t)nprob + 1, sizeof(int64_t));
    int64_t *bo = (int64_t *)R_alloc((size_t)nprob + 1, sizeof(int64_t));
    for (int i = 0; i <= nprob; i++) { o[i] = (int64_t)REAL(off)[i]; bo[i] = (int64_t)REAL(bad_off)[i]; }
    if (nprob > 0 && ((int64_t)length(lx) != o[nprob] || (int64_t)length(ly) != o[nprob] || (int64_t)length(bad) != bo[nprob]))
        error("TADpole: label or bad-position vectors do not match the offsets");
    const int *pm = INTEGER(problems);                    /* column-major: pad_left, pad_right, ntads */
    SEXP curves = PROTECT(allocVector(REALSXP, nprob > 0 ? (size_t)o[nprob] : 0));
    SEXP totals = PROTECT(allocVector(REALSXP, nprob));
    SEXP null = PROTECT(allocMatrix(REALSXP, P, nprob));
    SEXP status = PROTECT(allocVector(INTSXP, nprob));
    int rc = tp_difft_multi(ctx_of(ctx), nprob, o, INTEGER(lx), INTEGER(ly), pm, pm + nprob, pm + 2 * (size_t)nprob, bo,
                            length(bad) ? INTEGER(bad) : NULL, (unsigned long long)asReal(seed), P, REAL(curves),
                            REAL(totals), REAL(null), INTEGER(status));
    if (rc != TP_OK) {
        UNPROTECT(4);
        error("%s", tp_last_error());
    }
    SEXP out = PROTECT(allocVector(VECSXP, 4));
    SET_VECTOR_ELT(out, 0, curves);
    SET_VECTOR_ELT(out, 1, totals);
    SET_VECTOR_ELT(out, 2, null);
    SET_VECTOR_ELT(out, 3, status);
    UNPROTECT(5);
    return out;
}

/* several GPUs: one R process per GPU; rank 0 makes the id, every rank joins (csrc/comm.cu) */
SEXP C_tp_comm_unique_id(void) {
    SEXP id = PROTECT(allocVector(RAWSXP, 128));
    if (tp_comm_unique_id(RAW(id)) != TP_OK) {
        UNPROTECT(1);
        error("%s", tp_last_error());
    }
    UNPROTECT(1);
    return id;
}

SEXP C_tp_ctx_comm_init(SEXP ctx, SEXP id, SEXP rank, SEXP nranks, SEXP slot) {
    if (length(id) != 128) error("TADpole: the communicator id must be 128 raw bytes");
    if (tp_ctx_comm_init(ctx_of(ctx), RAW(id), asInteger(rank), asInteger(nranks), asInteger(slot)) != TP_OK)
        error("%s", tp_last_error());
    return R_NilValue;
}

SEXP C_tp_ctx_comm_select(SEXP ctx, SEXP slot) {
    if (tp_ctx_comm_select(ctx_of(ctx), asInteger(slot)) != TP_OK) error("%s", tp_last_error());
    return R_NilValue;
}

static const R_CallMethodDef call_table[] = {
    {"C_tp_ctx", (DL_FUNC)&C_tp_ctx, 1},
    {"C_tp_ingest", (DL_FUNC)&C_tp_ingest, 2},
    {"C_tp_ingested_matrix", (DL_FUNC)&C_tp_ingested_matrix, 1},
    {"C_tp_ingest_coo", (DL_FUNC)&C_tp_ingest_coo, 6},
    {"C_tp_ingest_coo_file", (DL_FUNC)&C_tp_ingest_coo_file, 4},
    {"C_tp_filter", (DL_FUNC)&C_tp_filter, 3},
    {"C_tp_call_arm", (DL_FUNC)&C_tp_call_arm, 4},
    {"C_tp_recall", (DL_FUNC)&C_tp_recall, 4},
    {"C_tp_dendro", (DL_FUNC)&C_tp_dendro, 3},
    {"C_tp_generation", (DL_FUNC)&C_tp_generation, 1},
    {"C_tp_get_filtered", (DL_FUNC)&C_tp_get_filtered, 2},
    {"C_tp_find_groups", (DL_FUNC)&C_tp_find_groups, 1},
    {"C_tp_call_arms", (DL_FUNC)&C_tp_call_arms, 5},
    {"C_tp_call_batch", (DL_FUNC)&C_tp_call_batch, 6},
    {"C_tp_genome", (DL_FUNC)&C_tp_genome, 6},
    {"C_tp_genome_file", (DL_FUNC)&C_tp_genome_file, 4},
    {"C_tp_call_genome", (DL_FUNC)&C_tp_call_genome, 8},
    {"C_tp_split", (DL_FUNC)&C_tp_split, 2},
    {"C_tp_call_batch_arms", (DL_FUNC)&C_tp_call_batch_arms, 6},
    {"C_tp_call_genome_arms", (DL_FUNC)&C_tp_call_genome_arms, 8},
    {"C_tp_levels", (DL_FUNC)&C_tp_levels, 5},
    {"C_tp_labels", (DL_FUNC)&C_tp_labels, 5},
    {"C_tp_difft", (DL_FUNC)&C_tp_difft, 5},
    {"C_tp_difft_null", (DL_FUNC)&C_tp_difft_null, 8},
    {"C_tp_difft_multi", (DL_FUNC)&C_tp_difft_multi, 8},
    {"C_tp_comm_unique_id", (DL_FUNC)&C_tp_comm_unique_id, 0},
    {"C_tp_ctx_comm_init", (DL_FUNC)&C_tp_ctx_comm_init, 5},
    {"C_tp_ctx_comm_select", (DL_FUNC)&C_tp_ctx_comm_select, 2},
    {"C_tp_ctx_set", (DL_FUNC)&C_tp_ctx_set, 3},
    {"C_tp_batch_recall", (DL_FUNC)&C_tp_batch_recall, 6},
    {"C_tp_batch_dendro", (DL_FUNC)&C_tp_batch_dendro, 4},
    {"C_tp_genome_depth", (DL_FUNC)&C_tp_genome_depth, 3},
    {"C_tp_genome_downsample", (DL_FUNC)&C_tp_genome_downsample, 5},
    {"C_tp_genome_pixels", (DL_FUNC)&C_tp_genome_pixels, 4},
    {"C_tp_genome_coarsen", (DL_FUNC)&C_tp_genome_coarsen, 4},
    {"C_tp_genome_pairs_file", (DL_FUNC)&C_tp_genome_pairs_file, 6},
    {NULL, NULL, 0}};

void R_init_TADpoleB200(DllInfo *dll) {
    R_registerRoutines(dll, NULL, call_table, NULL, NULL);
    R_useDynamicSymbols(dll, FALSE);
}
