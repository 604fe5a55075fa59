# R host of TADpoleB200: the exported functions of the reference package (NAMESPACE:3-8 there) with their
# signatures, messages and returned objects, every numeric step delegated to libtadpole_b200 through .Call.
# Written against the C ABI in include/tadpole_b200.h; the same logic runs (and is tested) as tadpole_b200/api.py.
# NOTE: R is not available in the build image, so this file is exercised only through its .Call targets
# (tests/test_r_shim_*.py drive src/r_shim.c with a stand-in R runtime); it has not been run under R.
# plot_hierarchy() and CH_map() of the reference only read the returned object: source them from the reference
# package unchanged (they are graphics, outside this package).

.tp_state <- new.env(parent = emptyenv())

# One context per device set.  options(tadpole.gpus = 0:7) makes every call of this session spread over those GPUs: the
# library then owns one host thread per GPU (R stays single-threaded), as registerDoParallel(detectCores()) made the
# reference spread over every core.
.tp_ctx <- function(devices = getOption("tadpole.gpus", 0L)) {
    devices <- as.integer(devices)
    key <- paste0("ctx", paste(devices, collapse = "_"))
    if (is.null(.tp_state[[key]])) .tp_state[[key]] <- .Call(C_tp_ctx, devices)
    .tp_state[[key]]
}

# chclust / hclust object from the seqdist vector the GPU returns (rioja builds the same fields from its C result);
# merge = rioja's .find.groups rule, computed in the library (union-find, O(n log n): the interpreted loop of repeated
# which.min is minutes at 25k bins)
.tp_dendro <- function(seqdist, labels) {
    n <- length(seqdist) + 1L
    structure(list(merge = .Call(C_tp_find_groups, as.numeric(seqdist)), height = sort(seqdist), seqdist = seqdist,
                   order = seq_len(n), labels = as.character(labels), method = "coniss",
                   call = quote(rioja::chclust(d = dist(pcs))), dist.method = "euclidean"),
              class = c("chclust", "hclust"))
}

# bad-column bookkeeping of load_mat after the GPU has flagged the columns
.tp_split <- function(bad, centromere_search) {
    n <- length(bad)
    idx <- which(bad)
    message(paste(length(idx), "bad columns found at position(s):"))
    message(paste(idx, collapse = " "))
    whole <- list(keep = which(!bad), bad_columns = as.character(idx))
    if (!centromere_search || length(idx) == 0L) return(whole)
    # the split itself (longest bad run, quirk Q3 kept) is the library's tp_centromere_split
    s <- .Call(C_tp_split, bad, FALSE)
    message(paste("centromere position:", s[[1L]][2L], s[[1L]][3L]))
    if (!s[[1L]][1L]) {
        message("longest stretch of bad rows/columns at the ends, not splitting the matrix.")
        return(whole)
    }
    list(p = list(keep = s[[2L]], bad_columns = s[[3L]]), q = list(keep = s[[4L]], bad_columns = s[[5L]]),
         centromere = s[[1L]][2L]:s[[1L]][3L])
}

# the numeric core of load_mat on the GPU: which bins stay (index lists; the matrix itself stays in HBM)
# A contact matrix given by its upper-triangle pixels (cooler dump / HiC-Pro): accepted wherever a matrix file is.
# sparse_counts(bin1, bin2, count, n_bins) from vectors, sparse_counts(path = ) for a three-column text file
# (n_bins = NULL: largest bin + 1).  A Matrix::sparseMatrix is accepted directly by TADpole() / load_mat().
sparse_counts <- function(bin1 = NULL, bin2 = NULL, count = NULL, n_bins = NULL, index_base = 0L, path = NULL) {
    if (is.null(path)) stopifnot(!is.null(bin1), !is.null(bin2), !is.null(count), !is.null(n_bins),
                                 length(bin1) == length(bin2), length(bin1) == length(count))
    structure(list(bin1 = as.integer(bin1), bin2 = as.integer(bin2), count = as.numeric(count),
                   n_bins = if (is.null(n_bins)) 0L else as.integer(n_bins), index_base = as.integer(index_base), path = path),
              class = "tadpole_pixels")
}

.tp_load <- function(ctx, mat_file, bad_frac, centromere_search) {
    if (inherits(mat_file, "sparseMatrix")) {                   # Matrix package: triplet form, 0-based slots i / j
        t <- methods::as(mat_file, "TsparseMatrix")
        mat_file <- sparse_counts(t@i, t@j, t@x, nrow(t), 0L)
    }
    if (inherits(mat_file, "tadpole_pixels")) {
        if (!is.null(mat_file$path)) .Call(C_tp_ingest_coo_file, ctx, path.expand(mat_file$path), mat_file$n_bins, mat_file$index_base)
        else .Call(C_tp_ingest_coo, ctx, mat_file$bin1, mat_file$bin2, mat_file$count, mat_file$n_bins, mat_file$index_base)
        bad <- .Call(C_tp_filter, ctx, NULL, as.numeric(bad_frac))
    } else if (is.character(mat_file)) {
        .Call(C_tp_ingest, ctx, path.expand(mat_file))          # the file's text is parsed on the GPU
        bad <- .Call(C_tp_filter, ctx, NULL, as.numeric(bad_frac))
    } else {
        bad <- .Call(C_tp_filter, ctx, as.matrix(mat_file) + 0, as.numeric(bad_frac))
    }
    structure(.tp_split(bad, centromere_search), n_bins = length(bad))
}

# mat[keep, keep] as the reference returns it: dimnames = original bin numbers, attr 'bad_columns'
.tp_part_matrix <- function(ctx, part) {
    m <- .Call(C_tp_get_filtered, ctx, as.integer(part$keep - 1L))
    dimnames(m) <- list(as.character(part$keep), as.character(part$keep))
    attr(m, "bad_columns") <- part$bad_columns
    m
}

# Same return value as the reference (R/TADpole.R:85,88-90): the filtered numeric matrix carrying attr 'bad_columns', or
# list(p = , q = , centromere = ) of such matrices.  (The plots of R/TADpole.R:24-53 are not drawn.)
load_mat <- function(mat_file, chr, start, end, resol, bad_frac = 0.01, centromere_search = FALSE) {
    ctx <- .tp_ctx()
    parts <- .tp_load(ctx, mat_file, bad_frac, centromere_search)
    if (is.null(parts$p)) return(.tp_part_matrix(ctx, parts))
    list(p = .tp_part_matrix(ctx, parts$p), q = .tp_part_matrix(ctx, parts$q), centromere = parts$centromere)
}

# one matrix or one arm: list(n_pcs, optimal_n_clusters, dendro, clusters, scores, labels_optimal)
.tp_pack_part <- function(res, part) {
    n_pcs <- res[[1L]]; n_clusters <- res[[2L]]; seqdist <- res[[3L]]; scores <- res[[4L]]
    dimnames(scores) <- list(as.character(seq_len(nrow(scores))), as.character(seq_len(ncol(scores))))
    message(paste("Optimal number of PCs:", n_pcs))
    message(paste("Optimal number of clusters:", n_clusters))
    levels <- which(!is.na(scores[n_pcs, ]))
    no_bad <- is.null(part$bad_columns)
    bad <- if (no_bad) integer(0) else as.integer(part$bad_columns)
    tabs <- .Call(C_tp_levels, seqdist, as.integer(levels), as.integer(part$keep), bad, no_bad)
    clusters <- lapply(tabs, function(m) data.frame(start = m[, 1L], end = m[, 2L]))
    names(clusters) <- as.character(levels)
    list(n_pcs = n_pcs, optimal_n_clusters = n_clusters, dendro = .tp_dendro(seqdist, part$keep),
         clusters = clusters, scores = scores,
         labels_optimal = .Call(C_tp_labels, seqdist, as.integer(n_clusters), as.integer(part$keep), bad, no_bad))
}

TADpole <- function(mat_file, max_pcs = 200, min_clusters = 2, bad_frac = 0.01,
                    chr, start, end, resol, centromere_search = FALSE) {
    ctx <- .tp_ctx()
    mat <- .tp_load(ctx, mat_file, bad_frac, centromere_search)
    if (!centromere_search) {
        res <- .Call(C_tp_call_arm, ctx, as.integer(mat$keep - 1L), as.integer(max_pcs), as.integer(min_clusters))
        r <- .tp_pack_part(res, mat)
        out <- structure(list(n_pcs = r$n_pcs, optimal_n_clusters = r$optimal_n_clusters, dendro = r$dendro,
                              clusters = r$clusters, scores = r$scores), class = "tadpole")
        attr(out, "resident") <- list(ctx = ctx, generation = res[[5L]], part = mat[c("keep", "bad_columns")])
        return(out)
    }
    if (is.null(mat$p)) stop("centromere_search = TRUE but load_mat did not split the matrix")
    # both arms in one .Call: on several GPUs the two halves of the devices work on the two arms at the same time
    both <- .Call(C_tp_call_arms, ctx, as.integer(mat$p$keep - 1L), as.integer(mat$q$keep - 1L),
                  as.integer(max_pcs), as.integer(min_clusters))
    names(both) <- c("p", "q")
    .tp_arms_object(both, mat)
}

# the tadpole object of a split chromosome (R/TADpole.R:376-442): both = list(p, q) of arm results (as C_tp_call_arm
# returns them), parts = list(p, q, centromere) of list(keep, bad_columns)
.tp_arms_object <- function(both, parts) {
    out <- structure(list(), class = "tadpole")
    joined <- integer(0)
    for (arm in c("p", "q")) {
        message(paste("Processing arm", arm))
        r <- .tp_pack_part(both[[arm]], parts[[arm]])
        out[[arm]] <- list(n_pcs = r$n_pcs, optimal_n_clusters = r$optimal_n_clusters, dendro = r$dendro,
                           cluster = r$clusters)
        joined <- c(joined, r$labels_optimal, rep(0L, length(parts$centromere)))
    }
    joined <- joined[seq_len(length(joined) - length(parts$centromere))]
    runs <- rle(joined)
    ends <- cumsum(runs$lengths)
    coord <- data.frame(start = c(1, ends[-length(ends)] + 1), end = ends)
    out$merging_arms <- coord[runs$values != 0, ]
    out
}

# one item of C_tp_call_batch_arms / C_tp_call_genome_arms: list(bad, centromere, p, q), each arm
# list(n_pcs, optimal_n_clusters, seqdist, scores, keep, bad_columns)
.tp_arms_batch_object <- function(r) {
    message(paste(sum(r[[1L]]), "bad columns found at position(s):"))
    message(paste(which(r[[1L]]), collapse = " "))
    message(paste("centromere position:", r[[2L]][1L], r[[2L]][length(r[[2L]])]))
    parts <- list(p = list(keep = r[[3L]][[5L]], bad_columns = r[[3L]][[6L]]),
                  q = list(keep = r[[4L]][[5L]], bad_columns = r[[4L]][[6L]]), centromere = r[[2L]])
    .tp_arms_object(list(p = r[[3L]], q = r[[4L]]), parts)
}

# TADpole() on a list of matrices (genome-wide use: one per chromosome), `inflight` calls per GPU kept in flight by the
# library's own threads over every GPU of options(tadpole.gpus); same objects, same order, as calling TADpole() on each
# centromere_search = TRUE: every matrix is split at its centromere and both arms run in those threads; a matrix that does
# not split stops, as TADpole(centromere_search = TRUE) does
TADpole_batch <- function(mats, max_pcs = 200, min_clusters = 2, bad_frac = 0.01, inflight = 8L, centromere_search = FALSE) {
    ctx <- .tp_ctx()
    mats <- lapply(mats, function(m) if (is.character(m)) {
        .Call(C_tp_ingest, ctx, path.expand(m)); .Call(C_tp_ingested_matrix, ctx) } else as.matrix(m) + 0)
    if (centromere_search) {
        res <- .Call(C_tp_call_batch_arms, ctx, mats, as.integer(max_pcs), as.integer(min_clusters), as.numeric(bad_frac),
                     as.integer(inflight))
        return(lapply(res, function(r) {
            if (is.character(r)) stop(r)
            .tp_arms_batch_object(r)
        }))
    }
    res <- .Call(C_tp_call_batch, ctx, mats, as.integer(max_pcs), as.integer(min_clusters), as.numeric(bad_frac),
                 as.integer(inflight))
    lapply(res, function(r) {
        if (is.character(r)) stop(r)
        .tp_batch_object(r)
    })
}

# the tadpole object of one item of a batch (C_tp_call_batch, C_tp_call_genome)
.tp_batch_object <- function(r) {
    bad <- r[[1L]]; scores <- r[[5L]]; keep <- which(!bad)
    dimnames(scores) <- list(as.character(seq_len(nrow(scores))), as.character(seq_len(ncol(scores))))
    clusters <- lapply(r[[7L]], function(m) data.frame(start = m[, 1L], end = m[, 2L]))
    names(clusters) <- as.character(r[[6L]])
    structure(list(n_pcs = r[[2L]], optimal_n_clusters = r[[3L]], dendro = .tp_dendro(r[[4L]], keep),
                   clusters = clusters, scores = scores), class = "tadpole")
}

# chromosome names and bins per chromosome of a bin table: a path (HiC-Pro *_abs.bed, `cooler dump -t bins`, header
# line allowed), a data.frame with the chromosome of every bin in column 1, or a named integer vector of bin counts
.tp_bin_table <- function(bins) {
    if (is.numeric(bins) && !is.null(names(bins))) {
        if (anyDuplicated(names(bins))) stop("a chromosome appears twice in the bin table")
        return(list(names = names(bins), n = as.integer(bins)))
    }
    if (is.character(bins) && length(bins) == 1L) {
        first <- strsplit(readLines(bins, n = 1L), "[ \t]+")[[1L]]
        header <- first[1L] == "chrom" || (length(first) >= 2L && !grepl("^[+-]?[0-9]+$", first[2L]))
        bins <- utils::read.table(path.expand(bins), header = FALSE, skip = if (header) 1L else 0L, sep = "",
                                  colClasses = "character", comment.char = "", fill = TRUE)
    }
    runs <- rle(as.character(bins[[1L]]))
    if (anyDuplicated(runs$values))
        stop("chromosome ", runs$values[anyDuplicated(runs$values)], " reappears after another chromosome in the bin table")
    list(names = runs$values, n = as.integer(runs$lengths))
}

# TADpole() on every chromosome of one genome-wide pixel list: pixels = sparse_counts(bin1, bin2, count, index_base =)
# or sparse_counts(path = , index_base = 1L) with GLOBAL bin ids (HiC-Pro *.matrix, cooler dump -t pixels), bins = the
# bin table.  The pixels are split by chromosome on the GPU and each chromosome's dense matrix exists only in HBM while
# its call runs.  A named list of tadpole objects (bin-table order, or chroms order), attr(, "failed") = the messages
# of the chromosomes whose call failed.  centromere_search = TRUE: as TADpole(centromere_search = TRUE) on each
# chromosome; one that does not split fails.
TADpole_genome <- function(pixels, bins, chroms = NULL, max_pcs = 200, min_clusters = 2, bad_frac = 0.01, inflight = 8L,
                           centromere_search = FALSE) {
    stopifnot(inherits(pixels, "tadpole_pixels"))
    ctx <- .tp_ctx()
    tab <- .tp_bin_table(bins)
    sel <- if (is.null(chroms)) tab$names else as.character(chroms)
    idx <- match(sel, tab$names)
    if (anyNA(idx)) stop("unknown chromosome(s): ", paste(sel[is.na(idx)], collapse = ", "))
    g <- if (is.null(pixels$path)) .Call(C_tp_genome, ctx, tab$n, pixels$bin1, pixels$bin2, pixels$count, pixels$index_base)
         else .Call(C_tp_genome_file, ctx, tab$n, path.expand(pixels$path), pixels$index_base)
    res <- if (centromere_search)
        .Call(C_tp_call_genome_arms, ctx, g[[1L]], as.integer(idx - 1L), as.integer(max_pcs), as.integer(min_clusters),
              as.numeric(bad_frac), as.integer(inflight), FALSE)
    else .Call(C_tp_call_genome, ctx, g[[1L]], as.integer(idx - 1L), as.integer(max_pcs), as.integer(min_clusters),
               as.numeric(bad_frac), as.integer(inflight), TRUE)
    out <- list()
    failed <- list()
    for (i in seq_along(sel)) {
        message(paste("Processing chromosome", sel[i]))
        r <- res[[i]]
        if (is.character(r)) { failed[[sel[i]]] <- r; next }
        if (centromere_search) { out[[sel[i]]] <- .tp_arms_batch_object(r); next }
        message(paste(sum(r[[1L]]), "bad columns found at position(s):"))
        message(paste(which(r[[1L]]), collapse = " "))
        message(paste("Optimal number of PCs:", r[[2L]]))
        message(paste("Optimal number of clusters:", r[[3L]]))
        out[[sel[i]]] <- .tp_batch_object(r)
    }
    attr(out, "failed") <- failed
    out
}

# the n_pcs sweep again with another max_pcs / min_clusters on the PC scores that are still on the GPU
tadpole_recall <- function(tadpole, max_pcs = 200, min_clusters = 2) {
    h <- attr(tadpole, "resident")
    if (is.null(h)) stop("this tadpole object carries no device handle")
    # the shim stops when the context has been used for another matrix since (generation), and sizes every buffer from
    # the context, never from this object
    res <- .Call(C_tp_recall, h$ctx, h$generation, as.integer(max_pcs), as.integer(min_clusters))
    r <- .tp_pack_part(res, h$part)
    out <- structure(list(n_pcs = r$n_pcs, optimal_n_clusters = r$optimal_n_clusters, dendro = r$dendro,
                          clusters = r$clusters, scores = r$scores), class = "tadpole")
    h$generation <- res[[5L]]               # the sweep state was replaced: `tadpole` itself is stale from here on
    attr(out, "resident") <- h
    out
}

# dendrogram of the candidate that clusters on the first n_pcs components (what CH_map / plot_hierarchy browse)
tadpole_dendro <- function(tadpole, n_pcs) {
    h <- attr(tadpole, "resident")
    if (is.null(h)) stop("this tadpole object carries no device handle")
    .tp_dendro(.Call(C_tp_dendro, h$ctx, h$generation, as.integer(n_pcs)), h$part$keep)
}

.tp_bin_index <- function(bed, size) {
    lab <- integer(size)
    for (i in seq_len(nrow(bed))) {
        pos <- seq(bed[i, 2], bed[i, 3]) - bed[1, 2] + 1
        lab[pos] <- i
    }
    lab
}

.tp_padded_labels <- function(bed_x, bed_y) {
    if (nrow(bed_x) != nrow(bed_y)) stop("Both calls must have the same number of TADs.")
    sx <- bed_x[1, 2]; sy <- bed_y[1, 2]; ex <- bed_x[nrow(bed_x), 3]; ey <- bed_y[nrow(bed_y), 3]
    tx <- .tp_bin_index(bed_x, ex - sx + 1)
    ty <- .tp_bin_index(bed_y, ey - sy + 1)
    tx <- c(rep(1L, max(0, sx - sy)), tx, rep(max(tx), max(0, ey - ex)))
    ty <- c(rep(1L, max(0, sy - sx)), ty, rep(max(ty), max(0, ex - ey)))
    stopifnot(length(tx) == length(ty))
    list(x = tx, y = ty, pad_left_y = max(0, sy - sx), pad_right_y = max(0, ex - ey))
}

diffT <- function(bed_x, bed_y) {
    lab <- .tp_padded_labels(bed_x, bed_y)
    .Call(C_tp_difft, .tp_ctx(), as.integer(lab$x), as.integer(lab$y), length(lab$x), 1L)
}

# random_bed: one draw, generated on the GPU (uniform subsets of bins[-1], as sample() draws them)
random_bed <- function(bed, bad_columns = NULL, seed = sample.int(.Machine$integer.max, 1L)) {
    size <- bed[nrow(bed), 3] - bed[1, 2] + 1
    bad <- if (is.null(bad_columns)) integer(0) else as.integer(bad_columns)
    res <- .Call(C_tp_difft_null, .tp_ctx(), rep(1L, size), 0L, 0L, nrow(bed), bad, as.numeric(seed), 1L)
    borders <- res[[1L]][, 1L] + bed[1, 2]
    data.frame(chrom = bed[, 1], start = c(bed[1, 2], borders - 1), end = c(borders - 2, bed[1, 2] + size - 1))
}

# diffT(bed_x, random_bed(bed_y, bad_columns)) for nperm random partitions, drawn and scored on the GPU
diffT_null <- function(bed_x, bed_y = bed_x, nperm = 1000L, bad_columns = NULL, seed = 0) {
    lab <- .tp_padded_labels(bed_x, bed_y)
    bad <- if (is.null(bad_columns)) integer(0) else as.integer(bad_columns)
    res <- .Call(C_tp_difft_null, .tp_ctx(), as.integer(lab$x), as.integer(lab$pad_left_y), as.integer(lab$pad_right_y),
                 nrow(bed_y), bad, as.numeric(seed), as.integer(nperm))
    list(borders = t(res[[1L]]) + bed_y[1, 2], totals = res[[2L]], curves = t(res[[3L]]))
}
