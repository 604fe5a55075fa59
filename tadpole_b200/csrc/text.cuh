// text.cuh -- text input shared by ingest.cu and pairs.cu: a host buffer or a file read by byte range, uploaded to the
// device through the context's two pinned buffers, and the byte offsets of its line ends found there (ingest.cu).
#pragma once
#include "common.cuh"
#include <errno.h>
#include <unistd.h>

struct TextSource {
    const unsigned char *mem = nullptr;
    int fd = -1;
    size_t size = 0;
    int fetch(size_t off, size_t len, void *dst) const {
        if (mem) { memcpy(dst, mem + off, len); return TP_OK; }
        size_t got = 0;
        while (got < len) {
            ssize_t k = pread(fd, (char *)dst + got, len - got, (off_t)(off + got));
            if (k < 0 && errno == EINTR) continue;
            if (k <= 0) { tp_set_error("tp_ingest_tsv_file: read failed at byte %zu (%s)", off + got, k < 0 ? strerror(errno) : "unexpected end of file"); return TP_ERR_ARG; }
            got += (size_t)k;
        }
        return TP_OK;
    }
};

// open `path` as a regular file (the caller closes src->fd)
int open_text_file(const char *path, const char *who, TextSource *src);
// Upload bytes [off, off + nbytes) of src through the two pinned buffers and count its rows: on return *text_out is the
// device copy (ctx->itext) with a newline and readable padding appended, offs[0..nb] the newline offsets per 16 KB tile
// (offs[nb] = rows, the appended newline included).  Synchronises the stream once, after the count.
int text_rows(tp_ctx *ctx, const TextSource &src, size_t off, size_t nbytes, unsigned char **text_out, int *nb_out,
              long long **offs_out, long long *nrows_out);
// the byte offset of every row end of what text_rows uploaded, in order, into ctx->irows (stream ordered, no sync)
int text_line_ends(tp_ctx *ctx, const unsigned char *text, size_t nbytes, int nb, const long long *offs, long long nrows,
                   long long **row_end_out);
