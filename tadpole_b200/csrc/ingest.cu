// ingest.cu -- input side of load_mat (reference R/TADpole.R:17): a header-less, tab-separated N x N text matrix
// becomes the N x N FP64 matrix in HBM that stage 1 (filter.cu) reads, without a host-side parse.
//
//   mat <- bigmemory::read.big.matrix(mat_file, type = 'double', sep = '\t')[, ]          (R/TADpole.R:17)
//
// The text is what crosses PCIe (2-3 bytes per count instead of 8 per double; 1.5 GB instead of 5 GB at N = 25 000);
// it is read through two pinned staging buffers so that the file read and the upload overlap.  On the device:
//   1. newline_count_kernel / newline_scan_kernel / newline_pos_kernel: byte offsets of the row ends (HBM-bound byte
//      pass, 16-byte loads, vector compares, block scan; the text is read twice);
//   2. parse_rows_kernel: one CTA per row; 4 KB tiles of the row staged in shared memory, a block scan of the
//      separator counts gives every thread the column of the first field that starts in its 16 bytes, each field is
//      converted with np_parse_field (numparse.cuh: exact decimal -> binary64) and stored at out[row * N + column];
//      a row with a field count != N raises the "not square" error.
// Fields the device cannot decide exactly (> 19 significant digits on a rounding boundary, or a spelling the device
// grammar does not know) are listed, converted by strtod on the host and scattered back -- that list is empty for
// count matrices and for the usual 6-17 digit normalised matrices.  Algorithmic traffic: file bytes read once + 8 N^2 written.
#include "common.cuh"
#include "numparse.cuh"
#include <errno.h>
#include <fcntl.h>
#include <stdlib.h>
#include <sys/stat.h>
#include <unistd.h>
#include <chrono>

static const uint64_t h_pow5[] = {
#include "pow5_table.inc"
};
__device__ const uint64_t d_pow5[] = {
#include "pow5_table.inc"
};
#define P10_LIST 1e0, 1e1, 1e2, 1e3, 1e4, 1e5, 1e6, 1e7, 1e8, 1e9, 1e10, 1e11, 1e12, 1e13, 1e14, 1e15, 1e16, 1e17, 1e18, 1e19, 1e20, 1e21, 1e22
static const double h_pow10[23] = {P10_LIST};
__device__ const double d_pow10[23] = {P10_LIST};

#define IG_THREADS 256
#define IG_SPAN 64                                  // bytes per thread in the newline passes
#define IG_TILE (IG_THREADS * IG_SPAN)              // 16 KB per CTA
#define PR_TILE (IG_THREADS * 16)                   // 4 KB of a row per step of the parse kernel
#define PR_HALO 80                                  // a field may run this far past the tile it starts in
#define PR_MAXTOK 64
#define IG_PAD (PR_TILE + 256)                      // readable bytes after the text

// exclusive scan of one int per thread over the CTA; *total_out = sum (valid for every thread)
__device__ __forceinline__ int block_excl_scan(int v, int *s_warp, int *total_out) {
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    int inc = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        int t = __shfl_up_sync(0xffffffffu, inc, o);
        if (lane >= o) inc += t;
    }
    __syncthreads();                                 // s_warp may still be read from the previous call
    if (lane == 31) s_warp[wid] = inc;
    __syncthreads();
    int base = 0, tot = 0;
#pragma unroll
    for (int w = 0; w < IG_THREADS / 32; w++) {
        const int x = s_warp[w];
        if (w < wid) base += x;
        tot += x;
    }
    *total_out = tot;
    return base + inc - v;
}

__device__ __forceinline__ int count_eq16(uint4 v, unsigned pat) {
    return (__popc(__vcmpeq4(v.x, pat)) + __popc(__vcmpeq4(v.y, pat)) + __popc(__vcmpeq4(v.z, pat)) +
            __popc(__vcmpeq4(v.w, pat))) >> 3;
}

// newlines per 16 KB tile; bytes at or past `limit` do not count
__global__ void __launch_bounds__(IG_THREADS)
newline_count_kernel(const unsigned char *__restrict__ text, long long limit, int *__restrict__ counts) {
    __shared__ int s_warp[IG_THREADS / 32];
    const long long base = (long long)blockIdx.x * IG_TILE;
    int c = 0;
#pragma unroll
    for (int j = 0; j < IG_SPAN / 16; j++) {
        const long long off = base + ((long long)j * IG_THREADS + threadIdx.x) * 16;
        if (off + 16 <= limit) c += count_eq16(*(const uint4 *)(text + off), 0x0a0a0a0au);
        else for (long long p = off; p < limit; p++) c += text[p] == '\n';
    }
    for (int o = 16; o > 0; o >>= 1) c += __shfl_xor_sync(0xffffffffu, c, o);
    if ((threadIdx.x & 31) == 0) s_warp[threadIdx.x >> 5] = c;
    __syncthreads();
    if (threadIdx.x == 0) {
        int t = 0;
        for (int w = 0; w < IG_THREADS / 32; w++) t += s_warp[w];
        counts[blockIdx.x] = t;
    }
}

// exclusive scan of the tile counts (one CTA, chunks of 256); offs[nb] = total
__global__ void __launch_bounds__(IG_THREADS)
newline_scan_kernel(const int *__restrict__ counts, int nb, long long *__restrict__ offs) {
    __shared__ int s_warp[IG_THREADS / 32];
    long long carry = 0;
    for (int b0 = 0; b0 < nb; b0 += IG_THREADS) {
        const int b = b0 + threadIdx.x;
        const int v = b < nb ? counts[b] : 0;
        int tot;
        const int ex = block_excl_scan(v, s_warp, &tot);
        if (b < nb) offs[b] = carry + ex;
        carry += tot;
    }
    if (threadIdx.x == 0) offs[nb] = carry;
}

// byte offset of every newline, in order
__global__ void __launch_bounds__(IG_THREADS)
newline_pos_kernel(const unsigned char *__restrict__ text, long long limit, const long long *__restrict__ offs,
                   long long *__restrict__ row_end) {
    __shared__ __align__(16) unsigned char tile[IG_TILE];
    __shared__ int s_warp[IG_THREADS / 32];
    const long long base = (long long)blockIdx.x * IG_TILE;
#pragma unroll
    for (int j = 0; j < IG_SPAN / 16; j++) {
        const int v = j * IG_THREADS + threadIdx.x;
        const long long off = base + (long long)v * 16;
        uint4 x = make_uint4(0, 0, 0, 0);
        if (off < limit) x = *(const uint4 *)(text + off);           // the pad after the text is readable
        *(uint4 *)(tile + v * 16) = x;
    }
    __syncthreads();
    const unsigned char *mine = tile + threadIdx.x * IG_SPAN;
    const long long p0 = base + (long long)threadIdx.x * IG_SPAN;
    int c = 0;
    if (p0 + IG_SPAN <= limit) {
#pragma unroll
        for (int j = 0; j < IG_SPAN / 16; j++) c += count_eq16(*(const uint4 *)(mine + 16 * j), 0x0a0a0a0au);
    } else {
        for (int j = 0; j < IG_SPAN; j++) c += (p0 + j < limit) && mine[j] == '\n';
    }
    int tot;
    int ex = block_excl_scan(c, s_warp, &tot);
    if (c) {
        long long o = offs[blockIdx.x] + ex;
        for (int j = 0; j < IG_SPAN; j++)
            if ((p0 + j < limit) && mine[j] == '\n') row_end[o++] = p0 + j;
    }
}

struct SlowTok { long long off; unsigned row, col; };

// status words: [0..1] one 64-bit word, (INT_MAX - first row with a wrong field count) << 32 | its field count; [2] slow-list overflow
__global__ void __launch_bounds__(IG_THREADS)
parse_rows_kernel(const unsigned char *__restrict__ text, const long long *__restrict__ row_end, int nrows, int ncols,
                  unsigned sep, double *__restrict__ out, SlowTok *__restrict__ slow, unsigned *__restrict__ slow_count,
                  unsigned slow_cap, int *__restrict__ status) {
    __shared__ __align__(16) unsigned char tile[16 + PR_TILE + PR_HALO];
    __shared__ int s_warp[IG_THREADS / 32];
    const int r = blockIdx.x;
    const long long s = r ? row_end[r - 1] + 1 : 0;
    const long long e = row_end[r];
    const long long a0 = s & ~15LL;
    double *orow = out + (size_t)r * ncols;
    int field_base = 0;
    for (long long t0 = a0; t0 < e || t0 == a0; t0 += PR_TILE) {
        // stage [t0 - 16, t0 + PR_TILE + PR_HALO)
        *(uint4 *)(tile + 16 + threadIdx.x * 16) = *(const uint4 *)(text + t0 + threadIdx.x * 16);
        if (threadIdx.x < PR_HALO / 16) *(uint4 *)(tile + 16 + PR_TILE + threadIdx.x * 16) = *(const uint4 *)(text + t0 + PR_TILE + threadIdx.x * 16);
        if (threadIdx.x == PR_HALO / 16) *(uint4 *)tile = t0 >= 16 ? *(const uint4 *)(text + t0 - 16) : make_uint4(0, 0, 0, 0);
        __syncthreads();
        const unsigned char *mine = tile + 16 + threadIdx.x * 16;
        const long long p0 = t0 + threadIdx.x * 16;
        unsigned sepmask = 0, valid = 0;
#pragma unroll
        for (int j = 0; j < 16; j++) {
            const bool v = p0 + j >= s && p0 + j < e;
            valid |= (unsigned)v << j;
            sepmask |= (unsigned)(v && mine[j] == sep) << j;
        }
        int tot;
        int f = field_base + block_excl_scan(__popc(sepmask), s_warp, &tot);
        field_base += tot;
        // a field starts at the first byte of the row and after every separator
        unsigned starts = (sepmask << 1) & valid;
        if (p0 > s && p0 < e && mine[-1] == sep) starts |= 1;
        if (p0 <= s && s < p0 + 16 && s < e) starts |= 1u << (int)(s - p0);
        unsigned todo = starts;
        while (todo) {
            const int j = __ffs(todo) - 1;
            todo &= todo - 1;
            const int col = f + __popc(sepmask & ((1u << j) - 1));
            const unsigned char *tok = mine + j;
            const long long room = e - (p0 + j);
            const int lim = room < PR_MAXTOK ? (int)room : PR_MAXTOK;
            int len = 0;
            while (len < lim && tok[len] != sep) len++;
            if (col < ncols) {
                double v;
                int st = (len == PR_MAXTOK && room > PR_MAXTOK) ? NP_HOST : np_parse_field(tok, len, d_pow10, d_pow5, &v);
                if (st == NP_OK) orow[col] = v;
                else {
                    const unsigned k = atomicAdd(slow_count, 1u);
                    if (k < slow_cap) { slow[k].off = p0 + j; slow[k].row = r; slow[k].col = col; }
                    else status[2] = 1;
                    orow[col] = __longlong_as_double(0x7ff8000000000000LL);
                }
            }
        }
        __syncthreads();
    }
    // an empty row is one empty field; a row ending in a separator has an empty last field
    if (threadIdx.x == 0) {
        int nfields = field_base + 1;
        if (e == s || text[e - 1] == sep) {
            if (nfields - 1 < ncols && nfields >= 1) orow[nfields - 1] = __longlong_as_double(0x7ff8000000000000LL);
        }
        if (nfields != ncols)          // the lowest offending row wins: (INT_MAX - row) in the high word, its field count below
            atomicMax((unsigned long long *)status, ((unsigned long long)(unsigned)(0x7fffffff - r) << 32) | (unsigned)nfields);
    }
}

__global__ void scatter_kernel(double *__restrict__ out, const long long *__restrict__ idx, const double *__restrict__ val, int m) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < m) out[idx[i]] = val[i];
}

// ---- sparse input: pixels (bin1, bin2, count) of the upper triangle -------------------------------------------------
// status64[0]: lowest index of an entry whose bins are outside [0, n) (~0 = none); status64[1]: entries below the diagonal
// (ignored: the reference reads the upper triangle only, Matrix::forceSymmetric(uplo = 'U'), R/TADpole.R:20);
// status64[2]: lowest index (>= 1) of a text row that is not "int sep int sep number"; status64[3]: largest bin seen + 1;
// status64[4]: row 0 is not such a row (a header line).
__global__ void __launch_bounds__(256)
coo_scatter_kernel(double *__restrict__ out, int n, const int *__restrict__ b1, const int *__restrict__ b2,
                   const double *__restrict__ v, unsigned m, int base, unsigned long long first,
                   unsigned long long *__restrict__ status64) {
    const unsigned e = blockIdx.x * blockDim.x + threadIdx.x;
    bool below = false;
    if (e < m) {
        const long long i = (long long)b1[e] - base, j = (long long)b2[e] - base;
        if (i < 0 || j < 0 || i >= n || j >= n) atomicMin(status64, first + e);
        else if (i > j) below = true;
        else atomicAdd(out + (size_t)i * n + j, v[e]);      // duplicates add up, as Matrix::sparseMatrix(i, j, x) has them
    }
    const unsigned bal = __ballot_sync(0xffffffffu, below);
    if (bal && (threadIdx.x & 31) == 0) atomicAdd(status64 + 1, (unsigned long long)__popc(bal));
}

// one text row per thread: "bin1 <sep> bin2 <sep> count"; the count goes through np_parse_field like a matrix field
__global__ void __launch_bounds__(256)
coo_parse_kernel(const unsigned char *__restrict__ text, const long long *__restrict__ row_end, unsigned nrows, unsigned sep,
                 double *__restrict__ v, int *__restrict__ b1, int *__restrict__ b2, SlowTok *__restrict__ slow,
                 unsigned *__restrict__ slow_count, unsigned slow_cap, unsigned long long *__restrict__ status64) {
    const unsigned r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= nrows) return;
    long long p = r ? row_end[r - 1] + 1 : 0;
    const long long e = row_end[r];
    bool ok = true;
    int bins[2] = {0, 0};
#pragma unroll
    for (int f = 0; f < 2; f++) {
        while (p < e && text[p] == ' ' && sep != ' ') p++;       // blanks around a bin, unless the blank separates
        long long x = 0;
        int nd = 0;
        while (p < e && text[p] - '0' < 10u && nd < 10) { x = x * 10 + (text[p] - '0'); p++; nd++; }
        while (p < e && text[p] == ' ' && sep != ' ') p++;
        ok = ok && nd > 0 && nd < 10 && p < e && text[p] == sep;
        bins[f] = (int)x;
        p++;
    }
    long long q = p;
    while (ok && q < e && text[q] != sep) q++;
    ok = ok && q == e && p <= e;
    if (!ok) {                                   // row 0 may be a header line (cooler dump --header): flagged apart
        if (r == 0) status64[4] = 1; else atomicMin(status64 + 2, (unsigned long long)r);
        b1[r] = b2[r] = 0; v[r] = 0.0;
        return;
    }
    double val;
    if (np_parse_field(text + p, (int)(e - p), d_pow10, d_pow5, &val) != NP_OK) {
        const unsigned k = atomicAdd(slow_count, 1u);
        if (k < slow_cap) { slow[k].off = p; slow[k].row = r; slow[k].col = 2; }
        else atomicMin(status64 + 2, ~0ull - 1);                 // list overflow
        val = 0.0;
    }
    b1[r] = bins[0]; b2[r] = bins[1]; v[r] = val;
    const int mx = bins[0] > bins[1] ? bins[0] : bins[1];
    atomicMax(status64 + 3, (unsigned long long)mx + 1);
}

__global__ void scatter_f64_kernel(double *__restrict__ out, const unsigned *__restrict__ idx, const double *__restrict__ val, int m) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < m) out[idx[i]] = val[i];
}

// ---- host side -----------------------------------------------------------------------------------------------------
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

// Upload the text (through the two pinned buffers) and count its rows: on return *text_out is the device copy with a
// newline and IG_PAD readable bytes appended, offs[0..nb] the newline offsets per 16 KB tile (offs[nb] = rows).
static int text_rows(tp_ctx *ctx, const TextSource &src, const char *who, unsigned char **text_out, size_t *nbytes_out,
                     int *nb_out, long long **offs_out, long long *nrows_out) {
    cudaStream_t st = ctx->stream;
    // drop trailing newlines / blanks: the last row ends at the single '\n' appended on the device
    size_t nbytes = src.size;
    {
        unsigned char tail[4096];
        while (nbytes > 0) {
            const size_t k = nbytes < sizeof(tail) ? nbytes : sizeof(tail);
            TP_TRY(src.fetch(nbytes - k, k, tail));
            size_t j = k;
            while (j > 0 && (tail[j - 1] == '\n' || tail[j - 1] == '\r' || tail[j - 1] == ' ')) j--;
            nbytes -= k - j;
            if (j > 0) break;
        }
    }
    if (nbytes == 0) { tp_set_error("%s: the input holds no data", who); return TP_ERR_ARG; }
    if (nbytes >= ((size_t)1 << 40)) { tp_set_error("%s: input too large", who); return TP_ERR_ARG; }
    const long long limit = (long long)nbytes + 1;
    TP_TRY(ctx->itext.reserve(nbytes + IG_PAD + 16));
    unsigned char *text = ctx->itext.as<unsigned char>();
    TP_CUDA(cudaMemsetAsync(text + nbytes, '\n', IG_PAD + 16, st));
    // upload through two pinned buffers: the read of chunk c + 1 overlaps the copy of chunk c
    const size_t CH = (size_t)32 << 20;
    if (!ctx->ipin[0]) {
        for (int b = 0; b < 2; b++) {
            TP_CUDA(cudaMallocHost(&ctx->ipin[b], CH));
            TP_CUDA(cudaEventCreateWithFlags(&ctx->ipin_ev[b], cudaEventDisableTiming));
        }
    }
    int c = 0;
    for (size_t off = 0; off < nbytes; off += CH, c++) {
        const int b = c & 1;
        const size_t k = nbytes - off < CH ? nbytes - off : CH;
        if (c >= 2) TP_CUDA(cudaEventSynchronize(ctx->ipin_ev[b]));
        TP_TRY(src.fetch(off, k, ctx->ipin[b]));
        TP_CUDA(cudaMemcpyAsync(text + off, ctx->ipin[b], k, cudaMemcpyHostToDevice, st));
        TP_CUDA(cudaEventRecord(ctx->ipin_ev[b], st));
    }
    TP_MARK(ctx, EV_INGEST0);
    const int nb = (int)((limit + IG_TILE - 1) / IG_TILE);
    TP_TRY(ctx->icounts.reserve((size_t)nb * sizeof(int) + (size_t)(nb + 1) * sizeof(long long) + 64));
    long long *offs = ctx->icounts.as<long long>();
    int *counts = (int *)(offs + nb + 1);
    newline_count_kernel<<<nb, IG_THREADS, 0, st>>>(text, limit, counts);
    newline_scan_kernel<<<1, IG_THREADS, 0, st>>>(counts, nb, offs);
    TP_CUDA(cudaGetLastError());
    long long nrows_ll = 0;
    TP_CUDA(cudaMemcpyAsync(&nrows_ll, offs + nb, sizeof(long long), cudaMemcpyDeviceToHost, st));
    TP_CUDA(tp_stream_sync(ctx));
    ctx->launches += 2;
    *text_out = text; *nbytes_out = nbytes; *nb_out = nb; *offs_out = offs; *nrows_out = nrows_ll;
    return TP_OK;
}

// One field of the text that the device left to the host: [off, end of field) converted by strtod.
static int host_field(const TextSource &src, size_t nbytes, size_t off, int sep, std::vector<char> &buf, double *out, const char *who,
                      unsigned row, unsigned col) {
    size_t len = 0;
    for (;;) {                                   // find the end of the field
        const size_t want = buf.size() - 1;
        const size_t k = nbytes - off < want ? nbytes - off : want;
        TP_TRY(src.fetch(off, k, buf.data()));
        len = 0;
        while (len < k && buf[len] != (char)sep && buf[len] != '\n') len++;
        if (len < k || k == nbytes - off) break;
        buf.resize(buf.size() * 2);
    }
    while (len > 0 && (buf[len - 1] == '\r' || buf[len - 1] == ' ')) len--;
    buf[len] = 0;
    char *endp = nullptr;
    const double v = strtod(buf.data(), &endp);
    if (endp == buf.data() || *endp != 0) {
        if (len > 40) buf[40] = 0;
        tp_set_error("%s: row %u, column %u: '%s' is not a number", who, row + 1, col + 1, buf.data());
        return TP_ERR_ARG;
    }
    *out = v;
    return TP_OK;
}

static int ingest_core(tp_ctx *ctx, const TextSource &src, int sep, int *n_out) {
    TP_ARG(sep > 0 && sep < 128 && sep != '\n' && sep != '\r' && sep != '.' && sep != '-' && sep != '+', "tp_ingest_tsv: bad separator");
    TP_CUDA(cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->stream;
    const auto t_begin = std::chrono::steady_clock::now();
    unsigned char *text = nullptr;
    size_t nbytes = 0;
    int nb = 0;
    long long *offs = nullptr, nrows_ll = 0;
    TP_TRY(text_rows(ctx, src, "tp_ingest_tsv", &text, &nbytes, &nb, &offs, &nrows_ll));
    const long long limit = (long long)nbytes + 1;
    TP_ARG(nrows_ll >= 2, "tp_ingest_tsv: the matrix must have at least 2 rows");
    TP_ARG(nrows_ll <= 200000, "tp_ingest_tsv: more than 200000 rows");
    const int n = (int)nrows_ll;
    const unsigned slow_cap = 1u << 20;
    TP_TRY(ctx->irows.reserve((size_t)n * sizeof(long long)));
    TP_TRY(ctx->islow.reserve((size_t)slow_cap * sizeof(SlowTok) + 64));
    TP_TRY(ctx->raw_own.reserve((size_t)n * n * sizeof(double)));
    long long *row_end = ctx->irows.as<long long>();
    int *status = ctx->islow.as<int>();                 // 16 ints of status, then the list
    unsigned *slow_count = (unsigned *)(status + 8);
    SlowTok *slow = (SlowTok *)(status + 16);
    double *out = ctx->raw_own.as<double>();
    TP_CUDA(cudaMemsetAsync(status, 0, 64, st));
    newline_pos_kernel<<<nb, IG_THREADS, 0, st>>>(text, limit, offs, row_end);
    parse_rows_kernel<<<n, IG_THREADS, 0, st>>>(text, row_end, n, n, (unsigned)sep, out, slow, slow_count, slow_cap, status);
    TP_CUDA(cudaGetLastError());
    ctx->launches += 2;
    TP_MARK(ctx, EV_INGEST1);
    int hstat[16];
    TP_CUDA(cudaMemcpyAsync(hstat, status, 64, cudaMemcpyDeviceToHost, st));
    TP_CUDA(tp_stream_sync(ctx));
    ctx->raw = nullptr; ctx->n = 0;
    ctx->have_X = ctx->have_C = ctx->have_scores = ctx->have_sweep = false;
    if (hstat[1]) {                                         // little endian: hstat[1] is the high word
        tp_set_error("tp_ingest_tsv: row %d has %d fields but the file has %d rows; a square, header-less, "
                     "separator-delimited matrix is expected (R/TADpole.R:17)", 0x7fffffff - hstat[1] + 1, hstat[0], n);
        return TP_ERR_ARG;
    }
    if (hstat[2]) {
        tp_set_error("tp_ingest_tsv: more than %u fields need the host conversion path", slow_cap);
        return TP_ERR_ARG;
    }
    const unsigned nslow = (unsigned)hstat[8];
    if (nslow) {
        std::vector<SlowTok> list(nslow);
        TP_CUDA(cudaMemcpy(list.data(), slow, (size_t)nslow * sizeof(SlowTok), cudaMemcpyDeviceToHost));
        std::vector<long long> idx(nslow);
        std::vector<double> val(nslow);
        std::vector<char> buf(4096 + 1);
        for (unsigned i = 0; i < nslow; i++) {
            double v = 0.0;
            TP_TRY(host_field(src, nbytes, (size_t)list[i].off, sep, buf, &v, "tp_ingest_tsv", list[i].row, list[i].col));
            idx[i] = (long long)list[i].row * n + list[i].col;
            val[i] = v;
        }
        // reuse the slow list's memory for the scatter operands
        long long *didx = (long long *)slow;
        double *dval = (double *)(didx + nslow);
        TP_CUDA(cudaMemcpyAsync(didx, idx.data(), (size_t)nslow * sizeof(long long), cudaMemcpyHostToDevice, st));
        TP_CUDA(cudaMemcpyAsync(dval, val.data(), (size_t)nslow * sizeof(double), cudaMemcpyHostToDevice, st));
        scatter_kernel<<<(nslow + 255) / 256, 256, 0, st>>>(out, didx, dval, (int)nslow);
        TP_CUDA(cudaGetLastError());
        TP_CUDA(tp_stream_sync(ctx));
        ctx->launches += 1;
    }
    ctx->raw = out;
    ctx->n = n;
    ctx->colmajor = 0;
    ctx->ingested_n = n;
    ctx->generation++;
    float ms = 0.f;
    cudaEventElapsedTime(&ms, ctx->ev[EV_INGEST0], ctx->ev[EV_INGEST1]);
    ctx->ingest_stats[0] = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t_begin).count();
    ctx->ingest_stats[1] = ms;
    ctx->ingest_stats[2] = (double)nbytes;
    ctx->ingest_stats[3] = (double)nslow;
    if (n_out) *n_out = n;
    return TP_OK;
}

extern "C" int tp_ingest_tsv(tp_ctx *ctx, const char *text, size_t nbytes, int sep, int *n_out) {
    TP_ARG(ctx && text, "tp_ingest_tsv: null argument");
    TextSource src;
    src.mem = (const unsigned char *)text;
    src.size = nbytes;
    return ingest_core(ctx, src, sep, n_out);
}

extern "C" int tp_ingest_tsv_file(tp_ctx *ctx, const char *path, int sep, int *n_out) {
    TP_ARG(ctx && path, "tp_ingest_tsv_file: null argument");
    TextSource src;
    src.fd = open(path, O_RDONLY);
    if (src.fd < 0) {
        tp_set_error("tp_ingest_tsv_file: cannot open '%s' (%s)", path, strerror(errno));
        return TP_ERR_ARG;
    }
    struct stat sb;
    if (fstat(src.fd, &sb) != 0 || !S_ISREG(sb.st_mode)) {
        close(src.fd);
        tp_set_error("tp_ingest_tsv_file: '%s' is not a regular file", path);
        return TP_ERR_ARG;
    }
    src.size = (size_t)sb.st_size;
#ifdef POSIX_FADV_SEQUENTIAL
    posix_fadvise(src.fd, 0, 0, POSIX_FADV_SEQUENTIAL);
#endif
    const int rc = ingest_core(ctx, src, sep, n_out);
    close(src.fd);
    return rc;
}

// ---- sparse input, host side ------------------------------------------------------------------------------------------
static int coo_status_init(tp_ctx *ctx, unsigned long long **status_out) {
    TP_TRY(ctx->islow.reserve(((size_t)1 << 20) * sizeof(SlowTok) + 128));
    unsigned long long *status64 = ctx->islow.as<unsigned long long>();          // 8 words, then the slow list
    const unsigned long long init[8] = {~0ull, 0, ~0ull, 0, 0, 0, 0, 0};
    TP_CUDA(cudaMemcpyAsync(status64, init, sizeof(init), cudaMemcpyHostToDevice, ctx->stream));
    *status_out = status64;
    return TP_OK;
}

static int coo_dense_alloc(tp_ctx *ctx, int n, double **out) {
    TP_TRY(ctx->raw_own.reserve((size_t)n * n * sizeof(double)));
    *out = ctx->raw_own.as<double>();
    TP_CUDA(cudaMemsetAsync(*out, 0, (size_t)n * n * sizeof(double), ctx->stream));
    return TP_OK;
}

static void coo_done(tp_ctx *ctx, double *out, int n, std::chrono::steady_clock::time_point t_begin, double bytes, double nslow) {
    ctx->raw = out;
    ctx->n = n;
    ctx->colmajor = 0;
    ctx->ingested_n = n;
    ctx->generation++;
    float ms = 0.f;
    cudaEventElapsedTime(&ms, ctx->ev[EV_INGEST0], ctx->ev[EV_INGEST1]);
    ctx->ingest_stats[0] = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t_begin).count();
    ctx->ingest_stats[1] = ms;
    ctx->ingest_stats[2] = bytes;
    ctx->ingest_stats[3] = nslow;
}

extern "C" int tp_ingest_coo(tp_ctx *ctx, const int32_t *bin1, const int32_t *bin2, const double *count, size_t nnz, int n,
                             int index_base, unsigned long long *below_out) {
    TP_ARG(ctx && (nnz == 0 || (bin1 && bin2 && count)), "tp_ingest_coo: null argument");
    TP_ARG(n >= 2 && n <= 200000, "tp_ingest_coo: the number of bins must be in 2..200000");
    TP_ARG(index_base == 0 || index_base == 1, "tp_ingest_coo: index_base must be 0 or 1");
    TP_CUDA(cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->stream;
    const auto t_begin = std::chrono::steady_clock::now();
    ctx->raw = nullptr; ctx->n = 0; ctx->ingested_n = 0;
    ctx->have_X = ctx->have_C = ctx->have_scores = ctx->have_sweep = false;
    unsigned long long *status64 = nullptr;
    TP_TRY(coo_status_init(ctx, &status64));
    double *out = nullptr;
    TP_TRY(coo_dense_alloc(ctx, n, &out));
    // 16 bytes per pixel cross PCIe: the three arrays go up whole (pageable arrays through the staging lanes of filter.cu),
    // then one scatter pass per 2^30 pixels
    TP_TRY(ctx->icoo.reserve(nnz * 16 + 16));
    double *dv = ctx->icoo.as<double>();
    int *d1 = (int *)(dv + nnz), *d2 = d1 + nnz;
    TP_MARK(ctx, EV_INGEST0);
    TP_TRY(tp_upload_range(ctx, dv, count, nnz * 8, st));
    TP_TRY(tp_upload_range(ctx, d1, bin1, nnz * 4, st));
    TP_TRY(tp_upload_range(ctx, d2, bin2, nnz * 4, st));
    const size_t M = (size_t)1 << 30;
    for (size_t off = 0; off < nnz; off += M) {
        const size_t m = nnz - off < M ? nnz - off : M;
        coo_scatter_kernel<<<(unsigned)((m + 255) / 256), 256, 0, st>>>(out, n, d1 + off, d2 + off, dv + off, (unsigned)m, index_base,
                                                                         (unsigned long long)off, status64);
        ctx->launches += 1;
    }
    TP_CUDA(cudaGetLastError());
    TP_MARK(ctx, EV_INGEST1);
    unsigned long long hs[8];
    TP_CUDA(cudaMemcpyAsync(hs, status64, sizeof(hs), cudaMemcpyDeviceToHost, st));
    TP_CUDA(tp_stream_sync(ctx));
    if (hs[0] != ~0ull) {
        tp_set_error("tp_ingest_coo: entry %llu is (%d, %d): outside the %d bins (index_base %d)", hs[0] + 1,
                     bin1[hs[0]], bin2[hs[0]], n, index_base);
        return TP_ERR_ARG;
    }
    if (below_out) *below_out = hs[1];
    coo_done(ctx, out, n, t_begin, (double)nnz * 16.0, 0.0);
    return TP_OK;
}

static int open_text_file(const char *path, const char *who, TextSource *src) {
    src->fd = open(path, O_RDONLY);
    if (src->fd < 0) {
        tp_set_error("%s: cannot open '%s' (%s)", who, path, strerror(errno));
        return TP_ERR_ARG;
    }
    struct stat sb;
    if (fstat(src->fd, &sb) != 0 || !S_ISREG(sb.st_mode)) {
        tp_set_error("%s: '%s' is not a regular file", who, path);
        return TP_ERR_ARG;
    }
    src->size = (size_t)sb.st_size;
#ifdef POSIX_FADV_SEQUENTIAL
    posix_fadvise(src->fd, 0, 0, POSIX_FADV_SEQUENTIAL);
#endif
    return TP_OK;
}

// fail with a plain message when `bytes` more cannot fit on ctx's device (`held`: bytes of the buffer about to be grown,
// which its reserve frees first)
static int device_room(tp_ctx *ctx, double bytes, size_t held, const char *who, const char *what) {
    size_t fr = 0, tot = 0;
    if (cudaMemGetInfo(&fr, &tot) != cudaSuccess) { (void)cudaGetLastError(); return TP_OK; }
    if (bytes > (double)fr + (double)held) {
        tp_set_error("%s: %s need %.2f GB on device %d and %.2f GB are free; inputs larger than the device memory are not "
                     "supported", who, what, bytes / 1e9, ctx->device, ((double)fr + (double)held) / 1e9);
        return TP_ERR_NOMEM;
    }
    return TP_OK;
}

// The pixels of a three-column text "bin1 <sep> bin2 <sep> count", parsed on ctx's device: on return row r of the file is
// (d1[r], d2[r], dv[r]) in ctx->icoo, rows [first, nrows) are pixels (first = 1 after a header line), status64 (8 words,
// then the slow list, in ctx->islow) as coo_parse_kernel left it.
static int coo_text_pixels(tp_ctx *ctx, const TextSource &src, int sep, const char *who, double *extra_per_row, int **d1_out,
                           int **d2_out, double **dv_out, long long *nrows_out, unsigned *first_out, unsigned *nslow_out,
                           size_t *nbytes_out, unsigned long long **status_out) {
    cudaStream_t st = ctx->stream;
    unsigned char *text = nullptr;
    size_t nbytes = 0;
    int nb = 0;
    long long *offs = nullptr, nrows = 0;
    TP_TRY(text_rows(ctx, src, who, &text, &nbytes, &nb, &offs, &nrows));
    if (nrows < 1 || nrows >= 0x7fffffffLL) {
        tp_set_error("%s: the file must hold between 1 and 2^31 - 2 rows", who);
        return TP_ERR_ARG;
    }
    if (extra_per_row) TP_TRY(device_room(ctx, (24.0 + *extra_per_row) * (double)nrows, ctx->irows.cap + ctx->icoo.cap, who, "the pixels"));
    const long long limit = (long long)nbytes + 1;
    const unsigned slow_cap = 1u << 20;
    unsigned long long *status64 = nullptr;
    TP_TRY(coo_status_init(ctx, &status64));
    unsigned *slow_count = (unsigned *)(status64 + 5);
    SlowTok *slow = (SlowTok *)(status64 + 8);
    TP_TRY(ctx->irows.reserve((size_t)nrows * sizeof(long long)));
    TP_TRY(ctx->icoo.reserve((size_t)nrows * 16));
    long long *row_end = ctx->irows.as<long long>();
    double *dv = ctx->icoo.as<double>();
    int *d1 = (int *)(dv + nrows), *d2 = d1 + nrows;
    newline_pos_kernel<<<nb, IG_THREADS, 0, st>>>(text, limit, offs, row_end);
    coo_parse_kernel<<<(unsigned)((nrows + 255) / 256), 256, 0, st>>>(text, row_end, (unsigned)nrows, (unsigned)sep, dv, d1, d2, slow,
                                                                    slow_count, slow_cap, status64);
    TP_CUDA(cudaGetLastError());
    ctx->launches += 2;
    unsigned long long hs[8];
    TP_CUDA(cudaMemcpyAsync(hs, status64, sizeof(hs), cudaMemcpyDeviceToHost, st));
    TP_CUDA(tp_stream_sync(ctx));
    if (hs[2] == ~0ull - 1) {
        tp_set_error("%s: more than %u counts need the host conversion path", who, slow_cap);
        return TP_ERR_ARG;
    }
    if (hs[2] != ~0ull) {
        tp_set_error("%s: row %llu is not 'bin1 <sep> bin2 <sep> count' with non-negative integer bins", who, hs[2] + 1);
        return TP_ERR_ARG;
    }
    const unsigned first = hs[4] ? 1u : 0u;                     // a header line is skipped
    if ((unsigned long long)nrows <= first) {
        tp_set_error("%s: the file holds a header and no pixels", who);
        return TP_ERR_ARG;
    }
    const unsigned nslow = (unsigned)(hs[5] & 0xffffffffu);
    if (nslow) {
        std::vector<SlowTok> list(nslow);
        TP_CUDA(cudaMemcpy(list.data(), slow, (size_t)nslow * sizeof(SlowTok), cudaMemcpyDeviceToHost));
        std::vector<unsigned> idx(nslow);
        std::vector<double> val(nslow);
        std::vector<char> buf(4096 + 1);
        for (unsigned i = 0; i < nslow; i++) {
            TP_TRY(host_field(src, nbytes, (size_t)list[i].off, sep, buf, &val[i], who, list[i].row, 2));
            idx[i] = list[i].row;
        }
        unsigned *didx = (unsigned *)slow;
        double *dval = (double *)(slow + ((size_t)nslow + 1) / 2 + 1);            // past the indices, 8-byte aligned
        TP_CUDA(cudaMemcpyAsync(didx, idx.data(), (size_t)nslow * sizeof(unsigned), cudaMemcpyHostToDevice, st));
        TP_CUDA(cudaMemcpyAsync(dval, val.data(), (size_t)nslow * sizeof(double), cudaMemcpyHostToDevice, st));
        scatter_f64_kernel<<<(nslow + 255) / 256, 256, 0, st>>>(dv, didx, dval, (int)nslow);
        TP_CUDA(cudaGetLastError());
        TP_CUDA(tp_stream_sync(ctx));
        ctx->launches += 1;
    }
    *d1_out = d1; *d2_out = d2; *dv_out = dv; *nrows_out = nrows; *first_out = first; *nslow_out = nslow;
    *nbytes_out = nbytes; *status_out = status64;
    return TP_OK;
}

extern "C" int tp_ingest_coo_file(tp_ctx *ctx, const char *path, int sep, int n, int index_base, int *n_out,
                                  unsigned long long *nnz_out, unsigned long long *below_out) {
    TP_ARG(ctx && path, "tp_ingest_coo_file: null argument");
    TP_ARG(sep > 0 && sep < 128 && sep != '\n' && sep != '\r' && sep != '.' && sep != '-' && sep != '+' && !(sep >= '0' && sep <= '9'),
           "tp_ingest_coo_file: bad separator");
    TP_ARG(n <= 200000, "tp_ingest_coo_file: more than 200000 bins");
    TP_ARG(index_base == 0 || index_base == 1, "tp_ingest_coo_file: index_base must be 0 or 1");
    TextSource src;
    TP_TRY(open_text_file(path, "tp_ingest_coo_file", &src));
    struct Closer { int fd; ~Closer() { close(fd); } } closer{src.fd};
    TP_CUDA(cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->stream;
    const auto t_begin = std::chrono::steady_clock::now();
    ctx->raw = nullptr; ctx->n = 0; ctx->ingested_n = 0;
    ctx->have_X = ctx->have_C = ctx->have_scores = ctx->have_sweep = false;
    int *d1 = nullptr, *d2 = nullptr;
    double *dv = nullptr;
    long long nrows = 0;
    unsigned first = 0, nslow = 0;
    size_t nbytes = 0;
    unsigned long long *status64 = nullptr;
    TP_TRY(coo_text_pixels(ctx, src, sep, "tp_ingest_coo_file", nullptr, &d1, &d2, &dv, &nrows, &first, &nslow, &nbytes, &status64));
    unsigned long long hs[8];
    if (n <= 0) {
        TP_CUDA(cudaMemcpy(hs, status64, sizeof(hs), cudaMemcpyDeviceToHost));
        const long long nn = (long long)hs[3] - index_base;
        if (nn < 2 || nn > 200000) {
            tp_set_error("tp_ingest_coo_file: the largest bin in the file gives %lld bins; 2..200000 are supported", nn);
            return TP_ERR_ARG;
        }
        n = (int)nn;
    }
    TP_ARG(n >= 2, "tp_ingest_coo_file: the number of bins must be at least 2");
    double *out = nullptr;
    TP_TRY(coo_dense_alloc(ctx, n, &out));
    const unsigned m = (unsigned)nrows - first;
    coo_scatter_kernel<<<(m + 255) / 256, 256, 0, st>>>(out, n, d1 + first, d2 + first, dv + first, m, index_base, (unsigned long long)first,
                                                        status64);
    TP_CUDA(cudaGetLastError());
    ctx->launches += 1;
    TP_MARK(ctx, EV_INGEST1);
    TP_CUDA(cudaMemcpyAsync(hs, status64, sizeof(hs), cudaMemcpyDeviceToHost, st));
    TP_CUDA(tp_stream_sync(ctx));
    if (hs[0] != ~0ull) {
        tp_set_error("tp_ingest_coo_file: row %llu names a bin outside the %d bins (index_base %d)", hs[0] + 1, n, index_base);
        return TP_ERR_ARG;
    }
    if (n_out) *n_out = n;
    if (nnz_out) *nnz_out = m;
    if (below_out) *below_out = hs[1];
    coo_done(ctx, out, n, t_begin, (double)nbytes, (double)nslow);
    return TP_OK;
}

// ---- genome-wide pixels (S0c): one pixel list over every chromosome -> one bucket of local pixels per chromosome ------
// Bins are global ids; chromosome c holds [starts[c], starts[c + 1]) (0-based, starts[0] = 0).  A pixel is out of range
// (a bin outside the table: the lowest entry index goes to status64[0]), trans (two chromosomes: counted in status64[6]
// and dropped), below the diagonal (counted in status64[1] and dropped, as S0b does) or cis (kept, in chromosome-local
// bins).  Any number of chromosomes up to 2^20: a binary search over the starts finds the one of a bin.
__device__ __forceinline__ int genome_chrom_of(const int *__restrict__ starts, int nchrom, int x) {
    int lo = 0, hi = nchrom - 1;
    while (lo < hi) {
        const int mid = (lo + hi + 1) >> 1;
        if (__ldg(starts + mid) <= x) lo = mid; else hi = mid - 1;
    }
    return lo;
}

// the chromosome whose bucket pixel e goes to, and its local bins; -1 when the pixel is dropped
__device__ __forceinline__ int genome_route(const int *__restrict__ b1, const int *__restrict__ b2, unsigned e, unsigned m, int base,
                                            const int *__restrict__ starts, int nchrom, unsigned long long first,
                                            unsigned long long *__restrict__ status64, bool count, int *li, int *lj) {
    bool trans = false, below = false;
    int c = -1;
    if (e < m) {
        const long long x = (long long)b1[e] - base, y = (long long)b2[e] - base, total = starts[nchrom];
        if (x < 0 || y < 0 || x >= total || y >= total) {
            if (count) atomicMin(status64, first + e);
        } else {
            const int cx = genome_chrom_of(starts, nchrom, (int)x), cy = genome_chrom_of(starts, nchrom, (int)y);
            if (cx != cy) trans = true;
            else if (x > y) below = true;
            else { c = cx; *li = (int)x - starts[c]; *lj = (int)y - starts[c]; }
        }
    }
    if (count) {
        const unsigned bt = __ballot_sync(0xffffffffu, trans), bb = __ballot_sync(0xffffffffu, below);
        if ((threadIdx.x & 31) == 0) {
            if (bt) atomicAdd(status64 + 6, (unsigned long long)__popc(bt));
            if (bb) atomicAdd(status64 + 1, (unsigned long long)__popc(bb));
        }
    }
    return c;
}

// pass 1: cis pixels per chromosome (one atomic per distinct chromosome in a warp)
__global__ void __launch_bounds__(256)
genome_route_kernel(const int *__restrict__ b1, const int *__restrict__ b2, unsigned m, int base, const int *__restrict__ starts,
                    int nchrom, unsigned long long first, unsigned long long *__restrict__ hist,
                    unsigned long long *__restrict__ status64) {
    const unsigned e = blockIdx.x * blockDim.x + threadIdx.x;
    int li = 0, lj = 0;
    const int c = genome_route(b1, b2, e, m, base, starts, nchrom, first, status64, true, &li, &lj);
    const unsigned grp = __match_any_sync(0xffffffffu, c);
    if (c >= 0 && (threadIdx.x & 31) == __ffs(grp) - 1) atomicAdd(hist + c, (unsigned long long)__popc(grp));
}

// pass 2: every cis pixel into its chromosome's bucket as local (i, j, count); cursor[c] starts at the bucket's offset
__global__ void __launch_bounds__(256)
genome_bucket_kernel(const int *__restrict__ b1, const int *__restrict__ b2, const double *__restrict__ v, unsigned m, int base,
                     const int *__restrict__ starts, int nchrom, unsigned long long *__restrict__ cursor,
                     double *__restrict__ ov, int *__restrict__ oi, int *__restrict__ oj) {
    const unsigned e = blockIdx.x * blockDim.x + threadIdx.x;
    const int lane = threadIdx.x & 31;
    int li = 0, lj = 0;
    const int c = genome_route(b1, b2, e, m, base, starts, nchrom, 0, nullptr, false, &li, &lj);
    const unsigned grp = __match_any_sync(0xffffffffu, c);
    const int leader = __ffs(grp) - 1;
    unsigned long long pos = 0;
    if (c >= 0 && lane == leader) pos = atomicAdd(cursor + c, (unsigned long long)__popc(grp));
    pos = __shfl_sync(0xffffffffu, pos, leader) + (unsigned long long)__popc(grp & ((1u << lane) - 1));
    if (c >= 0) { ov[pos] = v[e]; oi[pos] = li; oj[pos] = lj; }
}

static int genome_new(const int32_t *chrom_bins, int nchrom, int index_base, const char *who, tp_genome **out) {
    if (!(nchrom >= 1 && nchrom <= (1 << 20))) { tp_set_error("%s: the number of chromosomes must be in 1..2^20", who); return TP_ERR_ARG; }
    if (index_base != 0 && index_base != 1) { tp_set_error("%s: index_base must be 0 or 1", who); return TP_ERR_ARG; }
    long long total = 0;
    for (int c = 0; c < nchrom; c++) {
        if (chrom_bins[c] < 1) { tp_set_error("%s: chromosome %d has %d bins; at least 1 is needed", who, c, chrom_bins[c]); return TP_ERR_ARG; }
        total += chrom_bins[c];
    }
    if (total >= 0x7fffffffLL) { tp_set_error("%s: the bin table holds %lld bins; at most 2^31 - 2 are supported", who, total); return TP_ERR_ARG; }
    tp_genome *g = new tp_genome();
    g->bins.assign(chrom_bins, chrom_bins + nchrom);
    *out = g;
    return TP_OK;
}

// Route the pixels (d1, d2, dv: m of them on ctx's device; pixel e is entry first + e of the input) into g's buckets.
// hb1 / hb2: the host arrays, to name the bins of an entry outside the table (NULL for a file: the row is named).
static int genome_bucket(tp_ctx *ctx, tp_genome *g, const int *d1, const int *d2, const double *dv, size_t m, int index_base,
                         unsigned long long first, unsigned long long *status64, const int32_t *hb1, const int32_t *hb2,
                         const char *who) {
    cudaStream_t st = ctx->stream;
    const int nchrom = (int)g->bins.size();
    std::vector<int> starts((size_t)nchrom + 1, 0);
    for (int c = 0; c < nchrom; c++) starts[c + 1] = starts[c] + g->bins[c];
    struct Aux { DevBuf b; ~Aux() { b.release(); } } aux;         // hist[nchrom], cursor[nchrom] (u64), starts[nchrom + 1]
    TP_TRY(aux.b.reserve((size_t)nchrom * 16 + ((size_t)nchrom + 1) * sizeof(int)));
    unsigned long long *hist = aux.b.as<unsigned long long>(), *cursor = hist + nchrom;
    int *dstarts = (int *)(cursor + nchrom);
    TP_CUDA(cudaMemsetAsync(hist, 0, (size_t)nchrom * 8, st));
    TP_CUDA(cudaMemcpyAsync(dstarts, starts.data(), starts.size() * sizeof(int), cudaMemcpyHostToDevice, st));
    const size_t M = (size_t)1 << 30;
    for (size_t off = 0; off < m; off += M) {
        const unsigned k = (unsigned)(m - off < M ? m - off : M);
        genome_route_kernel<<<(k + 255) / 256, 256, 0, st>>>(d1 + off, d2 + off, k, index_base, dstarts, nchrom, first + off, hist, status64);
        ctx->launches += 1;
    }
    TP_CUDA(cudaGetLastError());
    std::vector<unsigned long long> h((size_t)nchrom);
    unsigned long long hs[8];
    TP_CUDA(cudaMemcpyAsync(h.data(), hist, (size_t)nchrom * 8, cudaMemcpyDeviceToHost, st));
    TP_CUDA(cudaMemcpyAsync(hs, status64, sizeof(hs), cudaMemcpyDeviceToHost, st));
    TP_CUDA(tp_stream_sync(ctx));
    if (hs[0] != ~0ull) {
        if (hb1) tp_set_error("%s: entry %llu is (%d, %d): outside the %d bins of the bin table (index_base %d)", who, hs[0] + 1,
                              hb1[hs[0]], hb2[hs[0]], starts[nchrom], index_base);
        else tp_set_error("%s: row %llu names a bin outside the %d bins of the bin table (index_base %d)", who, hs[0] + 1,
                          starts[nchrom], index_base);
        return TP_ERR_ARG;
    }
    g->offs.assign((size_t)nchrom + 1, 0);
    for (int c = 0; c < nchrom; c++) g->offs[c + 1] = g->offs[c] + h[c];
    g->below = hs[1];
    g->trans = hs[6];
    const size_t ncis = g->offs[nchrom];
    TP_TRY(device_room(ctx, 16.0 * (double)ncis, 0, who, "the buckets of the cis pixels"));
    TP_TRY(g->px.reserve(ncis * 16 + 16));
    double *ov = g->px.as<double>();
    int *oi = (int *)(ov + ncis), *oj = oi + ncis;
    TP_CUDA(cudaMemcpyAsync(cursor, g->offs.data(), (size_t)nchrom * 8, cudaMemcpyHostToDevice, st));
    for (size_t off = 0; off < m; off += M) {
        const unsigned k = (unsigned)(m - off < M ? m - off : M);
        genome_bucket_kernel<<<(k + 255) / 256, 256, 0, st>>>(d1 + off, d2 + off, dv + off, k, index_base, dstarts, nchrom, cursor, ov, oi, oj);
        ctx->launches += 1;
    }
    TP_CUDA(cudaGetLastError());
    TP_MARK(ctx, EV_INGEST1);
    TP_CUDA(tp_stream_sync(ctx));
    return TP_OK;
}

static void genome_done(tp_ctx *ctx, std::chrono::steady_clock::time_point t_begin, double bytes, double nslow) {
    // the parse arrays are not needed any more: their memory goes back to the calls
    ctx->icoo.release();
    ctx->irows.release();
    float ms = 0.f;
    cudaEventElapsedTime(&ms, ctx->ev[EV_INGEST0], ctx->ev[EV_INGEST1]);
    ctx->ingest_stats[0] = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t_begin).count();
    ctx->ingest_stats[1] = ms;
    ctx->ingest_stats[2] = bytes;
    ctx->ingest_stats[3] = nslow;
}

struct GenomeOwner { tp_genome *g = nullptr; ~GenomeOwner() { if (g) tp_genome_free(g); } };

extern "C" int tp_genome_ingest(tp_ctx *ctx, const int32_t *chrom_bins, int nchrom, const int32_t *bin1, const int32_t *bin2,
                                const double *count, size_t nnz, int index_base, tp_genome **out) {
    TP_ARG(ctx && chrom_bins && out && (nnz == 0 || (bin1 && bin2 && count)), "tp_genome_ingest: null argument");
    TP_CUDA(cudaSetDevice(ctx->device));
    const auto t_begin = std::chrono::steady_clock::now();
    GenomeOwner own;
    TP_TRY(genome_new(chrom_bins, nchrom, index_base, "tp_genome_ingest", &own.g));
    own.g->device = ctx->device;
    cudaStream_t st = ctx->stream;
    unsigned long long *status64 = nullptr;
    TP_TRY(coo_status_init(ctx, &status64));
    TP_TRY(device_room(ctx, 16.0 * (double)nnz, ctx->icoo.cap, "tp_genome_ingest", "the pixels"));
    TP_TRY(ctx->icoo.reserve(nnz * 16 + 16));
    double *dv = ctx->icoo.as<double>();
    int *d1 = (int *)(dv + nnz), *d2 = d1 + nnz;
    TP_MARK(ctx, EV_INGEST0);
    TP_TRY(tp_upload_range(ctx, dv, count, nnz * 8, st));
    TP_TRY(tp_upload_range(ctx, d1, bin1, nnz * 4, st));
    TP_TRY(tp_upload_range(ctx, d2, bin2, nnz * 4, st));
    TP_TRY(genome_bucket(ctx, own.g, d1, d2, dv, nnz, index_base, 0, status64, bin1, bin2, "tp_genome_ingest"));
    genome_done(ctx, t_begin, (double)nnz * 16.0, 0.0);
    *out = own.g;
    own.g = nullptr;
    return TP_OK;
}

extern "C" int tp_genome_ingest_file(tp_ctx *ctx, const int32_t *chrom_bins, int nchrom, const char *path, int sep, int index_base,
                                     tp_genome **out) {
    TP_ARG(ctx && chrom_bins && path && out, "tp_genome_ingest_file: null argument");
    TP_ARG(sep > 0 && sep < 128 && sep != '\n' && sep != '\r' && sep != '.' && sep != '-' && sep != '+' && !(sep >= '0' && sep <= '9'),
           "tp_genome_ingest_file: bad separator");
    GenomeOwner own;
    TP_TRY(genome_new(chrom_bins, nchrom, index_base, "tp_genome_ingest_file", &own.g));
    TextSource src;
    TP_TRY(open_text_file(path, "tp_genome_ingest_file", &src));
    struct Closer { int fd; ~Closer() { close(fd); } } closer{src.fd};
    TP_CUDA(cudaSetDevice(ctx->device));
    own.g->device = ctx->device;
    const auto t_begin = std::chrono::steady_clock::now();
    int *d1 = nullptr, *d2 = nullptr;
    double *dv = nullptr;
    long long nrows = 0;
    unsigned first = 0, nslow = 0;
    size_t nbytes = 0;
    unsigned long long *status64 = nullptr;
    double per_row = 16.0;                       // the buckets, if every row is a cis pixel
    TP_TRY(coo_text_pixels(ctx, src, sep, "tp_genome_ingest_file", &per_row, &d1, &d2, &dv, &nrows, &first, &nslow, &nbytes,
                           &status64));
    ctx->itext.release();                        // the text is parsed
    const size_t m = (size_t)nrows - first;
    TP_TRY(genome_bucket(ctx, own.g, d1 + first, d2 + first, dv + first, m, index_base, first, status64, nullptr, nullptr,
                         "tp_genome_ingest_file"));
    genome_done(ctx, t_begin, (double)nbytes, (double)nslow);
    *out = own.g;
    own.g = nullptr;
    return TP_OK;
}

extern "C" int tp_genome_stats(const tp_genome *g, unsigned long long *cis_out, unsigned long long *trans_out,
                               unsigned long long *below_out) {
    TP_ARG(g, "tp_genome_stats: null handle");
    if (cis_out)
        for (size_t c = 0; c + 1 < g->offs.size(); c++) cis_out[c] = g->offs[c + 1] - g->offs[c];
    if (trans_out) *trans_out = g->trans;
    if (below_out) *below_out = g->below;
    return TP_OK;
}

int tp_genome_dense(tp_ctx *c, const tp_genome *g, int chrom, double **out) {
    TP_ARG(chrom >= 0 && chrom < (int)g->bins.size(), "tp_genome: chromosome index out of range");
    TP_CUDA(cudaSetDevice(c->device));
    const int n = g->bins[(size_t)chrom];
    const size_t ncis = g->offs.back(), o = g->offs[(size_t)chrom], m = g->offs[(size_t)chrom + 1] - o;
    const double *v = g->px.as<double>() + o;
    const int *bi = (const int *)(g->px.as<double>() + ncis) + o, *bj = bi + ncis;
    const bool remote = c->device != g->device;
    // status words of the scatter (every bucket pixel is in range and on or above the diagonal: never written)
    TP_TRY(c->icoo.reserve(64 + (remote ? m * 16 : 0)));
    unsigned long long *status64 = c->icoo.as<unsigned long long>();
    TP_CUDA(cudaMemsetAsync(status64, 0, 64, c->stream));
    if (remote && m) {
        double *pv = (double *)(status64 + 8);
        int *pi = (int *)(pv + m), *pj = pi + m;
        TP_CUDA(cudaMemcpyPeerAsync(pv, c->device, v, g->device, m * 8, c->stream));
        TP_CUDA(cudaMemcpyPeerAsync(pi, c->device, bi, g->device, m * 4, c->stream));
        TP_CUDA(cudaMemcpyPeerAsync(pj, c->device, bj, g->device, m * 4, c->stream));
        v = pv; bi = pi; bj = pj;
    }
    c->raw = nullptr; c->n = 0; c->ingested_n = 0;
    c->have_X = c->have_C = c->have_scores = c->have_sweep = false;
    c->generation++;
    TP_TRY(coo_dense_alloc(c, n, out));
    const size_t M = (size_t)1 << 30;
    for (size_t off = 0; off < m; off += M) {
        const unsigned k = (unsigned)(m - off < M ? m - off : M);
        coo_scatter_kernel<<<(k + 255) / 256, 256, 0, c->stream>>>(*out, n, bi + off, bj + off, v + off, k, 0, off, status64);
        c->launches += 1;
    }
    TP_CUDA(cudaGetLastError());
    return TP_OK;
}

extern "C" int tp_genome_matrix(tp_ctx *ctx, const tp_genome *g, int chrom, double *out) {
    TP_ARG(ctx && g && out, "tp_genome_matrix: null argument");
    TP_ARG(chrom >= 0 && chrom < (int)g->bins.size(), "tp_genome_matrix: chromosome index out of range");
    double *dev = nullptr;
    TP_TRY(tp_genome_dense(ctx, g, chrom, &dev));
    const size_t n = (size_t)g->bins[(size_t)chrom];
    TP_CUDA(cudaMemcpyAsync(out, dev, n * n * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    TP_CUDA(tp_stream_sync(ctx));
    return TP_OK;
}

extern "C" int tp_genome_free(tp_genome *g) {
    if (!g) return TP_OK;
    cudaSetDevice(g->device);
    g->px.release();
    delete g;
    return TP_OK;
}

extern "C" int tp_ingested(tp_ctx *ctx, const double **dev_out, int *n_out) {
    TP_ARG(ctx, "tp_ingested: null context");
    TP_ARG(ctx->ingested_n > 0 && ctx->raw_own.p, "tp_ingested: no matrix has been ingested on this context");
    if (dev_out) *dev_out = ctx->raw_own.as<double>();
    if (n_out) *n_out = ctx->ingested_n;
    return TP_OK;
}

extern "C" int tp_get_ingested(tp_ctx *ctx, double *out) {
    TP_ARG(ctx && out, "tp_get_ingested: null argument");
    TP_ARG(ctx->ingested_n > 0 && ctx->raw_own.p, "tp_get_ingested: no matrix has been ingested on this context");
    TP_CUDA(cudaSetDevice(ctx->device));
    const size_t n = (size_t)ctx->ingested_n;
    TP_CUDA(cudaMemcpyAsync(out, ctx->raw_own.p, n * n * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    TP_CUDA(tp_stream_sync(ctx));
    return TP_OK;
}

extern "C" int tp_ingest_stats(tp_ctx *ctx, double *out4) {
    TP_ARG(ctx && out4, "tp_ingest_stats: null argument");
    for (int i = 0; i < 4; i++) out4[i] = ctx->ingest_stats[i];
    return TP_OK;
}

// host-only test hook: the field conversion exactly as the parse kernel runs it (no GPU needed)
extern "C" int tp_test_parse_field(const char *s, int len, double *out) {
    if (!s || !out || len < 0) return -1;
    return np_parse_field((const unsigned char *)s, len, h_pow10, h_pow5, out);
}
