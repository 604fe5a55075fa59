// pairs.cu -- a genome from read-pair files (S0f): tp_genome_ingest_pairs_file streams text files of read pairs (4DN
// .pairs, HiC-Pro *.allValidPairs, Juicer merged_nodups.txt) through fixed-size device windows, bins every pair at
// `binsize` bp on the device and merges the cells of all the files into one tp_genome.
//
// A window is a run of whole lines of at most `window` bytes: it ends at its last '\n', and the bytes after it start the
// next window.  Per window:
//   1. text_rows / text_line_ends (ingest.cu): the upload through the context's two pinned buffers, the line count and
//      the byte offset of every line end, found on the device.
//   2. Table growth: before a window of r lines, a cell table with occupied + r > capacity / 2 is rehashed
//      (pr_rehash_kernel) into a power-of-two table at least twice as large, so no insert of the window can fill it.
//   3. pr_parse_kernel, one thread per line: the four fields, the chromosome names looked up in a table sorted by 64-bit
//      hash (the bytes are compared after the hash matches, so names that share a hash resolve), the positions parsed and
//      checked, the pair classified, and a cis cell ((S_c + I) << 31) | (S_c + J) inserted into the open-addressing table
//      with CAS on the key and an FP64 atomicAdd of 1.  Pair lines, cis, trans, unplaced and newly occupied slots are
//      counted with warp-aggregated atomics; the lowest bad line goes to one atomicMin word.
// The host reads window w + 1 while the device parses window w.  It waits on the stream once per window, after the line
// count the growth check needs; the counters of the windows before come back in that same wait.  After the last window
// cs_count_kernel / cs_scatter_kernel (genome_util.cuh) write the buckets.
// Counts are integer sums of 1.0 (exact below 2^53 in any order), so the cells, the counts and the stats do not depend on
// the window size, the table growth or the file order.  Memory: the window + 16 KB, 8 bytes per line of a window, 16 bytes
// per table slot (2 to 4 slots per distinct cell), then 16 bytes per cell for the buckets while the table is held.
#include "genome_util.cuh"
#include "text.cuh"
#include <fcntl.h>
#include <stdlib.h>
#include <algorithm>
#include <chrono>
#include <string>
#include <unordered_set>

#define PR_THREADS 256
#define PR_WINDOW ((size_t)64 << 20)          // default window: two of the 32 MB pinned chunks of text_rows
#define PR_MAXCOL 63

// status words: counts, then the lowest bad line as (1-based line << 2) | kind (~0 = none)
enum { PR_LINES = 0, PR_CIS, PR_TRANS, PR_UNPLACED, PR_OCC, PR_BAD, PR_NSTATUS = 8 };
enum { PR_BAD_FIELDS = 1, PR_BAD_DIGITS = 2, PR_BAD_RANGE = 3 };

// the chromosome table on the device
struct PrTable {
    const u64 *hash;                 // name hashes, ascending
    const int *idx;                  // the chromosome of hash[k]
    const long long *noff;           // name c = blob[noff[c], noff[c + 1])
    const unsigned char *blob;
    const long long *len;            // length in bp
    const int *starts;               // first global bin
    int nchrom;
};
struct PrCols { int c[4]; int maxcol; };    // 0-based columns of chrom1, pos1, chrom2, pos2; the largest

// FNV-1a, 64 bits
__host__ __device__ __forceinline__ u64 pr_name_hash(const unsigned char *s, long long n) {
    u64 h = 0xcbf29ce484222325ULL;
    for (long long i = 0; i < n; i++) { h ^= s[i]; h *= 0x100000001b3ULL; }
    return h;
}

// the chromosome named by bytes s[0, n), or -1
__device__ __forceinline__ int pr_lookup(const PrTable &T, const unsigned char *s, long long n) {
    const u64 h = pr_name_hash(s, n);
    int lo = 0, hi = T.nchrom;
    while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        if (__ldg(T.hash + mid) < h) lo = mid + 1; else hi = mid;
    }
    for (int k = lo; k < T.nchrom && __ldg(T.hash + k) == h; k++) {
        const int c = __ldg(T.idx + k);
        const long long o = __ldg(T.noff + c);
        if (__ldg(T.noff + c + 1) - o != n) continue;
        long long i = 0;
        while (i < n && __ldg(T.blob + o + i) == s[i]) i++;
        if (i == n) return c;
    }
    return -1;
}

// 1-18 ASCII digits
__device__ __forceinline__ bool pr_position(const unsigned char *s, long long n, long long *out) {
    if (n < 1 || n > 18) return false;
    long long x = 0;
    for (long long i = 0; i < n; i++) {
        const unsigned d = (unsigned)s[i] - '0';
        if (d > 9) return false;
        x = x * 10 + d;
    }
    *out = x;
    return true;
}

__device__ __forceinline__ bool pr_blank(unsigned char b) { return b == ' ' || b == '\t'; }

__device__ __forceinline__ void pr_insert(u64 *__restrict__ tkeys, double *__restrict__ tval, u64 mask, u64 key, double v,
                                          bool *fresh) {
    u64 s = ds_hash(key) & mask;
    while (true) {
        u64 k = tkeys[s];
        if (k == CS_EMPTY) {
            k = atomicCAS(tkeys + s, CS_EMPTY, key);
            if (k == CS_EMPTY) *fresh = true;
        }
        if (k == CS_EMPTY || k == key) { atomicAdd(tval + s, v); break; }
        s = (s + 1) & mask;
    }
}

// one line per thread; line r of the window is line line0 + r + 1 of its file
__global__ void __launch_bounds__(PR_THREADS)
pr_parse_kernel(const unsigned char *__restrict__ text, const long long *__restrict__ row_end, unsigned nrows, u64 line0,
                PrCols cols, PrTable T, long long binsize, int base, u64 *__restrict__ tkeys, double *__restrict__ tval,
                u64 mask, u64 *__restrict__ status) {
    const unsigned r = blockIdx.x * PR_THREADS + threadIdx.x;
    int kind = 0;                                     // 0: no pair (comment, blank, beyond the window) 1: unplaced 2: trans 3: cis
    bool fresh = false;
    int bad = 0;
    if (r < nrows) {
        const long long p = r ? row_end[r - 1] + 1 : 0;
        long long e = row_end[r];
        if (e > p && text[e - 1] == '\r') e--;       // CRLF
        long long q = p;
        while (q < e && (pr_blank(text[q]) || text[q] == '\r')) q++;
        if (q < e && text[p] != '#') {
            long long fs[4] = {0, 0, 0, 0}, fl[4] = {0, 0, 0, 0};
            int f = 0;
            q = p;
            while (f <= cols.maxcol) {
                while (q < e && pr_blank(text[q])) q++;
                if (q >= e) break;
                const long long s0 = q;
                while (q < e && !pr_blank(text[q])) q++;
#pragma unroll
                for (int k = 0; k < 4; k++)
                    if (cols.c[k] == f) { fs[k] = s0; fl[k] = q - s0; }
                f++;
            }
            long long p1 = 0, p2 = 0;
            if (f <= cols.maxcol) bad = PR_BAD_FIELDS;
            else if (!pr_position(text + fs[1], fl[1], &p1) || !pr_position(text + fs[3], fl[3], &p2)) bad = PR_BAD_DIGITS;
            else {
                const int c1 = pr_lookup(T, text + fs[0], fl[0]), c2 = pr_lookup(T, text + fs[2], fl[2]);
                const bool out1 = c1 >= 0 && (p1 < base || p1 - base >= __ldg(T.len + c1));
                const bool out2 = c2 >= 0 && (p2 < base || p2 - base >= __ldg(T.len + c2));
                if (out1 || out2) bad = PR_BAD_RANGE;
                else if (c1 < 0 || c2 < 0) kind = 1;
                else if (c1 != c2) kind = 2;
                else {
                    kind = 3;
                    const long long b1 = (p1 - base) / binsize, b2 = (p2 - base) / binsize;
                    const long long s0 = __ldg(T.starts + c1);
                    const u64 key = ((u64)(s0 + (b1 < b2 ? b1 : b2)) << 31) | (u64)(s0 + (b1 < b2 ? b2 : b1));
                    pr_insert(tkeys, tval, mask, key, 1.0, &fresh);
                }
            }
            if (bad) atomicMin(status + PR_BAD, ((line0 + r + 1) << 2) | (u64)bad);
        }
    }
    const unsigned bl = __ballot_sync(CS_FULL, kind > 0), bc = __ballot_sync(CS_FULL, kind == 3),
                   bt = __ballot_sync(CS_FULL, kind == 2), bu = __ballot_sync(CS_FULL, kind == 1),
                   bf = __ballot_sync(CS_FULL, fresh);
    if ((threadIdx.x & 31) == 0) {
        if (bl) atomicAdd(status + PR_LINES, (u64)__popc(bl));
        if (bc) atomicAdd(status + PR_CIS, (u64)__popc(bc));
        if (bt) atomicAdd(status + PR_TRANS, (u64)__popc(bt));
        if (bu) atomicAdd(status + PR_UNPLACED, (u64)__popc(bu));
        if (bf) atomicAdd(status + PR_OCC, (u64)__popc(bf));
    }
}

// every cell of the old table into the new one (keys are distinct: each claims its own slot)
__global__ void __launch_bounds__(DS_THREADS)
pr_rehash_kernel(const u64 *__restrict__ okeys, const double *__restrict__ oval, u64 ocap, u64 *__restrict__ tkeys,
                 double *__restrict__ tval, u64 mask) {
    const u64 stride = (u64)gridDim.x * DS_THREADS;
    for (u64 e = (u64)blockIdx.x * DS_THREADS + threadIdx.x; e < ocap; e += stride) {
        const u64 key = okeys[e];
        if (key == CS_EMPTY) continue;
        u64 s = ds_hash(key) & mask;
        while (atomicCAS(tkeys + s, CS_EMPTY, key) != CS_EMPTY) s = (s + 1) & mask;
        tval[s] = oval[e];
    }
}

// ---- host side ------------------------------------------------------------------------------------------------------------
struct PrTableBuf {
    DevBuf b;
    u64 cap = 0;
    u64 *keys() const { return b.as<u64>(); }
    double *vals() const { return (double *)(b.as<u64>() + cap); }
};

struct PrBufs {
    DevBuf names, aux;
    PrTableBuf tab[2];
    cudaEvent_t ev[2] = {nullptr, nullptr};
    int fd = -1;
    ~PrBufs() {
        names.release(); aux.release(); tab[0].b.release(); tab[1].b.release();
        for (int i = 0; i < 2; i++) if (ev[i]) cudaEventDestroy(ev[i]);
        if (fd >= 0) close(fd);
    }
};

static int pr_table_new(tp_ctx *ctx, PrTableBuf *t, u64 cap, const char *who) {
    TP_TRY(device_room(ctx, 16.0 * (double)cap, t->b.cap, who, "the cell table"));
    t->b.release();
    TP_TRY(t->b.reserve((size_t)cap * 16));
    t->cap = cap;
    TP_CUDA(cudaMemsetAsync(t->keys(), 0xff, (size_t)cap * 8, ctx->stream));
    TP_CUDA(cudaMemsetAsync(t->vals(), 0, (size_t)cap * 8, ctx->stream));
    return TP_OK;
}

// the offset of the last '\n' in src's bytes [lo, hi), or -1
static int pr_last_newline(const TextSource &src, size_t lo, size_t hi, long long *out) {
    unsigned char buf[4096];
    *out = -1;
    while (hi > lo) {
        const size_t k = hi - lo < sizeof(buf) ? hi - lo : sizeof(buf);
        TP_TRY(src.fetch(hi - k, k, buf));
        for (size_t j = k; j > 0; j--)
            if (buf[j - 1] == '\n') { *out = (long long)(hi - k + j - 1); return TP_OK; }
        hi -= k;
    }
    return TP_OK;
}

// the message of the lowest bad line, (line << 2) | kind
static int pr_line_error(const char *who, const char *path, u64 bad, int base) {
    const u64 line = bad >> 2;
    const int kind = (int)(bad & 3);
    if (kind == PR_BAD_FIELDS)
        tp_set_error("%s: '%s' line %llu: fewer fields than the columns need", who, path, line);
    else if (kind == PR_BAD_DIGITS)
        tp_set_error("%s: '%s' line %llu: a position is not 1 to 18 digits", who, path, line);
    else
        tp_set_error("%s: '%s' line %llu: a position lies outside its chromosome (positions %d .. length - 1 + %d)", who,
                     path, line, base, base);
    return TP_ERR_ARG;
}

extern "C" int tp_genome_ingest_pairs_file(tp_ctx *ctx, const char *const *paths, int npaths, const char *const *names,
                                           const int64_t *lengths, int nchrom, int64_t binsize, const int cols[4],
                                           int index_base, unsigned long long counts_out[4], tp_genome **out) {
    const char *who = "tp_genome_ingest_pairs_file";
    TP_ARG(ctx && paths && names && lengths && cols && out, "tp_genome_ingest_pairs_file: null argument");
    TP_ARG(npaths >= 1, "tp_genome_ingest_pairs_file: at least one file is needed");
    for (int i = 0; i < npaths; i++) TP_ARG(paths[i], "tp_genome_ingest_pairs_file: null path");
    TP_ARG(binsize >= 1, "tp_genome_ingest_pairs_file: binsize must be >= 1");
    TP_ARG(index_base == 0 || index_base == 1, "tp_genome_ingest_pairs_file: index_base must be 0 or 1");
    TP_ARG(nchrom >= 1 && nchrom <= (1 << 20), "tp_genome_ingest_pairs_file: the number of chromosomes must be in 1..2^20");
    PrCols pc;
    pc.maxcol = 0;
    for (int k = 0; k < 4; k++) {
        TP_ARG(cols[k] >= 0 && cols[k] <= PR_MAXCOL, "tp_genome_ingest_pairs_file: columns must be in 0..63");
        for (int l = 0; l < k; l++) TP_ARG(cols[k] != cols[l], "tp_genome_ingest_pairs_file: the four columns must differ");
        pc.c[k] = cols[k];
        pc.maxcol = std::max(pc.maxcol, cols[k]);
    }
    // the chromosome table: names, lengths, bins
    std::vector<int32_t> bins((size_t)nchrom);
    std::vector<long long> len((size_t)nchrom), noff((size_t)nchrom + 1, 0);
    std::vector<int> starts((size_t)nchrom + 1, 0);
    std::unordered_set<std::string> seen;
    long long total = 0;
    for (int c = 0; c < nchrom; c++) {
        const char *nm = names[c];
        TP_ARG(nm, "tp_genome_ingest_pairs_file: null chromosome name");
        const size_t n = strlen(nm);
        if (n == 0) { tp_set_error("%s: chromosome %d has an empty name", who, c); return TP_ERR_ARG; }
        for (size_t i = 0; i < n; i++)
            if (strchr(" \t\r\n\v\f", nm[i])) {
                tp_set_error("%s: chromosome name '%s' contains whitespace", who, nm);
                return TP_ERR_ARG;
            }
        if (!seen.insert(std::string(nm, n)).second) { tp_set_error("%s: chromosome '%s' appears twice", who, nm); return TP_ERR_ARG; }
        if (lengths[c] < 1) { tp_set_error("%s: chromosome '%s' has length %lld; at least 1 bp is needed", who, nm, (long long)lengths[c]); return TP_ERR_ARG; }
        len[c] = lengths[c];
        noff[c + 1] = noff[c] + (long long)n;
        const long long nb = (lengths[c] - 1) / binsize + 1;
        total += nb;
        if (total >= 0x7fffffffLL) {
            tp_set_error("%s: %lld bp bins give more than 2^31 - 2 bins in all; at most 2^31 - 2 are supported", who, (long long)binsize);
            return TP_ERR_ARG;
        }
        bins[c] = (int32_t)nb;
        starts[c + 1] = starts[c] + (int)nb;
    }
    GenomeOwnerDs own;
    TP_TRY(genome_new(bins.data(), nchrom, index_base, who, &own.g));
    size_t window = PR_WINDOW;
    if (const char *e = getenv("TADPOLE_PAIRS_WINDOW")) {          // test hook: small windows straddle lines, grow the table
        const long long w = atoll(e);
        if (w >= 1) window = (size_t)w;
    }

    TP_CUDA(cudaSetDevice(ctx->device));
    own.g->device = ctx->device;
    cudaStream_t st = ctx->stream;
    const auto t_begin = std::chrono::steady_clock::now();
    PrBufs B;
    for (int i = 0; i < 2; i++) TP_CUDA(cudaEventCreate(&B.ev[i]));

    // the name table sorted by hash, the name blob, lengths and bin starts
    std::vector<std::pair<u64, int>> order((size_t)nchrom);
    std::vector<unsigned char> blob((size_t)noff[nchrom] + 1);
    for (int c = 0; c < nchrom; c++) {
        memcpy(blob.data() + noff[c], names[c], (size_t)(noff[c + 1] - noff[c]));
        order[c] = {pr_name_hash(blob.data() + noff[c], noff[c + 1] - noff[c]), c};
    }
    std::sort(order.begin(), order.end());
    std::vector<u64> hs((size_t)nchrom);
    std::vector<int> hidx((size_t)nchrom);
    for (int k = 0; k < nchrom; k++) { hs[k] = order[k].first; hidx[k] = order[k].second; }
    const size_t n8 = (size_t)nchrom * 8, n8p = ((size_t)nchrom + 1) * 8, n4 = (size_t)nchrom * 4, n4p = ((size_t)nchrom + 1) * 4;
    TP_TRY(B.names.reserve(n8 + n8 + n8p + n4 + n4p + blob.size() + 64));
    PrTable T;
    {
        char *p = B.names.as<char>();
        u64 *dh = (u64 *)p; long long *dlen = (long long *)(p + n8), *dnoff = dlen + nchrom;
        int *didx = (int *)(dnoff + nchrom + 1), *dstarts = didx + nchrom;
        unsigned char *dblob = (unsigned char *)(dstarts + nchrom + 1);
        TP_CUDA(cudaMemcpyAsync(dh, hs.data(), n8, cudaMemcpyHostToDevice, st));
        TP_CUDA(cudaMemcpyAsync(dlen, len.data(), n8, cudaMemcpyHostToDevice, st));
        TP_CUDA(cudaMemcpyAsync(dnoff, noff.data(), n8p, cudaMemcpyHostToDevice, st));
        TP_CUDA(cudaMemcpyAsync(didx, hidx.data(), n4, cudaMemcpyHostToDevice, st));
        TP_CUDA(cudaMemcpyAsync(dstarts, starts.data(), n4p, cudaMemcpyHostToDevice, st));
        TP_CUDA(cudaMemcpyAsync(dblob, blob.data(), blob.size(), cudaMemcpyHostToDevice, st));
        T = PrTable{dh, didx, dnoff, dblob, dlen, dstarts, nchrom};
    }
    // status words on the device, read back through pinned memory so that the read does not stall the host
    TP_TRY(B.aux.reserve(PR_NSTATUS * 8 + (size_t)nchrom * 16));
    u64 *status = B.aux.as<u64>(), *hist = status + PR_NSTATUS, *cursor = hist + nchrom;
    const u64 init[PR_NSTATUS] = {0, 0, 0, 0, 0, ~0ull, 0, 0};
    TP_CUDA(cudaMemcpyAsync(status, init, sizeof(init), cudaMemcpyHostToDevice, st));
    TP_TRY(tp_pin_reserve(ctx, PR_NSTATUS * 8));
    volatile u64 *hstat = (volatile u64 *)ctx->pin;
    int cur = 0;
    TP_TRY(pr_table_new(ctx, &B.tab[cur], 1024, who));

    double dev_ms = 0.0, bytes = 0.0;
    long long windows = 0;
    bool timed = false;                                          // B.ev holds a window's kernels not yet read
    u64 lines_before = 0;
    for (int fi = 0; fi < npaths; fi++) {
        const char *path = paths[fi];
        TextSource src;
        const int rc = open_text_file(path, who, &src);
        B.fd = src.fd;
        if (rc != TP_OK) return rc;
        unsigned char magic[2] = {0, 0};
        if (src.size >= 2) TP_TRY(src.fetch(0, 2, magic));
        if (magic[0] == 0x1f && magic[1] == 0x8b) {
            tp_set_error("%s: '%s' is gzip-compressed; compressed input is not read (decompress it first)", who, path);
            return TP_ERR_ARG;
        }
        u64 line0 = 0;                                           // lines of this file before the window
        size_t off = 0;
        while (off < src.size) {
            size_t end = src.size, next = src.size;
            if (src.size - off > window) {
                long long nl = -1;
                TP_TRY(pr_last_newline(src, off, off + window, &nl));
                if (nl < 0) {
                    // the windows before come first: their lowest bad line is the lowest of the file
                    TP_CUDA(cudaMemcpyAsync((void *)hstat, status, PR_NSTATUS * 8, cudaMemcpyDeviceToHost, st));
                    TP_CUDA(tp_stream_sync(ctx));
                    if (hstat[PR_BAD] != ~0ull) return pr_line_error(who, path, hstat[PR_BAD], index_base);
                    tp_set_error("%s: '%s' line %llu is longer than the device window (%zu bytes)", who, path,
                                 (unsigned long long)(line0 + 1), window);
                    return TP_ERR_ARG;
                }
                end = (size_t)nl;
                next = end + 1;
            } else {
                unsigned char last = 0;
                TP_TRY(src.fetch(src.size - 1, 1, &last));
                if (last == '\n') end = src.size - 1;                // text_rows appends the last line's '\n'
            }
            // the counters of the windows before come back with the line count of this one
            TP_CUDA(cudaMemcpyAsync((void *)hstat, status, PR_NSTATUS * 8, cudaMemcpyDeviceToHost, st));
            unsigned char *text = nullptr;
            int nb = 0;
            long long *offs = nullptr, nrows = 0;
            TP_TRY(text_rows(ctx, src, off, end - off, &text, &nb, &offs, &nrows));
            if (hstat[PR_BAD] != ~0ull) return pr_line_error(who, path, hstat[PR_BAD], index_base);
            if (timed) {
                float ms = 0.f;
                TP_CUDA(cudaEventElapsedTime(&ms, B.ev[0], B.ev[1]));
                dev_ms += ms;
            }
            if (nrows >= 0x7fffffffLL) { tp_set_error("%s: a window of more than 2^31 - 2 lines", who); return TP_ERR_ARG; }
            // growth: occupied + r <= capacity / 2 before the window
            const u64 need = hstat[PR_OCC] + (u64)nrows;
            if (need > B.tab[cur].cap / 2) {
                u64 cap = B.tab[cur].cap * 2;
                while (cap < 2 * need) cap <<= 1;
                PrTableBuf &o = B.tab[cur], &t = B.tab[cur ^ 1];
                TP_TRY(pr_table_new(ctx, &t, cap, who));
                pr_rehash_kernel<<<ds_grid(ctx, o.cap), DS_THREADS, 0, st>>>(o.keys(), o.vals(), o.cap, t.keys(), t.vals(), cap - 1);
                TP_CUDA(cudaGetLastError());
                ctx->launches += 1;
                cur ^= 1;
                TP_CUDA(tp_stream_sync(ctx));                        // the old table is released before the next growth
                B.tab[cur ^ 1].b.release();
                B.tab[cur ^ 1].cap = 0;
            }
            long long *row_end = nullptr;
            TP_CUDA(cudaEventRecord(B.ev[0], st));
            TP_TRY(text_line_ends(ctx, text, end - off, nb, offs, nrows, &row_end));
            pr_parse_kernel<<<(unsigned)((nrows + PR_THREADS - 1) / PR_THREADS), PR_THREADS, 0, st>>>(
                text, row_end, (unsigned)nrows, line0, pc, T, (long long)binsize, index_base, B.tab[cur].keys(),
                B.tab[cur].vals(), B.tab[cur].cap - 1, status);
            TP_CUDA(cudaGetLastError());
            TP_CUDA(cudaEventRecord(B.ev[1], st));
            ctx->launches += 1;
            timed = true;
            windows++;
            bytes += (double)(next - off);
            line0 += (u64)nrows;
            off = next;
        }
        TP_CUDA(cudaMemcpyAsync((void *)hstat, status, PR_NSTATUS * 8, cudaMemcpyDeviceToHost, st));
        TP_CUDA(tp_stream_sync(ctx));
        if (hstat[PR_BAD] != ~0ull) return pr_line_error(who, path, hstat[PR_BAD], index_base);
        if (hstat[PR_LINES] == lines_before) {
            tp_set_error("%s: '%s' holds no pair lines", who, path);
            return TP_ERR_ARG;
        }
        lines_before = hstat[PR_LINES];
        close(src.fd);
        B.fd = -1;
    }
    if (timed) {
        float ms = 0.f;
        TP_CUDA(cudaEventElapsedTime(&ms, B.ev[0], B.ev[1]));
        dev_ms += ms;
    }
    const u64 counts[4] = {hstat[PR_LINES], hstat[PR_CIS], hstat[PR_TRANS], hstat[PR_UNPLACED]};
    ctx->itext.release();                                        // the text is parsed
    ctx->irows.release();

    // the buckets
    const PrTableBuf &tb = B.tab[cur];
    int *dstarts = (int *)T.starts;
    TP_CUDA(cudaMemsetAsync(hist, 0, (size_t)nchrom * 8, st));
    cs_count_kernel<<<ds_grid(ctx, tb.cap), DS_THREADS, 0, st>>>(tb.keys(), tb.vals(), tb.cap, dstarts, nchrom, hist);
    ctx->launches += 1;
    TP_CUDA(cudaGetLastError());
    std::vector<u64> h((size_t)nchrom, 0);
    TP_CUDA(cudaMemcpyAsync(h.data(), hist, (size_t)nchrom * 8, cudaMemcpyDeviceToHost, st));
    TP_CUDA(tp_stream_sync(ctx));
    own.g->offs.assign((size_t)nchrom + 1, 0);
    for (int c = 0; c < nchrom; c++) own.g->offs[c + 1] = own.g->offs[c] + h[c];
    own.g->trans = counts[2];
    own.g->below = 0;
    const u64 ncell = own.g->offs[nchrom];
    TP_TRY(device_room(ctx, 16.0 * (double)ncell, 0, who, "the buckets of the cis cells"));
    TP_TRY(own.g->px.reserve((size_t)ncell * 16 + 16));
    if (ncell) {
        double *ov = own.g->px.as<double>();
        int *oi = (int *)(ov + ncell), *oj = oi + ncell;
        TP_CUDA(cudaMemcpyAsync(cursor, own.g->offs.data(), (size_t)nchrom * 8, cudaMemcpyHostToDevice, st));
        cs_scatter_kernel<<<ds_grid(ctx, tb.cap), DS_THREADS, 0, st>>>(tb.keys(), tb.vals(), tb.cap, dstarts, nchrom, cursor, ov,
                                                                      oi, oj);
        ctx->launches += 1;
        TP_CUDA(cudaGetLastError());
    }
    TP_CUDA(tp_stream_sync(ctx));
    ctx->ingest_stats[0] = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t_begin).count();
    ctx->ingest_stats[1] = dev_ms;
    ctx->ingest_stats[2] = bytes;
    ctx->ingest_stats[3] = (double)windows;
    if (counts_out) for (int k = 0; k < 4; k++) counts_out[k] = counts[k];
    *out = own.g;
    own.g = nullptr;
    return TP_OK;
}
