// api.cu -- C ABI of libsnacc_b200.so (see include/snacc_b200.h): argument checks, the context lock, the corpus upload,
// the dispatch of sizes calls to the codec drivers (lz4_driver.cuh, deflate.cuh, bzip2.cuh) and the epilogues.  No
// torch, no C++ types across the boundary, no exceptions escape.
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>
#include <stdlib.h>
#include <string>
#include <vector>
#include <charconv>
#include <thread>
#include <cmath>
#include <cstdio>
#include <algorithm>
#include <mutex>

#include "../../include/snacc_b200.h"
// The kernel headers come first, in this order, and the LZ4 driver (which instantiates the packed kernel templates)
// last: the order in which kernels enter the module steers the device compiler's inlining -- with the driver earlier,
// dfl_alone_kernel no longer inlines dfl_flush_block and spills.
#include "common.cuh"
#include "lz4.cuh"
#include "pack.cuh"
#include "lz4_packed.cuh"
#include "deflate.cuh"
#include "upgma.cuh"
#include "bzip2.cuh"
#include "lz4_driver.cuh"

using namespace snacc;

#define SNACC_VERSION 100   /* 0.1.0 */

struct snacc_ctx {
    int device = 0;
    cudaStream_t stream = nullptr;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    std::string err;
    std::mutex mu;                 // serialises calls: the single-job shim may be hit from many threads

    // corpus (device)
    int32_t n_seqs = 0;
    uint8_t *d_corpus = nullptr;   // padded layout
    uint64_t corpus_bytes = 0;
    uint64_t *d_off = nullptr;     // n_seqs offsets into d_corpus
    uint32_t *d_len = nullptr;     // n_seqs lengths
    std::vector<uint64_t> h_off;
    std::vector<uint32_t> h_len;

    // codec state (corpus-derived caches, working memory, options, statistics)
    Lz4State lz4;
    DeflateState dfl;
    BzState bz;

    // working memory, grown on demand and never freed between calls (all use is ordered on `stream`): upload staging,
    // the job arrays and sizes of a call, the NCD epilogue's arrays, and the LZ4 byte-wise tables or bzip2 global-sort
    // scratch (one buffer: a session that mixes codecs holds the larger of the two, not both)
    DevBuf staging, jobx, joby, out, ncd_c, ncd_s, ncd_d, work;

    // instrumentation
    double last_ms = 0.0; int64_t last_launches = 0;
    double last_main_ms = 0.0;              // dominant kernel only (lz4_stream_kernel / deflate pair kernel)
};

#define CK(call) do { cudaError_t e_ = (call); if (e_ != cudaSuccess) { \
        char b_[512]; snprintf(b_, sizeof b_, "%s failed at %s:%d: %s", #call, __FILE__, __LINE__, cudaGetErrorString(e_)); \
        ctx->err = b_; return SNACC_ERR_CUDA; } } while (0)
#define FAIL(code, msg) do { ctx->err = (msg); return (code); } while (0)

// the uploaded corpus as the codec drivers see it
static Corpus corpus(const snacc_ctx *ctx)
{
    return Corpus{ctx->d_corpus, ctx->d_off, ctx->d_len, ctx->h_off.data(), ctx->h_len.data(), ctx->n_seqs};
}


// ---------------------------------------------------------------------------------------------
// K0: scatter records into the padded corpus, optionally reverse-complementing each record
// (Biopython ambiguous-DNA table, case preserving; pairwise_ncd.py:33-34)
// ---------------------------------------------------------------------------------------------
__constant__ uint8_t c_complement[256];

static void build_complement_table(uint8_t *t)
{
    for (int i = 0; i < 256; ++i) t[i] = (uint8_t)i;
    const char *a = "ACGTMRWSYKVHDBXNU";
    const char *b = "TGCAKYWSRMBDHVXNA";
    for (int i = 0; a[i]; ++i) {
        t[(uint8_t)a[i]] = (uint8_t)b[i];
        t[(uint8_t)(a[i] | 0x20)] = (uint8_t)(b[i] | 0x20);
    }
}

__global__ void scatter_records_kernel(const uint8_t *__restrict__ src, uint64_t total,
                                       const uint64_t *__restrict__ rec_off, int64_t n_recs,
                                       const uint64_t *__restrict__ rec_dst, int rc,
                                       uint8_t *__restrict__ dst)
{
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += stride) {
        // record containing source byte i: last r with rec_off[r] <= i
        int64_t lo = 0, hi = n_recs;
        while (hi - lo > 1) {
            int64_t mid = (lo + hi) >> 1;
            if (rec_off[mid] <= i) lo = mid; else hi = mid;
        }
        const uint64_t a = rec_off[lo], b = rec_off[lo + 1];
        const uint64_t k = i - a;
        uint8_t v = src[i];
        if (rc) dst[rec_dst[lo] + (b - a - 1 - k)] = c_complement[v];
        else    dst[rec_dst[lo] + k] = v;
    }
}

// ---------------------------------------------------------------------------------------------
// K4: NCD epilogue in float64 (two correctly rounded divides and a min, like the reference)
// ---------------------------------------------------------------------------------------------
__global__ void ncd_kernel(const int64_t *__restrict__ C, const int64_t *__restrict__ S, int32_t n,
                           int formula, int64_t bias, double *__restrict__ D)
{
    const int64_t total = (int64_t)n * n;
    for (int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; k < total;
         k += (int64_t)gridDim.x * blockDim.x) {
        const int32_t i = (int32_t)(k / n), j = (int32_t)(k % n);
        const int64_t x = C[i] + bias, y = C[j] + bias;
        const int64_t lo = x < y ? x : y, hi = x < y ? y : x;
        const int64_t cxy = S[(int64_t)i * n + j] + bias;
        const double d1 = __ddiv_rn((double)(cxy - lo), (double)hi);
        if (formula == SNACC_NCD_ONE_ORDER) { D[k] = d1; continue; }
        const int64_t cyx = S[(int64_t)j * n + i] + bias;
        const double d2 = __ddiv_rn((double)(cyx - lo), (double)hi);
        D[k] = d1 < d2 ? d1 : d2;
    }
}

// ---------------------------------------------------------------------------------------------
extern "C" int snacc_version(void) { return SNACC_VERSION; }

// Host-side FASTA record scan (no GPU involved): the residues of every record of `raw` with the reference's line
// handling -- the file is read in text mode (universal newlines: "\n", "\r\n" and a lone "\r" all end a line), a
// record starts at a line that begins with '>', everything before the first one is ignored, every sequence line is
// right-stripped of white space (9-13, 32) and loses its blanks (pairwise_ncd.py:32-36 over Bio.SeqIO /
// SimpleFastaParser).  out needs room for n bytes.  Returns the number of records (their lengths in
// rec_len[0 .. min(records, max_recs))), *out_len = residues written.
namespace {
struct FastaScan {
    uint8_t *out; uint64_t *rec_len; int64_t max_recs;
    uint64_t w = 0, cur = 0; int64_t recs = 0; bool in_rec = false;
    static bool is_ws(uint8_t c) { return (c >= 9 && c <= 13) || c == 32; }
    void close_record() { if (in_rec && recs - 1 < max_recs && rec_len) rec_len[recs - 1] = cur; }
    void line(const uint8_t *a, const uint8_t *b)                 // one line without its terminator
    {
        if (b > a && *a == '>') { close_record(); in_rec = true; ++recs; cur = 0; return; }
        if (!in_rec) return;
        while (b > a && is_ws(b[-1])) --b;
        if (b == a) return;
        if (!memchr(a, ' ', (size_t)(b - a))) {                   // the usual line: nothing to drop inside it
            memcpy(out + w, a, (size_t)(b - a)); w += (uint64_t)(b - a); cur += (uint64_t)(b - a);
        } else {
            for (; a < b; ++a) if (*a != ' ') { out[w++] = *a; ++cur; }
        }
    }
};
}  // namespace

// ---- CSV of the distance matrix (host side, no GPU) -----------------------------------------------------------------
// What DataFrame.pivot(...).to_csv writes for the reference (cli.py:138-142): one row per file, cells = the float64 as
// Python's repr() prints it -- the shortest digit string that reads back to the same double, fixed notation when the
// decimal exponent is in (-4, 16], exponent notation (two exponent digits at least) otherwise, ".0" appended to whole
// numbers, NaN as an empty cell.  std::to_chars produces the shortest digits; the layout rules are applied here.
namespace {
static char *csv_put_double(char *o, double v)
{
    if (v != v) return o;                                         // NaN: empty cell
    if (v == HUGE_VAL || v == -HUGE_VAL) { if (v < 0) *o++ = '-'; memcpy(o, "inf", 3); return o + 3; }
    char buf[40];
    // scientific, shortest round trip: [-]d[.ddd]e[+-]XX
    const std::to_chars_result r = std::to_chars(buf, buf + sizeof buf, v, std::chars_format::scientific);
    const char *p = buf, *end = r.ptr;
    if (*p == '-') { *o++ = '-'; ++p; }
    const char *e = p;
    while (e < end && *e != 'e') ++e;
    char digits[24]; int nd = 0;
    for (const char *q = p; q < e; ++q) if (*q != '.') digits[nd++] = *q;
    int ex = 0;
    {
        const char *q = e + 1; bool neg = false;
        if (*q == '-') { neg = true; ++q; } else if (*q == '+') ++q;
        for (; q < end; ++q) ex = ex * 10 + (*q - '0');
        if (neg) ex = -ex;
    }
    const int decpt = ex + 1;                                     // value = 0.d1d2... x 10^decpt
    if (decpt > -4 && decpt <= 16) {
        if (decpt <= 0) {
            *o++ = '0'; *o++ = '.';
            for (int k = 0; k < -decpt; ++k) *o++ = '0';
            memcpy(o, digits, (size_t)nd); o += nd;
        } else if (decpt >= nd) {
            memcpy(o, digits, (size_t)nd); o += nd;
            for (int k = nd; k < decpt; ++k) *o++ = '0';
            *o++ = '.'; *o++ = '0';
        } else {
            memcpy(o, digits, (size_t)decpt); o += decpt;
            *o++ = '.';
            memcpy(o, digits + decpt, (size_t)(nd - decpt)); o += nd - decpt;
        }
    } else {
        *o++ = digits[0];
        if (nd > 1) { *o++ = '.'; memcpy(o, digits + 1, (size_t)(nd - 1)); o += nd - 1; }
        *o++ = 'e';
        int x = decpt - 1;
        if (x < 0) { *o++ = '-'; x = -x; } else *o++ = '+';
        if (x >= 100) { *o++ = (char)('0' + x / 100); x %= 100; *o++ = (char)('0' + x / 10); *o++ = (char)('0' + x % 10); }
        else { *o++ = (char)('0' + x / 10); *o++ = (char)('0' + x % 10); }
    }
    return o;
}
}  // namespace

extern "C" int snacc_csv_write(const char *path, const char *header_line, const char *const *row_labels, const double *D,
                               int64_t n, const int32_t *order, int threads)
{
    if (!path || !header_line || !row_labels || !D || !order || n < 0) return SNACC_ERR_ARG;
    FILE *f = fopen(path, "wb");
    if (!f) return SNACC_ERR_ARG;
    bool ok = fputs(header_line, f) >= 0 && fputc('\n', f) != EOF;
    // rows are formatted in blocks by a few threads, each into its own buffer, and written in order
    const int T = (int)std::max<int64_t>(1, std::min<int64_t>(threads > 0 ? threads : (int)std::thread::hardware_concurrency(), 64));
    const int64_t rows_per_block = std::max<int64_t>(1, std::min<int64_t>(256, (4 << 20) / std::max<int64_t>(1, n)));
    const int64_t per_round = rows_per_block * T;
    std::vector<std::vector<char>> bufs((size_t)T);
    for (int64_t r0 = 0; r0 < n && ok; r0 += per_round) {
        std::vector<std::thread> pool;
        for (int t = 0; t < T; ++t) {
            const int64_t a = r0 + t * rows_per_block, b = std::min<int64_t>(n, a + rows_per_block);
            bufs[(size_t)t].clear();
            if (a >= b) continue;
            pool.emplace_back([&, t, a, b]() {
                std::vector<char> &buf = bufs[(size_t)t];
                size_t labels = 0;
                for (int64_t r = a; r < b; ++r) labels += strlen(row_labels[order[r]]);
                buf.resize(labels + (size_t)(b - a) * ((size_t)n * 26 + 2));
                char *o = buf.data();
                for (int64_t r = a; r < b; ++r) {
                    const int32_t i = order[r];
                    const size_t ll = strlen(row_labels[i]);
                    memcpy(o, row_labels[i], ll); o += ll;
                    const double *row = D + (size_t)i * (size_t)n;
                    for (int64_t c = 0; c < n; ++c) { *o++ = ','; o = csv_put_double(o, row[order[c]]); }
                    *o++ = '\n';
                }
                buf.resize((size_t)(o - buf.data()));
            });
        }
        for (std::thread &th : pool) th.join();
        for (int t = 0; t < T && ok; ++t)
            if (!bufs[(size_t)t].empty()) ok = fwrite(bufs[(size_t)t].data(), 1, bufs[(size_t)t].size(), f) == bufs[(size_t)t].size();
    }
    ok = (fclose(f) == 0) && ok;
    return ok ? SNACC_OK : SNACC_ERR_ARG;
}

extern "C" int64_t snacc_fasta_parse(const uint8_t *raw, uint64_t n, uint8_t *out, uint64_t *out_len, uint64_t *rec_len,
                                     int64_t max_recs)
{
    if ((n && !raw) || !out || !out_len) return SNACC_ERR_ARG;
    FastaScan sc{out, rec_len, max_recs};
    for (uint64_t a = 0; a < n;) {
        const uint8_t *nl = (const uint8_t *)memchr(raw + a, '\n', n - a);
        const uint64_t b = nl ? (uint64_t)(nl - raw) : n;        // raw[a, b): text up to the next "\n"
        const uint8_t *cr = b > a ? (const uint8_t *)memchr(raw + a, '\r', b - a) : nullptr;
        if (!cr || (uint64_t)(cr - raw) == b - 1) {
            sc.line(raw + a, raw + b - (cr ? 1 : 0));            // no carriage return, or the "\r" of a "\r\n"
        } else {
            uint64_t s = a;                                      // lone carriage returns end lines too
            while (cr) {
                sc.line(raw + s, cr);
                s = (uint64_t)(cr - raw) + 1;
                cr = s < b ? (const uint8_t *)memchr(raw + s, '\r', b - s) : nullptr;
            }
            if (s < b || !nl) sc.line(raw + s, raw + b);         // (an "\r" right before the "\n" is one terminator)
        }
        a = b + 1;
    }
    sc.close_record();
    *out_len = sc.w;
    return sc.recs;
}

extern "C" const char *snacc_last_error(const snacc_ctx *ctx) { return ctx ? ctx->err.c_str() : "null context"; }

static void free_corpus(snacc_ctx *ctx)
{
    cudaFree(ctx->d_corpus); ctx->d_corpus = nullptr;
    cudaFree(ctx->d_off); ctx->d_off = nullptr;
    cudaFree(ctx->d_len); ctx->d_len = nullptr;
    ctx->n_seqs = 0;
    lz4_free_corpus(ctx->lz4);
    bz_free_corpus(ctx->bz);
    deflate_free_corpus(ctx->dfl);
}

// forget every per-sequence precomputation (prefix checkpoints, RLE1, deflate records ...) of every codec
static void invalidate_caches(snacc_ctx *ctx)
{
    lz4_invalidate(ctx->lz4);
    bz_invalidate(ctx->bz);
    deflate_invalidate(ctx->dfl);
}

extern "C" int snacc_ctx_create(int device_id, snacc_ctx **out)
{
    if (!out) return SNACC_ERR_ARG;
    *out = nullptr;
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess || device_id < 0 || device_id >= n) return SNACC_ERR_CUDA;
    snacc_ctx *ctx = new (std::nothrow) snacc_ctx();
    if (!ctx) return SNACC_ERR_ARG;
    ctx->device = device_id;
    if (cudaSetDevice(device_id) != cudaSuccess ||
        cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking) != cudaSuccess ||
        cudaEventCreate(&ctx->ev0) != cudaSuccess || cudaEventCreate(&ctx->ev1) != cudaSuccess) {
        delete ctx;
        return SNACC_ERR_CUDA;
    }
    uint8_t tab[256];
    build_complement_table(tab);
    if (cudaMemcpyToSymbol(c_complement, tab, 256) != cudaSuccess) { delete ctx; return SNACC_ERR_CUDA; }
    *out = ctx;
    return SNACC_OK;
}

extern "C" void snacc_ctx_destroy(snacc_ctx *ctx)
{
    if (!ctx) return;
    cudaSetDevice(ctx->device);
    cudaStreamSynchronize(ctx->stream);
    free_corpus(ctx);
    lz4_free_work(ctx->lz4);
    bz_free_work(ctx->bz);
    deflate_free_work(ctx->dfl);
    for (DevBuf *b : {&ctx->staging, &ctx->jobx, &ctx->joby, &ctx->out, &ctx->ncd_c, &ctx->ncd_s, &ctx->ncd_d, &ctx->work})
        b->release();
    cudaEventDestroy(ctx->ev0); cudaEventDestroy(ctx->ev1);
    cudaStreamDestroy(ctx->stream);
    delete ctx;
}

static int upload_impl(snacc_ctx *ctx, const void *bytes, bool on_device, const uint64_t *seq_offsets,
                       int32_t n_seqs, const uint64_t *rec_offsets, int64_t n_recs, int rc)
{
    NvtxRange nvtx_("snacc_b200: upload (scatter records, reverse complement)");
    if (!ctx) return SNACC_ERR_ARG;
    std::lock_guard<std::mutex> lock(ctx->mu);
    ctx->err.clear();
    if (!seq_offsets || n_seqs <= 0) FAIL(SNACC_ERR_ARG, "snacc_upload: no sequences");
    if (rc && (!rec_offsets || n_recs <= 0)) FAIL(SNACC_ERR_ARG, "snacc_upload: reverse complement needs record offsets");
    const uint64_t total = seq_offsets[n_seqs] - seq_offsets[0];
    if (!bytes && total) FAIL(SNACC_ERR_ARG, "snacc_upload: null bytes");
    for (int32_t i = 0; i < n_seqs; ++i) {
        if (seq_offsets[i + 1] < seq_offsets[i]) FAIL(SNACC_ERR_ARG, "snacc_upload: offsets not monotone");
        const uint64_t l = seq_offsets[i + 1] - seq_offsets[i];
        if (l == 0) {
            char b[128]; snprintf(b, sizeof b, "sequence %d is empty (no sequence extracted)", i);
            FAIL(SNACC_ERR_EMPTY, b);
        }
        if (l >= 0x7fffffffull) FAIL(SNACC_ERR_TOO_LARGE, "snacc_upload: sequence of 2 GiB or more");
    }
    // records default to whole sequences
    std::vector<uint64_t> recs;
    if (!rec_offsets) { recs.assign(seq_offsets, seq_offsets + n_seqs + 1); n_recs = n_seqs; }
    else recs.assign(rec_offsets, rec_offsets + n_recs + 1);
    if (recs.front() != seq_offsets[0] || recs.back() != seq_offsets[n_seqs])
        FAIL(SNACC_ERR_ARG, "snacc_upload: record offsets do not cover the sequences");

    // everything is validated before the previous corpus is dropped: a rejected upload leaves the context as it was
    std::vector<uint64_t> h_off((size_t)n_seqs);
    std::vector<uint32_t> h_len((size_t)n_seqs);
    uint64_t pos = 0;
    for (int32_t i = 0; i < n_seqs; ++i) {
        h_off[i] = pos;
        h_len[i] = (uint32_t)(seq_offsets[i + 1] - seq_offsets[i]);
        pos += ((uint64_t)h_len[i] + SEQ_PAD + SEQ_ALIGN - 1) & ~(uint64_t)(SEQ_ALIGN - 1);
    }
    // destination of every record
    std::vector<uint64_t> rec_dst((size_t)n_recs);
    {
        int32_t si = 0;
        for (int64_t r = 0; r < n_recs; ++r) {
            if (recs[r + 1] < recs[r]) FAIL(SNACC_ERR_ARG, "snacc_upload: record offsets not monotone");
            if (recs[r + 1] == recs[r]) { rec_dst[r] = 0; continue; }   // empty record: moves no bytes
            while (si < n_seqs && recs[r] >= seq_offsets[si + 1]) ++si;
            if (si >= n_seqs || recs[r] < seq_offsets[si] || recs[r + 1] > seq_offsets[si + 1])
                FAIL(SNACC_ERR_ARG, "snacc_upload: a record straddles two sequences or lies outside them");
            rec_dst[r] = h_off[si] + (recs[r] - seq_offsets[si]);
        }
    }
    CK(cudaSetDevice(ctx->device));
    // a corpus of the same shape as the previous one (same sequence lengths: every e2e step of bench.py, any re-upload
    // with another reverse-complement flag) keeps every device buffer -- tens of GB for the deflate codecs -- and only
    // forgets what was computed from the old bytes
    const bool same_shape = ctx->n_seqs == n_seqs && ctx->d_corpus && ctx->h_len == h_len;
    if (same_shape) {
        invalidate_caches(ctx);
        ctx->n_seqs = 0;                                     // (restored below; a failure in between leaves no corpus)
    } else {
        free_corpus(ctx);
    }
    ctx->h_off.swap(h_off); ctx->h_len.swap(h_len);
    ctx->corpus_bytes = pos + 64;
    for (auto &v : recs) v -= seq_offsets[0];

    if (!ctx->d_corpus) CK(cudaMalloc(&ctx->d_corpus, ctx->corpus_bytes));
    CK(cudaMemsetAsync(ctx->d_corpus, 0, ctx->corpus_bytes, ctx->stream));
    if (!ctx->d_off) CK(cudaMalloc(&ctx->d_off, sizeof(uint64_t) * n_seqs));
    if (!ctx->d_len) CK(cudaMalloc(&ctx->d_len, sizeof(uint32_t) * n_seqs));
    CK(cudaMemcpyAsync(ctx->d_off, ctx->h_off.data(), sizeof(uint64_t) * n_seqs, cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaMemcpyAsync(ctx->d_len, ctx->h_len.data(), sizeof(uint32_t) * n_seqs, cudaMemcpyHostToDevice, ctx->stream));

    uint8_t *d_src = nullptr; uint64_t *d_rec_off = nullptr, *d_rec_dst = nullptr;
    const uint8_t *src_dev = nullptr;
    if (on_device) src_dev = (const uint8_t *)bytes + 0;
    else {
        CK(ctx->staging.grow(total ? total : 1, ctx->stream));    // staging copy of the host bytes (kept: no malloc per upload)
        d_src = ctx->staging.get<uint8_t>();
        CK(cudaMemcpyAsync(d_src, (const uint8_t *)bytes + seq_offsets[0], total, cudaMemcpyHostToDevice, ctx->stream));
        src_dev = d_src;
    }
    if (on_device) src_dev += seq_offsets[0];
    CK(cudaMalloc(&d_rec_off, sizeof(uint64_t) * (n_recs + 1)));
    CK(cudaMalloc(&d_rec_dst, sizeof(uint64_t) * n_recs));
    CK(cudaMemcpyAsync(d_rec_off, recs.data(), sizeof(uint64_t) * (n_recs + 1), cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaMemcpyAsync(d_rec_dst, rec_dst.data(), sizeof(uint64_t) * n_recs, cudaMemcpyHostToDevice, ctx->stream));
    {
        const int threads = 256;
        const uint64_t want = (total + threads - 1) / threads;
        const int blocks = (int)std::min<uint64_t>(std::max<uint64_t>(want, 1), 148ull * 16);
        scatter_records_kernel<<<blocks, threads, 0, ctx->stream>>>(src_dev, total, d_rec_off, n_recs, d_rec_dst,
                                                                    rc ? 1 : 0, ctx->d_corpus);
        CK(cudaGetLastError());
    }

    CK(cudaStreamSynchronize(ctx->stream));
    cudaFree(d_rec_off); cudaFree(d_rec_dst);
    ctx->n_seqs = n_seqs;
    return lz4_prepare(ctx->lz4, corpus(ctx), ctx->stream, ctx->err);
}

extern "C" int snacc_upload(snacc_ctx *ctx, const uint8_t *bytes, const uint64_t *seq_offsets, int32_t n_seqs,
                            const uint64_t *rec_offsets, int64_t n_recs, int reverse_complement)
{
    return upload_impl(ctx, bytes, false, seq_offsets, n_seqs, rec_offsets, n_recs, reverse_complement);
}

extern "C" int snacc_upload_device(snacc_ctx *ctx, const void *d_bytes, const uint64_t *seq_offsets, int32_t n_seqs,
                                   const uint64_t *rec_offsets, int64_t n_recs, int reverse_complement)
{
    return upload_impl(ctx, d_bytes, true, seq_offsets, n_seqs, rec_offsets, n_recs, reverse_complement);
}

extern "C" int snacc_download_sequence(snacc_ctx *ctx, int32_t i, uint8_t *out)
{
    if (!ctx || !out) return SNACC_ERR_ARG;
    std::lock_guard<std::mutex> lock(ctx->mu);
    if (!ctx->n_seqs) FAIL(SNACC_ERR_STATE, "nothing uploaded");
    if (i < 0 || i >= ctx->n_seqs) FAIL(SNACC_ERR_ARG, "sequence index out of range");
    CK(cudaSetDevice(ctx->device));
    CK(cudaMemcpy(out, ctx->d_corpus + ctx->h_off[i], ctx->h_len[i], cudaMemcpyDeviceToHost));
    return SNACC_OK;
}

static int64_t wrapper_bytes(int codec) { return codec == SNACC_GZIP9 ? 18 : codec == SNACC_ZLIB6 ? 6 : 0; }

// a tile of the ordered-pair matrix: rows [row0, row0 + n_rows) x columns [col0, col0 + n_cols), jobs in row-major order
struct Tile { int32_t row0, n_rows, col0, n_cols; };

// The sizes of a job list (xs, ys; ys null for singles) or, with xs null, of a tile, into out[0, n_jobs).  The whole
// call holds the lock: validation, the codec's run (an LZ4 tile that is uniform enough as one rectangle, everything
// else as a job list), the copy to the host, the LZ4 redo of handed-off streams, the wrapper bytes.
static int sizes_impl(snacc_ctx *ctx, int codec, const int32_t *xs, const int32_t *ys, int64_t n_jobs, const Tile *tile,
                      int64_t *out)
{
    if (!ctx) return SNACC_ERR_ARG;
    std::lock_guard<std::mutex> lock(ctx->mu);
    ctx->err.clear();
    if (!ctx->n_seqs) FAIL(SNACC_ERR_STATE, "nothing uploaded");
    if (codec != SNACC_LZ4F && codec != SNACC_GZIP9 && codec != SNACC_ZLIB6 && codec != SNACC_BZIP2_9)
        FAIL(SNACC_ERR_CODEC, "codec not supported on the GPU path (supported: lz4, gzip, zlib, bzip2)");
    if (n_jobs < 0 || (n_jobs && ((!tile && !xs) || !out))) FAIL(SNACC_ERR_ARG, "bad job list");
    if (n_jobs == 0) return SNACC_OK;
    if (tile) {
        if ((int64_t)tile->row0 + tile->n_rows > ctx->n_seqs || (int64_t)tile->col0 + tile->n_cols > ctx->n_seqs)
            FAIL(SNACC_ERR_ARG, "sequence index out of range");
        uint32_t max_x = 0, max_y = 0;
        for (int32_t r = 0; r < tile->n_rows; ++r) max_x = std::max(max_x, ctx->h_len[tile->row0 + r]);
        for (int32_t c = 0; c < tile->n_cols; ++c) max_y = std::max(max_y, ctx->h_len[tile->col0 + c]);
        if ((uint64_t)max_x + max_y >= 0x7fffffffull) FAIL(SNACC_ERR_TOO_LARGE, "pair stream of 2 GiB or more");
    } else {
        for (int64_t k = 0; k < n_jobs; ++k) {
            if (xs[k] < 0 || xs[k] >= ctx->n_seqs || (ys && (ys[k] < 0 || ys[k] >= ctx->n_seqs)))
                FAIL(SNACC_ERR_ARG, "sequence index out of range");
            if (ys && (uint64_t)ctx->h_len[xs[k]] + ctx->h_len[ys[k]] >= 0x7fffffffull)
                FAIL(SNACC_ERR_TOO_LARGE, "pair stream of 2 GiB or more");
        }
    }
    CK(cudaSetDevice(ctx->device));
    const Corpus c = corpus(ctx);
    CK(ctx->out.grow(sizeof(int64_t) * n_jobs, ctx->stream, true));
    int64_t *d_out = ctx->out.get<int64_t>();
    const int regime = tile && codec == SNACC_LZ4F
                     ? lz4_rect_regime(ctx->lz4, c, tile->row0, tile->n_rows, tile->col0, tile->n_cols) : 0;
    std::vector<int32_t> txs, tys;
    if (tile && !regime) {
        txs.resize((size_t)n_jobs); tys.resize((size_t)n_jobs);
        for (int32_t r = 0; r < tile->n_rows; ++r)
            for (int32_t col = 0; col < tile->n_cols; ++col) {
                txs[(size_t)r * tile->n_cols + col] = tile->row0 + r;
                tys[(size_t)r * tile->n_cols + col] = tile->col0 + col;
            }
        xs = txs.data(); ys = tys.data();
    }
    if (!regime) {
        CK(ctx->jobx.grow(sizeof(int32_t) * n_jobs, ctx->stream, true));
        CK(cudaMemcpyAsync(ctx->jobx.p, xs, sizeof(int32_t) * n_jobs, cudaMemcpyHostToDevice, ctx->stream));
        if (ys) {
            CK(ctx->joby.grow(sizeof(int32_t) * n_jobs, ctx->stream, true));
            CK(cudaMemcpyAsync(ctx->joby.p, ys, sizeof(int32_t) * n_jobs, cudaMemcpyHostToDevice, ctx->stream));
        }
    }
    const int32_t *d_xs = ctx->jobx.get<int32_t>(), *d_ys = ys ? ctx->joby.get<int32_t>() : nullptr;
    int64_t *launches = &ctx->last_launches;
    *launches = 0;
    CK(cudaEventRecord(ctx->ev0, ctx->stream));
    int r;
    if (regime)
        r = lz4_run_rect(ctx->lz4, c, regime, tile->row0, tile->n_rows, tile->col0, tile->n_cols, d_out, ctx->stream,
                         launches, ctx->err);
    else if (codec == SNACC_LZ4F)
        r = lz4_run(ctx->lz4, c, xs, ys, d_xs, d_ys, n_jobs, d_out, ctx->work, ctx->stream, launches, ctx->err);
    else if (codec == SNACC_BZIP2_9)
        r = bz_run(ctx->bz, c, xs, ys, d_xs, n_jobs, d_out, ctx->work, ctx->stream, launches, ctx->err);
    else
        r = deflate_run(ctx->dfl, c, codec == SNACC_GZIP9 ? 9 : 6, xs, ys, d_xs, n_jobs, d_out, ctx->stream, launches,
                        ctx->err);
    if (r) return r;
    CK(cudaEventRecord(ctx->ev1, ctx->stream));
    CK(cudaMemcpyAsync(out, d_out, sizeof(int64_t) * n_jobs, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    float ms = 0.f;
    CK(cudaEventElapsedTime(&ms, ctx->ev0, ctx->ev1));
    ctx->last_ms = ms;
    if (codec == SNACC_LZ4F) {
        r = lz4_finish(ctx->lz4, c, xs, ys, tile ? tile->row0 : 0, tile ? tile->col0 : 0, tile ? tile->n_cols : 0, n_jobs,
                       out, d_out, ctx->work, ctx->stream, launches, ctx->err);
        if (r) return r;
        ctx->last_main_ms = ctx->lz4.main_ms;
    } else if (codec == SNACC_BZIP2_9) {
        ctx->last_main_ms = ctx->bz.ms[1] + ctx->bz.ms[2];
    } else {
        ctx->last_main_ms = ctx->dfl.main_ms;
    }
    const int64_t wb = wrapper_bytes(codec);
    if (wb) for (int64_t k = 0; k < n_jobs; ++k) out[k] += wb;
    return SNACC_OK;
}

extern "C" int snacc_single_sizes(snacc_ctx *ctx, int codec, const int32_t *idx, int64_t n, int64_t *out)
{
    return sizes_impl(ctx, codec, idx, nullptr, n, nullptr, out);
}

extern "C" int snacc_pair_sizes(snacc_ctx *ctx, int codec, const int32_t *xs, const int32_t *ys, int64_t n_jobs,
                                int64_t *out)
{
    if (n_jobs && !ys) return SNACC_ERR_ARG;
    return sizes_impl(ctx, codec, xs, ys, n_jobs, nullptr, out);
}

extern "C" int snacc_tile_sizes(snacc_ctx *ctx, int codec, int32_t row0, int32_t n_rows, int32_t col0,
                                int32_t n_cols, int64_t *out)
{
    if (!ctx) return SNACC_ERR_ARG;
    if (n_rows < 0 || n_cols < 0 || row0 < 0 || col0 < 0) return SNACC_ERR_ARG;
    const Tile tile{row0, n_rows, col0, n_cols};
    return sizes_impl(ctx, codec, nullptr, nullptr, (int64_t)n_rows * n_cols, &tile, out);
}

// ---- multi-GPU: exchange of per-sequence prefix state between ranks that prepared different sequences ----
extern "C" int64_t snacc_prefix_record_bytes(const snacc_ctx *ctx, int codec)
{
    if (!ctx) return SNACC_ERR_ARG;
    // LZ4: every rank parses every x itself (one sequence per CTA: the pass costs the latency of ONE sequence however
    // many a rank owns, so there is nothing to gain from sharing); deflate: checkpoint + size of the sequence alone
    return (codec == SNACC_GZIP9 || codec == SNACC_ZLIB6) ? (int64_t)sizeof(DflPrefixRecord) : 0;
}

static int prefix_xfer(snacc_ctx *ctx, int codec, const int32_t *seqs, int64_t n, void *buf, bool do_export)
{
    if (!ctx) return SNACC_ERR_ARG;
    std::lock_guard<std::mutex> lock(ctx->mu);
    ctx->err.clear();
    if (!ctx->n_seqs) FAIL(SNACC_ERR_STATE, "nothing uploaded");
    if (codec != SNACC_GZIP9 && codec != SNACC_ZLIB6) FAIL(SNACC_ERR_CODEC, "this codec has no prefix records to exchange");
    if (n < 0 || (n && (!seqs || !buf))) FAIL(SNACC_ERR_ARG, "bad sequence list");
    CK(cudaSetDevice(ctx->device));
    const Corpus dc = corpus(ctx);
    const int level = codec == SNACC_GZIP9 ? 9 : 6;
    const int r = do_export ? deflate_export_prefix(ctx->dfl, dc, level, seqs, n, (DflPrefixRecord *)buf, ctx->stream, ctx->err)
                            : deflate_import_prefix(ctx->dfl, dc, level, seqs, n, (const DflPrefixRecord *)buf, ctx->stream, ctx->err);
    return r ? SNACC_ERR_CUDA : SNACC_OK;
}

extern "C" int snacc_export_prefix(snacc_ctx *ctx, int codec, const int32_t *seqs, int64_t n, void *out)
{
    return prefix_xfer(ctx, codec, seqs, n, out, true);
}

extern "C" int snacc_import_prefix(snacc_ctx *ctx, int codec, const int32_t *seqs, int64_t n, const void *in)
{
    return prefix_xfer(ctx, codec, seqs, n, const_cast<void *>(in), false);
}

extern "C" int snacc_ncd(snacc_ctx *ctx, const int64_t *C, const int64_t *S, int32_t n, int formula, int32_t bias,
                         double *D)
{
    NvtxRange nvtx_("snacc_b200: ncd epilogue");
    if (!ctx) return SNACC_ERR_ARG;
    std::lock_guard<std::mutex> lock(ctx->mu);
    ctx->err.clear();
    if (n <= 0 || !C || !S || !D) FAIL(SNACC_ERR_ARG, "snacc_ncd: bad arguments");
    if (formula != SNACC_NCD_REFERENCE && formula != SNACC_NCD_ONE_ORDER) FAIL(SNACC_ERR_ARG, "snacc_ncd: bad formula");
    CK(cudaSetDevice(ctx->device));
    const size_t nn = (size_t)n * n;
    CK(ctx->ncd_c.grow(sizeof(int64_t) * n, ctx->stream));           // kept across calls: no malloc per step
    CK(ctx->ncd_s.grow(sizeof(int64_t) * nn, ctx->stream));
    CK(ctx->ncd_d.grow(sizeof(double) * nn, ctx->stream));
    int64_t *dC = ctx->ncd_c.get<int64_t>(), *dS = ctx->ncd_s.get<int64_t>();
    double *dD = ctx->ncd_d.get<double>();
    CK(cudaMemcpyAsync(dC, C, sizeof(int64_t) * n, cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaMemcpyAsync(dS, S, sizeof(int64_t) * nn, cudaMemcpyHostToDevice, ctx->stream));
    const int threads = 256;
    const int blocks = (int)std::min<size_t>((nn + threads - 1) / threads, 148 * 8);
    ncd_kernel<<<blocks, threads, 0, ctx->stream>>>(dC, dS, n, formula, bias, dD);
    CK(cudaGetLastError());
    CK(cudaMemcpyAsync(D, dD, sizeof(double) * nn, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    return SNACC_OK;
}

// scipy's label(): the merges, sorted by height, name their clusters by slot; a union-find over the leaves turns each
// slot into the id of the cluster that holds it (n, n+1, ... in row order), smaller id first
static void upgma_label(double *Z, int32_t n)
{
    std::vector<int32_t> parent(2 * (size_t)n - 1), count(2 * (size_t)n - 1, 1);
    for (int32_t i = 0; i < 2 * n - 1; ++i) parent[i] = i;
    auto find = [&](int32_t a) {
        int32_t r = a;
        while (parent[r] != r) r = parent[r];
        while (parent[a] != r) { const int32_t p = parent[a]; parent[a] = r; a = p; }
        return r;
    };
    for (int32_t k = 0; k + 1 < n; ++k) {
        const int32_t a = find((int32_t)Z[4 * (size_t)k]), b = find((int32_t)Z[4 * (size_t)k + 1]);
        Z[4 * (size_t)k + 0] = (double)std::min(a, b);
        Z[4 * (size_t)k + 1] = (double)std::max(a, b);
        parent[a] = parent[b] = n + k;
        count[n + k] = count[a] + count[b];
        Z[4 * (size_t)k + 3] = (double)count[n + k];
    }
}

// downstream of the distance matrix: metrify (misc.py:20-25) + UPGMA (distmatrix_to_tree.py:9-15) -> scipy's linkage matrix
extern "C" int snacc_upgma(snacc_ctx *ctx, const double *D, int32_t n, int metrify, double *Z)
{
    if (!ctx) return SNACC_ERR_ARG;
    std::lock_guard<std::mutex> lock(ctx->mu);
    ctx->err.clear();
    if (n < 2 || !D || !Z) FAIL(SNACC_ERR_ARG, "snacc_upgma: needs a matrix of at least 2 x 2");
    NvtxRange nvtx_("snacc_b200: metrify + upgma");
    CK(cudaSetDevice(ctx->device));
    const size_t nn = (size_t)n * n;
    double *dD = nullptr, *dM = nullptr, *dZ = nullptr;
    int32_t *d_size = nullptr, *d_chain = nullptr;
    int *d_flags = nullptr;
    auto release = [&]() {
        cudaFree(dD); cudaFree(dM); cudaFree(dZ); cudaFree(d_size); cudaFree(d_chain); cudaFree(d_flags);
    };
#define UCK(call) do { cudaError_t e_ = (call); if (e_ != cudaSuccess) { release(); \
        ctx->err = std::string(#call " failed: ") + cudaGetErrorString(e_); return SNACC_ERR_CUDA; } } while (0)
    UCK(cudaMalloc(&dD, sizeof(double) * nn));
    UCK(cudaMalloc(&dM, sizeof(double) * nn));
    UCK(cudaMalloc(&dZ, sizeof(double) * 4 * (size_t)(n - 1)));
    UCK(cudaMalloc(&d_size, sizeof(int32_t) * n));
    UCK(cudaMalloc(&d_chain, sizeof(int32_t) * n));
    UCK(cudaMalloc(&d_flags, sizeof(int)));
    UCK(cudaMemcpyAsync(dD, D, sizeof(double) * nn, cudaMemcpyHostToDevice, ctx->stream));
    UCK(cudaMemsetAsync(d_flags, 0, sizeof(int), ctx->stream));
    const unsigned grid = (unsigned)std::min<size_t>((nn + 255) / 256, 148 * 8);
    metrify_kernel<<<grid, 256, 0, ctx->stream>>>(dD, n, metrify ? 1 : 0, dM);
    UCK(cudaGetLastError());
    // what scipy's squareform and linkage refuse: checked on the matrix to be clustered, before the UPGMA launch
    upgma_check_kernel<<<grid, 256, 0, ctx->stream>>>(dM, n, metrify ? 0 : 1, d_flags);
    UCK(cudaGetLastError());
    int flags = 0;
    UCK(cudaMemcpyAsync(&flags, d_flags, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
    UCK(cudaStreamSynchronize(ctx->stream));
    if (flags) {
        release();
        std::string msg = "snacc_upgma: the distance matrix";
        if (flags & UPGMA_NONFINITE) msg += " must contain only finite values;";
        if (flags & UPGMA_ASYMMETRIC) msg += " must be symmetric;";
        if (flags & UPGMA_DIAGONAL) msg += " must have a zero diagonal;";
        msg.back() = ' ';
        msg += metrify ? "(after metrify)" : "(metrify is off)";
        FAIL(SNACC_ERR_ARG, msg);
    }
    upgma_kernel<<<1, UPGMA_THREADS, 0, ctx->stream>>>(dM, n, dZ, d_size, d_chain);
    UCK(cudaGetLastError());
    UCK(cudaMemcpyAsync(Z, dZ, sizeof(double) * 4 * (size_t)(n - 1), cudaMemcpyDeviceToHost, ctx->stream));
    UCK(cudaStreamSynchronize(ctx->stream));
#undef UCK
    release();
    // the rows come in merge order with slot ids: sort them stably by height (numpy's mergesort), then scipy's labels
    std::vector<double> raw(Z, Z + 4 * (size_t)(n - 1));
    std::vector<int32_t> order(n - 1);
    for (int32_t k = 0; k + 1 < n; ++k) order[k] = k;
    std::stable_sort(order.begin(), order.end(), [&](int32_t a, int32_t b) { return raw[4 * (size_t)a + 2] < raw[4 * (size_t)b + 2]; });
    for (int32_t k = 0; k + 1 < n; ++k)
        for (int c = 0; c < 4; ++c) Z[4 * (size_t)k + c] = raw[4 * (size_t)order[k] + c];
    upgma_label(Z, n);
    return SNACC_OK;
}

extern "C" int snacc_last_kernel_ms(const snacc_ctx *ctx, double *ms, int64_t *launches)
{
    if (!ctx) return SNACC_ERR_ARG;
    if (ms) *ms = ctx->last_ms;
    if (launches) *launches = ctx->last_launches;
    return SNACC_OK;
}

extern "C" int snacc_get_stat(const snacc_ctx *ctx, const char *name, double *out)
{
    if (!ctx || !name || !out) return SNACC_ERR_ARG;
    if (!strcmp(name, "main_kernel_ms")) { *out = ctx->last_main_ms; return SNACC_OK; }
    if (!strcmp(name, "total_kernel_ms")) { *out = ctx->last_ms; return SNACC_OK; }
    if (!strcmp(name, "launches")) { *out = (double)ctx->last_launches; return SNACC_OK; }
    if (!strcmp(name, "packed_jobs")) { *out = (double)ctx->lz4.packed_jobs; return SNACC_OK; }
    if (!strcmp(name, "bytewise_jobs")) { *out = (double)ctx->lz4.bytewise_jobs; return SNACC_OK; }
    if (!strcmp(name, "lz4_segments")) { *out = (double)ctx->lz4.segments; return SNACC_OK; }
    if (!strcmp(name, "deflate_serial_jobs")) { *out = (double)ctx->dfl.serial_jobs; return SNACC_OK; }
    if (!strcmp(name, "deflate_parallel_prep_seqs")) { *out = (double)ctx->dfl.parallel_prep_seqs; return SNACC_OK; }
    if (!strcmp(name, "deflate_bands")) { *out = (double)ctx->dfl.bands; return SNACC_OK; }
    if (!strcmp(name, "deflate_state_bytes")) { *out = (double)ctx->dfl.peak; return SNACC_OK; }
    if (!strcmp(name, "deflate_prepared_seqs")) { *out = (double)ctx->dfl.prepared_seqs; return SNACC_OK; }
    if (!strcmp(name, "bzip2_blocks")) { *out = (double)ctx->bz.n_blocks; return SNACC_OK; }
    if (!strcmp(name, "bzip2_smem_blocks")) { *out = (double)ctx->bz.smem_blocks; return SNACC_OK; }
    if (!strcmp(name, "bzip2_prefix_blocks")) { *out = (double)ctx->bz.prefix_blocks; return SNACC_OK; }
    if (!strcmp(name, "bzip2_rle_gather_ms")) { *out = ctx->bz.ms[0]; return SNACC_OK; }
    if (!strcmp(name, "bzip2_bwt_small_ms")) { *out = ctx->bz.ms[1]; return SNACC_OK; }
    if (!strcmp(name, "bzip2_bwt_large_ms")) { *out = ctx->bz.ms[2]; return SNACC_OK; }
    if (!strcmp(name, "bzip2_bits_ms")) { *out = ctx->bz.ms[3]; return SNACC_OK; }
    return SNACC_ERR_ARG;
}

extern "C" int snacc_set_option(snacc_ctx *ctx, const char *name, int64_t value)
{
    if (!ctx || !name) return SNACC_ERR_ARG;
    std::lock_guard<std::mutex> lock(ctx->mu);
    if (!strcmp(name, "streams_in_flight")) { ctx->lz4.streams_in_flight = value; return SNACC_OK; }
    if (!strcmp(name, "lz4_packed")) { ctx->lz4.use_packed = value ? 1 : 0; return SNACC_OK; }
    if (!strcmp(name, "lz4_segments")) { ctx->lz4.pk_segments = value < 0 ? 0 : value; return SNACC_OK; }
    if (!strcmp(name, "deflate_canonical")) { ctx->dfl.use_canon = value ? 1 : 0; return SNACC_OK; }
    if (!strcmp(name, "deflate_index6")) { ctx->dfl.use_index6 = value ? 1 : 0; return SNACC_OK; }
    if (!strcmp(name, "deflate_parallel_prep")) { ctx->dfl.use_parallel_prep = value ? 1 : 0; return SNACC_OK; }
    if (!strcmp(name, "deflate_tail_index")) { ctx->dfl.use_tail_index = value ? 1 : 0; return SNACC_OK; }
    if (!strcmp(name, "deflate_junction")) { ctx->dfl.junction_impl = value == 2 ? 2 : 3; return SNACC_OK; }
    if (!strcmp(name, "deflate_band_bytes")) { ctx->dfl.band_bytes = value < 0 ? 0 : value; return SNACC_OK; }
    if (!strcmp(name, "bzip2_smem")) { ctx->bz.use_smem = value ? 1 : 0; return SNACC_OK; }
    if (!strcmp(name, "bzip2_prefix")) { ctx->bz.use_prefix = value ? 1 : 0; bz_invalidate(ctx->bz); return SNACC_OK; }
    if (!strcmp(name, "invalidate_caches")) {
        // forget every per-sequence precomputation (prefix checkpoints ...) so the next sizes call
        // redoes the whole job; used by bench.py so that no step reuses work of an earlier step
        invalidate_caches(ctx);
        return SNACC_OK;
    }
    ctx->err = std::string("unknown option: ") + name;
    return SNACC_ERR_ARG;
}
