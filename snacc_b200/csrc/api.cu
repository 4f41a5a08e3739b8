// api.cu -- C ABI of libsnacc_b200.so (see include/snacc_b200.h) and the host-side orchestration of
// the sm_100a kernels.  No torch, no C++ types across the boundary, no exceptions escape.
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
#include "common.cuh"
#include "lz4.cuh"
#include "pack.cuh"
#include "lz4_packed.cuh"
#include "deflate.cuh"
#include "upgma.cuh"
#include "bzip2.cuh"

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

    // LZ4 prefix checkpoints
    int32_t *d_slot_of = nullptr;          // per sequence: checkpoint slot or -1
    std::vector<int32_t> h_slot_of;
    std::vector<uint8_t> ckpt_done;        // per sequence
    int32_t n_slots = 0;
    uint8_t *d_ckpt_tab = nullptr;
    uint64_t *d_ckpt_total = nullptr;

    // 2-bit packed copy + packed-path prefix checkpoints (lz4_packed.cuh)
    int use_packed = 1;                    // option "lz4_packed": 0 forces the byte-wise kernels
    int sm_count = 148;
    uint64_t *d_pk_words = nullptr, *d_pk_woff = nullptr;
    uint16_t *d_alias5 = nullptr, *d_alias4 = nullptr;
    uint32_t *d_ck_tab = nullptr; PkState *d_ck_state = nullptr;
    std::vector<uint8_t> h_packable, h_ck_have;   // per sequence; h_packable 0: no 2-bit copy usable, 1: clean, 2: a few bytes
                                                  // outside the alphabet (flagged in the per-base mask); h_ck_have bit0:
                                                  // single-block regime, bit1: linked
    // sequences with a few bytes outside the alphabet (EXC kernels; allocated only for corpora that have any)
    int corpus_dirty = 0;
    uint32_t *d_pk_mask = nullptr; uint64_t *d_pk_moff = nullptr; uint64_t mask_words = 0;
    uint16_t *d_b2s = nullptr;
    uint32_t *d_ck_ovf = nullptr, *d_ovf_work = nullptr; size_t ovf_work_tabs = 0;
    PkAlphabet alphabet;
    uint32_t nslot5 = 1024;                // distinct hash buckets the 1024 5-mers of the alphabet reach
    int64_t last_packed_jobs = 0, last_bytewise_jobs = 0;
    int64_t pk_segments = 0, last_pk_segments = 1;     // tile segments of the linked pair kernel: 0 = choose per launch

    // working memory
    uint8_t *d_work = nullptr; size_t work_bytes = 0;
    void *d_scratch[23] = {nullptr}; size_t scratch_cap[23] = {0};   // per-call argument arrays, grown on demand, never
                                                                   // freed between calls (all use is ordered on `stream`)
    unsigned long long *d_counter = nullptr;
    int32_t *d_jobx = nullptr, *d_joby = nullptr; int64_t job_cap = 0;
    int64_t *d_out = nullptr; int64_t out_cap = 0;

    // options / instrumentation
    int64_t streams_in_flight = 0;         // 0 = default
    double last_ms = 0.0; int64_t last_launches = 0;
    double last_main_ms = 0.0;              // dominant kernel only (lz4_stream_kernel / deflate pair kernel)
    cudaEvent_t evm0 = nullptr, evm1 = nullptr;

    DeflateState dfl;

    // bzip2 (bzip2.cuh): RLE1 of every sequence, its emission-start flags (a host copy plans the block cuts), where the
    // open block of each sequence alone starts, and the bits of its closed blocks once computed
    int bz_use_smem = 1, bz_use_prefix = 1;     // options "bzip2_smem", "bzip2_prefix" (0: for tests, same results)
    bool bz_ready = false;
    uint8_t *d_bz_rle = nullptr, *d_bz_flag = nullptr; BzSeq *d_bz_info = nullptr; uint64_t bz_rle_cap = 0;
    unsigned long long *d_bz_seq_bits = nullptr;
    std::vector<BzSeq> h_bz_info; std::vector<uint8_t> h_bz_flag, h_bz_pdone;
    std::vector<uint32_t> h_bz_open, h_bz_nclosed;
    int64_t bz_blocks = 0, bz_smem_blocks = 0, bz_prefix_blocks = 0;
    double bz_ms[4] = {0, 0, 0, 0};            // RLE1 + gather, BWT small, BWT large, MTF + selection + bits
    cudaEvent_t bz_ev[5] = {nullptr, nullptr, nullptr, nullptr, nullptr};
};

#define CK(call) do { cudaError_t e_ = (call); if (e_ != cudaSuccess) { \
        char b_[512]; snprintf(b_, sizeof b_, "%s failed at %s:%d: %s", #call, __FILE__, __LINE__, cudaGetErrorString(e_)); \
        ctx->err = b_; return SNACC_ERR_CUDA; } } while (0)
#define FAIL(code, msg) do { ctx->err = (msg); return (code); } while (0)

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
    cudaFree(ctx->d_slot_of); ctx->d_slot_of = nullptr;
    cudaFree(ctx->d_ckpt_tab); ctx->d_ckpt_tab = nullptr;
    cudaFree(ctx->d_ckpt_total); ctx->d_ckpt_total = nullptr;
    cudaFree(ctx->d_pk_words); ctx->d_pk_words = nullptr;
    cudaFree(ctx->d_pk_woff); ctx->d_pk_woff = nullptr;
    cudaFree(ctx->d_alias5); ctx->d_alias5 = nullptr;
    cudaFree(ctx->d_alias4); ctx->d_alias4 = nullptr;
    cudaFree(ctx->d_ck_tab); ctx->d_ck_tab = nullptr;
    cudaFree(ctx->d_ck_state); ctx->d_ck_state = nullptr;
    cudaFree(ctx->d_pk_mask); ctx->d_pk_mask = nullptr; ctx->mask_words = 0;
    cudaFree(ctx->d_pk_moff); ctx->d_pk_moff = nullptr;
    cudaFree(ctx->d_b2s); ctx->d_b2s = nullptr;
    cudaFree(ctx->d_ck_ovf); ctx->d_ck_ovf = nullptr;
    ctx->corpus_dirty = 0;
    ctx->h_packable.clear(); ctx->h_ck_have.clear();
    ctx->n_seqs = 0; ctx->n_slots = 0;
    cudaFree(ctx->d_bz_rle); ctx->d_bz_rle = nullptr;
    cudaFree(ctx->d_bz_flag); ctx->d_bz_flag = nullptr;
    cudaFree(ctx->d_bz_info); ctx->d_bz_info = nullptr;
    cudaFree(ctx->d_bz_seq_bits); ctx->d_bz_seq_bits = nullptr;
    ctx->bz_rle_cap = 0; ctx->bz_ready = false;
    deflate_free_corpus(ctx->dfl);
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
        cudaEventCreate(&ctx->ev0) != cudaSuccess || cudaEventCreate(&ctx->ev1) != cudaSuccess ||
        cudaEventCreate(&ctx->evm0) != cudaSuccess || cudaEventCreate(&ctx->evm1) != cudaSuccess ||
        cudaMalloc(&ctx->d_counter, 64) != cudaSuccess) {
        delete ctx;
        return SNACC_ERR_CUDA;
    }
    for (cudaEvent_t &e : ctx->bz_ev) if (cudaEventCreate(&e) != cudaSuccess) {
        delete ctx;
        return SNACC_ERR_CUDA;
    }
    cudaDeviceGetAttribute(&ctx->sm_count, cudaDevAttrMultiProcessorCount, device_id);
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
    deflate_free_work(ctx->dfl);
    cudaFree(ctx->d_work); cudaFree(ctx->d_counter); cudaFree(ctx->d_ovf_work);
    for (void *p : ctx->d_scratch) cudaFree(p);
    cudaFree(ctx->d_jobx); cudaFree(ctx->d_joby); cudaFree(ctx->d_out);
    cudaEventDestroy(ctx->ev0); cudaEventDestroy(ctx->ev1);
    cudaEventDestroy(ctx->evm0); cudaEventDestroy(ctx->evm1);
    for (cudaEvent_t e : ctx->bz_ev) cudaEventDestroy(e);
    cudaStreamDestroy(ctx->stream);
    delete ctx;
}

// ---------------------------------------------------------------------------------------------
// K0b: measure the corpus alphabet on the device, then keep a 2-bit copy of every sequence that only
// uses the four most frequent byte values (pack.cuh)
// ---------------------------------------------------------------------------------------------
static int pack_corpus(snacc_ctx *ctx)
{
    NvtxRange nvtx_("snacc_b200: alphabet + 2-bit pack");
    const int32_t n = ctx->n_seqs;
    unsigned long long *d_hist = nullptr;
    CK(cudaMalloc(&d_hist, 256 * sizeof(unsigned long long)));
    CK(cudaMemsetAsync(d_hist, 0, 256 * sizeof(unsigned long long), ctx->stream));
    uint32_t max_len = 0;
    for (int32_t i = 0; i < n; ++i) max_len = std::max(max_len, ctx->h_len[i]);
    {
        dim3 grid(std::min<uint32_t>((max_len + 65535) / 65536, 64), (unsigned)std::min<int32_t>(n, 1024));
        pk_hist_kernel<<<grid, 256, 0, ctx->stream>>>(ctx->d_corpus, ctx->d_off, ctx->d_len, n, d_hist);
        CK(cudaGetLastError());
    }
    unsigned long long hist[256];
    CK(cudaMemcpyAsync(hist, d_hist, sizeof hist, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    cudaFree(d_hist);
    ctx->alphabet = pk_choose_alphabet(hist);
    uint16_t a5[1024], a4[256];
    ctx->nslot5 = pk_slot_lut(ctx->alphabet, false, a5);
    pk_slot_lut(ctx->alphabet, true, a4);
    if (!ctx->d_alias5) CK(cudaMalloc(&ctx->d_alias5, sizeof a5));
    if (!ctx->d_alias4) CK(cudaMalloc(&ctx->d_alias4, sizeof a4));
    CK(cudaMemcpyAsync(ctx->d_alias5, a5, sizeof a5, cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaMemcpyAsync(ctx->d_alias4, a4, sizeof a4, cudaMemcpyHostToDevice, ctx->stream));

    PkCodes codes;
    memcpy(codes.c, ctx->alphabet.code_of, 256);
    std::vector<uint64_t> woff((size_t)n), moff((size_t)n);
    uint64_t w = 0, mw = 0;
    for (int32_t i = 0; i < n; ++i) { woff[i] = w; w += pk_words(ctx->h_len[i]); moff[i] = mw; mw += pk_mask_words(ctx->h_len[i]); }
    // bytes outside the alphabet anywhere in the corpus?  Then the packed copy carries a per-base mask of them and the
    // EXC kernels run (lz4_packed.cuh: pk_step_exact)
    unsigned long long outside = 0;
    for (int i = 0; i < 256; ++i) if (ctx->alphabet.code_of[i] > 3) outside += hist[i];
    ctx->corpus_dirty = outside ? 1 : 0;
    int32_t *d_nexc = nullptr;
    if (!ctx->d_pk_words) CK(cudaMalloc(&ctx->d_pk_words, w * sizeof(uint64_t)));
    if (!ctx->d_pk_woff) CK(cudaMalloc(&ctx->d_pk_woff, sizeof(uint64_t) * n));
    CK(cudaMalloc(&d_nexc, sizeof(int32_t) * n));
    CK(cudaMemsetAsync(d_nexc, 0, sizeof(int32_t) * n, ctx->stream));
    CK(cudaMemcpyAsync(ctx->d_pk_woff, woff.data(), sizeof(uint64_t) * n, cudaMemcpyHostToDevice, ctx->stream));
    if (ctx->corpus_dirty) {
        if (ctx->d_pk_mask && ctx->mask_words < mw) { cudaFree(ctx->d_pk_mask); ctx->d_pk_mask = nullptr; }
        if (!ctx->d_pk_mask) { CK(cudaMalloc(&ctx->d_pk_mask, (mw + 64) * sizeof(uint32_t))); ctx->mask_words = mw; }
        if (!ctx->d_pk_moff) CK(cudaMalloc(&ctx->d_pk_moff, sizeof(uint64_t) * n));
        if (!ctx->d_b2s) CK(cudaMalloc(&ctx->d_b2s, sizeof(uint16_t) * PK_OVF_ENTRIES));
        if (!ctx->d_ck_ovf) CK(cudaMalloc(&ctx->d_ck_ovf, sizeof(uint32_t) * PK_OVF_ENTRIES * (size_t)n));
        CK(cudaMemsetAsync(ctx->d_pk_mask, 0, (mw + 64) * sizeof(uint32_t), ctx->stream));
        CK(cudaMemsetAsync(ctx->d_ck_ovf, 0, sizeof(uint32_t) * PK_OVF_ENTRIES * (size_t)n, ctx->stream));
        CK(cudaMemcpyAsync(ctx->d_pk_moff, moff.data(), sizeof(uint64_t) * n, cudaMemcpyHostToDevice, ctx->stream));
        uint16_t b2s[PK_OVF_ENTRIES];
        for (uint32_t i = 0; i < PK_OVF_ENTRIES; ++i) b2s[i] = 0xffff;
        for (uint32_t c = 0; c < 1024; ++c) b2s[pk_bucket(ctx->alphabet, c, false)] = a5[c];
        CK(cudaMemcpyAsync(ctx->d_b2s, b2s, sizeof b2s, cudaMemcpyHostToDevice, ctx->stream));
    }
    {
        dim3 grid(std::min<uint32_t>((pk_words(max_len) + 255) / 256, 256), (unsigned)std::min<int32_t>(n, 4096));
        pk_pack_kernel<<<grid, 256, 0, ctx->stream>>>(ctx->d_corpus, ctx->d_off, ctx->d_len, ctx->d_pk_woff, n,
                                                      ctx->d_pk_words, d_nexc, ctx->corpus_dirty ? ctx->d_pk_mask : nullptr,
                                                      ctx->d_pk_moff, codes);
        CK(cudaGetLastError());
    }
    std::vector<int32_t> nexc((size_t)n);
    CK(cudaMemcpyAsync(nexc.data(), d_nexc, sizeof(int32_t) * n, cudaMemcpyDeviceToHost, ctx->stream));
    if (!ctx->d_ck_tab) CK(cudaMalloc(&ctx->d_ck_tab, (size_t)n * 2 * PK_CKPT_TAB * sizeof(uint32_t)));
    if (!ctx->d_ck_state) CK(cudaMalloc(&ctx->d_ck_state, (size_t)n * 2 * sizeof(PkState)));
    CK(cudaStreamSynchronize(ctx->stream));
    cudaFree(d_nexc);
    // a sequence keeps to the tile kernels while its flagged bases are sparse: an isolated one costs every stream that
    // meets it a handful of byte-exact steps (about what 450 ordinary probes cost a warp), so the tile kernels stay
    // ahead of the byte-wise ones up to roughly one flagged base in 64; denser sequences -- proteins, heavily
    // soft-masked assemblies -- take the byte-wise kernels
    ctx->h_packable.assign(n, 0);
    for (int32_t i = 0; i < n; ++i)
        ctx->h_packable[i] = nexc[i] == 0 ? 1 : ((uint64_t)nexc[i] <= (uint64_t)ctx->h_len[i] / 64 + 8 ? 2 : 0);
    ctx->h_ck_have.assign(n, 0);
    return SNACC_OK;
}

static int scratch(snacc_ctx *ctx, int slot, size_t bytes, void **out);

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
        std::fill(ctx->ckpt_done.begin(), ctx->ckpt_done.end(), 0);
        deflate_invalidate(ctx->dfl);
        ctx->bz_ready = false;
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
        int rs = scratch(ctx, 8, total ? total : 1, (void **)&d_src);      // staging copy of the host bytes (kept: no malloc per upload)
        if (rs) return rs;
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

    // LZ4 checkpoint slots for sequences that own at least one full 64 KiB block
    ctx->h_slot_of.assign(n_seqs, -1);
    ctx->ckpt_done.assign(n_seqs, 0);
    ctx->n_slots = 0;
    for (int32_t i = 0; i < n_seqs; ++i)
        if (ctx->h_len[i] >= LZ4_BLOCK) ctx->h_slot_of[i] = ctx->n_slots++;
    if (!ctx->d_slot_of) CK(cudaMalloc(&ctx->d_slot_of, sizeof(int32_t) * n_seqs));
    CK(cudaMemcpyAsync(ctx->d_slot_of, ctx->h_slot_of.data(), sizeof(int32_t) * n_seqs, cudaMemcpyHostToDevice, ctx->stream));
    if (ctx->n_slots) {
        if (!ctx->d_ckpt_tab) CK(cudaMalloc(&ctx->d_ckpt_tab, (size_t)ctx->n_slots * LZ4_TABLE_BYTES));
        if (!ctx->d_ckpt_total) CK(cudaMalloc(&ctx->d_ckpt_total, sizeof(uint64_t) * ctx->n_slots));
    }
    ctx->n_seqs = n_seqs;
    CK(cudaStreamSynchronize(ctx->stream));
    cudaFree(d_rec_off); cudaFree(d_rec_dst);
    return pack_corpus(ctx);
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

// ---------------------------------------------------------------------------------------------
static int ensure_job_buffers(snacc_ctx *ctx, int64_t n)
{
    if (n > ctx->job_cap) {
        cudaFree(ctx->d_jobx); cudaFree(ctx->d_joby); ctx->d_jobx = ctx->d_joby = nullptr; ctx->job_cap = 0;
        CK(cudaMalloc(&ctx->d_jobx, sizeof(int32_t) * n));
        CK(cudaMalloc(&ctx->d_joby, sizeof(int32_t) * n));
        ctx->job_cap = n;
    }
    if (n > ctx->out_cap) {
        cudaFree(ctx->d_out); ctx->d_out = nullptr; ctx->out_cap = 0;
        CK(cudaMalloc(&ctx->d_out, sizeof(int64_t) * n));
        ctx->out_cap = n;
    }
    return SNACC_OK;
}

// device scratch array `slot` with room for `bytes` (argument arrays of the launches: no cudaMalloc / cudaFree per call)
static int scratch(snacc_ctx *ctx, int slot, size_t bytes, void **out)
{
    if (bytes > ctx->scratch_cap[slot]) {
        CK(cudaStreamSynchronize(ctx->stream));              // an earlier launch may still read the old array
        cudaFree(ctx->d_scratch[slot]); ctx->d_scratch[slot] = nullptr; ctx->scratch_cap[slot] = 0;
        const size_t cap = std::max<size_t>(bytes + bytes / 4, 4096);
        CK(cudaMalloc(&ctx->d_scratch[slot], cap));
        ctx->scratch_cap[slot] = cap;
    }
    *out = ctx->d_scratch[slot];
    return SNACC_OK;
}

static int ensure_work(snacc_ctx *ctx, size_t bytes)
{
    if (bytes > ctx->work_bytes) {
        cudaFree(ctx->d_work); ctx->d_work = nullptr; ctx->work_bytes = 0;
        CK(cudaMalloc(&ctx->d_work, bytes));
        ctx->work_bytes = bytes;
    }
    return SNACC_OK;
}

// LZ4: make sure every x that starts a linked-regime stream has its prefix checkpoint
static int lz4_prepare_prefixes(snacc_ctx *ctx, const int32_t *xs, int64_t n)
{
    std::vector<int32_t> todo;
    for (int64_t k = 0; k < n; ++k) {
        const int32_t x = xs[k];
        if (ctx->h_slot_of[x] >= 0 && !ctx->ckpt_done[x]) { ctx->ckpt_done[x] = 1; todo.push_back(x); }
    }
    if (todo.empty()) return SNACC_OK;
    int32_t *d_todo = nullptr;
    CK(cudaMalloc(&d_todo, sizeof(int32_t) * todo.size()));
    CK(cudaMemcpyAsync(d_todo, todo.data(), sizeof(int32_t) * todo.size(), cudaMemcpyHostToDevice, ctx->stream));
    const int threads = 32;
    const int blocks = (int)((todo.size() + threads - 1) / threads);
    lz4_prefix_kernel<<<blocks, threads, 0, ctx->stream>>>(ctx->d_corpus, ctx->d_off, ctx->d_len, d_todo,
                                                           (int32_t)todo.size(), ctx->d_slot_of, ctx->d_ckpt_tab,
                                                           ctx->d_ckpt_total);
    ctx->last_launches++;
    CK(cudaGetLastError());
    CK(cudaStreamSynchronize(ctx->stream));
    cudaFree(d_todo);
    return SNACC_OK;
}

// byte-wise kernels (lz4.cuh) on the jobs `sel` (host list; null = all n_jobs jobs) of the uploaded job arrays
static int run_lz4_bytewise(snacc_ctx *ctx, const int32_t *h_x, const std::vector<int64_t> *sel, int64_t n_jobs,
                            bool pairs)
{
    NvtxRange nvtx_("snacc_b200: lz4 byte-wise streams");
    const int64_t n = sel ? (int64_t)sel->size() : n_jobs;
    if (n == 0) return SNACC_OK;
    std::vector<int32_t> xs((size_t)n);
    for (int64_t k = 0; k < n; ++k) xs[k] = h_x[sel ? (*sel)[k] : k];
    int r = lz4_prepare_prefixes(ctx, xs.data(), n);
    if (r) return r;
    // linked-regime streams each own a 16 KiB table that is hit at random: keep the set L2 resident
    // (one warp per SM); single-block streams are short and want many more threads in flight
    bool any_linked = false;
    for (int64_t k = 0; k < n && !any_linked; ++k) any_linked = ctx->h_len[xs[k]] >= LZ4_BLOCK / 2;
    int64_t inflight = ctx->streams_in_flight > 0 ? ctx->streams_in_flight : (any_linked ? 148 * 32 : 148 * 1024);
    const int threads = 32;
    int64_t blocks = (std::min<int64_t>(inflight, n) + threads - 1) / threads;
    if (blocks < 1) blocks = 1;
    r = ensure_work(ctx, (size_t)blocks * threads * LZ4_TABLE_BYTES);
    if (r) return r;
    int64_t *d_sel = nullptr;
    if (sel) {
        CK(cudaMalloc(&d_sel, sizeof(int64_t) * n));
        CK(cudaMemcpyAsync(d_sel, sel->data(), sizeof(int64_t) * n, cudaMemcpyHostToDevice, ctx->stream));
    }
    CK(cudaMemsetAsync(ctx->d_counter, 0, sizeof(unsigned long long), ctx->stream));
    if (!ctx->last_packed_jobs) CK(cudaEventRecord(ctx->evm0, ctx->stream));
    lz4_stream_kernel<<<(unsigned)blocks, threads, 0, ctx->stream>>>(
        ctx->d_corpus, ctx->d_off, ctx->d_len, ctx->d_jobx, pairs ? ctx->d_joby : nullptr, d_sel, n, ctx->d_slot_of,
        ctx->d_ckpt_tab, ctx->d_ckpt_total, ctx->d_work, ctx->d_counter, ctx->d_out);
    if (!ctx->last_packed_jobs) CK(cudaEventRecord(ctx->evm1, ctx->stream));
    ctx->last_launches++;
    ctx->last_bytewise_jobs += n;
    CK(cudaGetLastError());
    if (d_sel) { CK(cudaStreamSynchronize(ctx->stream)); cudaFree(d_sel); }
    return SNACC_OK;
}

// what the EXC kernels take on top of the packed corpus; `tabs` overflow tables of working memory are made available
static int pk_exc_corpus(snacc_ctx *ctx, size_t tabs, PkExcCorpus *xc)
{
    if (tabs > ctx->ovf_work_tabs) {
        CK(cudaStreamSynchronize(ctx->stream));
        cudaFree(ctx->d_ovf_work); ctx->d_ovf_work = nullptr; ctx->ovf_work_tabs = 0;
        CK(cudaMalloc(&ctx->d_ovf_work, tabs * PK_OVF_ENTRIES * sizeof(uint32_t)));
        ctx->ovf_work_tabs = tabs;
    }
    *xc = PkExcCorpus{ctx->d_pk_mask, ctx->d_pk_moff, ctx->d_corpus, ctx->d_off, ctx->d_b2s, ctx->d_ovf_work, ctx->d_ck_ovf};
    return SNACC_OK;
}

// packed path, step 1: singles and/or prefix checkpoints of the listed sequences (lz4_pk_single_kernel)
static int run_pk_single(snacc_ctx *ctx, const std::vector<int32_t> &seqs, const std::vector<int32_t> &want,
                         const std::vector<int64_t> &out_idx)
{
    NvtxRange nvtx_("snacc_b200: lz4 singles + prefix checkpoints");
    const int32_t n = (int32_t)seqs.size();
    if (!n) return SNACC_OK;
    int32_t *d_seqs = nullptr, *d_want = nullptr; int64_t *d_idx = nullptr;
    int rs = scratch(ctx, 0, sizeof(int32_t) * n, (void **)&d_seqs); if (rs) return rs;
    rs = scratch(ctx, 1, sizeof(int32_t) * n, (void **)&d_want); if (rs) return rs;
    rs = scratch(ctx, 2, sizeof(int64_t) * n, (void **)&d_idx); if (rs) return rs;
    CK(cudaMemcpyAsync(d_seqs, seqs.data(), sizeof(int32_t) * n, cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaMemcpyAsync(d_want, want.data(), sizeof(int32_t) * n, cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaMemcpyAsync(d_idx, out_idx.data(), sizeof(int64_t) * n, cudaMemcpyHostToDevice, ctx->stream));
    const PkCorpus pc{ctx->d_pk_words, ctx->d_pk_woff, ctx->d_len};
    PkExcCorpus xc{};
    if (ctx->corpus_dirty) {
        rs = pk_exc_corpus(ctx, (size_t)n, &xc); if (rs) return rs;
        lz4_pk_single_kernel<true><<<n, 64, 0, ctx->stream>>>(pc, xc, d_seqs, d_want, n, ctx->d_ck_tab, ctx->d_ck_state,
                                                              ctx->d_alias5, ctx->d_alias4, d_idx, ctx->d_out);
    } else {
        lz4_pk_single_kernel<false><<<n, 64, 0, ctx->stream>>>(pc, xc, d_seqs, d_want, n, ctx->d_ck_tab, ctx->d_ck_state,
                                                               ctx->d_alias5, ctx->d_alias4, d_idx, ctx->d_out);
    }
    ctx->last_launches++;
    CK(cudaGetLastError());
    return SNACC_OK;
}

// tile geometry of lz4_pk_pair_kernel.  Linked regime: 16-bit slots + epoch bit plane (PkTab KIND 2: 2 bytes +
// 1 bit per slot, as many slots as the alphabet's 5-mers reach), as many streams as fit one SM's shared memory:
// 4 warps x 26 lanes = 104 for A/C/G/T (one warp per scheduler).  Single-block regime: 12 warps x 32 lanes,
// 512 B table per stream.
constexpr int PK_S_LANES = 32, PK_S_WARPS = 12;
constexpr size_t PK_SMEM_MAX = 232448 - 16;       // 227 KiB per CTA minus the kernel's static shared memory
constexpr size_t PK_S_SMEM = PK_RING_BYTES + 256 * 2 + (size_t)PK_S_WARPS * 256 * PK_S_LANES * 2;

struct PkJob { int32_t y, x; int64_t j; };

struct PkGeometry { uint32_t nslot; int lanes, warps; size_t smem; int T; bool exc; };

static PkGeometry pk_geometry(const snacc_ctx *ctx, bool u16)
{
    PkGeometry g;
    g.exc = false;
    if (u16) { g.nslot = 256; g.lanes = PK_S_LANES; g.warps = PK_S_WARPS; g.smem = PK_S_SMEM; g.T = PK_S_LANES * PK_S_WARPS; return g; }
    // linked regime: as many streams as one SM's shared memory holds (A/C/G/T: 894 slots -> 1900 B per stream
    // -> 104 streams = 4 warps x 26 lanes; a full 1024-slot alphabet: 90 -> 2 warps x 32 lanes)
    g.nslot = (ctx->nslot5 + 1) & ~1u;
    const size_t l_stream = (size_t)g.nslot * 2 + ((g.nslot + 31) / 32) * 4;        // bytes of table per linked stream
    // a corpus with flagged bases runs the EXC kernel (same geometry: its dirty ring lives inside the ring)
    g.exc = ctx->corpus_dirty != 0;
    const size_t l_fixed = PK_RING_BYTES + 1024 * 2;
    const size_t l_fit = (PK_SMEM_MAX - l_fixed) / l_stream;
    g.lanes = l_fit >= 104 ? 26 : l_fit >= 100 ? 25 : 32;
    g.warps = l_fit >= 100 ? 4 : (int)std::max<size_t>(1, l_fit / 32);
    g.smem = l_fixed + (size_t)g.warps * g.lanes * l_stream;
    g.T = g.lanes * g.warps;
    return g;
}

// split `cnt` jobs of one y into near-equal tiles of at most T streams
static void pk_split(std::vector<PkTile> &tiles, int32_t y, size_t first, size_t cnt, int T)
{
    const size_t nt = (cnt + T - 1) / T;
    for (size_t t = 0; t < nt; ++t) {
        const size_t a = first + cnt * t / nt, b = first + cnt * (t + 1) / nt;
        tiles.push_back(PkTile{y, (int32_t)(b - a), (int64_t)a});
    }
}

// How many segments to cut the tiles of a linked-regime launch into (PkSegStore): the launch takes
// ceil(tiles * k / SMs) / k tile times, so k > 1 pays when tiles / SMs has a large fractional part relative to its
// value (320 tiles on 148 SMs: 3 -> 2.25 tile times with k = 8).  Every tile needs at least 2 k ring states, and the
// records (2 KB per stream, + a 16 KB overflow table with flagged bases) must stay modest.
static int pk_choose_segments(const snacc_ctx *ctx, const PkGeometry &g, const std::vector<PkTile> &tiles)
{
    uint32_t min_runs = 0xffffffffu;
    for (const PkTile &t : tiles) {
        PkRing rg; uint32_t w0, w1;
        rg.start(ctx->h_len[t.y], w0, w1, g.exc ? PK_RING_COVER_EXC : PK_RING_WORDS);
        min_runs = std::min(min_runs, rg.runs());
    }
    const size_t per_stream = (size_t)g.nslot * 2 + ((g.nslot + 31) / 32) * 4 + sizeof(PkState) + 4 +
                              (g.exc ? PK_OVF_ENTRIES * sizeof(uint32_t) : 0);
    if (tiles.size() * g.T * per_stream > ((size_t)6 << 30)) return 1;
    if (ctx->pk_segments > 0) return (int)std::min<int64_t>(ctx->pk_segments, std::max<uint32_t>(1, min_runs / 2));
    const double sms = (double)ctx->sm_count, nt = (double)tiles.size();
    int best = 1;
    double best_t = std::ceil(nt / sms);
    for (int k : {2, 4, 8}) {
        if ((uint32_t)(2 * k) > min_runs) break;
        const double t = std::max(1.0, std::ceil(nt * k / sms) / k);      // (the segments of one tile run one after the other)
        if (t < best_t * 0.985) { best = k; best_t = t; }
    }
    return best;
}

// launch lz4_pk_pair_kernel on prepared tiles; tout empty = rectangle mode (out_stride, col0)
static int pk_launch(snacc_ctx *ctx, bool u16, const PkGeometry &g, const std::vector<PkTile> &tiles,
                     const std::vector<int32_t> &tx, const std::vector<int64_t> &tout, int64_t out_stride, int32_t col0,
                     int64_t n_jobs)
{
    NvtxRange nvtx_("snacc_b200: lz4 pair tiles");
    PkTile *d_tiles = nullptr; int32_t *d_tx = nullptr; int64_t *d_tout = nullptr;
    int rs = scratch(ctx, u16 ? 3 : 5, sizeof(PkTile) * tiles.size(), (void **)&d_tiles); if (rs) return rs;
    rs = scratch(ctx, u16 ? 4 : 6, sizeof(int32_t) * tx.size(), (void **)&d_tx); if (rs) return rs;
    CK(cudaMemcpyAsync(d_tiles, tiles.data(), sizeof(PkTile) * tiles.size(), cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaMemcpyAsync(d_tx, tx.data(), sizeof(int32_t) * tx.size(), cudaMemcpyHostToDevice, ctx->stream));
    if (!tout.empty()) {
        rs = scratch(ctx, 7, sizeof(int64_t) * tout.size(), (void **)&d_tout); if (rs) return rs;
        CK(cudaMemcpyAsync(d_tout, tout.data(), sizeof(int64_t) * tout.size(), cudaMemcpyHostToDevice, ctx->stream));
    }
    unsigned long long *counter = ctx->d_counter + (u16 ? 1 : 2);
    CK(cudaMemsetAsync(counter, 0, sizeof(unsigned long long), ctx->stream));
    const PkCorpus pc{ctx->d_pk_words, ctx->d_pk_woff, ctx->d_len};
    const int32_t nt = (int32_t)tiles.size();
    const int n_seg = u16 ? 1 : pk_choose_segments(ctx, g, tiles);
    ctx->last_pk_segments = n_seg;
    const int grid = (int)std::min<size_t>(tiles.size() * n_seg, (size_t)ctx->sm_count);
    PkSegStore ss{};
    if (n_seg > 1) {
        // the records of every stream of the launch, carved out of one array; flags zeroed per launch
        const size_t ns = tiles.size() * g.T, nw = (g.nslot + 31) / 32;
        const size_t b_tab = (ns * g.nslot * 2 + 15) & ~(size_t)15, b_ep = (ns * nw * 4 + 15) & ~(size_t)15,
                     b_st = ns * sizeof(PkState), b_eb = ns * 4;
        uint8_t *base = nullptr;
        rs = scratch(ctx, 12, b_tab + b_ep + b_st + b_eb, (void **)&base); if (rs) return rs;
        ss.tab = (uint16_t *)base; ss.ep = (uint32_t *)(base + b_tab); ss.st = (PkState *)(base + b_tab + b_ep);
        ss.eb = (uint32_t *)(base + b_tab + b_ep + b_st);
        rs = scratch(ctx, 13, sizeof(int32_t) * tiles.size(), (void **)&ss.flag); if (rs) return rs;
        CK(cudaMemsetAsync(ss.flag, 0, sizeof(int32_t) * tiles.size(), ctx->stream));
    }
    CK(cudaEventRecord(ctx->evm0, ctx->stream));
    PkExcCorpus xc{};
    if (g.exc) { rs = pk_exc_corpus(ctx, n_seg > 1 ? tiles.size() * g.T : (size_t)grid * g.T, &xc); if (rs) return rs; }
#define PK_GO(KIND_, LANES_, EXC_, lut_) do {                                                                        \
        CK(cudaFuncSetAttribute(lz4_pk_pair_kernel<KIND_, LANES_, EXC_>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)g.smem)); \
        lz4_pk_pair_kernel<KIND_, LANES_, EXC_><<<grid, g.warps * 32, g.smem, ctx->stream>>>(                          \
            pc, xc, d_tiles, nt, d_tx, d_tout, ctx->d_ck_tab, ctx->d_ck_state, lut_, g.nslot, out_stride, col0, counter, ctx->d_out, n_seg, ss); \
    } while (0)
    if (u16) PK_GO(1, PK_S_LANES, false, ctx->d_alias4);
    else if (g.exc && g.lanes == 26) PK_GO(2, 26, true, ctx->d_alias5);
    else if (g.exc && g.lanes == 25) PK_GO(2, 25, true, ctx->d_alias5);
    else if (g.exc) PK_GO(2, 32, true, ctx->d_alias5);
    else if (g.lanes == 26) PK_GO(2, 26, false, ctx->d_alias5);
    else if (g.lanes == 25) PK_GO(2, 25, false, ctx->d_alias5);
    else PK_GO(2, 32, false, ctx->d_alias5);
#undef PK_GO
    CK(cudaEventRecord(ctx->evm1, ctx->stream));
    ctx->last_launches++;
    ctx->last_packed_jobs += n_jobs;
    CK(cudaGetLastError());
    return SNACC_OK;
}

static int run_pk_pairs(snacc_ctx *ctx, std::vector<PkJob> &jobs, bool u16)
{
    if (jobs.empty()) return SNACC_OK;
    const PkGeometry g = pk_geometry(ctx, u16);
    std::sort(jobs.begin(), jobs.end(), [&](const PkJob &a, const PkJob &b) {
        const uint32_t la = ctx->h_len[a.y], lb = ctx->h_len[b.y];
        return la != lb ? la > lb : a.y != b.y ? a.y < b.y : a.j < b.j;       // longest y first, jobs of one y together
    });
    std::vector<PkTile> tiles;
    std::vector<int32_t> tx(jobs.size());
    std::vector<int64_t> tout(jobs.size());
    for (size_t k = 0; k < jobs.size();) {
        size_t e = k;
        while (e < jobs.size() && jobs[e].y == jobs[k].y) ++e;
        pk_split(tiles, jobs[k].y, k, e - k, g.T);
        k = e;
    }
    for (size_t k = 0; k < jobs.size(); ++k) { tx[k] = jobs[k].x; tout[k] = jobs[k].j; }
    return pk_launch(ctx, u16, g, tiles, tx, tout, 0, 0, (int64_t)jobs.size());
}

// make sure the listed sequences have their packed prefix checkpoint for the regimes in `need` (bit 0 / bit 1)
static int pk_ensure_ckpts(snacc_ctx *ctx, const std::vector<int32_t> &need)
{
    std::vector<int32_t> seqs, want; std::vector<int64_t> idx;
    for (int32_t s = 0; s < ctx->n_seqs; ++s) {
        const int32_t missing = need[s] & ~ctx->h_ck_have[s];
        if (missing) { seqs.push_back(s); want.push_back(missing); idx.push_back(-1); ctx->h_ck_have[s] |= (uint8_t)missing; }
    }
    return run_pk_single(ctx, seqs, want, idx);
}

// Rectangle rows [row0, row0+n_rows) x cols [col0, col0+n_cols) of the ordered-pair matrix on the packed path
// without building per-job arrays (c3: 10^8 jobs).  Returns 1 when the rectangle is not uniform enough (some
// sequence outside the alphabet, a y shorter than 16, or pairs on both sides of the 64 KiB regime boundary):
// the caller then takes the per-job path.
static int run_pk_rect(snacc_ctx *ctx, int32_t row0, int32_t n_rows, int32_t col0, int32_t n_cols)
{
    uint32_t min_x = 0xffffffffu, max_x = 0, min_y = 0xffffffffu, max_y = 0;
    bool any_flagged = false;
    for (int32_t r = row0; r < row0 + n_rows; ++r) {
        if (!ctx->h_packable[r]) return 1;
        any_flagged |= ctx->h_packable[r] == 2;
        min_x = std::min(min_x, ctx->h_len[r]); max_x = std::max(max_x, ctx->h_len[r]);
    }
    for (int32_t c = col0; c < col0 + n_cols; ++c) {
        if (!ctx->h_packable[c]) return 1;
        any_flagged |= ctx->h_packable[c] == 2;
        min_y = std::min(min_y, ctx->h_len[c]); max_y = std::max(max_y, ctx->h_len[c]);
    }
    if (min_y < 16) return 1;
    const bool all_small = (uint64_t)max_x + max_y <= LZ4_BLOCK, all_linked = (uint64_t)min_x + min_y > LZ4_BLOCK;
    if (!all_small && !all_linked) return 1;
    if (all_small && any_flagged) return 1;            // flagged bases: linked regime only (per-job path sorts it out)
    const bool u16 = all_small;
    std::vector<int32_t> need((size_t)ctx->n_seqs, 0);
    for (int32_t r = row0; r < row0 + n_rows; ++r) need[r] = u16 ? 1 : 2;
    int rc = pk_ensure_ckpts(ctx, need);
    if (rc) return rc;
    const PkGeometry g = pk_geometry(ctx, u16);
    std::vector<int32_t> cols((size_t)n_cols), tx((size_t)n_rows);
    for (int32_t c = 0; c < n_cols; ++c) cols[c] = col0 + c;
    std::stable_sort(cols.begin(), cols.end(), [&](int32_t a, int32_t b) { return ctx->h_len[a] > ctx->h_len[b]; });
    for (int32_t r = 0; r < n_rows; ++r) tx[r] = row0 + r;
    std::vector<PkTile> tiles;
    for (int32_t y : cols) pk_split(tiles, y, 0, (size_t)n_rows, g.T);
    return pk_launch(ctx, u16, g, tiles, tx, std::vector<int64_t>(), n_cols, col0, (int64_t)n_rows * n_cols);
}

// LZ4 driver: jobs whose operands have a 2-bit copy take the packed tile kernels, the rest the byte-wise kernel
static int run_lz4(snacc_ctx *ctx, const int32_t *h_x, const int32_t *h_y, int64_t n_jobs)
{
    const bool pairs = h_y != nullptr;
    ctx->last_packed_jobs = ctx->last_bytewise_jobs = 0;
    if (!ctx->use_packed) return run_lz4_bytewise(ctx, h_x, nullptr, n_jobs, pairs);
    std::vector<int64_t> bytewise;
    int r;
    if (!pairs) {
        std::vector<int32_t> seqs, want; std::vector<int64_t> idx;
        for (int64_t k = 0; k < n_jobs; ++k) {
            // (a sequence with flagged bases that is a single-block stream has no byte-exact step: byte-wise kernel)
            if (ctx->h_packable[h_x[k]] == 1 || (ctx->h_packable[h_x[k]] == 2 && ctx->h_len[h_x[k]] > LZ4_BLOCK)) {
                // the same pass leaves the prefix checkpoints a later pair call with this x would need (the extra work
                // is a re-run of the last partial block), so that call does not have to parse the sequence again
                const int32_t sq = h_x[k];
                const int32_t all = 2 | (ctx->h_len[sq] < LZ4_BLOCK ? 1 : 0);
                const int32_t missing = all & ~ctx->h_ck_have[sq];
                ctx->h_ck_have[sq] |= (uint8_t)missing;
                seqs.push_back(sq); want.push_back(missing); idx.push_back(k);
            }
            else bytewise.push_back(k);
        }
        ctx->last_packed_jobs = (int64_t)seqs.size();
        CK(cudaEventRecord(ctx->evm0, ctx->stream));
        r = run_pk_single(ctx, seqs, want, idx);
        if (r) return r;
        CK(cudaEventRecord(ctx->evm1, ctx->stream));
    } else {
        std::vector<PkJob> small, linked;
        std::vector<int32_t> need((size_t)ctx->n_seqs, 0);
        for (int64_t k = 0; k < n_jobs; ++k) {
            const int32_t x = h_x[k], y = h_y[k];
            if (!ctx->h_packable[x] || !ctx->h_packable[y] || ctx->h_len[y] < 16) { bytewise.push_back(k); continue; }
            const bool u16 = (uint64_t)ctx->h_len[x] + ctx->h_len[y] <= LZ4_BLOCK;
            if (u16 && (ctx->h_packable[x] == 2 || ctx->h_packable[y] == 2)) { bytewise.push_back(k); continue; }
            (u16 ? small : linked).push_back(PkJob{y, x, k});
            need[x] |= u16 ? 1 : 2;
        }
        r = pk_ensure_ckpts(ctx, need);
        if (r) return r;
        r = run_pk_pairs(ctx, small, true);
        if (r) return r;
        r = run_pk_pairs(ctx, linked, false);
        if (r) return r;
    }
    if (!bytewise.empty()) return run_lz4_bytewise(ctx, h_x, &bytewise, n_jobs, pairs);
    return SNACC_OK;
}

// ---------------------------------------------------------------------------------------------
// K5: bzip2 (bzip2.cuh).  RLE1 of every sequence once per upload; then per call the host cuts every job into blocks
// (x's closed blocks once per x, the rest of each job from x's open tail, the junction and RLE1(y)) and the blocks go
// through fixed-size batches: gather, BWT (shared memory up to BZ_SMEM_MAX_N bytes, else global scratch), MTF + table
// choice + bit count.  Device memory of a batch is bounded by BZ_BATCH_BYTES whatever the number of jobs.
// ---------------------------------------------------------------------------------------------
constexpr uint64_t BZ_BATCH_BYTES = 192ull << 20;
constexpr size_t BZ_BATCH_BLOCKS = 1 << 16;

static int bz_prepare(snacc_ctx *ctx)
{
    NvtxRange nvtx_("snacc_b200: bzip2 RLE1");
    const int32_t n = ctx->n_seqs;
    ctx->h_bz_info.assign((size_t)n, BzSeq{});
    uint64_t cap = 0;
    for (int32_t i = 0; i < n; ++i) { ctx->h_bz_info[i].roff = cap; cap += (uint64_t)ctx->h_len[i] / 4 * 5 + 16; }
    if (cap > ctx->bz_rle_cap) {
        cudaFree(ctx->d_bz_rle); cudaFree(ctx->d_bz_flag); ctx->d_bz_rle = ctx->d_bz_flag = nullptr; ctx->bz_rle_cap = 0;
        CK(cudaMalloc(&ctx->d_bz_rle, cap));
        CK(cudaMalloc(&ctx->d_bz_flag, cap));
        ctx->bz_rle_cap = cap;
    }
    if (!ctx->d_bz_info) CK(cudaMalloc(&ctx->d_bz_info, sizeof(BzSeq) * n));
    if (!ctx->d_bz_seq_bits) CK(cudaMalloc(&ctx->d_bz_seq_bits, sizeof(unsigned long long) * n));
    CK(cudaMemsetAsync(ctx->d_bz_seq_bits, 0, sizeof(unsigned long long) * n, ctx->stream));
    CK(cudaMemcpyAsync(ctx->d_bz_info, ctx->h_bz_info.data(), sizeof(BzSeq) * n, cudaMemcpyHostToDevice, ctx->stream));
    std::vector<int32_t> all((size_t)n);
    for (int32_t i = 0; i < n; ++i) all[i] = i;
    int32_t *d_all = nullptr;
    int rs = scratch(ctx, 14, sizeof(int32_t) * n, (void **)&d_all); if (rs) return rs;
    CK(cudaMemcpyAsync(d_all, all.data(), sizeof(int32_t) * n, cudaMemcpyHostToDevice, ctx->stream));
    bz_rle_kernel<<<(n + 31) / 32, 32, 0, ctx->stream>>>(ctx->d_corpus, ctx->d_off, ctx->d_len, d_all, n, ctx->d_bz_rle,
                                                         ctx->d_bz_flag, ctx->d_bz_info);
    CK(cudaGetLastError());
    ctx->last_launches++;
    ctx->h_bz_flag.resize(cap);
    CK(cudaMemcpyAsync(ctx->h_bz_info.data(), ctx->d_bz_info, sizeof(BzSeq) * n, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaMemcpyAsync(ctx->h_bz_flag.data(), ctx->d_bz_flag, cap, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    // where the last block of each sequence alone starts: the blocks before it close the same way in every x.y
    ctx->h_bz_open.assign((size_t)n, 0); ctx->h_bz_nclosed.assign((size_t)n, 0); ctx->h_bz_pdone.assign((size_t)n, 0);
    std::vector<BzWin> wins;
    for (int32_t i = 0; i < n; ++i) {
        const BzSeq &si = ctx->h_bz_info[i];
        if (si.rlen <= BZ_NBLOCK_MAX) continue;
        const uint8_t *f = ctx->h_bz_flag.data() + si.roff;
        wins.clear();
        bz_cut(bz_view_single(0, si.rlen), f, f, wins);
        ctx->h_bz_open[i] = wins.back().v0;
        ctx->h_bz_nclosed[i] = (uint32_t)wins.size() - 1;
    }
    ctx->bz_ready = true;
    return SNACC_OK;
}

static int bz_run_batch(snacc_ctx *ctx, const BzBlock *blocks, size_t nb, uint64_t bytes,
                        unsigned long long *d_job_bits)
{
    NvtxRange nvtx_("snacc_b200: bzip2 batch");
    std::vector<int32_t> small, large;
    for (size_t k = 0; k < nb; ++k)
        ((ctx->bz_use_smem && blocks[k].n <= BZ_SMEM_MAX_N) ? small : large).push_back((int32_t)k);
    BzBlock *d_blocks = nullptr; int32_t *d_small = nullptr, *d_large = nullptr;
    uint8_t *d_buf = nullptr, *d_bwt = nullptr; uint16_t *d_mtf = nullptr; uint32_t *d_sort = nullptr;
    int rs = scratch(ctx, 15, sizeof(BzBlock) * nb, (void **)&d_blocks); if (rs) return rs;
    rs = scratch(ctx, 16, sizeof(int32_t) * (small.size() + 1), (void **)&d_small); if (rs) return rs;
    rs = scratch(ctx, 17, sizeof(int32_t) * (large.size() + 1), (void **)&d_large); if (rs) return rs;
    rs = scratch(ctx, 18, bytes, (void **)&d_buf); if (rs) return rs;
    rs = scratch(ctx, 19, bytes, (void **)&d_bwt); if (rs) return rs;
    rs = scratch(ctx, 20, sizeof(uint16_t) * (bytes + nb), (void **)&d_mtf); if (rs) return rs;
    if (!large.empty()) {
        // the global-memory sort's 4 arrays of 32-bit words per block byte
        rs = ensure_work(ctx, 16 * bytes); if (rs) return rs;
        d_sort = (uint32_t *)ctx->d_work;
    }
    CK(cudaMemcpyAsync(d_blocks, blocks, sizeof(BzBlock) * nb, cudaMemcpyHostToDevice, ctx->stream));
    if (!small.empty()) CK(cudaMemcpyAsync(d_small, small.data(), sizeof(int32_t) * small.size(), cudaMemcpyHostToDevice, ctx->stream));
    if (!large.empty()) CK(cudaMemcpyAsync(d_large, large.data(), sizeof(int32_t) * large.size(), cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaEventRecord(ctx->bz_ev[0], ctx->stream));
    bz_gather_kernel<<<(unsigned)nb, 256, 0, ctx->stream>>>(d_blocks, ctx->d_bz_info, ctx->d_bz_rle, ctx->d_bz_flag, d_buf);
    CK(cudaGetLastError());
    CK(cudaEventRecord(ctx->bz_ev[1], ctx->stream));
    if (!small.empty()) {
        CK(cudaFuncSetAttribute(bz_bwt_smem_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)BZ_SMEM_BYTES));
        bz_bwt_smem_kernel<<<(unsigned)small.size(), BZ_SORT_THREADS, BZ_SMEM_BYTES, ctx->stream>>>(d_blocks, d_small, d_buf, d_bwt);
        CK(cudaGetLastError());
    }
    CK(cudaEventRecord(ctx->bz_ev[2], ctx->stream));
    if (!large.empty()) {
        bz_bwt_global_kernel<<<(unsigned)large.size(), BZ_SORT_THREADS, 0, ctx->stream>>>(d_blocks, d_large, d_buf, d_bwt, d_sort);
        CK(cudaGetLastError());
    }
    CK(cudaEventRecord(ctx->bz_ev[3], ctx->stream));
    CK(cudaFuncSetAttribute(bz_bits_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)BZ_BITS_DYN_SMEM));
    bz_bits_kernel<<<(unsigned)nb, BZ_BITS_THREADS, BZ_BITS_DYN_SMEM, ctx->stream>>>(d_blocks, d_bwt, d_mtf, d_job_bits,
                                                                                    ctx->d_bz_seq_bits);
    CK(cudaGetLastError());
    CK(cudaEventRecord(ctx->bz_ev[4], ctx->stream));
    CK(cudaEventSynchronize(ctx->bz_ev[4]));
    for (int s = 0; s < 4; ++s) {
        float ms = 0.f;
        CK(cudaEventElapsedTime(&ms, ctx->bz_ev[s], ctx->bz_ev[s + 1]));
        ctx->bz_ms[s] += ms;
    }
    ctx->last_launches += 2 + !small.empty() + !large.empty();
    ctx->bz_blocks += (int64_t)nb;
    ctx->bz_smem_blocks += (int64_t)small.size();
    return SNACC_OK;
}

static int run_bzip2(snacc_ctx *ctx, const int32_t *xs, const int32_t *ys, int64_t n_jobs)
{
    ctx->bz_blocks = ctx->bz_smem_blocks = ctx->bz_prefix_blocks = 0;
    for (double &m : ctx->bz_ms) m = 0;
    if (!ctx->bz_ready) {
        CK(cudaEventRecord(ctx->bz_ev[0], ctx->stream));
        int r = bz_prepare(ctx);
        if (r) return r;
        CK(cudaEventRecord(ctx->bz_ev[1], ctx->stream));
        CK(cudaEventSynchronize(ctx->bz_ev[1]));
        float ms = 0.f;
        CK(cudaEventElapsedTime(&ms, ctx->bz_ev[0], ctx->bz_ev[1]));
        ctx->bz_ms[0] += ms;
    }
    unsigned long long *d_job_bits = nullptr; uint8_t *d_use_prefix = nullptr;
    int rs = scratch(ctx, 21, sizeof(unsigned long long) * n_jobs, (void **)&d_job_bits); if (rs) return rs;
    rs = scratch(ctx, 22, (size_t)n_jobs, (void **)&d_use_prefix); if (rs) return rs;
    CK(cudaMemsetAsync(d_job_bits, 0, sizeof(unsigned long long) * n_jobs, ctx->stream));
    std::vector<uint8_t> use_prefix((size_t)n_jobs, 0);
    std::vector<BzBlock> batch;
    batch.reserve(BZ_BATCH_BLOCKS);
    uint64_t bytes = 0;
    std::vector<BzWin> wins;
    const uint8_t *hf = ctx->h_bz_flag.data();
    int64_t computed_closed = 0, used_closed = 0;
    // blocks of the view v of job/sequence `dst` go into the batch, which runs whenever it is full
    auto add = [&](int64_t dst, int32_t x, int32_t y, const BzView &v) -> int {
        const BzSeq &sx = ctx->h_bz_info[x], &sy = ctx->h_bz_info[y < 0 ? x : y];
        wins.clear();
        bz_cut(v, hf + sx.roff, hf + sy.roff, wins);
        for (const BzWin &w : wins) {
            if (batch.size() == BZ_BATCH_BLOCKS || bytes + w.n > BZ_BATCH_BYTES) {
                int r = bz_run_batch(ctx, batch.data(), batch.size(), bytes, d_job_bits);
                if (r) return r;
                batch.clear(); bytes = 0;
            }
            batch.push_back(BzBlock{dst, bytes, x, y, w.v0, w.n, v});
            bytes += (w.n + 15) & ~15u;
        }
        return SNACC_OK;
    };
    for (int64_t k = 0; k < n_jobs; ++k) {
        const int32_t x = xs[k], y = ys ? ys[k] : -1;
        const uint32_t open = ctx->h_bz_open[x];
        int r;
        if (open) {
            if (ctx->bz_use_prefix) {
                use_prefix[k] = 1;
                used_closed += ctx->h_bz_nclosed[x];
                if (!ctx->h_bz_pdone[x]) {
                    ctx->h_bz_pdone[x] = 1;
                    computed_closed += ctx->h_bz_nclosed[x];
                    if ((r = add(-1 - (int64_t)x, x, -1, bz_view_single(0, open)))) return r;
                }
            } else if ((r = add(k, x, -1, bz_view_single(0, open)))) return r;
        }
        const BzSeq &sx = ctx->h_bz_info[x];
        if ((r = add(k, x, y, y < 0 ? bz_view_single(open, sx.rlen) : bz_view_pair(sx, open, ctx->h_bz_info[y])))) return r;
    }
    if (!batch.empty()) { int r = bz_run_batch(ctx, batch.data(), batch.size(), bytes, d_job_bits); if (r) return r; }
    ctx->bz_prefix_blocks = used_closed - computed_closed;
    CK(cudaMemcpyAsync(d_use_prefix, use_prefix.data(), (size_t)n_jobs, cudaMemcpyHostToDevice, ctx->stream));
    const int blocks = (int)std::min<int64_t>((n_jobs + 255) / 256, 148 * 8);
    bz_finish_kernel<<<blocks, 256, 0, ctx->stream>>>(d_job_bits, ctx->d_bz_seq_bits, ctx->d_jobx, d_use_prefix, n_jobs, ctx->d_out);
    CK(cudaGetLastError());
    ctx->last_launches++;
    return SNACC_OK;
}

static int64_t wrapper_bytes(int codec) { return codec == SNACC_GZIP9 ? 18 : codec == SNACC_ZLIB6 ? 6 : 0; }

// common driver: job lists on host -> sizes on host
static int sizes_impl(snacc_ctx *ctx, int codec, const int32_t *xs, const int32_t *ys, int64_t n_jobs, int64_t *out)
{
    if (!ctx) return SNACC_ERR_ARG;
    std::lock_guard<std::mutex> lock(ctx->mu);
    ctx->err.clear();
    if (!ctx->n_seqs) FAIL(SNACC_ERR_STATE, "nothing uploaded");
    if (codec != SNACC_LZ4F && codec != SNACC_GZIP9 && codec != SNACC_ZLIB6 && codec != SNACC_BZIP2_9)
        FAIL(SNACC_ERR_CODEC, "codec not supported on the GPU path (supported: lz4, gzip, zlib, bzip2)");
    if (n_jobs < 0 || (n_jobs && (!xs || !out))) FAIL(SNACC_ERR_ARG, "bad job list");
    if (n_jobs == 0) return SNACC_OK;
    for (int64_t k = 0; k < n_jobs; ++k) {
        if (xs[k] < 0 || xs[k] >= ctx->n_seqs || (ys && (ys[k] < 0 || ys[k] >= ctx->n_seqs)))
            FAIL(SNACC_ERR_ARG, "sequence index out of range");
        if (ys && (uint64_t)ctx->h_len[xs[k]] + ctx->h_len[ys[k]] >= 0x7fffffffull)
            FAIL(SNACC_ERR_TOO_LARGE, "pair stream of 2 GiB or more");
    }
    CK(cudaSetDevice(ctx->device));
    int r = ensure_job_buffers(ctx, n_jobs);
    if (r) return r;
    CK(cudaMemcpyAsync(ctx->d_jobx, xs, sizeof(int32_t) * n_jobs, cudaMemcpyHostToDevice, ctx->stream));
    if (ys) CK(cudaMemcpyAsync(ctx->d_joby, ys, sizeof(int32_t) * n_jobs, cudaMemcpyHostToDevice, ctx->stream));
    ctx->last_launches = 0;
    CK(cudaEventRecord(ctx->ev0, ctx->stream));
    if (codec == SNACC_LZ4F) r = run_lz4(ctx, xs, ys, n_jobs);
    else if (codec == SNACC_BZIP2_9) r = run_bzip2(ctx, xs, ys, n_jobs);
    else {
        DeflateCorpus dc{ctx->d_corpus, ctx->d_off, ctx->d_len, ctx->h_off.data(), ctx->h_len.data(), ctx->n_seqs};
        r = deflate_run(ctx->dfl, dc, codec == SNACC_GZIP9 ? 9 : 6, xs, ys, ctx->d_jobx, ys ? ctx->d_joby : nullptr,
                        n_jobs, ctx->d_out, ctx->stream, ctx->streams_in_flight, &ctx->last_launches, ctx->err);
    }
    if (r) return r;
    CK(cudaEventRecord(ctx->ev1, ctx->stream));
    CK(cudaMemcpyAsync(out, ctx->d_out, sizeof(int64_t) * n_jobs, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    float ms = 0.f;
    CK(cudaEventElapsedTime(&ms, ctx->ev0, ctx->ev1));
    ctx->last_ms = ms;
    if (codec == SNACC_GZIP9 || codec == SNACC_ZLIB6) ctx->last_main_ms = ctx->dfl.main_ms;
    if (codec == SNACC_BZIP2_9) ctx->last_main_ms = ctx->bz_ms[1] + ctx->bz_ms[2];
    if (codec == SNACC_LZ4F) {
        CK(cudaEventElapsedTime(&ms, ctx->evm0, ctx->evm1)); ctx->last_main_ms = ms;
        // packed pair streams that could not use their checkpoint exactly (-1) are redone byte-wise
        std::vector<int64_t> redo;
        if (ctx->last_packed_jobs && ys) for (int64_t k = 0; k < n_jobs; ++k) if (out[k] < 0) redo.push_back(k);
        if (!redo.empty()) {
            ctx->last_packed_jobs -= (int64_t)redo.size();
            r = run_lz4_bytewise(ctx, xs, &redo, n_jobs, true);
            if (r) return r;
            CK(cudaMemcpyAsync(out, ctx->d_out, sizeof(int64_t) * n_jobs, cudaMemcpyDeviceToHost, ctx->stream));
            CK(cudaStreamSynchronize(ctx->stream));
        }
    }
    const int64_t wb = wrapper_bytes(codec);
    if (wb) for (int64_t k = 0; k < n_jobs; ++k) out[k] += wb;
    return SNACC_OK;
}

extern "C" int snacc_single_sizes(snacc_ctx *ctx, int codec, const int32_t *idx, int64_t n, int64_t *out)
{
    return sizes_impl(ctx, codec, idx, nullptr, n, out);
}

extern "C" int snacc_pair_sizes(snacc_ctx *ctx, int codec, const int32_t *xs, const int32_t *ys, int64_t n_jobs,
                                int64_t *out)
{
    if (n_jobs && !ys) return SNACC_ERR_ARG;
    return sizes_impl(ctx, codec, xs, ys, n_jobs, out);
}

// rectangle on the packed LZ4 path; returns 1 when the rectangle has to take the per-job path
static int tile_sizes_rect(snacc_ctx *ctx, int32_t row0, int32_t n_rows, int32_t col0, int32_t n_cols, int64_t *out)
{
    std::unique_lock<std::mutex> lock(ctx->mu);
    ctx->err.clear();
    if (!ctx->n_seqs || !ctx->use_packed) return 1;
    if (row0 + n_rows > ctx->n_seqs || col0 + n_cols > ctx->n_seqs) return 1;      // the per-job path reports the error
    const int64_t n = (int64_t)n_rows * n_cols;
    if (n == 0) return 1;
    CK(cudaSetDevice(ctx->device));
    if (n > ctx->out_cap) {
        cudaFree(ctx->d_out); ctx->d_out = nullptr; ctx->out_cap = 0;
        CK(cudaMalloc(&ctx->d_out, sizeof(int64_t) * n));
        ctx->out_cap = n;
    }
    ctx->last_launches = 0;
    ctx->last_packed_jobs = ctx->last_bytewise_jobs = 0;
    CK(cudaEventRecord(ctx->ev0, ctx->stream));
    int r = run_pk_rect(ctx, row0, n_rows, col0, n_cols);
    if (r) return r;
    CK(cudaEventRecord(ctx->ev1, ctx->stream));
    CK(cudaMemcpyAsync(out, ctx->d_out, sizeof(int64_t) * n, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    float ms = 0.f;
    CK(cudaEventElapsedTime(&ms, ctx->ev0, ctx->ev1)); ctx->last_ms = ms;
    CK(cudaEventElapsedTime(&ms, ctx->evm0, ctx->evm1)); ctx->last_main_ms = ms;
    // streams that could not use their checkpoint exactly (-1): redo those jobs on the per-job path
    std::vector<int64_t> redo;
    for (int64_t k = 0; k < n; ++k) if (out[k] < 0) redo.push_back(k);
    if (!redo.empty()) {
        std::vector<int32_t> xs(redo.size()), ys(redo.size());
        std::vector<int64_t> got(redo.size());
        for (size_t k = 0; k < redo.size(); ++k) { xs[k] = row0 + (int32_t)(redo[k] / n_cols); ys[k] = col0 + (int32_t)(redo[k] % n_cols); }
        const int64_t packed = ctx->last_packed_jobs - (int64_t)redo.size();
        ctx->use_packed = 0;
        lock.unlock();
        r = sizes_impl(ctx, SNACC_LZ4F, xs.data(), ys.data(), (int64_t)redo.size(), got.data());
        lock.lock();
        ctx->use_packed = 1;
        if (r) return r;
        for (size_t k = 0; k < redo.size(); ++k) out[redo[k]] = got[k];
        ctx->last_packed_jobs = packed; ctx->last_bytewise_jobs = (int64_t)redo.size();
    }
    return SNACC_OK;
}

extern "C" int snacc_tile_sizes(snacc_ctx *ctx, int codec, int32_t row0, int32_t n_rows, int32_t col0,
                                int32_t n_cols, int64_t *out)
{
    if (!ctx) return SNACC_ERR_ARG;
    if (n_rows < 0 || n_cols < 0 || row0 < 0 || col0 < 0) return SNACC_ERR_ARG;
    if (codec == SNACC_LZ4F && out) {
        const int r = tile_sizes_rect(ctx, row0, n_rows, col0, n_cols, out);
        if (r != 1) return r;
    }
    const int64_t n = (int64_t)n_rows * n_cols;
    std::vector<int32_t> xs((size_t)n), ys((size_t)n);
    for (int32_t r = 0; r < n_rows; ++r)
        for (int32_t c = 0; c < n_cols; ++c) {
            xs[(size_t)r * n_cols + c] = row0 + r;
            ys[(size_t)r * n_cols + c] = col0 + c;
        }
    return sizes_impl(ctx, codec, xs.data(), ys.data(), n, out);
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
    DeflateCorpus dc{ctx->d_corpus, ctx->d_off, ctx->d_len, ctx->h_off.data(), ctx->h_len.data(), ctx->n_seqs};
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
    int64_t *dC = nullptr, *dS = nullptr; double *dD = nullptr;
    const size_t nn = (size_t)n * n;
    int rs = scratch(ctx, 9, sizeof(int64_t) * n, (void **)&dC); if (rs) return rs;       // kept across calls: no malloc per step
    rs = scratch(ctx, 10, sizeof(int64_t) * nn, (void **)&dS); if (rs) return rs;
    rs = scratch(ctx, 11, sizeof(double) * nn, (void **)&dD); if (rs) return rs;
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
    double *dD = nullptr, *dM = nullptr, *dZ = nullptr, *d_nnv = nullptr;
    int32_t *d_size = nullptr, *d_label = nullptr, *d_nni = nullptr, *d_todo = nullptr;
    uint8_t *d_active = nullptr;
    auto release = [&]() {
        cudaFree(dD); cudaFree(dM); cudaFree(dZ); cudaFree(d_nnv); cudaFree(d_size); cudaFree(d_label); cudaFree(d_nni);
        cudaFree(d_todo); cudaFree(d_active);
    };
#define UCK(call) do { cudaError_t e_ = (call); if (e_ != cudaSuccess) { release(); \
        ctx->err = std::string(#call " failed: ") + cudaGetErrorString(e_); return SNACC_ERR_CUDA; } } while (0)
    UCK(cudaMalloc(&dD, sizeof(double) * nn));
    UCK(cudaMalloc(&dM, sizeof(double) * nn));
    UCK(cudaMalloc(&dZ, sizeof(double) * 4 * (size_t)(n - 1)));
    UCK(cudaMalloc(&d_nnv, sizeof(double) * n));
    UCK(cudaMalloc(&d_size, sizeof(int32_t) * n));
    UCK(cudaMalloc(&d_label, sizeof(int32_t) * n));
    UCK(cudaMalloc(&d_nni, sizeof(int32_t) * n));
    UCK(cudaMalloc(&d_todo, sizeof(int32_t) * (n + 1)));
    UCK(cudaMalloc(&d_active, (size_t)n));
    UCK(cudaMemcpyAsync(dD, D, sizeof(double) * nn, cudaMemcpyHostToDevice, ctx->stream));
    metrify_kernel<<<(unsigned)std::min<size_t>((nn + 255) / 256, 148 * 8), 256, 0, ctx->stream>>>(dD, n, metrify ? 1 : 0, dM);
    UCK(cudaGetLastError());
    upgma_kernel<<<1, UPGMA_THREADS, 0, ctx->stream>>>(dM, n, dZ, d_size, d_label, d_nni, d_nnv, d_active, d_todo);
    UCK(cudaGetLastError());
    UCK(cudaMemcpyAsync(Z, dZ, sizeof(double) * 4 * (size_t)(n - 1), cudaMemcpyDeviceToHost, ctx->stream));
    UCK(cudaStreamSynchronize(ctx->stream));
#undef UCK
    release();
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
    if (!strcmp(name, "packed_jobs")) { *out = (double)ctx->last_packed_jobs; return SNACC_OK; }
    if (!strcmp(name, "bytewise_jobs")) { *out = (double)ctx->last_bytewise_jobs; return SNACC_OK; }
    if (!strcmp(name, "lz4_segments")) { *out = (double)ctx->last_pk_segments; return SNACC_OK; }
    if (!strcmp(name, "deflate_serial_jobs")) { *out = (double)ctx->dfl.serial_jobs; return SNACC_OK; }
    if (!strcmp(name, "deflate_parallel_prep_seqs")) { *out = (double)ctx->dfl.parallel_prep_seqs; return SNACC_OK; }
    if (!strcmp(name, "deflate_bands")) { *out = (double)ctx->dfl.bands; return SNACC_OK; }
    if (!strcmp(name, "deflate_state_bytes")) { *out = (double)ctx->dfl.peak; return SNACC_OK; }
    if (!strcmp(name, "deflate_prepared_seqs")) { *out = (double)ctx->dfl.prepared_seqs; return SNACC_OK; }
    if (!strcmp(name, "bzip2_blocks")) { *out = (double)ctx->bz_blocks; return SNACC_OK; }
    if (!strcmp(name, "bzip2_smem_blocks")) { *out = (double)ctx->bz_smem_blocks; return SNACC_OK; }
    if (!strcmp(name, "bzip2_prefix_blocks")) { *out = (double)ctx->bz_prefix_blocks; return SNACC_OK; }
    if (!strcmp(name, "bzip2_rle_gather_ms")) { *out = ctx->bz_ms[0]; return SNACC_OK; }
    if (!strcmp(name, "bzip2_bwt_small_ms")) { *out = ctx->bz_ms[1]; return SNACC_OK; }
    if (!strcmp(name, "bzip2_bwt_large_ms")) { *out = ctx->bz_ms[2]; return SNACC_OK; }
    if (!strcmp(name, "bzip2_bits_ms")) { *out = ctx->bz_ms[3]; return SNACC_OK; }
    return SNACC_ERR_ARG;
}

extern "C" int snacc_set_option(snacc_ctx *ctx, const char *name, int64_t value)
{
    if (!ctx || !name) return SNACC_ERR_ARG;
    std::lock_guard<std::mutex> lock(ctx->mu);
    if (!strcmp(name, "streams_in_flight")) { ctx->streams_in_flight = value; return SNACC_OK; }
    if (!strcmp(name, "lz4_packed")) { ctx->use_packed = value ? 1 : 0; return SNACC_OK; }
    if (!strcmp(name, "lz4_segments")) { ctx->pk_segments = value < 0 ? 0 : value; return SNACC_OK; }
    if (!strcmp(name, "deflate_canonical")) { ctx->dfl.use_canon = value ? 1 : 0; return SNACC_OK; }
    if (!strcmp(name, "deflate_index6")) { ctx->dfl.use_index6 = value ? 1 : 0; return SNACC_OK; }
    if (!strcmp(name, "deflate_parallel_prep")) { ctx->dfl.use_parallel_prep = value ? 1 : 0; return SNACC_OK; }
    if (!strcmp(name, "deflate_tail_index")) { ctx->dfl.use_tail_index = value ? 1 : 0; return SNACC_OK; }
    if (!strcmp(name, "deflate_junction")) { ctx->dfl.junction_impl = value == 2 ? 2 : 3; return SNACC_OK; }
    if (!strcmp(name, "deflate_band_bytes")) { ctx->dfl.band_bytes = value < 0 ? 0 : value; return SNACC_OK; }
    if (!strcmp(name, "bzip2_smem")) { ctx->bz_use_smem = value ? 1 : 0; return SNACC_OK; }
    if (!strcmp(name, "bzip2_prefix")) { ctx->bz_use_prefix = value ? 1 : 0; ctx->bz_ready = false; return SNACC_OK; }
    if (!strcmp(name, "invalidate_caches")) {
        // forget every per-sequence precomputation (prefix checkpoints ...) so the next sizes call
        // redoes the whole job; used by bench.py so that no step reuses work of an earlier step
        std::fill(ctx->ckpt_done.begin(), ctx->ckpt_done.end(), 0);
        std::fill(ctx->h_ck_have.begin(), ctx->h_ck_have.end(), 0);
        deflate_invalidate(ctx->dfl);
        ctx->bz_ready = false;
        return SNACC_OK;
    }
    ctx->err = std::string("unknown option: ") + name;
    return SNACC_ERR_ARG;
}
