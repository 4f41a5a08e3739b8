// lz4_driver.cuh -- host side of the LZ4 codec: the 2-bit packed copy of the corpus (pack.cuh), the prefix checkpoints
// of both paths and the launches of the byte-wise (lz4.cuh) and packed tile kernels (lz4_packed.cuh).  Jobs whose
// operands have a 2-bit copy take the packed kernels, the rest the byte-wise kernel.  Called from api.cu with the
// context lock held.
#pragma once
#include "common.cuh"
#include "lz4.cuh"
#include "pack.cuh"
#include "lz4_packed.cuh"

#ifdef __CUDACC__
#include <string.h>
#include <algorithm>
#include <cmath>
#include <string>
#include <vector>

namespace snacc {

struct Lz4State {
    // byte-wise prefix checkpoints (lz4_prefix_kernel) of the sequences that own at least one full 64 KiB block
    int32_t *d_slot_of = nullptr;          // per sequence: checkpoint slot or -1
    std::vector<int32_t> h_slot_of;
    std::vector<uint8_t> ckpt_done;        // per sequence
    int32_t n_slots = 0;
    uint8_t *d_ckpt_tab = nullptr;
    uint64_t *d_ckpt_total = nullptr;

    // 2-bit packed copy + packed-path prefix checkpoints
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
    uint32_t *d_ck_ovf = nullptr;
    PkAlphabet alphabet;
    uint32_t nslot5 = 1024;                // distinct hash buckets the 1024 5-mers of the alphabet reach

    // working memory: argument arrays of the launches (tiles and their x lists per regime: index 1 single-block, 0
    // linked), EXC overflow tables, tile-segment records
    DevBuf single_seqs, single_want, single_idx, tiles[2], tile_x[2], tile_out, seg_rec, seg_flag, ovf_work;
    unsigned long long *d_counter = nullptr;
    cudaEvent_t evm0 = nullptr, evm1 = nullptr;   // around the dominant kernel of a call
    int sm_count = 148;

    // options
    int use_packed = 1;                    // "lz4_packed": 0 forces the byte-wise kernels
    int64_t pk_segments = 0;               // "lz4_segments": tile segments of the linked pair kernel, 0 = choose per launch
    int64_t streams_in_flight = 0;         // "streams_in_flight": byte-wise streams per launch, 0 = default

    // statistics of the last call
    int64_t packed_jobs = 0, bytewise_jobs = 0, segments = 1;
    double main_ms = 0.0;
};

static inline void lz4_free_corpus(Lz4State &st)
{
    cudaFree(st.d_slot_of); st.d_slot_of = nullptr;
    cudaFree(st.d_ckpt_tab); st.d_ckpt_tab = nullptr;
    cudaFree(st.d_ckpt_total); st.d_ckpt_total = nullptr;
    cudaFree(st.d_pk_words); st.d_pk_words = nullptr;
    cudaFree(st.d_pk_woff); st.d_pk_woff = nullptr;
    cudaFree(st.d_alias5); st.d_alias5 = nullptr;
    cudaFree(st.d_alias4); st.d_alias4 = nullptr;
    cudaFree(st.d_ck_tab); st.d_ck_tab = nullptr;
    cudaFree(st.d_ck_state); st.d_ck_state = nullptr;
    cudaFree(st.d_pk_mask); st.d_pk_mask = nullptr; st.mask_words = 0;
    cudaFree(st.d_pk_moff); st.d_pk_moff = nullptr;
    cudaFree(st.d_b2s); st.d_b2s = nullptr;
    cudaFree(st.d_ck_ovf); st.d_ck_ovf = nullptr;
    st.corpus_dirty = 0;
    st.h_packable.clear(); st.h_ck_have.clear();
    st.n_slots = 0;
}

static inline void lz4_free_work(Lz4State &st)
{
    for (DevBuf *b : {&st.single_seqs, &st.single_want, &st.single_idx, &st.tiles[0], &st.tiles[1], &st.tile_x[0],
                      &st.tile_x[1], &st.tile_out, &st.seg_rec, &st.seg_flag, &st.ovf_work})
        b->release();
    cudaFree(st.d_counter); st.d_counter = nullptr;
    if (st.evm0) cudaEventDestroy(st.evm0);
    if (st.evm1) cudaEventDestroy(st.evm1);
    st.evm0 = st.evm1 = nullptr;
}

// forget every prefix checkpoint: the next call parses its x again
static inline void lz4_invalidate(Lz4State &st)
{
    std::fill(st.ckpt_done.begin(), st.ckpt_done.end(), 0);
    std::fill(st.h_ck_have.begin(), st.h_ck_have.end(), 0);
}

// After an upload: the byte-wise checkpoint slots, then the corpus alphabet measured on the device and a 2-bit copy
// of every sequence that only uses the four most frequent byte values (pack.cuh).  Buffers of a corpus of the same
// shape are reused.
static int lz4_prepare(Lz4State &st, const Corpus &c, cudaStream_t stream, std::string &err)
{
    NvtxRange nvtx_("snacc_b200: alphabet + 2-bit pack");
    const int32_t n = c.n_seqs;
    if (!st.d_counter) {
        int dev = 0;
        DCK(cudaGetDevice(&dev));
        DCK(cudaDeviceGetAttribute(&st.sm_count, cudaDevAttrMultiProcessorCount, dev));
        DCK(cudaMalloc(&st.d_counter, 64));
        DCK(cudaEventCreate(&st.evm0));
        DCK(cudaEventCreate(&st.evm1));
    }
    st.h_slot_of.assign(n, -1);
    st.ckpt_done.assign(n, 0);
    st.n_slots = 0;
    for (int32_t i = 0; i < n; ++i)
        if (c.h_len[i] >= LZ4_BLOCK) st.h_slot_of[i] = st.n_slots++;
    if (!st.d_slot_of) DCK(cudaMalloc(&st.d_slot_of, sizeof(int32_t) * n));
    DCK(cudaMemcpyAsync(st.d_slot_of, st.h_slot_of.data(), sizeof(int32_t) * n, cudaMemcpyHostToDevice, stream));
    if (st.n_slots) {
        if (!st.d_ckpt_tab) DCK(cudaMalloc(&st.d_ckpt_tab, (size_t)st.n_slots * LZ4_TABLE_BYTES));
        if (!st.d_ckpt_total) DCK(cudaMalloc(&st.d_ckpt_total, sizeof(uint64_t) * st.n_slots));
    }

    unsigned long long *d_hist = nullptr;
    DCK(cudaMalloc(&d_hist, 256 * sizeof(unsigned long long)));
    DCK(cudaMemsetAsync(d_hist, 0, 256 * sizeof(unsigned long long), stream));
    uint32_t max_len = 0;
    for (int32_t i = 0; i < n; ++i) max_len = std::max(max_len, c.h_len[i]);
    {
        dim3 grid(std::min<uint32_t>((max_len + 65535) / 65536, 64), (unsigned)std::min<int32_t>(n, 1024));
        pk_hist_kernel<<<grid, 256, 0, stream>>>(c.d_corpus, c.d_off, c.d_len, n, d_hist);
        DCK(cudaGetLastError());
    }
    unsigned long long hist[256];
    DCK(cudaMemcpyAsync(hist, d_hist, sizeof hist, cudaMemcpyDeviceToHost, stream));
    DCK(cudaStreamSynchronize(stream));
    cudaFree(d_hist);
    st.alphabet = pk_choose_alphabet(hist);
    uint16_t a5[1024], a4[256];
    st.nslot5 = pk_slot_lut(st.alphabet, false, a5);
    pk_slot_lut(st.alphabet, true, a4);
    if (!st.d_alias5) DCK(cudaMalloc(&st.d_alias5, sizeof a5));
    if (!st.d_alias4) DCK(cudaMalloc(&st.d_alias4, sizeof a4));
    DCK(cudaMemcpyAsync(st.d_alias5, a5, sizeof a5, cudaMemcpyHostToDevice, stream));
    DCK(cudaMemcpyAsync(st.d_alias4, a4, sizeof a4, cudaMemcpyHostToDevice, stream));

    PkCodes codes;
    memcpy(codes.c, st.alphabet.code_of, 256);
    std::vector<uint64_t> woff((size_t)n), moff((size_t)n);
    uint64_t w = 0, mw = 0;
    for (int32_t i = 0; i < n; ++i) { woff[i] = w; w += pk_words(c.h_len[i]); moff[i] = mw; mw += pk_mask_words(c.h_len[i]); }
    // bytes outside the alphabet anywhere in the corpus?  Then the packed copy carries a per-base mask of them and the
    // EXC kernels run (lz4_packed.cuh: pk_step_exact)
    unsigned long long outside = 0;
    for (int i = 0; i < 256; ++i) if (st.alphabet.code_of[i] > 3) outside += hist[i];
    st.corpus_dirty = outside ? 1 : 0;
    int32_t *d_nexc = nullptr;
    if (!st.d_pk_words) DCK(cudaMalloc(&st.d_pk_words, w * sizeof(uint64_t)));
    if (!st.d_pk_woff) DCK(cudaMalloc(&st.d_pk_woff, sizeof(uint64_t) * n));
    DCK(cudaMalloc(&d_nexc, sizeof(int32_t) * n));
    DCK(cudaMemsetAsync(d_nexc, 0, sizeof(int32_t) * n, stream));
    DCK(cudaMemcpyAsync(st.d_pk_woff, woff.data(), sizeof(uint64_t) * n, cudaMemcpyHostToDevice, stream));
    if (st.corpus_dirty) {
        if (st.d_pk_mask && st.mask_words < mw) { cudaFree(st.d_pk_mask); st.d_pk_mask = nullptr; }
        if (!st.d_pk_mask) { DCK(cudaMalloc(&st.d_pk_mask, (mw + 64) * sizeof(uint32_t))); st.mask_words = mw; }
        if (!st.d_pk_moff) DCK(cudaMalloc(&st.d_pk_moff, sizeof(uint64_t) * n));
        if (!st.d_b2s) DCK(cudaMalloc(&st.d_b2s, sizeof(uint16_t) * PK_OVF_ENTRIES));
        if (!st.d_ck_ovf) DCK(cudaMalloc(&st.d_ck_ovf, sizeof(uint32_t) * PK_OVF_ENTRIES * (size_t)n));
        DCK(cudaMemsetAsync(st.d_pk_mask, 0, (mw + 64) * sizeof(uint32_t), stream));
        DCK(cudaMemsetAsync(st.d_ck_ovf, 0, sizeof(uint32_t) * PK_OVF_ENTRIES * (size_t)n, stream));
        DCK(cudaMemcpyAsync(st.d_pk_moff, moff.data(), sizeof(uint64_t) * n, cudaMemcpyHostToDevice, stream));
        uint16_t b2s[PK_OVF_ENTRIES];
        for (uint32_t i = 0; i < PK_OVF_ENTRIES; ++i) b2s[i] = 0xffff;
        for (uint32_t cc = 0; cc < 1024; ++cc) b2s[pk_bucket(st.alphabet, cc, false)] = a5[cc];
        DCK(cudaMemcpyAsync(st.d_b2s, b2s, sizeof b2s, cudaMemcpyHostToDevice, stream));
    }
    {
        dim3 grid(std::min<uint32_t>((pk_words(max_len) + 255) / 256, 256), (unsigned)std::min<int32_t>(n, 4096));
        pk_pack_kernel<<<grid, 256, 0, stream>>>(c.d_corpus, c.d_off, c.d_len, st.d_pk_woff, n, st.d_pk_words, d_nexc,
                                                 st.corpus_dirty ? st.d_pk_mask : nullptr, st.d_pk_moff, codes);
        DCK(cudaGetLastError());
    }
    std::vector<int32_t> nexc((size_t)n);
    DCK(cudaMemcpyAsync(nexc.data(), d_nexc, sizeof(int32_t) * n, cudaMemcpyDeviceToHost, stream));
    if (!st.d_ck_tab) DCK(cudaMalloc(&st.d_ck_tab, (size_t)n * 2 * PK_CKPT_TAB * sizeof(uint32_t)));
    if (!st.d_ck_state) DCK(cudaMalloc(&st.d_ck_state, (size_t)n * 2 * sizeof(PkState)));
    DCK(cudaStreamSynchronize(stream));
    cudaFree(d_nexc);
    // a sequence keeps to the tile kernels while its flagged bases are sparse: an isolated one costs every stream that
    // meets it a handful of byte-exact steps (about what 450 ordinary probes cost a warp), so the tile kernels stay
    // ahead of the byte-wise ones up to roughly one flagged base in 64; denser sequences -- proteins, heavily
    // soft-masked assemblies -- take the byte-wise kernels
    st.h_packable.assign(n, 0);
    for (int32_t i = 0; i < n; ++i)
        st.h_packable[i] = nexc[i] == 0 ? 1 : ((uint64_t)nexc[i] <= (uint64_t)c.h_len[i] / 64 + 8 ? 2 : 0);
    st.h_ck_have.assign(n, 0);
    return 0;
}

// byte-wise path: make sure every x that starts a linked-regime stream has its prefix checkpoint
static int lz4_prepare_prefixes(Lz4State &st, const Corpus &c, const int32_t *xs, int64_t n, cudaStream_t stream,
                                int64_t *launches, std::string &err)
{
    std::vector<int32_t> todo;
    for (int64_t k = 0; k < n; ++k) {
        const int32_t x = xs[k];
        if (st.h_slot_of[x] >= 0 && !st.ckpt_done[x]) { st.ckpt_done[x] = 1; todo.push_back(x); }
    }
    if (todo.empty()) return 0;
    int32_t *d_todo = nullptr;
    DCK(cudaMalloc(&d_todo, sizeof(int32_t) * todo.size()));
    DCK(cudaMemcpyAsync(d_todo, todo.data(), sizeof(int32_t) * todo.size(), cudaMemcpyHostToDevice, stream));
    const int threads = 32;
    const int blocks = (int)((todo.size() + threads - 1) / threads);
    lz4_prefix_kernel<<<blocks, threads, 0, stream>>>(c.d_corpus, c.d_off, c.d_len, d_todo, (int32_t)todo.size(),
                                                      st.d_slot_of, st.d_ckpt_tab, st.d_ckpt_total);
    ++*launches;
    DCK(cudaGetLastError());
    DCK(cudaStreamSynchronize(stream));
    cudaFree(d_todo);
    return 0;
}

// byte-wise kernel (lz4.cuh) on the jobs `sel` (host list; null = all n_jobs jobs) of the device job arrays d_xs, d_ys
// (d_ys null: singles); h_x is the host copy of d_xs.  `work` holds one 16 KiB table per resident stream.
static int lz4_run_bytewise(Lz4State &st, const Corpus &c, const int32_t *h_x, const int32_t *d_xs, const int32_t *d_ys,
                            const std::vector<int64_t> *sel, int64_t n_jobs, int64_t *d_out, DevBuf &work,
                            cudaStream_t stream, int64_t *launches, std::string &err)
{
    NvtxRange nvtx_("snacc_b200: lz4 byte-wise streams");
    const int64_t n = sel ? (int64_t)sel->size() : n_jobs;
    if (n == 0) return 0;
    std::vector<int32_t> xs((size_t)n);
    for (int64_t k = 0; k < n; ++k) xs[k] = h_x[sel ? (*sel)[k] : k];
    int r = lz4_prepare_prefixes(st, c, xs.data(), n, stream, launches, err);
    if (r) return r;
    // linked-regime streams each own a 16 KiB table that is hit at random: keep the set L2 resident
    // (one warp per SM); single-block streams are short and want many more threads in flight
    bool any_linked = false;
    for (int64_t k = 0; k < n && !any_linked; ++k) any_linked = c.h_len[xs[k]] >= LZ4_BLOCK / 2;
    int64_t inflight = st.streams_in_flight > 0 ? st.streams_in_flight : (any_linked ? 148 * 32 : 148 * 1024);
    const int threads = 32;
    int64_t blocks = (std::min<int64_t>(inflight, n) + threads - 1) / threads;
    if (blocks < 1) blocks = 1;
    DCK(work.grow((size_t)blocks * threads * LZ4_TABLE_BYTES, stream, true));
    int64_t *d_sel = nullptr;
    if (sel) {
        DCK(cudaMalloc(&d_sel, sizeof(int64_t) * n));
        DCK(cudaMemcpyAsync(d_sel, sel->data(), sizeof(int64_t) * n, cudaMemcpyHostToDevice, stream));
    }
    DCK(cudaMemsetAsync(st.d_counter, 0, sizeof(unsigned long long), stream));
    if (!st.packed_jobs) DCK(cudaEventRecord(st.evm0, stream));
    lz4_stream_kernel<<<(unsigned)blocks, threads, 0, stream>>>(
        c.d_corpus, c.d_off, c.d_len, d_xs, d_ys, d_sel, n, st.d_slot_of, st.d_ckpt_tab, st.d_ckpt_total,
        work.get<uint8_t>(), st.d_counter, d_out);
    if (!st.packed_jobs) DCK(cudaEventRecord(st.evm1, stream));
    ++*launches;
    st.bytewise_jobs += n;
    DCK(cudaGetLastError());
    if (d_sel) { DCK(cudaStreamSynchronize(stream)); cudaFree(d_sel); }
    return 0;
}

// what the EXC kernels take on top of the packed corpus; `tabs` overflow tables of working memory are made available
static int pk_exc_corpus(Lz4State &st, const Corpus &c, size_t tabs, PkExcCorpus *xc, cudaStream_t stream,
                         std::string &err)
{
    DCK(st.ovf_work.grow(tabs * PK_OVF_ENTRIES * sizeof(uint32_t), stream, true));
    *xc = PkExcCorpus{st.d_pk_mask, st.d_pk_moff, c.d_corpus, c.d_off, st.d_b2s, st.ovf_work.get<uint32_t>(), st.d_ck_ovf};
    return 0;
}

// packed path, step 1: singles and/or prefix checkpoints of the listed sequences (lz4_pk_single_kernel)
static int run_pk_single(Lz4State &st, const Corpus &c, const std::vector<int32_t> &seqs, const std::vector<int32_t> &want,
                         const std::vector<int64_t> &out_idx, int64_t *d_out, cudaStream_t stream, int64_t *launches,
                         std::string &err)
{
    NvtxRange nvtx_("snacc_b200: lz4 singles + prefix checkpoints");
    const int32_t n = (int32_t)seqs.size();
    if (!n) return 0;
    DCK(st.single_seqs.grow(sizeof(int32_t) * n, stream));
    DCK(st.single_want.grow(sizeof(int32_t) * n, stream));
    DCK(st.single_idx.grow(sizeof(int64_t) * n, stream));
    int32_t *d_seqs = st.single_seqs.get<int32_t>(), *d_want = st.single_want.get<int32_t>();
    int64_t *d_idx = st.single_idx.get<int64_t>();
    DCK(cudaMemcpyAsync(d_seqs, seqs.data(), sizeof(int32_t) * n, cudaMemcpyHostToDevice, stream));
    DCK(cudaMemcpyAsync(d_want, want.data(), sizeof(int32_t) * n, cudaMemcpyHostToDevice, stream));
    DCK(cudaMemcpyAsync(d_idx, out_idx.data(), sizeof(int64_t) * n, cudaMemcpyHostToDevice, stream));
    const PkCorpus pc{st.d_pk_words, st.d_pk_woff, c.d_len};
    PkExcCorpus xc{};
    if (st.corpus_dirty) {
        const int rs = pk_exc_corpus(st, c, (size_t)n, &xc, stream, err); if (rs) return rs;
        lz4_pk_single_kernel<true><<<n, 64, 0, stream>>>(pc, xc, d_seqs, d_want, n, st.d_ck_tab, st.d_ck_state,
                                                         st.d_alias5, st.d_alias4, d_idx, d_out);
    } else {
        lz4_pk_single_kernel<false><<<n, 64, 0, stream>>>(pc, xc, d_seqs, d_want, n, st.d_ck_tab, st.d_ck_state,
                                                          st.d_alias5, st.d_alias4, d_idx, d_out);
    }
    ++*launches;
    DCK(cudaGetLastError());
    return 0;
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

static PkGeometry pk_geometry(const Lz4State &st, bool u16)
{
    PkGeometry g;
    g.exc = false;
    if (u16) { g.nslot = 256; g.lanes = PK_S_LANES; g.warps = PK_S_WARPS; g.smem = PK_S_SMEM; g.T = PK_S_LANES * PK_S_WARPS; return g; }
    // linked regime: as many streams as one SM's shared memory holds (A/C/G/T: 894 slots -> 1900 B per stream
    // -> 104 streams = 4 warps x 26 lanes; a full 1024-slot alphabet: 90 -> 2 warps x 32 lanes)
    g.nslot = (st.nslot5 + 1) & ~1u;
    const size_t l_stream = (size_t)g.nslot * 2 + ((g.nslot + 31) / 32) * 4;        // bytes of table per linked stream
    // a corpus with flagged bases runs the EXC kernel (same geometry: its dirty ring lives inside the ring)
    g.exc = st.corpus_dirty != 0;
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
static int pk_choose_segments(const Lz4State &st, const Corpus &c, const PkGeometry &g, const std::vector<PkTile> &tiles)
{
    uint32_t min_runs = 0xffffffffu;
    for (const PkTile &t : tiles) {
        PkRing rg; uint32_t w0, w1;
        rg.start(c.h_len[t.y], w0, w1, g.exc ? PK_RING_COVER_EXC : PK_RING_WORDS);
        min_runs = std::min(min_runs, rg.runs());
    }
    const size_t per_stream = (size_t)g.nslot * 2 + ((g.nslot + 31) / 32) * 4 + sizeof(PkState) + 4 +
                              (g.exc ? PK_OVF_ENTRIES * sizeof(uint32_t) : 0);
    if (tiles.size() * g.T * per_stream > ((size_t)6 << 30)) return 1;
    if (st.pk_segments > 0) return (int)std::min<int64_t>(st.pk_segments, std::max<uint32_t>(1, min_runs / 2));
    const double sms = (double)st.sm_count, nt = (double)tiles.size();
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
static int pk_launch(Lz4State &st, const Corpus &c, bool u16, const PkGeometry &g, const std::vector<PkTile> &tiles,
                     const std::vector<int32_t> &tx, const std::vector<int64_t> &tout, int64_t out_stride, int32_t col0,
                     int64_t n_jobs, int64_t *d_out, cudaStream_t stream, int64_t *launches, std::string &err)
{
    NvtxRange nvtx_("snacc_b200: lz4 pair tiles");
    DevBuf &b_tiles = st.tiles[u16], &b_tx = st.tile_x[u16];
    DCK(b_tiles.grow(sizeof(PkTile) * tiles.size(), stream));
    DCK(b_tx.grow(sizeof(int32_t) * tx.size(), stream));
    const PkTile *d_tiles = b_tiles.get<PkTile>();
    const int32_t *d_tx = b_tx.get<int32_t>();
    int64_t *d_tout = nullptr;
    DCK(cudaMemcpyAsync(b_tiles.p, tiles.data(), sizeof(PkTile) * tiles.size(), cudaMemcpyHostToDevice, stream));
    DCK(cudaMemcpyAsync(b_tx.p, tx.data(), sizeof(int32_t) * tx.size(), cudaMemcpyHostToDevice, stream));
    if (!tout.empty()) {
        DCK(st.tile_out.grow(sizeof(int64_t) * tout.size(), stream));
        d_tout = st.tile_out.get<int64_t>();
        DCK(cudaMemcpyAsync(d_tout, tout.data(), sizeof(int64_t) * tout.size(), cudaMemcpyHostToDevice, stream));
    }
    unsigned long long *counter = st.d_counter + (u16 ? 1 : 2);
    DCK(cudaMemsetAsync(counter, 0, sizeof(unsigned long long), stream));
    const PkCorpus pc{st.d_pk_words, st.d_pk_woff, c.d_len};
    const int32_t nt = (int32_t)tiles.size();
    const int n_seg = u16 ? 1 : pk_choose_segments(st, c, g, tiles);
    st.segments = n_seg;
    const int grid = (int)std::min<size_t>(tiles.size() * n_seg, (size_t)st.sm_count);
    PkSegStore ss{};
    if (n_seg > 1) {
        // the records of every stream of the launch, carved out of one array; flags zeroed per launch
        const size_t ns = tiles.size() * g.T, nw = (g.nslot + 31) / 32;
        const size_t b_tab = (ns * g.nslot * 2 + 15) & ~(size_t)15, b_ep = (ns * nw * 4 + 15) & ~(size_t)15,
                     b_st = ns * sizeof(PkState), b_eb = ns * 4;
        DCK(st.seg_rec.grow(b_tab + b_ep + b_st + b_eb, stream));
        uint8_t *base = st.seg_rec.get<uint8_t>();
        ss.tab = (uint16_t *)base; ss.ep = (uint32_t *)(base + b_tab); ss.st = (PkState *)(base + b_tab + b_ep);
        ss.eb = (uint32_t *)(base + b_tab + b_ep + b_st);
        DCK(st.seg_flag.grow(sizeof(int32_t) * tiles.size(), stream));
        ss.flag = st.seg_flag.get<int32_t>();
        DCK(cudaMemsetAsync(ss.flag, 0, sizeof(int32_t) * tiles.size(), stream));
    }
    DCK(cudaEventRecord(st.evm0, stream));
    PkExcCorpus xc{};
    if (g.exc) {
        const int rs = pk_exc_corpus(st, c, n_seg > 1 ? tiles.size() * g.T : (size_t)grid * g.T, &xc, stream, err);
        if (rs) return rs;
    }
#define PK_GO(KIND_, LANES_, EXC_, lut_) do {                                                                        \
        DCK(cudaFuncSetAttribute(lz4_pk_pair_kernel<KIND_, LANES_, EXC_>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)g.smem)); \
        lz4_pk_pair_kernel<KIND_, LANES_, EXC_><<<grid, g.warps * 32, g.smem, stream>>>(                               \
            pc, xc, d_tiles, nt, d_tx, d_tout, st.d_ck_tab, st.d_ck_state, lut_, g.nslot, out_stride, col0, counter, d_out, n_seg, ss); \
    } while (0)
    if (u16) PK_GO(1, PK_S_LANES, false, st.d_alias4);
    else if (g.exc && g.lanes == 26) PK_GO(2, 26, true, st.d_alias5);
    else if (g.exc && g.lanes == 25) PK_GO(2, 25, true, st.d_alias5);
    else if (g.exc) PK_GO(2, 32, true, st.d_alias5);
    else if (g.lanes == 26) PK_GO(2, 26, false, st.d_alias5);
    else if (g.lanes == 25) PK_GO(2, 25, false, st.d_alias5);
    else PK_GO(2, 32, false, st.d_alias5);
#undef PK_GO
    DCK(cudaEventRecord(st.evm1, stream));
    ++*launches;
    st.packed_jobs += n_jobs;
    DCK(cudaGetLastError());
    return 0;
}

static int run_pk_pairs(Lz4State &st, const Corpus &c, std::vector<PkJob> &jobs, bool u16, int64_t *d_out,
                        cudaStream_t stream, int64_t *launches, std::string &err)
{
    if (jobs.empty()) return 0;
    const PkGeometry g = pk_geometry(st, u16);
    std::sort(jobs.begin(), jobs.end(), [&](const PkJob &a, const PkJob &b) {
        const uint32_t la = c.h_len[a.y], lb = c.h_len[b.y];
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
    return pk_launch(st, c, u16, g, tiles, tx, tout, 0, 0, (int64_t)jobs.size(), d_out, stream, launches, err);
}

// make sure the listed sequences have their packed prefix checkpoint for the regimes in `need` (bit 0 / bit 1)
static int pk_ensure_ckpts(Lz4State &st, const Corpus &c, const std::vector<int32_t> &need, int64_t *d_out,
                           cudaStream_t stream, int64_t *launches, std::string &err)
{
    std::vector<int32_t> seqs, want; std::vector<int64_t> idx;
    for (int32_t s = 0; s < c.n_seqs; ++s) {
        const int32_t missing = need[s] & ~st.h_ck_have[s];
        if (missing) { seqs.push_back(s); want.push_back(missing); idx.push_back(-1); st.h_ck_have[s] |= (uint8_t)missing; }
    }
    return run_pk_single(st, c, seqs, want, idx, d_out, stream, launches, err);
}

// Whether rows [row0, row0+n_rows) x cols [col0, col0+n_cols) of the ordered-pair matrix can run on the packed path as
// one rectangle, without per-job arrays (c3: 10^8 jobs): 0 when it is not uniform enough (packed path off, some
// sequence outside the alphabet, a y shorter than 16, or pairs on both sides of the 64 KiB regime boundary), else the
// regime of all its pairs, 1 single-block or 2 linked (the checkpoint bit its x need).
static int lz4_rect_regime(const Lz4State &st, const Corpus &c, int32_t row0, int32_t n_rows, int32_t col0,
                           int32_t n_cols)
{
    if (!st.use_packed) return 0;
    uint32_t min_x = 0xffffffffu, max_x = 0, min_y = 0xffffffffu, max_y = 0;
    bool any_flagged = false;
    for (int32_t r = row0; r < row0 + n_rows; ++r) {
        if (!st.h_packable[r]) return 0;
        any_flagged |= st.h_packable[r] == 2;
        min_x = std::min(min_x, c.h_len[r]); max_x = std::max(max_x, c.h_len[r]);
    }
    for (int32_t cc = col0; cc < col0 + n_cols; ++cc) {
        if (!st.h_packable[cc]) return 0;
        any_flagged |= st.h_packable[cc] == 2;
        min_y = std::min(min_y, c.h_len[cc]); max_y = std::max(max_y, c.h_len[cc]);
    }
    if (min_y < 16) return 0;
    const bool all_small = (uint64_t)max_x + max_y <= LZ4_BLOCK, all_linked = (uint64_t)min_x + min_y > LZ4_BLOCK;
    if (!all_small && !all_linked) return 0;
    if (all_small && any_flagged) return 0;            // flagged bases: linked regime only (per-job path sorts it out)
    return all_small ? 1 : 2;
}

// the rectangle of lz4_rect_regime on the packed path; results go to d_out in row-major order
static int lz4_run_rect(Lz4State &st, const Corpus &c, int regime, int32_t row0, int32_t n_rows, int32_t col0,
                        int32_t n_cols, int64_t *d_out, cudaStream_t stream, int64_t *launches, std::string &err)
{
    st.packed_jobs = st.bytewise_jobs = 0;
    const bool u16 = regime == 1;
    std::vector<int32_t> need((size_t)c.n_seqs, 0);
    for (int32_t r = row0; r < row0 + n_rows; ++r) need[r] = regime;
    int rc = pk_ensure_ckpts(st, c, need, d_out, stream, launches, err);
    if (rc) return rc;
    const PkGeometry g = pk_geometry(st, u16);
    std::vector<int32_t> cols((size_t)n_cols), tx((size_t)n_rows);
    for (int32_t k = 0; k < n_cols; ++k) cols[k] = col0 + k;
    std::stable_sort(cols.begin(), cols.end(), [&](int32_t a, int32_t b) { return c.h_len[a] > c.h_len[b]; });
    for (int32_t r = 0; r < n_rows; ++r) tx[r] = row0 + r;
    std::vector<PkTile> tiles;
    for (int32_t y : cols) pk_split(tiles, y, 0, (size_t)n_rows, g.T);
    return pk_launch(st, c, u16, g, tiles, tx, std::vector<int64_t>(), n_cols, col0, (int64_t)n_rows * n_cols, d_out,
                     stream, launches, err);
}

// A job list (ys null: singles) into d_out.  d_xs, d_ys: the job arrays on the device.
static int lz4_run(Lz4State &st, const Corpus &c, const int32_t *xs, const int32_t *ys, const int32_t *d_xs,
                   const int32_t *d_ys, int64_t n_jobs, int64_t *d_out, DevBuf &work, cudaStream_t stream,
                   int64_t *launches, std::string &err)
{
    st.packed_jobs = st.bytewise_jobs = 0;
    if (!st.use_packed) return lz4_run_bytewise(st, c, xs, d_xs, d_ys, nullptr, n_jobs, d_out, work, stream, launches, err);
    std::vector<int64_t> bytewise;
    int r;
    if (!ys) {
        std::vector<int32_t> seqs, want; std::vector<int64_t> idx;
        for (int64_t k = 0; k < n_jobs; ++k) {
            // (a sequence with flagged bases that is a single-block stream has no byte-exact step: byte-wise kernel)
            if (st.h_packable[xs[k]] == 1 || (st.h_packable[xs[k]] == 2 && c.h_len[xs[k]] > LZ4_BLOCK)) {
                // the same pass leaves the prefix checkpoints a later pair call with this x would need (the extra work
                // is a re-run of the last partial block), so that call does not have to parse the sequence again
                const int32_t sq = xs[k];
                const int32_t all = 2 | (c.h_len[sq] < LZ4_BLOCK ? 1 : 0);
                const int32_t missing = all & ~st.h_ck_have[sq];
                st.h_ck_have[sq] |= (uint8_t)missing;
                seqs.push_back(sq); want.push_back(missing); idx.push_back(k);
            }
            else bytewise.push_back(k);
        }
        st.packed_jobs = (int64_t)seqs.size();
        DCK(cudaEventRecord(st.evm0, stream));
        r = run_pk_single(st, c, seqs, want, idx, d_out, stream, launches, err);
        if (r) return r;
        DCK(cudaEventRecord(st.evm1, stream));
    } else {
        std::vector<PkJob> small, linked;
        std::vector<int32_t> need((size_t)c.n_seqs, 0);
        for (int64_t k = 0; k < n_jobs; ++k) {
            const int32_t x = xs[k], y = ys[k];
            if (!st.h_packable[x] || !st.h_packable[y] || c.h_len[y] < 16) { bytewise.push_back(k); continue; }
            const bool u16 = (uint64_t)c.h_len[x] + c.h_len[y] <= LZ4_BLOCK;
            if (u16 && (st.h_packable[x] == 2 || st.h_packable[y] == 2)) { bytewise.push_back(k); continue; }
            (u16 ? small : linked).push_back(PkJob{y, x, k});
            need[x] |= u16 ? 1 : 2;
        }
        r = pk_ensure_ckpts(st, c, need, d_out, stream, launches, err);
        if (r) return r;
        r = run_pk_pairs(st, c, small, true, d_out, stream, launches, err);
        if (r) return r;
        r = run_pk_pairs(st, c, linked, false, d_out, stream, launches, err);
        if (r) return r;
    }
    if (!bytewise.empty()) return lz4_run_bytewise(st, c, xs, d_xs, d_ys, &bytewise, n_jobs, d_out, work, stream, launches, err);
    return 0;
}

// After the sizes of a call are on the host (out[0, n_jobs)): the time of its dominant kernel, then the packed pair
// streams that could not use their checkpoint exactly (-1) are redone on the byte-wise kernel.  The jobs are xs, ys,
// or with xs null the rectangle rows from row0 x n_cols columns from col0 (row-major).  The redo runs on its own
// compact job list, its sizes land in d_out[0, redo) and then in out.
static int lz4_finish(Lz4State &st, const Corpus &c, const int32_t *xs, const int32_t *ys, int32_t row0, int32_t col0,
                      int32_t n_cols, int64_t n_jobs, int64_t *out, int64_t *d_out, DevBuf &work, cudaStream_t stream,
                      int64_t *launches, std::string &err)
{
    float ms = 0.f;
    DCK(cudaEventElapsedTime(&ms, st.evm0, st.evm1));
    st.main_ms = ms;
    if (!st.packed_jobs || (xs && !ys)) return 0;
    std::vector<int64_t> redo;
    for (int64_t k = 0; k < n_jobs; ++k) if (out[k] < 0) redo.push_back(k);
    if (redo.empty()) return 0;
    const int64_t n = (int64_t)redo.size();
    std::vector<int32_t> rxy((size_t)(2 * n));            // x list, then y list
    for (int64_t k = 0; k < n; ++k) {
        const int64_t j = redo[k];
        rxy[k] = xs ? xs[j] : row0 + (int32_t)(j / n_cols);
        rxy[n + k] = xs ? ys[j] : col0 + (int32_t)(j % n_cols);
    }
    st.packed_jobs -= n;
    int32_t *d_rxy = nullptr;
    DCK(cudaMalloc(&d_rxy, sizeof(int32_t) * 2 * n));
    DCK(cudaMemcpyAsync(d_rxy, rxy.data(), sizeof(int32_t) * 2 * n, cudaMemcpyHostToDevice, stream));
    const int r = lz4_run_bytewise(st, c, rxy.data(), d_rxy, d_rxy + n, nullptr, n, d_out, work, stream, launches, err);
    if (r) { cudaFree(d_rxy); return r; }
    std::vector<int64_t> got((size_t)n);
    DCK(cudaMemcpyAsync(got.data(), d_out, sizeof(int64_t) * n, cudaMemcpyDeviceToHost, stream));
    DCK(cudaStreamSynchronize(stream));
    cudaFree(d_rxy);
    for (int64_t k = 0; k < n; ++k) out[redo[k]] = got[k];
    return 0;
}

}  // namespace snacc
#endif  // __CUDACC__
