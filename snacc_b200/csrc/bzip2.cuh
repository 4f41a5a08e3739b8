// bzip2.cuh -- K5: len(bz2.compress(b)) (libbz2 1.0.8, level 9, as CPython drives it: BZ_RUN, then BZ_FINISH).
//
// The size is a function of independent blocks, and the bits of a block depend only on its bytes:
//   RLE1 -> block cut -> BWT (last column of the sorted cyclic rotations; tied rotations are equal, so the sort
//   algorithm does not matter) -> MTF + RLE2 -> Huffman table choice (4 iterations) -> bit count.
// CRCs and origPtr are fixed-width fields, so nothing of the bit stream itself has to be produced.
//
// Everything below marked SNACC_BZ_HD is compiled for the host as well (tests/host_emu_bzip2.cu runs the same code
// against libbz2); the kernels (bz_*) compose those functions in parallel.
#pragma once
#include <stdint.h>
#include <algorithm>
#include <string>
#include <vector>
#include "common.cuh"

#define SNACC_BZ_HD __host__ __device__ inline

namespace snacc {

constexpr uint32_t BZ_NBLOCK_MAX = 100000u * 9u - 19u;     // a block closes before an emission once it holds this many
constexpr int BZ_G_SIZE = 50, BZ_N_ITERS = 4, BZ_N_GROUPS = 6, BZ_MAX_ALPHA = 258, BZ_MAX_CODE_LEN = 17;
constexpr int BZ_MAX_SELECTORS = (int)((BZ_NBLOCK_MAX + 5 + 1 + BZ_G_SIZE - 1) / BZ_G_SIZE);
constexpr int64_t BZ_STREAM_BITS = 32 + 48 + 32;            // "BZh9", end-of-stream magic, combined CRC
constexpr int64_t BZ_BLOCK_FIXED_BITS = 48 + 32 + 1 + 24;   // block magic, block CRC, randomised bit, origPtr
constexpr int BZ_HB_SCRATCH = (BZ_MAX_ALPHA + 2) + 2 * (2 * BZ_MAX_ALPHA);   // ints for bz_make_code_lengths

// ---- RLE1 (stage 1) ------------------------------------------------------------------------------------------------
// A maximal run of T equal bytes is emitted as chunks of 255 (then the remainder): a chunk of 1-3 bytes as itself, one
// of 4-255 as 4 bytes plus a count byte (length - 4).  RLE1 bytes of a chunk of length c:
SNACC_BZ_HD uint32_t bz_chunk_bytes(uint32_t c) { return c >= 4 ? 5u : c; }
SNACC_BZ_HD uint64_t bz_run_bytes(uint64_t T) { return (T / 255) * 5 + bz_chunk_bytes((uint32_t)(T % 255)); }

// byte t of the emissions of a run of T bytes b, and whether an emission starts there
SNACC_BZ_HD uint8_t bz_run_at(uint8_t b, uint64_t T, uint64_t t, bool *start)
{
    const uint64_t full = (T / 255) * 5;
    if (t < full) { const uint32_t k = (uint32_t)(t % 5); *start = k == 0; return k < 4 ? b : (uint8_t)251; }
    const uint32_t u = (uint32_t)(t - full), r = (uint32_t)(T % 255);
    *start = u == 0;
    return u < 4 ? b : (uint8_t)(r - 4);
}

// What a pair stream needs of a sequence besides its RLE1 bytes.
struct BzSeq {
    uint64_t roff;        // offset of the sequence's RLE1 bytes (and emission-start flags)
    uint32_t rlen;        // RLE1 bytes of the sequence alone (every emission, the final one included)
    uint32_t fin;         // where the final emission (the last chunk of the last run, 1-255 bytes long) starts
    uint32_t first_end;   // where the emissions of the first maximal run end
    uint32_t p;           // length of that final chunk
    uint32_t U;           // length of the first maximal run
    uint8_t blast, bfirst;
};

// RLE1 of one sequence: rle[0, rlen) and flag[t] = 1 where an emission starts (room for bz_run_bytes bound: n*5/4+5)
SNACC_BZ_HD void bz_rle_seq(const uint8_t *s, uint32_t n, uint8_t *rle, uint8_t *flag, BzSeq *info)
{
    uint32_t w = 0, i = 0, fin = 0, p = 0;
    info->bfirst = s[0];
    while (i < n) {
        const uint8_t b = s[i];
        uint32_t j = i + 1;
        while (j < n && s[j] == b) ++j;
        const uint32_t T = j - i;
        if (i == 0) info->U = T;
        for (uint32_t c0 = 0; c0 < T; c0 += 255) {
            const uint32_t c = T - c0 < 255 ? T - c0 : 255;
            fin = w; p = c;
            const uint32_t k = bz_chunk_bytes(c);
            for (uint32_t q = 0; q < k; ++q) { rle[w + q] = q < 4 ? b : (uint8_t)(c - 4); flag[w + q] = q == 0; }
            w += k;
        }
        if (i == 0) info->first_end = w;
        info->blast = b;
        i = j;
    }
    info->rlen = w; info->fin = fin; info->p = p;
}

// The stream a pair job still has to cut after x's closed blocks: A = RLE1(x)[a0, a1) (x's open tail without its final
// emission), then the junction -- the final chunk of x merged with y's first run when the bytes agree, else the two
// runs one after the other -- then B = RLE1(y)[b0, b1) (RLE1(x.y) equals RLE1(y) after y's first run).  A single or
// a closed block of x is a window of A alone (no junction, no B).
struct BzView {
    uint32_t a0, a1, b0, b1;
    uint32_t j0, j1;      // junction run lengths (j1 = 0: one run)
    uint8_t jb0, jb1;
    SNACC_BZ_HD uint64_t jlen() const { return (j0 ? bz_run_bytes(j0) : 0) + (j1 ? bz_run_bytes(j1) : 0); }
    SNACC_BZ_HD uint64_t total() const { return (uint64_t)(a1 - a0) + jlen() + (b1 - b0); }
    // does an emission start at byte t of the view?
    SNACC_BZ_HD bool starts(const uint8_t *fx, const uint8_t *fy, uint64_t t) const
    {
        const uint64_t la = a1 - a0;
        if (t < la) return fx[a0 + t] != 0;
        t -= la;
        const uint64_t lj = jlen();
        if (t >= lj) return fy[b0 + (t - lj)] != 0;
        bool st;
        const uint64_t l0 = j0 ? bz_run_bytes(j0) : 0;
        if (t < l0) bz_run_at(jb0, j0, t, &st); else bz_run_at(jb1, j1, t - l0, &st);
        return st;
    }
    // byte t of the view; *start: an emission starts at t
    SNACC_BZ_HD uint8_t at(const uint8_t *rx, const uint8_t *fx, const uint8_t *ry, const uint8_t *fy, uint64_t t,
                           bool *start) const
    {
        const uint64_t la = a1 - a0;
        if (t < la) { *start = fx[a0 + t] != 0; return rx[a0 + t]; }
        t -= la;
        const uint64_t l0 = j0 ? bz_run_bytes(j0) : 0;
        if (t < l0) return bz_run_at(jb0, j0, t, start);
        t -= l0;
        const uint64_t l1 = j1 ? bz_run_bytes(j1) : 0;
        if (t < l1) return bz_run_at(jb1, j1, t, start);
        t -= l1;
        *start = fy[b0 + t] != 0;
        return ry[b0 + t];
    }
};

SNACC_BZ_HD BzView bz_view_single(uint32_t a0, uint32_t a1)
{
    BzView v{}; v.a0 = a0; v.a1 = a1; return v;
}

// x's open tail (from `open`, the start of x's last block alone), junction, rest of y
SNACC_BZ_HD BzView bz_view_pair(const BzSeq &x, uint32_t open, const BzSeq &y)
{
    BzView v{};
    v.a0 = open; v.a1 = x.fin;
    v.jb0 = x.blast;
    if (y.bfirst == x.blast) { v.j0 = x.p + y.U; }
    else { v.j0 = x.p; v.jb1 = y.bfirst; v.j1 = y.U; }
    v.b0 = y.first_end; v.b1 = y.rlen;
    return v;
}

// Block cut (host planning): before each emission, the block closes if it already holds >= BZ_NBLOCK_MAX bytes, so a
// block ends at the first emission start at or after start + BZ_NBLOCK_MAX.  Appends (start, length) windows.
struct BzWin { uint32_t v0, n; };
inline void bz_cut(const BzView &v, const uint8_t *fx, const uint8_t *fy, std::vector<BzWin> &out)
{
    const uint64_t total = v.total();
    uint64_t pos = 0;
    while (pos < total) {
        uint64_t c = pos + BZ_NBLOCK_MAX;
        if (c >= total) { out.push_back(BzWin{(uint32_t)pos, (uint32_t)(total - pos)}); break; }
        while (c < total && !v.starts(fx, fy, c)) ++c;
        out.push_back(BzWin{(uint32_t)pos, (uint32_t)(c - pos)});
        pos = c;
    }
}

// ---- MTF + RLE2 ----------------------------------------------------------------------------------------------------
// L: the block's BWT; seq_of: in-use byte -> its index among the in-use bytes; yy: nInUse bytes of work space.
// Writes mtfv (at most n + 1 symbols), freq[0 .. nInUse + 2).  Returns nMTF (EOB included).
SNACC_BZ_HD uint32_t bz_mtf(const uint8_t *L, uint32_t n, const uint8_t *seq_of, int nInUse, uint8_t *yy,
                            uint16_t *mtfv, int32_t *freq)
{
    const int EOB = nInUse + 1;
    for (int i = 0; i <= EOB; ++i) freq[i] = 0;
    for (int i = 0; i < nInUse; ++i) yy[i] = (uint8_t)i;
    uint32_t wr = 0, zPend = 0;
    auto flush = [&]() {
        zPend--;
        for (;;) {
            const uint16_t s = (zPend & 1) ? 1 : 0;          // RUNB : RUNA
            mtfv[wr++] = s; freq[s]++;
            if (zPend < 2) break;
            zPend = (zPend - 2) / 2;
        }
        zPend = 0;
    };
    for (uint32_t i = 0; i < n; ++i) {
        const uint8_t ll = seq_of[L[i]];
        if (yy[0] == ll) { zPend++; continue; }
        if (zPend > 0) flush();
        uint8_t tmp = yy[1], prev = yy[0];
        yy[1] = prev;
        int j = 1;
        while (tmp != ll) { ++j; prev = tmp; tmp = yy[j]; yy[j] = prev; }
        yy[0] = tmp;
        mtfv[wr++] = (uint16_t)(j + 1); freq[j + 1]++;
    }
    if (zPend > 0) flush();
    mtfv[wr++] = (uint16_t)EOB; freq[EOB]++;
    return wr;
}

SNACC_BZ_HD int bz_n_groups(uint32_t nMTF)
{
    return nMTF < 200 ? 2 : nMTF < 600 ? 3 : nMTF < 1200 ? 4 : nMTF < 2400 ? 5 : 6;
}

// initial tables: the symbols split into nGroups parts of near-equal cumulative frequency; len[t * BZ_MAX_ALPHA + v]
SNACC_BZ_HD void bz_init_tables(uint8_t *len, int nGroups, int alphaSize, const int32_t *freq, uint32_t nMTF)
{
    for (int t = 0; t < BZ_N_GROUPS; ++t)
        for (int v = 0; v < alphaSize; ++v) len[t * BZ_MAX_ALPHA + v] = 15;
    int nPart = nGroups, remF = (int)nMTF, gs = 0;
    while (nPart > 0) {
        const int tFreq = remF / nPart;
        int ge = gs - 1, aFreq = 0;
        while (aFreq < tFreq && ge < alphaSize - 1) { ge++; aFreq += freq[ge]; }
        if (ge > gs && nPart != nGroups && nPart != 1 && ((nGroups - nPart) % 2 == 1)) { aFreq -= freq[ge]; ge--; }
        for (int v = 0; v < alphaSize; ++v) len[(nPart - 1) * BZ_MAX_ALPHA + v] = (v >= gs && v <= ge) ? 0 : 15;
        nPart--;
        gs = ge + 1;
        remF -= aFreq;
    }
}

// the table of least cost (first one on ties) for symbols mtfv[gs .. ge]; *cost receives that cost
SNACC_BZ_HD int bz_group_choose(const uint8_t *len, int nGroups, const uint16_t *mtfv, uint32_t gs, uint32_t ge,
                                uint32_t *cost)
{
    uint32_t c[BZ_N_GROUPS] = {0, 0, 0, 0, 0, 0};
    for (uint32_t i = gs; i <= ge; ++i) {
        const uint16_t v = mtfv[i];
        for (int t = 0; t < nGroups; ++t) c[t] += len[t * BZ_MAX_ALPHA + v];
    }
    int bt = 0;
    for (int t = 1; t < nGroups; ++t) if (c[t] < c[bt]) bt = t;
    *cost = c[bt];
    return bt;
}

// BZ2_hbMakeCodeLengths: weights (freq or 1) << 8 | depth, a binary heap whose tie order is part of the result,
// and while a code is longer than maxLen every weight is rescaled to 1 + (w >> 8) / 2 and the tree rebuilt.
SNACC_BZ_HD void bz_make_code_lengths(uint8_t *len, const int32_t *freq, int alphaSize, int maxLen, int32_t *scratch)
{
    int32_t *heap = scratch, *weight = scratch + (BZ_MAX_ALPHA + 2), *parent = weight + 2 * BZ_MAX_ALPHA;
    for (int i = 0; i < alphaSize; ++i) weight[i + 1] = (freq[i] == 0 ? 1 : freq[i]) << 8;
    for (;;) {
        int nNodes = alphaSize, nHeap = 0;
        heap[0] = 0; weight[0] = 0; parent[0] = -2;
        auto upheap = [&](int z) {
            const int tmp = heap[z];
            while (weight[tmp] < weight[heap[z >> 1]]) { heap[z] = heap[z >> 1]; z >>= 1; }
            heap[z] = tmp;
        };
        auto downheap = [&](int z) {
            const int tmp = heap[z];
            for (;;) {
                int y = z << 1;
                if (y > nHeap) break;
                if (y < nHeap && weight[heap[y + 1]] < weight[heap[y]]) y++;
                if (weight[tmp] < weight[heap[y]]) break;
                heap[z] = heap[y]; z = y;
            }
            heap[z] = tmp;
        };
        for (int i = 1; i <= alphaSize; ++i) { parent[i] = -1; heap[++nHeap] = i; upheap(nHeap); }
        while (nHeap > 1) {
            const int n1 = heap[1]; heap[1] = heap[nHeap]; nHeap--; downheap(1);
            const int n2 = heap[1]; heap[1] = heap[nHeap]; nHeap--; downheap(1);
            nNodes++;
            parent[n1] = parent[n2] = nNodes;
            const int32_t w1 = weight[n1], w2 = weight[n2];
            const int32_t d1 = w1 & 0xff, d2 = w2 & 0xff;
            weight[nNodes] = ((w1 & (int32_t)0xffffff00) + (w2 & (int32_t)0xffffff00)) | (1 + (d1 > d2 ? d1 : d2));
            parent[nNodes] = -1;
            heap[++nHeap] = nNodes; upheap(nHeap);
        }
        bool tooLong = false;
        for (int i = 1; i <= alphaSize; ++i) {
            int j = 0, k = i;
            while (parent[k] >= 0) { k = parent[k]; j++; }
            len[i - 1] = (uint8_t)j;
            if (j > maxLen) tooLong = true;
        }
        if (!tooLong) break;
        for (int i = 1; i <= alphaSize; ++i) { int j = weight[i] >> 8; j = 1 + (j / 2); weight[i] = j << 8; }
    }
}

// bits of a block besides the coded symbols: fixed fields, mapping table, selectors (MTF-coded, unary), code tables
SNACC_BZ_HD int64_t bz_header_bits(const uint8_t *in_use, const uint8_t *sel, int nSel, int nGroups, const uint8_t *len,
                                   int alphaSize)
{
    int64_t bits = BZ_BLOCK_FIXED_BITS + 16;
    for (int i = 0; i < 16; ++i) {
        bool any = false;
        for (int j = 0; j < 16; ++j) any |= in_use[i * 16 + j] != 0;
        if (any) bits += 16;
    }
    bits += 3 + 15;
    uint8_t pos[BZ_N_GROUPS];
    for (int i = 0; i < nGroups; ++i) pos[i] = (uint8_t)i;
    for (int i = 0; i < nSel; ++i) {
        const uint8_t ll = sel[i];
        int j = 0; uint8_t tmp = pos[0];
        while (ll != tmp) { j++; const uint8_t t2 = tmp; tmp = pos[j]; pos[j] = t2; }
        pos[0] = tmp;
        bits += j + 1;
    }
    for (int t = 0; t < nGroups; ++t) {
        int curr = len[t * BZ_MAX_ALPHA];
        bits += 5;
        for (int i = 0; i < alphaSize; ++i) {
            const int l = len[t * BZ_MAX_ALPHA + i];
            bits += 2 * (l > curr ? l - curr : curr - l) + 1;
            curr = l;
        }
    }
    return bits;
}

// In-use bytes of a block -> seq_of map; returns nInUse
SNACC_BZ_HD int bz_map(const uint8_t *in_use, uint8_t *seq_of)
{
    int k = 0;
    for (int i = 0; i < 256; ++i) if (in_use[i]) seq_of[i] = (uint8_t)k++;
    return k;
}

// Work space of the serial bit count (host emulation)
struct BzWork {
    std::vector<uint16_t> mtfv;
    std::vector<uint8_t> sel;
};

// The bits of one block from its BWT, serially (the host emulation; bz_bits_kernel runs the same steps in parallel)
inline int64_t bz_block_bits_serial(const uint8_t *L, uint32_t n, BzWork &w)
{
    uint8_t in_use[256] = {0}, seq_of[256], yy[256], len[BZ_N_GROUPS * BZ_MAX_ALPHA];
    int32_t freq[BZ_MAX_ALPHA], rfreq[BZ_N_GROUPS * BZ_MAX_ALPHA], scratch[BZ_HB_SCRATCH];
    for (uint32_t i = 0; i < n; ++i) in_use[L[i]] = 1;
    const int nInUse = bz_map(in_use, seq_of), alphaSize = nInUse + 2;
    w.mtfv.resize((size_t)n + 1);
    const uint32_t nMTF = bz_mtf(L, n, seq_of, nInUse, yy, w.mtfv.data(), freq);
    const int nGroups = bz_n_groups(nMTF);
    bz_init_tables(len, nGroups, alphaSize, freq, nMTF);
    const int nSel = (int)((nMTF + BZ_G_SIZE - 1) / BZ_G_SIZE);
    w.sel.resize((size_t)nSel);
    for (int iter = 0; iter < BZ_N_ITERS; ++iter) {
        for (int k = 0; k < BZ_N_GROUPS * BZ_MAX_ALPHA; ++k) rfreq[k] = 0;
        for (int g = 0; g < nSel; ++g) {
            const uint32_t gs = (uint32_t)g * BZ_G_SIZE, ge = gs + BZ_G_SIZE - 1 < nMTF ? gs + BZ_G_SIZE - 1 : nMTF - 1;
            uint32_t c;
            const int bt = bz_group_choose(len, nGroups, w.mtfv.data(), gs, ge, &c);
            w.sel[g] = (uint8_t)bt;
            for (uint32_t i = gs; i <= ge; ++i) rfreq[bt * BZ_MAX_ALPHA + w.mtfv[i]]++;
        }
        for (int t = 0; t < nGroups; ++t)
            bz_make_code_lengths(len + t * BZ_MAX_ALPHA, rfreq + t * BZ_MAX_ALPHA, alphaSize, BZ_MAX_CODE_LEN, scratch);
    }
    int64_t bits = bz_header_bits(in_use, w.sel.data(), nSel, nGroups, len, alphaSize);
    for (uint32_t i = 0; i < nMTF; ++i) bits += len[w.sel[i / BZ_G_SIZE] * BZ_MAX_ALPHA + w.mtfv[i]];
    return bits;
}

SNACC_BZ_HD int64_t bz_stream_bytes(int64_t block_bits) { return (BZ_STREAM_BITS + block_bits + 7) / 8; }

// ---- device kernels ------------------------------------------------------------------------------------------------
#ifdef __CUDACC__

// a block of a batch: the window [v0, v0 + n) of a view, its bits added to bits[dst]
struct BzBlock {
    int64_t dst;          // >= 0: job; < 0: -1 - x, the closed-block bits of sequence x
    uint64_t off;         // offset of its bytes in the batch
    int32_t x, y;         // y < 0: no second sequence
    uint32_t v0, n;
    BzView v;
};

// K5a: RLE1 of every listed sequence, one thread each
__global__ void bz_rle_kernel(const uint8_t *__restrict__ corpus, const uint64_t *__restrict__ off,
                              const uint32_t *__restrict__ len, const int32_t *__restrict__ seqs, int32_t n,
                              uint8_t *__restrict__ rle, uint8_t *__restrict__ flag, BzSeq *__restrict__ info)
{
    const int32_t k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= n) return;
    const int32_t s = seqs[k];
    BzSeq si = info[s];
    bz_rle_seq(corpus + off[s], len[s], rle + si.roff, flag + si.roff, &si);
    info[s] = si;
}

// K5b: the bytes of every block of a batch
__global__ void bz_gather_kernel(const BzBlock *__restrict__ blocks, const BzSeq *__restrict__ info,
                                 const uint8_t *__restrict__ rle, const uint8_t *__restrict__ flag, uint8_t *__restrict__ buf)
{
    const BzBlock bk = blocks[blockIdx.x];
    const uint8_t *rx = rle + info[bk.x].roff, *fx = flag + info[bk.x].roff;
    const uint8_t *ry = bk.y >= 0 ? rle + info[bk.y].roff : rx, *fy = bk.y >= 0 ? flag + info[bk.y].roff : fx;
    for (uint32_t t = threadIdx.x; t < bk.n; t += blockDim.x) {
        bool st;
        buf[bk.off + t] = bk.v.at(rx, fx, ry, fy, (uint64_t)bk.v0 + t, &st);
    }
}

// K5c: BWT of one block per CTA by prefix doubling over cyclic rotations.  Ranks are group-head positions; each round
// sorts by (rank[i], rank[i + h]) with stable 8-bit LSD radix passes (warp match ranking, 1024 threads), passes whose
// digit is the same for every element are skipped.  Rounds stop when every rank is distinct or h >= n (a periodic
// block: the remaining ties are equal rotations, with equal last bytes).
constexpr int BZ_SORT_THREADS = 1024;
constexpr int BZ_SORT_WARPS = BZ_SORT_THREADS / 32;

struct BzSortSmem {
    uint16_t wh[BZ_SORT_WARPS * 256];
    uint32_t cnt[256], base[256];
    uint32_t wtot[BZ_SORT_WARPS];
    uint32_t carry, groups;
    int skip;
};

template <typename I>
struct BzKey {
    const uint8_t *text; const I *rk; uint32_t n, h; int rbits;
    __device__ __forceinline__ uint64_t operator()(uint32_t i) const
    {
        if (!rk) {
            uint32_t k = 0;
            for (int q = 0; q < 4; ++q) { uint32_t j = i + q; j = j >= n ? j % n : j; k = (k << 8) | text[j]; }
            return k;
        }
        uint32_t j = i + h; if (j >= n) j -= n;
        return ((uint64_t)rk[i] << rbits) | rk[j];
    }
};

template <typename I, typename K>
__device__ bool bz_radix_pass(uint32_t n, const I *src, I *dst, const K &key, int shift, BzSortSmem &sm)
{
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    for (int d = tid; d < 256; d += BZ_SORT_THREADS) sm.cnt[d] = 0;
    __syncthreads();
    for (uint32_t i = tid; i < n; i += BZ_SORT_THREADS) atomicAdd(&sm.cnt[(key(src[i]) >> shift) & 255], 1u);
    __syncthreads();
    if (tid == 0) {
        uint32_t run = 0; int skip = 0;
        for (int d = 0; d < 256; ++d) { sm.base[d] = run; skip |= sm.cnt[d] == n; run += sm.cnt[d]; }
        sm.skip = skip;
    }
    __syncthreads();
    if (sm.skip) return false;
    const uint32_t lt = (1u << lane) - 1;
    for (uint32_t t0 = 0; t0 < n; t0 += BZ_SORT_THREADS) {
        for (int k = tid; k < BZ_SORT_WARPS * 256; k += BZ_SORT_THREADS) sm.wh[k] = 0;
        __syncthreads();
        const uint32_t i = t0 + tid;
        const bool valid = i < n;
        const I e = valid ? src[i] : (I)0;
        const uint32_t d = valid ? (uint32_t)((key(e) >> shift) & 255) : 256u;
        const uint32_t peers = __match_any_sync(0xffffffffu, d);
        const uint32_t r = __popc(peers & lt);
        if (valid && r == 0) sm.wh[warp * 256 + d] = (uint16_t)__popc(peers);
        __syncthreads();
        if (tid < 256) {
            uint32_t s = 0;
            for (int w = 0; w < BZ_SORT_WARPS; ++w) { const uint32_t v = sm.wh[w * 256 + tid]; sm.wh[w * 256 + tid] = (uint16_t)s; s += v; }
            sm.cnt[tid] = s;
        }
        __syncthreads();
        if (valid) dst[sm.base[d] + sm.wh[warp * 256 + d] + r] = e;
        __syncthreads();
        if (tid < 256) sm.base[tid] += sm.cnt[tid];
    }
    __syncthreads();
    return true;
}

// rank of every rotation after a sort: position of the first element of its group; returns the number of groups
template <typename I, typename K>
__device__ uint32_t bz_assign_ranks(uint32_t n, const I *sa, I *rk_out, const K &key, BzSortSmem &sm)
{
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    if (tid == 0) { sm.carry = 0; sm.groups = 0; }
    __syncthreads();
    for (uint32_t t0 = 0; t0 < n; t0 += BZ_SORT_THREADS) {
        const uint32_t i = t0 + tid;
        const bool valid = i < n;
        bool head = false;
        I e = 0;
        if (valid) { e = sa[i]; head = i == 0 || key(sa[i - 1]) != key(e); }
        uint32_t m = head ? i : 0;
        for (int o = 1; o < 32; o <<= 1) { const uint32_t v = __shfl_up_sync(0xffffffffu, m, o); if (lane >= o) m = m > v ? m : v; }
        if (lane == 31) sm.wtot[warp] = m;
        const int heads = __syncthreads_count(head);
        if (warp == 0) {
            uint32_t w = sm.wtot[lane];
            for (int o = 1; o < 32; o <<= 1) { const uint32_t v = __shfl_up_sync(0xffffffffu, w, o); if (lane >= o) w = w > v ? w : v; }
            sm.wtot[lane] = w;
        }
        __syncthreads();
        if (warp > 0) { const uint32_t p = sm.wtot[warp - 1]; m = m > p ? m : p; }
        m = m > sm.carry ? m : sm.carry;
        if (valid) rk_out[e] = (I)m;
        __syncthreads();
        if (tid == BZ_SORT_THREADS - 1) { sm.carry = m; sm.groups += (uint32_t)heads; }
        __syncthreads();
    }
    return sm.groups;
}

template <typename I>
__device__ void bz_sort_block(const uint8_t *text, uint32_t n, I *sa, I *sa2, I *rk, I *rk2, int rbits, uint8_t *out,
                              BzSortSmem &sm)
{
    for (uint32_t i = threadIdx.x; i < n; i += BZ_SORT_THREADS) sa[i] = (I)i;
    __syncthreads();
    BzKey<I> k0{text, nullptr, n, 0, rbits};
    for (int sh = 0; sh < 32; sh += 8)
        if (bz_radix_pass(n, sa, sa2, k0, sh, sm)) { I *t = sa; sa = sa2; sa2 = t; }
    uint32_t groups = bz_assign_ranks(n, sa, rk, k0, sm);
    for (uint32_t h = 4; groups < n && h < n; h *= 2) {
        BzKey<I> k{text, rk, n, h, rbits};
        for (int sh = 0; sh < 2 * rbits; sh += 8)
            if (bz_radix_pass(n, sa, sa2, k, sh, sm)) { I *t = sa; sa = sa2; sa2 = t; }
        groups = bz_assign_ranks(n, sa, rk2, k, sm);
        I *t = rk; rk = rk2; rk2 = t;
    }
    for (uint32_t i = threadIdx.x; i < n; i += BZ_SORT_THREADS) { const uint32_t s = sa[i]; out[i] = text[s ? s - 1 : n - 1]; }
}

// blocks of at most BZ_SMEM_MAX_N bytes sort with 16-bit indices and ranks in shared memory (4 arrays); larger ones
// with 32-bit arrays in global scratch (16 bytes per block byte, at 4 * off 32-bit words)
constexpr uint32_t BZ_SMEM_MAX_N = 24576;
constexpr size_t BZ_SMEM_BYTES = (size_t)4 * BZ_SMEM_MAX_N * sizeof(uint16_t);

__global__ void __launch_bounds__(BZ_SORT_THREADS, 1)
bz_bwt_smem_kernel(const BzBlock *__restrict__ blocks, const int32_t *__restrict__ list, const uint8_t *__restrict__ buf,
                   uint8_t *__restrict__ bwt)
{
    extern __shared__ __align__(16) uint16_t bz_dyn[];
    __shared__ BzSortSmem sm;
    const BzBlock bk = blocks[list[blockIdx.x]];
    const uint32_t n = bk.n;
    bz_sort_block<uint16_t>(buf + bk.off, n, bz_dyn, bz_dyn + n, bz_dyn + 2 * n, bz_dyn + 3 * n, 16, bwt + bk.off, sm);
}

__global__ void __launch_bounds__(BZ_SORT_THREADS, 1)
bz_bwt_global_kernel(const BzBlock *__restrict__ blocks, const int32_t *__restrict__ list, const uint8_t *__restrict__ buf,
                     uint8_t *__restrict__ bwt, uint32_t *__restrict__ scratch)
{
    __shared__ BzSortSmem sm;
    const BzBlock bk = blocks[list[blockIdx.x]];
    const uint32_t n = bk.n;
    uint32_t *w = scratch + 4 * bk.off;
    bz_sort_block<uint32_t>(buf + bk.off, n, w, w + n, w + 2 * n, w + 3 * n, 20, bwt + bk.off, sm);
}

// K5d: MTF + RLE2 (serial, thread 0), the 4 table-choice iterations (parallel over the groups of 50 symbols, code
// lengths one table per thread) and the bit count; one CTA per block.  mtfv: n + 1 symbols at off + block index.
constexpr int BZ_BITS_THREADS = 128;
constexpr size_t BZ_BITS_DYN_SMEM = sizeof(int32_t) * BZ_N_GROUPS * BZ_HB_SCRATCH;

__global__ void __launch_bounds__(BZ_BITS_THREADS)
bz_bits_kernel(const BzBlock *__restrict__ blocks, const uint8_t *__restrict__ bwt, uint16_t *__restrict__ mtfv_all,
               unsigned long long *__restrict__ job_bits, unsigned long long *__restrict__ seq_bits)
{
    __shared__ uint8_t in_use[256], seq_of[256], yy[256];
    __shared__ uint8_t len[BZ_N_GROUPS * BZ_MAX_ALPHA];
    __shared__ int32_t freq[BZ_MAX_ALPHA], rfreq[BZ_N_GROUPS * BZ_MAX_ALPHA];
    extern __shared__ int32_t bz_hb[];                     // BZ_N_GROUPS * BZ_HB_SCRATCH: one code-length build per table
    __shared__ uint8_t sel[BZ_MAX_SELECTORS];
    __shared__ uint32_t s_nmtf;
    __shared__ unsigned long long s_bits;
    const int tid = threadIdx.x;
    const BzBlock bk = blocks[blockIdx.x];
    const uint8_t *L = bwt + bk.off;
    uint16_t *mtfv = mtfv_all + bk.off + blockIdx.x;
    const uint32_t n = bk.n;
    for (int i = tid; i < 256; i += BZ_BITS_THREADS) in_use[i] = 0;
    if (tid == 0) s_bits = 0;
    __syncthreads();
    for (uint32_t i = tid; i < n; i += BZ_BITS_THREADS) in_use[L[i]] = 1;
    __syncthreads();
    __shared__ int s_nin;
    if (tid == 0) {
        const int nInUse = bz_map(in_use, seq_of);
        s_nin = nInUse;
        s_nmtf = bz_mtf(L, n, seq_of, nInUse, yy, mtfv, freq);
    }
    __syncthreads();
    const int alphaSize = s_nin + 2;
    const uint32_t nMTF = s_nmtf;
    const int nGroups = bz_n_groups(nMTF);
    const int nSel = (int)((nMTF + BZ_G_SIZE - 1) / BZ_G_SIZE);
    if (tid == 0) bz_init_tables(len, nGroups, alphaSize, freq, nMTF);
    __syncthreads();
    for (int iter = 0; iter < BZ_N_ITERS; ++iter) {
        for (int k = tid; k < BZ_N_GROUPS * BZ_MAX_ALPHA; k += BZ_BITS_THREADS) rfreq[k] = 0;
        __syncthreads();
        for (int g = tid; g < nSel; g += BZ_BITS_THREADS) {
            const uint32_t gs = (uint32_t)g * BZ_G_SIZE, ge = gs + BZ_G_SIZE - 1 < nMTF ? gs + BZ_G_SIZE - 1 : nMTF - 1;
            uint32_t c;
            const int bt = bz_group_choose(len, nGroups, mtfv, gs, ge, &c);
            sel[g] = (uint8_t)bt;
            for (uint32_t i = gs; i <= ge; ++i) atomicAdd(&rfreq[bt * BZ_MAX_ALPHA + mtfv[i]], 1);
        }
        __syncthreads();
        if (tid < nGroups)
            bz_make_code_lengths(len + tid * BZ_MAX_ALPHA, rfreq + tid * BZ_MAX_ALPHA, alphaSize, BZ_MAX_CODE_LEN, bz_hb + tid * BZ_HB_SCRATCH);
        __syncthreads();
    }
    unsigned long long mine = 0;
    for (int g = tid; g < nSel; g += BZ_BITS_THREADS) {
        const uint32_t gs = (uint32_t)g * BZ_G_SIZE, ge = gs + BZ_G_SIZE - 1 < nMTF ? gs + BZ_G_SIZE - 1 : nMTF - 1;
        const uint8_t *l = len + sel[g] * BZ_MAX_ALPHA;
        for (uint32_t i = gs; i <= ge; ++i) mine += l[mtfv[i]];
    }
    if (tid == 0) mine += (unsigned long long)bz_header_bits(in_use, sel, nSel, nGroups, len, alphaSize);
    atomicAdd(&s_bits, mine);
    __syncthreads();
    if (tid == 0) {
        if (bk.dst >= 0) atomicAdd(&job_bits[bk.dst], s_bits);
        else atomicAdd(&seq_bits[-1 - bk.dst], s_bits);
    }
}

// K5e: sizes from the summed block bits (x's closed blocks from seq_bits when `prefix`)
__global__ void bz_finish_kernel(const unsigned long long *__restrict__ job_bits, const unsigned long long *__restrict__ seq_bits,
                                 const int32_t *__restrict__ xs, const uint8_t *__restrict__ use_prefix, int64_t n,
                                 int64_t *__restrict__ out)
{
    for (int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; k < n; k += (int64_t)gridDim.x * blockDim.x) {
        int64_t bits = (int64_t)job_bits[k];
        if (use_prefix[k]) bits += (int64_t)seq_bits[xs[k]];
        out[k] = bz_stream_bytes(bits);
    }
}


// ---- host side (called from api.cu with the context lock held) ------------------------------------------------------
// RLE1 of every sequence once per upload; then per call the host cuts every job into blocks (x's closed blocks once per
// x, the rest of each job from x's open tail, the junction and RLE1(y)) and the blocks go through fixed-size batches:
// gather, BWT (shared memory up to BZ_SMEM_MAX_N bytes, else global scratch), MTF + table choice + bit count.  Device
// memory of a batch is bounded by BZ_BATCH_BYTES whatever the number of jobs.
constexpr uint64_t BZ_BATCH_BYTES = 192ull << 20;
constexpr size_t BZ_BATCH_BLOCKS = 1 << 16;

// RLE1 of every sequence, its emission-start flags (a host copy plans the block cuts), where the open block of each
// sequence alone starts, and the bits of its closed blocks once computed
struct BzState {
    bool ready = false;
    DevBuf rle, flag;
    BzSeq *d_info = nullptr;
    unsigned long long *d_seq_bits = nullptr;
    std::vector<BzSeq> h_info; std::vector<uint8_t> h_flag, h_pdone;
    std::vector<uint32_t> h_open, h_nclosed;
    // working memory: argument arrays and batch buffers
    DevBuf all, blocks, small, large, buf, bwt, mtf, job_bits, job_prefix;
    cudaEvent_t ev[5] = {nullptr, nullptr, nullptr, nullptr, nullptr};
    // options "bzip2_smem", "bzip2_prefix" (0: for tests, same results)
    int use_smem = 1, use_prefix = 1;
    // statistics of the last call
    int64_t n_blocks = 0, smem_blocks = 0, prefix_blocks = 0;
    double ms[4] = {0, 0, 0, 0};               // RLE1 + gather, BWT small, BWT large, MTF + selection + bits
};

static inline void bz_free_corpus(BzState &st)
{
    st.rle.release(); st.flag.release();
    cudaFree(st.d_info); st.d_info = nullptr;
    cudaFree(st.d_seq_bits); st.d_seq_bits = nullptr;
    st.ready = false;
}

static inline void bz_free_work(BzState &st)
{
    for (DevBuf *b : {&st.all, &st.blocks, &st.small, &st.large, &st.buf, &st.bwt, &st.mtf, &st.job_bits, &st.job_prefix})
        b->release();
    for (cudaEvent_t &e : st.ev) { if (e) cudaEventDestroy(e); e = nullptr; }
}

// the RLE1 of the corpus is computed again by the next call
static inline void bz_invalidate(BzState &st) { st.ready = false; }

static int bz_prepare(BzState &st, const Corpus &c, cudaStream_t stream, int64_t *launches, std::string &err)
{
    NvtxRange nvtx_("snacc_b200: bzip2 RLE1");
    const int32_t n = c.n_seqs;
    st.h_info.assign((size_t)n, BzSeq{});
    uint64_t cap = 0;
    for (int32_t i = 0; i < n; ++i) { st.h_info[i].roff = cap; cap += (uint64_t)c.h_len[i] / 4 * 5 + 16; }
    DCK(st.rle.grow(cap, stream, true));
    DCK(st.flag.grow(cap, stream, true));
    if (!st.d_info) DCK(cudaMalloc(&st.d_info, sizeof(BzSeq) * n));
    if (!st.d_seq_bits) DCK(cudaMalloc(&st.d_seq_bits, sizeof(unsigned long long) * n));
    DCK(cudaMemsetAsync(st.d_seq_bits, 0, sizeof(unsigned long long) * n, stream));
    DCK(cudaMemcpyAsync(st.d_info, st.h_info.data(), sizeof(BzSeq) * n, cudaMemcpyHostToDevice, stream));
    std::vector<int32_t> all((size_t)n);
    for (int32_t i = 0; i < n; ++i) all[i] = i;
    DCK(st.all.grow(sizeof(int32_t) * n, stream));
    DCK(cudaMemcpyAsync(st.all.p, all.data(), sizeof(int32_t) * n, cudaMemcpyHostToDevice, stream));
    bz_rle_kernel<<<(n + 31) / 32, 32, 0, stream>>>(c.d_corpus, c.d_off, c.d_len, st.all.get<int32_t>(), n,
                                                    st.rle.get<uint8_t>(), st.flag.get<uint8_t>(), st.d_info);
    DCK(cudaGetLastError());
    ++*launches;
    st.h_flag.resize(cap);
    DCK(cudaMemcpyAsync(st.h_info.data(), st.d_info, sizeof(BzSeq) * n, cudaMemcpyDeviceToHost, stream));
    DCK(cudaMemcpyAsync(st.h_flag.data(), st.flag.p, cap, cudaMemcpyDeviceToHost, stream));
    DCK(cudaStreamSynchronize(stream));
    // where the last block of each sequence alone starts: the blocks before it close the same way in every x.y
    st.h_open.assign((size_t)n, 0); st.h_nclosed.assign((size_t)n, 0); st.h_pdone.assign((size_t)n, 0);
    std::vector<BzWin> wins;
    for (int32_t i = 0; i < n; ++i) {
        const BzSeq &si = st.h_info[i];
        if (si.rlen <= BZ_NBLOCK_MAX) continue;
        const uint8_t *f = st.h_flag.data() + si.roff;
        wins.clear();
        bz_cut(bz_view_single(0, si.rlen), f, f, wins);
        st.h_open[i] = wins.back().v0;
        st.h_nclosed[i] = (uint32_t)wins.size() - 1;
    }
    st.ready = true;
    return 0;
}

// one batch of blocks; `work` holds the global-memory sort's 4 arrays of 32-bit words per block byte
static int bz_run_batch(BzState &st, const BzBlock *blocks, size_t nb, uint64_t bytes, unsigned long long *d_job_bits,
                        DevBuf &work, cudaStream_t stream, int64_t *launches, std::string &err)
{
    NvtxRange nvtx_("snacc_b200: bzip2 batch");
    std::vector<int32_t> small, large;
    for (size_t k = 0; k < nb; ++k)
        ((st.use_smem && blocks[k].n <= BZ_SMEM_MAX_N) ? small : large).push_back((int32_t)k);
    DCK(st.blocks.grow(sizeof(BzBlock) * nb, stream));
    DCK(st.small.grow(sizeof(int32_t) * (small.size() + 1), stream));
    DCK(st.large.grow(sizeof(int32_t) * (large.size() + 1), stream));
    DCK(st.buf.grow(bytes, stream));
    DCK(st.bwt.grow(bytes, stream));
    DCK(st.mtf.grow(sizeof(uint16_t) * (bytes + nb), stream));
    if (!large.empty()) DCK(work.grow(16 * bytes, stream, true));
    const BzBlock *d_blocks = st.blocks.get<BzBlock>();
    const int32_t *d_small = st.small.get<int32_t>(), *d_large = st.large.get<int32_t>();
    uint8_t *d_buf = st.buf.get<uint8_t>(), *d_bwt = st.bwt.get<uint8_t>();
    DCK(cudaMemcpyAsync(st.blocks.p, blocks, sizeof(BzBlock) * nb, cudaMemcpyHostToDevice, stream));
    if (!small.empty()) DCK(cudaMemcpyAsync(st.small.p, small.data(), sizeof(int32_t) * small.size(), cudaMemcpyHostToDevice, stream));
    if (!large.empty()) DCK(cudaMemcpyAsync(st.large.p, large.data(), sizeof(int32_t) * large.size(), cudaMemcpyHostToDevice, stream));
    DCK(cudaEventRecord(st.ev[0], stream));
    bz_gather_kernel<<<(unsigned)nb, 256, 0, stream>>>(d_blocks, st.d_info, st.rle.get<uint8_t>(), st.flag.get<uint8_t>(), d_buf);
    DCK(cudaGetLastError());
    DCK(cudaEventRecord(st.ev[1], stream));
    if (!small.empty()) {
        DCK(cudaFuncSetAttribute(bz_bwt_smem_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)BZ_SMEM_BYTES));
        bz_bwt_smem_kernel<<<(unsigned)small.size(), BZ_SORT_THREADS, BZ_SMEM_BYTES, stream>>>(d_blocks, d_small, d_buf, d_bwt);
        DCK(cudaGetLastError());
    }
    DCK(cudaEventRecord(st.ev[2], stream));
    if (!large.empty()) {
        bz_bwt_global_kernel<<<(unsigned)large.size(), BZ_SORT_THREADS, 0, stream>>>(d_blocks, d_large, d_buf, d_bwt,
                                                                                      work.get<uint32_t>());
        DCK(cudaGetLastError());
    }
    DCK(cudaEventRecord(st.ev[3], stream));
    DCK(cudaFuncSetAttribute(bz_bits_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)BZ_BITS_DYN_SMEM));
    bz_bits_kernel<<<(unsigned)nb, BZ_BITS_THREADS, BZ_BITS_DYN_SMEM, stream>>>(d_blocks, d_bwt, st.mtf.get<uint16_t>(),
                                                                               d_job_bits, st.d_seq_bits);
    DCK(cudaGetLastError());
    DCK(cudaEventRecord(st.ev[4], stream));
    DCK(cudaEventSynchronize(st.ev[4]));
    for (int s = 0; s < 4; ++s) {
        float ms = 0.f;
        DCK(cudaEventElapsedTime(&ms, st.ev[s], st.ev[s + 1]));
        st.ms[s] += ms;
    }
    *launches += 2 + !small.empty() + !large.empty();
    st.n_blocks += (int64_t)nb;
    st.smem_blocks += (int64_t)small.size();
    return 0;
}

// A job list (ys null: singles) into d_out.  d_xs: the x list on the device.
static int bz_run(BzState &st, const Corpus &c, const int32_t *xs, const int32_t *ys, const int32_t *d_xs,
                  int64_t n_jobs, int64_t *d_out, DevBuf &work, cudaStream_t stream, int64_t *launches, std::string &err)
{
    st.n_blocks = st.smem_blocks = st.prefix_blocks = 0;
    for (double &m : st.ms) m = 0;
    for (cudaEvent_t &e : st.ev) if (!e) DCK(cudaEventCreate(&e));
    if (!st.ready) {
        DCK(cudaEventRecord(st.ev[0], stream));
        int r = bz_prepare(st, c, stream, launches, err);
        if (r) return r;
        DCK(cudaEventRecord(st.ev[1], stream));
        DCK(cudaEventSynchronize(st.ev[1]));
        float ms = 0.f;
        DCK(cudaEventElapsedTime(&ms, st.ev[0], st.ev[1]));
        st.ms[0] += ms;
    }
    DCK(st.job_bits.grow(sizeof(unsigned long long) * n_jobs, stream));
    DCK(st.job_prefix.grow((size_t)n_jobs, stream));
    unsigned long long *d_job_bits = st.job_bits.get<unsigned long long>();
    DCK(cudaMemsetAsync(d_job_bits, 0, sizeof(unsigned long long) * n_jobs, stream));
    std::vector<uint8_t> use_prefix((size_t)n_jobs, 0);
    std::vector<BzBlock> batch;
    batch.reserve(BZ_BATCH_BLOCKS);
    uint64_t bytes = 0;
    std::vector<BzWin> wins;
    const uint8_t *hf = st.h_flag.data();
    int64_t computed_closed = 0, used_closed = 0;
    // blocks of the view v of job/sequence `dst` go into the batch, which runs whenever it is full
    auto add = [&](int64_t dst, int32_t x, int32_t y, const BzView &v) -> int {
        const BzSeq &sx = st.h_info[x], &sy = st.h_info[y < 0 ? x : y];
        wins.clear();
        bz_cut(v, hf + sx.roff, hf + sy.roff, wins);
        for (const BzWin &w : wins) {
            if (batch.size() == BZ_BATCH_BLOCKS || bytes + w.n > BZ_BATCH_BYTES) {
                int r = bz_run_batch(st, batch.data(), batch.size(), bytes, d_job_bits, work, stream, launches, err);
                if (r) return r;
                batch.clear(); bytes = 0;
            }
            batch.push_back(BzBlock{dst, bytes, x, y, w.v0, w.n, v});
            bytes += (w.n + 15) & ~15u;
        }
        return 0;
    };
    for (int64_t k = 0; k < n_jobs; ++k) {
        const int32_t x = xs[k], y = ys ? ys[k] : -1;
        const uint32_t open = st.h_open[x];
        int r;
        if (open) {
            if (st.use_prefix) {
                use_prefix[k] = 1;
                used_closed += st.h_nclosed[x];
                if (!st.h_pdone[x]) {
                    st.h_pdone[x] = 1;
                    computed_closed += st.h_nclosed[x];
                    if ((r = add(-1 - (int64_t)x, x, -1, bz_view_single(0, open)))) return r;
                }
            } else if ((r = add(k, x, -1, bz_view_single(0, open)))) return r;
        }
        const BzSeq &sx = st.h_info[x];
        if ((r = add(k, x, y, y < 0 ? bz_view_single(open, sx.rlen) : bz_view_pair(sx, open, st.h_info[y])))) return r;
    }
    if (!batch.empty()) {
        const int r = bz_run_batch(st, batch.data(), batch.size(), bytes, d_job_bits, work, stream, launches, err);
        if (r) return r;
    }
    st.prefix_blocks = used_closed - computed_closed;
    DCK(cudaMemcpyAsync(st.job_prefix.p, use_prefix.data(), (size_t)n_jobs, cudaMemcpyHostToDevice, stream));
    const int blocks = (int)std::min<int64_t>((n_jobs + 255) / 256, 148 * 8);
    bz_finish_kernel<<<blocks, 256, 0, stream>>>(d_job_bits, st.d_seq_bits, d_xs, st.job_prefix.get<uint8_t>(), n_jobs, d_out);
    DCK(cudaGetLastError());
    ++*launches;
    return 0;
}

#endif  // __CUDACC__

}  // namespace snacc
