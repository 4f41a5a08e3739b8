// host_emu_bzip2.cu -- the product's bzip2 size functions (snacc_b200/csrc/bzip2.cuh) compiled for the host, with a
// plain host rotation sort in place of the device BWT.  Test infrastructure only (tests/test_bzip2_host.py).
#include <stdint.h>
#include <algorithm>
#include <numeric>
#include <vector>
#include "../snacc_b200/csrc/bzip2.cuh"

using namespace snacc;

namespace {

// last column of the sorted cyclic rotations of t[0, n), by prefix doubling with std::sort
void host_bwt(const uint8_t *t, uint32_t n, std::vector<uint8_t> &L)
{
    std::vector<uint32_t> sa(n), rk(n), tmp(n);
    std::iota(sa.begin(), sa.end(), 0u);
    for (uint32_t i = 0; i < n; ++i) rk[i] = t[i];
    for (uint32_t h = 1;; h *= 2) {
        auto key = [&](uint32_t i) { return ((uint64_t)rk[i] << 32) | rk[(i + h) % n]; };
        std::sort(sa.begin(), sa.end(), [&](uint32_t a, uint32_t b) { return key(a) < key(b); });
        tmp[sa[0]] = 0;
        for (uint32_t i = 1; i < n; ++i) tmp[sa[i]] = tmp[sa[i - 1]] + (key(sa[i]) != key(sa[i - 1]));
        rk.swap(tmp);
        if (rk[sa[n - 1]] == n - 1 || h >= n) break;
    }
    L.resize(n);
    for (uint32_t i = 0; i < n; ++i) L[i] = t[sa[i] ? sa[i] - 1 : n - 1];
}

struct Rle {
    std::vector<uint8_t> r, f;
    BzSeq s{};
    Rle(const uint8_t *p, uint32_t n) : r((size_t)n * 5 / 4 + 8), f((size_t)n * 5 / 4 + 8) { bz_rle_seq(p, n, r.data(), f.data(), &s); }
};

int64_t view_bits(const BzView &v, const Rle &x, const Rle *y, std::vector<BzWin> *wins_out, int64_t *nblocks)
{
    std::vector<BzWin> wins;
    const uint8_t *ry = y ? y->r.data() : x.r.data(), *fy = y ? y->f.data() : x.f.data();
    bz_cut(v, x.f.data(), fy, wins);
    std::vector<uint8_t> blk, L;
    BzWork w;
    int64_t bits = 0;
    for (const BzWin &b : wins) {
        blk.resize(b.n);
        for (uint32_t t = 0; t < b.n; ++t) { bool st; blk[t] = v.at(x.r.data(), x.f.data(), ry, fy, (uint64_t)b.v0 + t, &st); }
        host_bwt(blk.data(), b.n, L);
        bits += bz_block_bits_serial(L.data(), b.n, w);
    }
    if (wins_out) *wins_out = wins;
    if (nblocks) *nblocks += (int64_t)wins.size();
    return bits;
}

// x alone: its closed blocks (all but the last of its own cut), and where the open block starts
int64_t closed_bits(const Rle &x, uint32_t *open, int64_t *nblocks)
{
    std::vector<BzWin> wins;
    bz_cut(bz_view_single(0, x.s.rlen), x.f.data(), x.f.data(), wins);
    *open = wins.back().v0;
    return *open ? view_bits(bz_view_single(0, *open), x, nullptr, nullptr, nblocks) : 0;
}

}  // namespace

extern "C" {

// len(bz2.compress(s)) the way the device computes a single: x's closed blocks + its open block
int64_t emu_bz2_single(const uint8_t *s, uint32_t n, int64_t *nblocks)
{
    Rle x(s, n);
    uint32_t open;
    int64_t bits = closed_bits(x, &open, nblocks);
    bits += view_bits(bz_view_single(open, x.s.rlen), x, nullptr, nullptr, nblocks);
    return bz_stream_bytes(bits);
}

// len(bz2.compress(x + y)) the way the device computes a pair: x's closed blocks, then the blocks of
// x's open tail + junction + RLE1(y) after its first run
int64_t emu_bz2_pair(const uint8_t *xs, uint32_t nx, const uint8_t *ys, uint32_t ny, int64_t *nblocks)
{
    Rle x(xs, nx), y(ys, ny);
    uint32_t open;
    int64_t bits = closed_bits(x, &open, nblocks);
    bits += view_bits(bz_view_pair(x.s, open, y.s), x, &y, nullptr, nblocks);
    return bz_stream_bytes(bits);
}

// RLE1 block lengths of s as the product cuts it (n_out: room in out); returns the number of blocks
int64_t emu_bz2_block_lengths(const uint8_t *s, uint32_t n, uint32_t *out, int64_t n_out)
{
    Rle x(s, n);
    std::vector<BzWin> wins;
    bz_cut(bz_view_single(0, x.s.rlen), x.f.data(), x.f.data(), wins);
    for (size_t k = 0; k < wins.size() && (int64_t)k < n_out; ++k) out[k] = wins[k].n;
    return (int64_t)wins.size();
}

// code lengths of one table (BZ2_hbMakeCodeLengths restated) for the given symbol frequencies
void emu_bz2_code_lengths(const int32_t *freq, int32_t alpha_size, int32_t max_len, uint8_t *len)
{
    int32_t scratch[BZ_HB_SCRATCH];
    bz_make_code_lengths(len, freq, alpha_size, max_len, scratch);
}

// last column of the sorted cyclic rotations of t[0, n) (the emulator's BWT)
void emu_bz2_bwt(const uint8_t *t, uint32_t n, uint8_t *L)
{
    std::vector<uint8_t> out;
    host_bwt(t, n, out);
    std::copy(out.begin(), out.end(), L);
}

// bits of one block from its last column L[0, n): MTF + RLE2, table choice and bit count, serially
int64_t emu_bz2_block_bits(const uint8_t *L, uint32_t n)
{
    BzWork w;
    return bz_block_bits_serial(L, n, w);
}

// how many of the code-length builds of a block's table choice (BZ_N_ITERS iterations x nGroups tables) hit the
// 17-bit cap and rescaled: the iterations of bz_block_bits_serial, each build repeated without the cap
int32_t emu_bz2_rescaled_builds(const uint8_t *L, uint32_t n)
{
    uint8_t in_use[256] = {0}, seq_of[256], yy[256], len[BZ_N_GROUPS * BZ_MAX_ALPHA], free_len[BZ_MAX_ALPHA];
    int32_t freq[BZ_MAX_ALPHA], rfreq[BZ_N_GROUPS * BZ_MAX_ALPHA], scratch[BZ_HB_SCRATCH];
    for (uint32_t i = 0; i < n; ++i) in_use[L[i]] = 1;
    const int nInUse = bz_map(in_use, seq_of), alphaSize = nInUse + 2;
    std::vector<uint16_t> mtfv((size_t)n + 1);
    const uint32_t nMTF = bz_mtf(L, n, seq_of, nInUse, yy, mtfv.data(), freq);
    const int nGroups = bz_n_groups(nMTF);
    bz_init_tables(len, nGroups, alphaSize, freq, nMTF);
    const int nSel = (int)((nMTF + BZ_G_SIZE - 1) / BZ_G_SIZE);
    int32_t rescaled = 0;
    for (int iter = 0; iter < BZ_N_ITERS; ++iter) {
        for (int k = 0; k < BZ_N_GROUPS * BZ_MAX_ALPHA; ++k) rfreq[k] = 0;
        for (int g = 0; g < nSel; ++g) {
            const uint32_t gs = (uint32_t)g * BZ_G_SIZE, ge = gs + BZ_G_SIZE - 1 < nMTF ? gs + BZ_G_SIZE - 1 : nMTF - 1;
            uint32_t c;
            const int bt = bz_group_choose(len, nGroups, mtfv.data(), gs, ge, &c);
            for (uint32_t i = gs; i <= ge; ++i) rfreq[bt * BZ_MAX_ALPHA + mtfv[i]]++;
        }
        for (int t = 0; t < nGroups; ++t) {
            bz_make_code_lengths(len + t * BZ_MAX_ALPHA, rfreq + t * BZ_MAX_ALPHA, alphaSize, BZ_MAX_CODE_LEN, scratch);
            // no code of alphaSize symbols is longer than alphaSize - 1 < BZ_MAX_ALPHA bits: this build never rescales
            bz_make_code_lengths(free_len, rfreq + t * BZ_MAX_ALPHA, alphaSize, BZ_MAX_ALPHA, scratch);
            rescaled += *std::max_element(free_len, free_len + alphaSize) > BZ_MAX_CODE_LEN;
        }
    }
    return rescaled;
}

}  // extern "C"
