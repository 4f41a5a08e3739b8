// common.cuh -- shared device helpers for libsnacc_b200 (sm_100a).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

// Device code is also compilable for the host so that tests/host_emu.cu can run the very same parse
// functions on the CPU against the oracle (test infrastructure; the product never does this).
#define SNACC_HD __host__ __device__ __forceinline__
#ifdef __CUDA_ARCH__
#define SNACC_LDG(p) __ldg(p)
#define SNACC_FFS32(x) __ffs((int)(x))
#define SNACC_FFS64(x) __ffsll((long long)(x))
#else
#define SNACC_LDG(p) (*(p))
#define SNACC_FFS32(x) __builtin_ffs((int)(x))
#define SNACC_FFS64(x) __builtin_ffsll((long long)(x))
#endif

// NVTX ranges around the phases of a call (upload / pack / singles / pair tiles / deflate stages / epilogue): visible to
// `ncu --nvtx` and any NVTX-aware tool; header-only NVTX3, a no-op when no tool is attached.  Host builds of the
// device headers (tests/host_emu.cu) do not need it.
#if defined(__CUDACC__) && !defined(SNACC_NO_NVTX) && __has_include(<nvtx3/nvToolsExt.h>)
#include <nvtx3/nvToolsExt.h>
namespace snacc { struct NvtxRange { explicit NvtxRange(const char *name) { nvtxRangePushA(name); } ~NvtxRange() { nvtxRangePop(); } }; }
#else
namespace snacc { struct NvtxRange { explicit NvtxRange(const char *) {} }; }
#endif

namespace snacc {

template <typename T> SNACC_HD T tmin(T a, T b) { return a < b ? a : b; }
template <typename T> SNACC_HD T tmax(T a, T b) { return a > b ? a : b; }

// Every sequence sits in the padded corpus at a 16-byte aligned offset and is followed by at least
// SEQ_PAD zero bytes, so 16-byte over-reads past either end of a stream segment are always legal.
constexpr uint32_t SEQ_ALIGN = 16;
constexpr uint32_t SEQ_PAD = 32;

// A compressor input as the reference builds it (pairwise_ncd.py:29-30): x, or x followed by y.
// Positions are byte offsets into the virtual concatenation; nothing is materialised.
struct Stream {
    const uint8_t *x;   // first segment
    const uint8_t *y;   // second segment (for a single: points at x's zero padding)
    uint32_t lx;        // length of x
    uint32_t n;         // total length lx + ly
};

// 2-bit packed copy of a sequence (pack.cuh): base k sits in bits 2(k%32) of 64-bit word k/32; the word
// count is even (16-byte vector copies) and PK_PAD_WORDS zero words follow, so reading 32 bases from any
// position below len + 64 is legal.
constexpr uint32_t PK_PAD_WORDS = 4;
SNACC_HD uint32_t pk_words(uint32_t len) { return ((((len + 31) >> 5) + 1) & ~1u) + PK_PAD_WORDS; }

SNACC_HD uint64_t ldu64(const uint8_t *p)
{
    // unaligned 8-byte little-endian load built from two aligned 8-byte loads
    uintptr_t a = reinterpret_cast<uintptr_t>(p);
    const uint64_t *q = reinterpret_cast<const uint64_t *>(a & ~uintptr_t(7));
    uint32_t sh = (uint32_t)(a & 7) * 8;
    uint64_t lo = SNACC_LDG(q);
    if (sh == 0) return lo;
    uint64_t hi = SNACC_LDG(q + 1);
    return (lo >> sh) | (hi << (64 - sh));
}

SNACC_HD uint64_t ld64(const Stream &s, uint32_t p)
{
    if (p >= s.lx) return ldu64(s.y + (p - s.lx));
    uint64_t a = ldu64(s.x + p);
    uint32_t k = s.lx - p;               // bytes of x available from p
    if (k >= 8) return a;
    uint64_t b = ldu64(s.y);             // straddles the x|y boundary
    return (a & ((1ull << (8 * k)) - 1)) | (b << (8 * k));
}

SNACC_HD uint8_t ld8(const Stream &s, uint32_t p)
{
    return p >= s.lx ? SNACC_LDG(s.y + (p - s.lx)) : SNACC_LDG(s.x + p);
}

#ifdef __CUDACC__
// ---- host side of the codec drivers ----------------------------------------------------------------------------------

// the uploaded corpus as the codec drivers see it (device arrays and their host copies)
struct Corpus {
    const uint8_t *d_corpus; const uint64_t *d_off; const uint32_t *d_len;
    const uint64_t *h_off; const uint32_t *h_len; int32_t n_seqs;
};

// A device array that grows on demand and is kept between calls (all its use is ordered on one stream).  Growing
// synchronises the stream first: an earlier launch may still read the old array.  Small argument arrays get 1.25x
// headroom (4 KiB at least) so that calls of slowly growing size do not reallocate every time; the large ones (job
// arrays, outputs, working tables) are sized exactly, since headroom there would be memory held between calls for nothing.
struct DevBuf {
    void *p = nullptr;
    size_t cap = 0;
    template <typename T> T *get() const { return (T *)p; }
    cudaError_t grow(size_t bytes, cudaStream_t stream, bool exact = false)
    {
        if (bytes <= cap) return cudaSuccess;
        cudaError_t e = cudaStreamSynchronize(stream);
        if (e != cudaSuccess) return e;
        release();
        const size_t want = exact ? bytes : (bytes + bytes / 4 > 4096 ? bytes + bytes / 4 : 4096);
        e = cudaMalloc(&p, want);
        if (e != cudaSuccess) { p = nullptr; return e; }
        cap = want;
        return cudaSuccess;
    }
    void release() { cudaFree(p); p = nullptr; cap = 0; }
};

// codec drivers: a failed CUDA call records its message in `err` (a std::string in scope) and the function returns
// SNACC_ERR_CUDA (-1)
#define DCK(call) do { cudaError_t e_ = (call); if (e_ != cudaSuccess) { \
        char b_[512]; snprintf(b_, sizeof b_, "%s failed at %s:%d: %s", #call, __FILE__, __LINE__, cudaGetErrorString(e_)); \
        err = b_; return -1; } } while (0)
#endif  // __CUDACC__

}  // namespace snacc
