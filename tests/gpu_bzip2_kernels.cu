// gpu_bzip2_kernels.cu -- the product's bzip2 device kernels (snacc_b200/csrc/bzip2.cuh) launched directly on
// caller-supplied blocks, so the BWT of each sort regime and the bit count can be compared with plain references.
// Test infrastructure only (tests/test_bzip2_kernels_gpu.py).  Every call frees what it allocated and returns 0, -1 for
// bad arguments, -2 when bits reached the wrong destination, or the CUDA error code.
#include <stdint.h>
#include <string.h>
#include <vector>
#include <cuda_runtime.h>
#include "../snacc_b200/csrc/bzip2.cuh"

using namespace snacc;

namespace {

struct Dev {
    void *p = nullptr;
    ~Dev() { if (p) cudaFree(p); }
    template <typename T> T *get() const { return (T *)p; }
};

#define KCK(x) do { const cudaError_t e_ = (x); if (e_ != cudaSuccess) return (int)e_; } while (0)

// the blocks at 16-byte-aligned offsets, as bz_run lays out a batch; returns the padded byte count (0: bad lengths)
uint64_t layout(const uint8_t *bytes, const uint32_t *lens, int32_t nb, uint32_t max_n, std::vector<BzBlock> &bl,
                std::vector<uint8_t> &padded)
{
    bl.assign((size_t)nb, BzBlock{});
    uint64_t off = 0;
    for (int32_t k = 0; k < nb; ++k) {
        if (lens[k] == 0 || lens[k] > max_n) return 0;
        bl[k].dst = k; bl[k].off = off; bl[k].x = 0; bl[k].y = -1; bl[k].v0 = 0; bl[k].n = lens[k];
        off += (lens[k] + 15) & ~15u;
    }
    padded.assign(off, 0);
    uint64_t in = 0;
    for (int32_t k = 0; k < nb; ++k) { memcpy(padded.data() + bl[k].off, bytes + in, lens[k]); in += lens[k]; }
    return off;
}

}  // namespace

extern "C" {

// L_out: the last column of every block (tightly packed, as `bytes` is).  regime 0: bz_bwt_smem_kernel (every block at
// most BZ_SMEM_MAX_N bytes); 1: bz_bwt_global_kernel (16 bytes of scratch per block byte)
int kbz_bwt(const uint8_t *bytes, const uint32_t *lens, int32_t nb, int32_t regime, uint8_t *L_out)
{
    if (!bytes || !lens || !L_out || nb <= 0 || (regime != 0 && regime != 1)) return -1;
    std::vector<BzBlock> bl;
    std::vector<uint8_t> h;
    const uint64_t total = layout(bytes, lens, nb, regime == 0 ? BZ_SMEM_MAX_N : BZ_NBLOCK_MAX + 4, bl, h);
    if (!total) return -1;
    std::vector<int32_t> list((size_t)nb);
    for (int32_t k = 0; k < nb; ++k) list[k] = k;
    Dev d_blocks, d_list, d_buf, d_bwt, d_work;
    KCK(cudaMalloc(&d_blocks.p, sizeof(BzBlock) * nb));
    KCK(cudaMalloc(&d_list.p, sizeof(int32_t) * nb));
    KCK(cudaMalloc(&d_buf.p, total));
    KCK(cudaMalloc(&d_bwt.p, total));
    KCK(cudaMemcpy(d_blocks.p, bl.data(), sizeof(BzBlock) * nb, cudaMemcpyHostToDevice));
    KCK(cudaMemcpy(d_list.p, list.data(), sizeof(int32_t) * nb, cudaMemcpyHostToDevice));
    KCK(cudaMemcpy(d_buf.p, h.data(), total, cudaMemcpyHostToDevice));
    KCK(cudaMemset(d_bwt.p, 0, total));
    if (regime == 0) {
        KCK(cudaFuncSetAttribute(bz_bwt_smem_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)BZ_SMEM_BYTES));
        bz_bwt_smem_kernel<<<(unsigned)nb, BZ_SORT_THREADS, BZ_SMEM_BYTES>>>(d_blocks.get<BzBlock>(), d_list.get<int32_t>(),
                                                                             d_buf.get<uint8_t>(), d_bwt.get<uint8_t>());
    } else {
        KCK(cudaMalloc(&d_work.p, 16 * total));
        bz_bwt_global_kernel<<<(unsigned)nb, BZ_SORT_THREADS>>>(d_blocks.get<BzBlock>(), d_list.get<int32_t>(),
                                                                d_buf.get<uint8_t>(), d_bwt.get<uint8_t>(), d_work.get<uint32_t>());
    }
    KCK(cudaGetLastError());
    KCK(cudaDeviceSynchronize());
    KCK(cudaMemcpy(h.data(), d_bwt.p, total, cudaMemcpyDeviceToHost));
    uint64_t out = 0;
    for (int32_t k = 0; k < nb; ++k) { memcpy(L_out + out, h.data() + bl[k].off, lens[k]); out += lens[k]; }
    return 0;
}

// bits_out[k]: the bits bz_bits_kernel counts for the last column L of block k (tightly packed).  Even blocks are
// job blocks (dst >= 0, summed into job bits), odd ones a sequence's closed blocks (dst < 0, into sequence bits).
int kbz_bits(const uint8_t *L, const uint32_t *lens, int32_t nb, int64_t *bits_out)
{
    if (!L || !lens || !bits_out || nb <= 0) return -1;
    std::vector<BzBlock> bl;
    std::vector<uint8_t> h;
    const uint64_t total = layout(L, lens, nb, BZ_NBLOCK_MAX + 4, bl, h);
    if (!total) return -1;
    for (int32_t k = 0; k < nb; ++k) bl[k].dst = (k & 1) ? -1 - (int64_t)k : (int64_t)k;
    Dev d_blocks, d_bwt, d_mtf, d_job, d_seq;
    KCK(cudaMalloc(&d_blocks.p, sizeof(BzBlock) * nb));
    KCK(cudaMalloc(&d_bwt.p, total));
    KCK(cudaMalloc(&d_mtf.p, sizeof(uint16_t) * (total + nb)));
    KCK(cudaMalloc(&d_job.p, sizeof(unsigned long long) * nb));
    KCK(cudaMalloc(&d_seq.p, sizeof(unsigned long long) * nb));
    KCK(cudaMemcpy(d_blocks.p, bl.data(), sizeof(BzBlock) * nb, cudaMemcpyHostToDevice));
    KCK(cudaMemcpy(d_bwt.p, h.data(), total, cudaMemcpyHostToDevice));
    KCK(cudaMemset(d_job.p, 0, sizeof(unsigned long long) * nb));
    KCK(cudaMemset(d_seq.p, 0, sizeof(unsigned long long) * nb));
    KCK(cudaFuncSetAttribute(bz_bits_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)BZ_BITS_DYN_SMEM));
    bz_bits_kernel<<<(unsigned)nb, BZ_BITS_THREADS, BZ_BITS_DYN_SMEM>>>(
        d_blocks.get<BzBlock>(), d_bwt.get<uint8_t>(), d_mtf.get<uint16_t>(), d_job.get<unsigned long long>(),
        d_seq.get<unsigned long long>());
    KCK(cudaGetLastError());
    KCK(cudaDeviceSynchronize());
    std::vector<unsigned long long> job((size_t)nb), seq((size_t)nb);
    KCK(cudaMemcpy(job.data(), d_job.p, sizeof(unsigned long long) * nb, cudaMemcpyDeviceToHost));
    KCK(cudaMemcpy(seq.data(), d_seq.p, sizeof(unsigned long long) * nb, cudaMemcpyDeviceToHost));
    for (int32_t k = 0; k < nb; ++k) {
        // the other array must be untouched: each record goes to exactly one destination
        if (((k & 1) ? job[k] : seq[k]) != 0) return -2;
        bits_out[k] = (int64_t)((k & 1) ? seq[k] : job[k]);
    }
    return 0;
}

}  // extern "C"
