// upgma.cuh -- K5: the downstream step of the distance matrix on the device (SURVEY.md 8f rank 4), sm_100a.
//   metrify      snacc/misc.py:20-25               D_sym = 0.5 (D + D^T), zero diagonal
//   hierarchical snacc/distmatrix_to_tree.py:9-15  scipy.cluster.hierarchy.linkage(squareform(D_sym), method='average')
// Output is scipy's linkage matrix Z ((n-1) x 4: cluster ids a < b, height, leaf count; new clusters are numbered n,
// n+1, ... in row order), bit for bit, ties included.  An NCD is a ratio of integer sizes, so real matrices have many
// equal distances, and with ties the order of the merges decides the tree.  So the kernel runs scipy's own algorithm,
// nn_chain (scipy/cluster/_hierarchy.pyx), not some other reducible-linkage order:
//   * the chain starts at the first active slot; each step takes the closest active cluster y of the chain's top x
//     (ties: smallest slot), and takes it only when it is strictly closer than the previous chain element;
//   * when the step returns the previous element, x and y merge: with x < y, the merged cluster goes to slot y and
//     slot x is dropped; the row (x, y, height, size) is recorded in merge order;
//   * the update is d(i, y) = (|x| d(i, x) + |y| d(i, y)) / (|x| + |y|) with every product and sum rounded on its own
//     (__dmul_rn / __dadd_rn / __ddiv_rn: a fused multiply-add would change the last bit of a height).
// The host (snacc_upgma) then sorts the rows stably by height and relabels them with a union-find, as scipy's
// label() does.  Input scipy rejects (non-finite values; with metrify off, an asymmetric matrix or a non-zero
// diagonal) is found by upgma_check_kernel and refused before upgma_kernel is launched.
//
// One CTA walks the chain (the steps are serial); each step is one parallel argmin over row x, a contiguous read of n
// doubles, and each merge one parallel update of row and column y.  The matrix stays in HBM / L2 (n = 10 000:
// 800 MB); nothing here is a dense contraction.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace snacc {

__global__ void metrify_kernel(const double *__restrict__ D, int32_t n, int do_metrify, double *__restrict__ M)
{
    const int64_t total = (int64_t)n * n;
    for (int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; k < total; k += (int64_t)gridDim.x * blockDim.x) {
        const int32_t i = (int32_t)(k / n), j = (int32_t)(k % n);
        M[k] = !do_metrify ? D[k] : (i == j ? 0.0 : 0.5 * (D[k] + D[(int64_t)j * n + i]));
    }
}

// what scipy refuses in the matrix to be clustered, OR-ed into *flags
constexpr int UPGMA_NONFINITE = 1, UPGMA_ASYMMETRIC = 2, UPGMA_DIAGONAL = 4;

__global__ void upgma_check_kernel(const double *__restrict__ M, int32_t n, int check_square_form, int *__restrict__ flags)
{
    const int64_t total = (int64_t)n * n;
    int f = 0;
    for (int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; k < total; k += (int64_t)gridDim.x * blockDim.x) {
        const int32_t i = (int32_t)(k / n), j = (int32_t)(k % n);
        const double v = M[k];
        if (i != j && !isfinite(v)) f |= UPGMA_NONFINITE;
        if (check_square_form) {
            if (i == j && v != 0.0) f |= UPGMA_DIAGONAL;
            if (i < j && !(v == M[(int64_t)j * n + i])) f |= UPGMA_ASYMMETRIC;
        }
    }
    if (f) atomicOr(flags, f);
}

constexpr int UPGMA_THREADS = 1024;

// the smaller of two (value, slot) candidates; ties: smaller slot
__device__ __forceinline__ void upgma_take_min(double &bv, int32_t &bi, double ov, int32_t oi)
{
    if (ov < bv || (ov == bv && oi < bi)) { bv = ov; bi = oi; }
}

// M: the symmetric n x n matrix, overwritten.  Z: the (n-1) x 4 merges in merge order, with slot ids (x < y) -- the
// host sorts and relabels them.  size: n ints (0 = dropped slot).  chain: n ints.
__global__ void __launch_bounds__(UPGMA_THREADS)
upgma_kernel(double *__restrict__ M, int32_t n, double *__restrict__ Z, int32_t *__restrict__ size, int32_t *__restrict__ chain)
{
    __shared__ double s_val[UPGMA_THREADS / 32];
    __shared__ int32_t s_idx[UPGMA_THREADS / 32];
    __shared__ int32_t s_x, s_y, s_len, s_first, s_merge;
    const int32_t tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    for (int32_t i = tid; i < n; i += UPGMA_THREADS) size[i] = 1;
    if (tid == 0) { s_len = 0; s_first = 0; }
    __syncthreads();
    for (int32_t k = 0; k + 1 < n; ++k) {
        if (tid == 0 && s_len == 0) {                        // an empty chain restarts at the first active slot
            while (!size[s_first]) ++s_first;
            chain[0] = s_first; s_len = 1;
        }
        // walk the chain until its top two are each other's nearest neighbours
        for (;;) {
            if (tid == 0) s_x = chain[s_len - 1];
            __syncthreads();
            const int32_t x = s_x;
            const double *row = M + (int64_t)x * n;
            double bv = 1.0 / 0.0;
            int32_t bi = 0x7fffffff;
            for (int32_t i = tid; i < n; i += UPGMA_THREADS)
                if (i != x && size[i]) upgma_take_min(bv, bi, row[i], i);
            for (int off = 16; off; off >>= 1)
                upgma_take_min(bv, bi, __shfl_down_sync(0xffffffffu, bv, off), __shfl_down_sync(0xffffffffu, bi, off));
            if (lane == 0) { s_val[warp] = bv; s_idx[warp] = bi; }
            __syncthreads();
            if (warp == 0) {
                bv = s_val[lane]; bi = s_idx[lane];
                for (int off = 16; off; off >>= 1)
                    upgma_take_min(bv, bi, __shfl_down_sync(0xffffffffu, bv, off), __shfl_down_sync(0xffffffffu, bi, off));
                if (lane == 0) {
                    const int32_t prev = s_len > 1 ? chain[s_len - 2] : -1;
                    if (prev >= 0 && !(bv < row[prev])) {        // the previous element is (one of) the closest: merge
                        s_y = prev; s_merge = 1;
                    } else {
                        chain[s_len++] = bi; s_merge = 0;
                    }
                }
            }
            __syncthreads();
            if (s_merge) break;
        }
        const int32_t x = min(s_x, s_y), y = max(s_x, s_y);
        const int32_t nx = size[x], ny = size[y];
        const double fx = (double)nx, fy = (double)ny, fxy = (double)(nx + ny);
        if (tid == 0) {
            Z[4 * (int64_t)k + 0] = (double)x;
            Z[4 * (int64_t)k + 1] = (double)y;
            Z[4 * (int64_t)k + 2] = M[(int64_t)x * n + y];
            Z[4 * (int64_t)k + 3] = fxy;
        }
        // the merged cluster replaces y; the reads of rows x and y and the writes of row y are contiguous
        for (int32_t i = tid; i < n; i += UPGMA_THREADS) {
            if (i == x || i == y || !size[i]) continue;
            const double d = __ddiv_rn(__dadd_rn(__dmul_rn(fx, M[(int64_t)x * n + i]), __dmul_rn(fy, M[(int64_t)y * n + i])), fxy);
            M[(int64_t)y * n + i] = d;
            M[(int64_t)i * n + y] = d;
        }
        __syncthreads();
        if (tid == 0) { size[x] = 0; size[y] = nx + ny; s_len -= 2; }
        __syncthreads();
    }
}

}  // namespace snacc
