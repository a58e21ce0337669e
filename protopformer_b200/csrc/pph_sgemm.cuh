// Generic CUDA-core FP32 tile GEMM used by the small / exact-precision pieces of the head
// (last layers, their backward, add-on backward, global-prototype gradients).
//
//   acc[m,n] = sum_{k in split} A(m,k) * B(n,k)        rs[m] = sum_{k in split} A(m,k)   (optional)
//   epi(m, n, acc, rs)                                 -- the functor writes / atomically accumulates the result
//
// A and B are functors `float operator()(int row, int k)` (row = m or n) that return 0 outside their range and
// carry `static constexpr bool kContigK` (true: consecutive k are contiguous in memory, false: consecutive rows
// are) so the tile loader issues coalesced requests either way.  64x64x16 tiles, 256 threads, 4x4 per thread.
// blockIdx.z splits the k range (`k_per_split` each); the epilogue must then accumulate atomically.
#pragma once

#include "pph_common.cuh"

namespace pph {

constexpr int kGemmBM = 64, kGemmBN = 64, kGemmBK = 16, kGemmThreads = 256, kGemmPad = 4;

template <class Op>
__device__ __forceinline__ void gemm_load_tile(float (*dst)[kGemmBM + kGemmPad], const Op& op, int row0, int k0,
                                               int k_end, int tid) {
    if (Op::kContigK) {
        const int k = tid & 15, r = tid >> 4;
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const int row = r + 16 * i;
            dst[k][row] = (k0 + k < k_end) ? op(row0 + row, k0 + k) : 0.0f;
        }
    } else {
        const int row = tid & 63, k = tid >> 6;
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const int kk = k + 4 * i;
            dst[kk][row] = (k0 + kk < k_end) ? op(row0 + row, k0 + kk) : 0.0f;
        }
    }
}

template <bool kRowSum, class AOp, class BOp, class Epi>
__global__ void __launch_bounds__(kGemmThreads)
sgemm_kernel(int M, int N, int Kd, int k_per_split, AOp a_op, BOp b_op, Epi epi) {
    __shared__ __align__(16) float As[kGemmBK][kGemmBM + kGemmPad];
    __shared__ __align__(16) float Bs[kGemmBK][kGemmBN + kGemmPad];
    const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
    const int m0 = blockIdx.y * kGemmBM, n0 = blockIdx.x * kGemmBN;
    const int k_begin = blockIdx.z * k_per_split;
    const int k_end = min(Kd, k_begin + k_per_split);
    float acc[4][4];
    float rs[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;

    for (int k0 = k_begin; k0 < k_end; k0 += kGemmBK) {
        gemm_load_tile(As, a_op, m0, k0, k_end, tid);
        gemm_load_tile(Bs, b_op, n0, k0, k_end, tid);
        __syncthreads();
#pragma unroll
        for (int kk = 0; kk < kGemmBK; ++kk) {
            const float4 a = *reinterpret_cast<const float4*>(&As[kk][ty * 4]);
            const float4 b = *reinterpret_cast<const float4*>(&Bs[kk][tx * 4]);
            const float av[4] = {a.x, a.y, a.z, a.w}, bv[4] = {b.x, b.y, b.z, b.w};
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                if (kRowSum) rs[i] += av[i];
#pragma unroll
                for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(av[i], bv[j], acc[i][j]);
            }
        }
        __syncthreads();
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const int m = m0 + ty * 4 + i;
        if (m >= M) continue;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int n = n0 + tx * 4 + j;
            if (n < N) epi(m, n, acc[i][j], rs[i]);
        }
    }
}

// plain strided operand: element (row, k) at base[row * ld_row + k * ld_k], zero outside [0,rows)
template <bool CONTIG_K>
struct StridedOp {
    static constexpr bool kContigK = CONTIG_K;
    const float* base;
    int rows;
    long ld_row, ld_k;
    __device__ __forceinline__ float operator()(int row, int k) const {
        return row < rows ? __ldg(base + (long)row * ld_row + (long)k * ld_k) : 0.0f;
    }
};

template <bool kRowSum, class AOp, class BOp, class Epi>
inline void launch_sgemm(int M, int N, int Kd, int splits, AOp a, BOp b, Epi e, cudaStream_t st) {
    splits = splits < 1 ? 1 : splits;
    int k_per_split = ceil_div(ceil_div(Kd, splits), kGemmBK) * kGemmBK;
    if (k_per_split < kGemmBK) k_per_split = kGemmBK;
    splits = ceil_div(Kd, k_per_split);
    if (splits < 1) splits = 1;
    dim3 grid(ceil_div(N, kGemmBN), ceil_div(M, kGemmBM), splits);
    launch_k(sgemm_kernel<kRowSum, AOp, BOp, Epi>, dim3(grid), dim3(kGemmThreads), (size_t)(0), st, M, N, Kd, k_per_split, a, b, e);
}

}  // namespace pph
