// Shared helpers for the prototype-head kernels (sm_100a only).
#pragma once

#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <stdint.h>
#include <stdio.h>

#include "../../include/protohead.h"

#if defined(__CUDA_ARCH__) && (__CUDA_ARCH__ < 1000)
#error "protohead_b200 is written for sm_100a only"
#endif

namespace pph {

// ---------------------------------------------------------------------------------------------------------------
// host-side error plumbing
// ---------------------------------------------------------------------------------------------------------------
void set_error(const char* fmt, ...);

#define PPH_REQUIRE(cond, code, ...)            \
    do {                                        \
        if (!(cond)) {                          \
            ::pph::set_error(__VA_ARGS__);      \
            return (code);                      \
        }                                       \
    } while (0)

inline int launch_status(const char* what) {
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) {
        set_error("%s: %s", what, cudaGetErrorString(e));
        return (int)e;
    }
    return 0;
}

inline cudaStream_t as_stream(pph_stream_t s) { return reinterpret_cast<cudaStream_t>(s); }

template <typename... KArgs, typename... Args>
inline void launch_k(void (*kern)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, Args... args) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid;
    cfg.blockDim = block;
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    (void)cudaLaunchKernelEx(&cfg, kern, static_cast<KArgs>(args)...);   // status is read by launch_status()
}

inline int ceil_div(int a, int b) { return (a + b - 1) / b; }

// Opt a kernel into `bytes` of dynamic shared memory AND ask for the maximum shared-memory carve-out: the L1 / shared
// split of an SM is set by the kernel that arrives first, and a kernel of a concurrent graph branch can only join that
// SM if its shared memory still fits the carve-out -- with the default (smallest sufficient) carve-out the branches of
// the step serialised instead of overlapping.
template <class K>
inline cudaError_t opt_in_smem(K kern, size_t bytes) {
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
    if (e == cudaSuccess)
        e = cudaFuncSetAttribute(kern, cudaFuncAttributePreferredSharedMemoryCarveout, (int)cudaSharedmemCarveoutMaxShared);
    return e;
}

// ---------------------------------------------------------------------------------------------------------------
// device helpers
// ---------------------------------------------------------------------------------------------------------------
// relu as torch computes it: NaN stays NaN (fmaxf(NaN, 0) would return 0 and hide a diverged step from the
// caller's isfinite(loss) check, tools/engine_proto.py:68-70)
__device__ __forceinline__ float relu_keep_nan(float x) { return x < 0.0f ? 0.0f : x; }

// Rank of element n of a score row in the selection order (larger first, lower index first on equal scores): the number of
// elements that beat it.  `s4` = the row in shared memory, padded to a multiple of 4 with -inf; v = s[n], never NaN (NaN is
// canonicalised to +inf when the row is staged).  Elements before n beat it when >=, elements after n when >: one compare
// per element instead of the (>, ==, index) triple.
__device__ __forceinline__ int rank_by_count(const float4* s4, int n, int n_pad, float v) {
    int rank = 0;
    const int nq = n >> 2;
    for (int j = 0; j < nq; ++j) {
        const float4 q = s4[j];
        rank += (q.x >= v) + (q.y >= v) + (q.z >= v) + (q.w >= v);
    }
    {
        const float4 q = s4[nq];
        const int r = n & 3;
        rank += (r > 0 ? q.x >= v : false) + (r > 1 ? q.y >= v : (r < 1 && q.y > v)) +
                (r > 2 ? q.z >= v : (r < 2 && q.z > v)) + (r < 3 && q.w > v);
    }
    for (int j = nq + 1; j < (n_pad >> 2); ++j) {
        const float4 q = s4[j];
        rank += (q.x > v) + (q.y > v) + (q.z > v) + (q.w > v);
    }
    return rank;
}

// ---- cp.async (LDGSTS): 16-byte global -> shared copies that bypass the register file ---------------------------
__device__ __forceinline__ void cp_async16(void* smem_dst, const void* gmem_src) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"((uint32_t)__cvta_generic_to_shared(smem_dst)),
                 "l"(gmem_src)
                 : "memory");
}
__device__ __forceinline__ void cp_async4(void* smem_dst, const void* gmem_src) {
    asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"((uint32_t)__cvta_generic_to_shared(smem_dst)),
                 "l"(gmem_src)
                 : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

// ---- grid-wide barrier for kernels whose CTAs are all co-resident (grid <= SM count x resident CTAs per SM) ------
// `counter` counts arrivals monotonically inside one launch (barrier i releases at i * n_ctas); the kernel's
// finisher (grid_finish) resets it, so a CUDA-graph replay starts from zero again.  The spin is bounded: a protocol
// bug traps (launch error reported to the caller) instead of hanging the device.
__device__ __forceinline__ unsigned int ld_acquire_u32(const unsigned int* p) {
    unsigned int v;
    asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void grid_barrier(unsigned int* counter, unsigned int target) {
    __syncthreads();
    if (threadIdx.x == 0) {
        __threadfence();
        atomicAdd(counter, 1u);
        const long long t0 = clock64();
        while (ld_acquire_u32(counter) < target) {
            if (clock64() - t0 > 4000000000LL) __trap();
        }
        __threadfence();
    }
    __syncthreads();
}
// Called by every participating CTA after its last barrier: the last one to arrive zeroes both counters.
__device__ __forceinline__ void grid_finish(unsigned int* counter, unsigned int* done, unsigned int n_ctas) {
    __syncthreads();
    if (threadIdx.x == 0) {
        __threadfence();
        if (atomicAdd(done, 1u) == n_ctas - 1u) {
            *counter = 0u;
            *done = 0u;
            __threadfence();
        }
    }
}
__device__ __forceinline__ float4 ldcg4(const float* p) { return __ldcg(reinterpret_cast<const float4*>(p)); }

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// activation of a distance, protopformer.py:228-234 (precise log/div: parity is 1e-4 on a cancelling quantity)
__device__ __forceinline__ float act_of_dist(float d, int act_fn, float eps) {
    return act_fn == PPH_ACT_LOG ? logf((d + 1.0f) / (d + eps)) : -d;
}

// d act / d d, including the relu mask of protopformer.py:216 (relu'(0) = 0 as in torch)
__device__ __forceinline__ float dact_of_dist(float d, int act_fn, float eps) {
    if (!(d > 0.0f)) return 0.0f;
    return act_fn == PPH_ACT_LOG ? (1.0f / (d + 1.0f) - 1.0f / (d + eps)) : -1.0f;
}

__device__ __forceinline__ uint16_t bf16_bits(float x) {
    return __bfloat16_as_ushort(__float2bfloat16_rn(x));
}
__device__ __forceinline__ float bf16_to_float(uint16_t b) {
    return __uint_as_float(((uint32_t)b) << 16);
}

// ---- backbone token rows: fp32 (float) or bf16 (uint16_t storage) ------------------------------------------------
// Every bf16 value is exact in fp32, so a bf16 token is widened at its load and nothing downstream changes: the
// results equal those of the fp32 kernels fed the widened tokens.  Token gradients are accumulated in fp32 and
// rounded to nearest-even once, at the store.
__device__ __forceinline__ float tok_f(float x) { return x; }
__device__ __forceinline__ float tok_f(uint16_t x) { return bf16_to_float(x); }
template <class T>
__device__ __forceinline__ float ldg_tok(const T* p) { return tok_f(__ldg(p)); }
// four consecutive tokens values (16-byte aligned fp32 / 8-byte aligned bf16)
__device__ __forceinline__ float4 ldg4_tok(const float* p) { return __ldg(reinterpret_cast<const float4*>(p)); }
__device__ __forceinline__ float4 ldg4_tok(const uint16_t* p) {
    const uint2 q = __ldg(reinterpret_cast<const uint2*>(p));
    return make_float4(__uint_as_float(q.x << 16), __uint_as_float(q.x & 0xffff0000u), __uint_as_float(q.y << 16),
                       __uint_as_float(q.y & 0xffff0000u));
}
__device__ __forceinline__ void st_tok(float* p, float v) { *p = v; }
__device__ __forceinline__ void st_tok(uint16_t* p, float v) { *p = bf16_bits(v); }
__device__ __forceinline__ void st2_tok(float* p, float a, float b) { *reinterpret_cast<float2*>(p) = make_float2(a, b); }
__device__ __forceinline__ void st2_tok(uint16_t* p, float a, float b) {
    *reinterpret_cast<uint32_t*>(p) = (uint32_t)bf16_bits(a) | ((uint32_t)bf16_bits(b) << 16);
}
__device__ __forceinline__ void st4_tok(float* p, float4 v) { *reinterpret_cast<float4*>(p) = v; }
__device__ __forceinline__ void st4_tok(uint16_t* p, float4 v) {
    *reinterpret_cast<uint2*>(p) = make_uint2((uint32_t)bf16_bits(v.x) | ((uint32_t)bf16_bits(v.y) << 16),
                                              (uint32_t)bf16_bits(v.z) | ((uint32_t)bf16_bits(v.w) << 16));
}

}  // namespace pph
