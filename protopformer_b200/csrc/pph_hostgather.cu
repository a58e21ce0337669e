// Selection-first input transfer for callers whose backbone tokens live in (pinned) HOST memory.
//
// The head consumes only the CLS row and the K selected token rows of every image (protopformer.py:156-166: the
// top-k of the CLS-attention scores, then the gather) -- at the CUB shape 82 of 197 rows.  Copying the whole
// (B, 1+N, Din) tensor over PCIe therefore moves 2.4x the bytes the path reads, and at B = 64 that copy (9.7 MB) takes
// longer than the whole training step.  This kernel reads exactly the consumed rows straight out of the mapped host
// buffer (zero-copy loads over PCIe) and drops them at their natural positions of the device-side token tensor; the
// other rows of that tensor are never read by the forward or the backward.  The scores (B x N floats) travel first by
// an ordinary copy and are ranked on the device (pph_select_topk), so the row list is the device's own.
#include "pph_common.cuh"

namespace pph {
namespace {

// small CTAs (few registers, no shared memory) slip in beside the step's one-CTA-per-SM kernels instead of holding SMs
// those kernels' grid barriers are waiting for; the loads in flight come from the batch depth instead
constexpr int kHgThreads = 128;
constexpr int kHgBatch = 8;

__device__ __forceinline__ float4 ld_host4(const float4* p) {
    float4 v;   // streaming, no L1 allocation: every byte is read once
    asm volatile("ld.global.L1::no_allocate.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "l"(p));
    return v;
}

// rows are moved as q 16-byte words (fp32: Din / 4, bf16: Din / 8): the kernel never looks at the element type
__global__ void __launch_bounds__(kHgThreads) host_rows_kernel(const float* __restrict__ src, const int* __restrict__ idx32,
                                                               int B, int N, int q, int K, float* __restrict__ dst) {
    const long long total = (long long)B * (K + 1) * q;
    const long long stride = (long long)gridDim.x * kHgThreads;
    for (long long i0 = (long long)blockIdx.x * kHgThreads + threadIdx.x; i0 < total; i0 += kHgBatch * stride) {
        float4 v[kHgBatch];
        long long at[kHgBatch];
#pragma unroll
        for (int k = 0; k < kHgBatch; ++k) {
            const long long i = i0 + k * stride;
            at[k] = -1;
            if (i < total) {
                const int r = (int)(i / q), c = (int)(i - (long long)r * q);
                const int b = r / (K + 1), j = r - b * (K + 1);
                const int row = j == K ? 0 : 1 + __ldg(idx32 + (size_t)b * K + j);      // token n sits at row 1 + n
                at[k] = ((long long)b * (N + 1) + row) * q + c;
                v[k] = ld_host4(reinterpret_cast<const float4*>(src) + at[k]);
            }
        }
#pragma unroll
        for (int k = 0; k < kHgBatch; ++k)
            if (at[k] >= 0) reinterpret_cast<float4*>(dst)[at[k]] = v[k];
    }
}

}  // namespace
}  // namespace pph

using namespace pph;

static int gather_rows_host(const char* name, const void* tokens_host, const int32_t* idx32, int B, int N, int Din, int K,
                            int elem_bytes, void* tokens_dev, int n_ctas, pph_stream_t stream) {
    const int per16 = 16 / elem_bytes;                       // elements per 16-byte word
    PPH_REQUIRE(tokens_host && idx32 && tokens_dev, PPH_EINVAL, "%s: null pointer", name);
    PPH_REQUIRE(B >= 0 && N >= 1 && K >= 1 && K <= N && Din >= per16 && Din % per16 == 0 && n_ctas >= 1 && n_ctas <= 1024,
                PPH_EINVAL, "%s: need 1 <= K <= N, Din a multiple of %d, 1 <= n_ctas <= 1024", name, per16);
    if (B == 0) return 0;
    const void* dev_view = nullptr;     // the device-side address of the mapped host allocation (equal under UVA)
    cudaError_t e = cudaHostGetDevicePointer(const_cast<void**>(&dev_view), const_cast<void*>(tokens_host), 0);
    if (e != cudaSuccess) {
        cudaGetLastError();
        set_error("%s: tokens_host is not pinned / mapped host memory (%s)", name, cudaGetErrorString(e));
        return PPH_EINVAL;
    }
    cudaFuncSetAttribute(host_rows_kernel, cudaFuncAttributePreferredSharedMemoryCarveout, (int)cudaSharedmemCarveoutMaxShared);
    host_rows_kernel<<<n_ctas, kHgThreads, 0, as_stream(stream)>>>(static_cast<const float*>(dev_view), idx32, B, N,
                                                                   Din / per16, K, static_cast<float*>(tokens_dev));
    return launch_status(name);
}

extern "C" int pph_gather_rows_host(const float* tokens_host, const int32_t* idx32, int B, int N, int Din, int K,
                                    float* tokens_dev, int n_ctas, pph_stream_t stream) {
    return gather_rows_host("pph_gather_rows_host", tokens_host, idx32, B, N, Din, K, 4, tokens_dev, n_ctas, stream);
}

extern "C" int pph_gather_rows_host_bf16tok(const uint16_t* tokens_host, const int32_t* idx32, int B, int N, int Din, int K,
                                            uint16_t* tokens_dev, int n_ctas, pph_stream_t stream) {
    return gather_rows_host("pph_gather_rows_host_bf16tok", tokens_host, idx32, B, N, Din, K, 2, tokens_dev, n_ctas, stream);
}
