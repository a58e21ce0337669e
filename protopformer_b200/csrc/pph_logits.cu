// (a6) prototype-to-class last layers + global/local combine (protopformer.py:297-300, 314-316) and the first
// step of their backward, collapsed with the similarity derivative into one scalar per (image, prototype).
// The last layers are frozen in the reference (protopformer.py:130-131); a caller that unfreezes them gets their weight
// gradients from pph_last_layer_wgrad (bottom of this file).
//
// Both are skinny FP32 contractions (B x C x (P+Pg) with B = 64): too small for a tensor-core tile grid, so they are
// laid out for L2 traffic and determinism instead:
//   forward : CTA = 8 images x 8 classes, the 256 threads split the prototype axis (coalesced row reads), 64
//             register accumulators per thread, one block reduction -> every logit has ONE writer (deterministic).
//   backward: transposed product G^T = W^T * upstream^T on tcgen05 through the manual-fill GEMM (pph_tcgemm.cuh).
#include "pph_common.cuh"
#include "pph_sgemm.cuh"
#include "pph_tcgemm.cuh"

namespace pph {

constexpr int kLogThreads = 256;
constexpr int kLogTB = 8, kLogTC = 8;

__global__ void __launch_bounds__(kLogThreads)
logits_fwd_kernel(const float* __restrict__ act_l, const float* __restrict__ act_g, const float* __restrict__ Wl,
                  const float* __restrict__ Wg, int B, int P, int Pg, int C, float gc,
                  float* __restrict__ logits, float* __restrict__ logits_g, float* __restrict__ logits_l) {
    pdl_sync();
    __shared__ float red[kLogThreads / 32][kLogTB * kLogTC];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int b0 = blockIdx.y * kLogTB, c0 = blockIdx.x * kLogTC;
    float res[2] = {0.f, 0.f};      // this thread's (b,c) output: local, global   (thread tid < 64 owns output tid)
    for (int branch = 0; branch < 2; ++branch) {
        const float* A = branch ? act_g : act_l;
        const float* W = branch ? Wg : Wl;
        const int Kd = branch ? Pg : P;
        float acc[kLogTB][kLogTC];
#pragma unroll
        for (int i = 0; i < kLogTB; ++i)
#pragma unroll
            for (int j = 0; j < kLogTC; ++j) acc[i][j] = 0.f;
        for (int p = tid; p < Kd; p += kLogThreads) {
            float a[kLogTB], w[kLogTC];
#pragma unroll
            for (int i = 0; i < kLogTB; ++i) a[i] = (b0 + i < B) ? __ldg(A + (size_t)(b0 + i) * Kd + p) : 0.f;
#pragma unroll
            for (int j = 0; j < kLogTC; ++j) w[j] = (c0 + j < C) ? __ldg(W + (size_t)(c0 + j) * Kd + p) : 0.f;
#pragma unroll
            for (int i = 0; i < kLogTB; ++i)
#pragma unroll
                for (int j = 0; j < kLogTC; ++j) acc[i][j] = fmaf(a[i], w[j], acc[i][j]);
        }
        // block reduction of the 64 accumulators: warp shuffles, then a fixed-order sum over the 8 warps
#pragma unroll
        for (int i = 0; i < kLogTB; ++i)
#pragma unroll
            for (int j = 0; j < kLogTC; ++j) {
                const float v = warp_sum(acc[i][j]);
                if (lane == 0) red[warp][i * kLogTC + j] = v;
            }
        __syncthreads();
        if (tid < kLogTB * kLogTC) {
            float s = 0.f;
#pragma unroll
            for (int w = 0; w < kLogThreads / 32; ++w) s += red[w][tid];
            res[branch] = s;
        }
        __syncthreads();
    }
    if (tid < kLogTB * kLogTC) {
        const int b = b0 + tid / kLogTC, c = c0 + tid % kLogTC;
        if (b < B && c < C) {
            const size_t o = (size_t)b * C + c;
            logits_l[o] = res[0];
            logits_g[o] = res[1];
            logits[o] = gc * res[1] + (1.0f - gc) * res[0];
        }
    }
}

// ---- backward on tcgen05 (pph_tcgemm.cuh): G^T[p, b] = sum_c W[c,p] * up[b,c], rows = local prototypes (padded to a
// 128 multiple) followed by the global ones, columns = images, contraction over the C classes (zero padded to 64).
// 32 CTAs at the CUB shape instead of a latency-bound CUDA-core tile loop; the epilogue applies the similarity
// derivative and writes g[b,p] directly (thread = prototype: loads and stores are coalesced without a transpose).
struct LbAOp {      // (row = m -> (branch, p), k = c) -> W[c, p]; consecutive lanes = consecutive prototypes
    static constexpr bool kContigK = false;
    const float *Wl, *Wg;
    int P, Plpad, Pg, C;
    __device__ __forceinline__ void load8(int m, int c0, float (&v)[8]) const {
        const bool global = m >= Plpad;
        const int p = global ? m - Plpad : m, np = global ? Pg : P;
        const float* W = global ? Wg : Wl;
#pragma unroll
        for (int i = 0; i < 8; ++i) v[i] = (p < np && c0 + i < C) ? __ldg(W + (size_t)(c0 + i) * np + p) : 0.f;
    }
};
struct LbBOp {      // (row = b, k = c) -> upstream gradient of the branch this CTA's rows belong to
    static constexpr bool kContigK = true;
    const float *dlogits, *dlogits_g, *dlogits_l;
    int B, C, Plpad;
    float gc;
    __device__ __forceinline__ void load8(int b, int c0, float (&v)[8]) const {
        const bool global = (int)blockIdx.x * kTgBM >= Plpad;
        const float coef = global ? gc : 1.0f - gc;
        const float* extra = global ? dlogits_g : dlogits_l;
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            float x = 0.f;
            if (b < B && c0 + i < C) {
                const size_t o = (size_t)b * C + c0 + i;
                x = coef * __ldg(dlogits + o);
                if (extra) x += __ldg(extra + o);
            }
            v[i] = x;
        }
    }
};
struct LbEpi {
    static constexpr bool kDirect = true;
    const float *dmin_l, *dmin_g;
    float *g_l, *g_g;
    int B, P, Plpad, Pg, act_fn;
    float eps;
    struct State { int dummy; };
    __device__ __forceinline__ void init(State& s) const { s.dummy = 0; }
    __device__ __forceinline__ void row_ptrs(int, void* (&)[3]) const {}
    __device__ __forceinline__ void transform(State&, int m, int n0, uint32_t (&acc)[32]) const {
        const bool global = m >= Plpad;
        const int p = global ? m - Plpad : m, np = global ? Pg : P;
        if (p >= np) return;
        const float* dmin = global ? dmin_g : dmin_l;
        float* g = global ? g_g : g_l;
#pragma unroll
        for (int j = 0; j < 32; ++j) {
            const int b = n0 + j;
            if (b < B) {
                const size_t o = (size_t)b * np + p;
                g[o] = __uint_as_float(acc[j]) * dact_of_dist(__ldg(dmin + o), act_fn, eps);
            }
        }
    }
    __device__ __forceinline__ void store2(void* const*, int, float, float) const {}
    __device__ __forceinline__ void finish(State&, int, int, int, float*, bool) const {}
};

// ---- backward on CUDA cores, exact FP32 FMA: g[b,p] = (sum_c up[b,c] W[c,p]) * act'(dmin[b,p]).  The tcgen05 version above
// rounds the upstream gradient to bf16 hi + lo (2^-17 relative per element); the CLS-token gradient then takes
// Z * sum_p g - sum_p g P, a difference of two sums that nearly cancel, and the rounding came out as 3.5e-4 of the largest
// token-gradient entry on the CLS rows (scripts/measure_tolerances.py).  This kernel is what the autograd path uses; the
// graphed step computes the same product in FP32 inside pph_head_mid.  Thread = prototype (coalesced W rows), 8 images per
// CTA in registers, the upstream rows of those images in shared memory.
constexpr int kLbfTB = 8, kLbfThreads = 256;

__global__ void __launch_bounds__(kLbfThreads)
logits_bwd_fma_kernel(const float* __restrict__ dlogits, const float* __restrict__ dlogits_g, const float* __restrict__ dlogits_l,
                      const float* __restrict__ Wl, const float* __restrict__ Wg, const float* __restrict__ dmin_l,
                      const float* __restrict__ dmin_g, int B, int P, int Pg, int C, int nbl, float gc, int act_fn, float eps,
                      float* __restrict__ g_l, float* __restrict__ g_g) {
    pdl_sync();
    extern __shared__ float up[];                      // [kLbfTB][C]
    const bool global = (int)blockIdx.x >= nbl;
    const int p = ((int)blockIdx.x - (global ? nbl : 0)) * kLbfThreads + threadIdx.x;
    const int np = global ? Pg : P;
    const float* W = global ? Wg : Wl;
    const float* extra = global ? dlogits_g : dlogits_l;
    const float coef = global ? gc : 1.0f - gc;
    const int b0 = blockIdx.y * kLbfTB;
    for (int i = threadIdx.x; i < kLbfTB * C; i += kLbfThreads) {
        const int bi = i / C, c = i - bi * C;
        float x = 0.f;
        if (b0 + bi < B) {
            const size_t o = (size_t)(b0 + bi) * C + c;
            x = coef * __ldg(dlogits + o);
            if (extra) x += __ldg(extra + o);
        }
        up[i] = x;
    }
    __syncthreads();
    if (p >= np) return;
    float acc[kLbfTB];
#pragma unroll
    for (int i = 0; i < kLbfTB; ++i) acc[i] = 0.f;
#pragma unroll 8
    for (int c = 0; c < C; ++c) {
        const float w = __ldg(W + (size_t)c * np + p);
#pragma unroll
        for (int i = 0; i < kLbfTB; ++i) acc[i] = fmaf(up[i * C + c], w, acc[i]);
    }
    const float* dmin = global ? dmin_g : dmin_l;
    float* g = global ? g_g : g_l;
#pragma unroll
    for (int i = 0; i < kLbfTB; ++i)
        if (b0 + i < B) {
            const size_t o = (size_t)(b0 + i) * np + p;
            g[o] = acc[i] * dact_of_dist(__ldg(dmin + o), act_fn, eps);
        }
}

// ---- last-layer weight gradients: dW[c,p] = sum_b (coef dlogits[b,c] + extra[b,c]) act[b,p], coef = 1-gc (local) | gc
// (global).  ONE FP32 tile GEMM (pph_sgemm.cuh) over both layers: rows = classes, columns [0, nl) the local prototypes
// (nl = P rounded up to the 64-wide column tile, so each CTA belongs to one layer), [nl, nl + Pg) the global ones,
// contraction over the B images NOT split -> every entry is one fixed-order sum, no atomics (bit-reproducible).
// Skinny-K (K = B) and bounded by the 4 C (P+Pg) bytes of output.
struct LwAOp {      // (row = c, k = b) -> upstream gradient of the layer this CTA's columns belong to
    static constexpr bool kContigK = false;
    const float *dlogits, *dlogits_g, *dlogits_l;
    int C, nl;
    float gc;
    __device__ __forceinline__ float operator()(int c, int b) const {
        if (c >= C) return 0.f;
        const bool global = (int)blockIdx.x * kGemmBN >= nl;
        const float* extra = global ? dlogits_g : dlogits_l;
        const size_t o = (size_t)b * C + c;
        float x = (global ? gc : 1.0f - gc) * __ldg(dlogits + o);
        if (extra) x += __ldg(extra + o);
        return x;
    }
};
// ng = Pg when dWg is computed, else 0: the loader's tail columns past the last requested one never touch act_g (which
// may then be NULL)
struct LwBOp {      // (row = column n, k = b) -> act[b, p]; consecutive columns are consecutive prototypes
    static constexpr bool kContigK = false;
    const float *act_l, *act_g;
    int P, Pg, ng, nl;
    __device__ __forceinline__ float operator()(int n, int b) const {
        const bool global = n >= nl;
        const int p = global ? n - nl : n;
        if (p >= (global ? ng : P)) return 0.f;
        return __ldg((global ? act_g : act_l) + (size_t)b * (global ? Pg : P) + p);
    }
};
struct LwEpi {
    float *dWl, *dWg;
    int P, Pg, ng, nl;
    __device__ __forceinline__ void operator()(int c, int n, float acc, float) const {
        const bool global = n >= nl;
        const int p = global ? n - nl : n;
        if (p < (global ? ng : P)) (global ? dWg : dWl)[(size_t)c * (global ? Pg : P) + p] = acc;
    }
};

}  // namespace pph

extern "C" int pph_logits_fwd(const float* act_l, const float* act_g, const float* Wl, const float* Wg,
                              int B, int P, int Pg, int C, float global_coe,
                              float* logits, float* logits_g, float* logits_l, pph_stream_t stream) {
    using namespace pph;
    PPH_REQUIRE(act_l && Wl && logits && logits_g && logits_l && (Pg == 0 || (act_g && Wg)), PPH_EINVAL,
                "pph_logits_fwd: null pointer");
    PPH_REQUIRE(B >= 0 && P >= 1 && Pg >= 0 && C >= 1, PPH_EINVAL, "pph_logits_fwd: bad dims");
    if (B == 0) return 0;
    dim3 grid(ceil_div(C, kLogTC), ceil_div(B, kLogTB));
    launch_k(logits_fwd_kernel, dim3(grid), dim3(kLogThreads), (size_t)(0), as_stream(stream), act_l, act_g, Wl, Wg, B, P, Pg, C, global_coe, logits, logits_g, logits_l);
    return launch_status("pph_logits_fwd");
}

extern "C" int pph_logits_bwd(const float* dlogits, const float* dlogits_g, const float* dlogits_l,
                              const float* Wl, const float* Wg, const float* dmin_l, const float* dmin_g,
                              int B, int P, int Pg, int C, float global_coe, int act_fn, float eps,
                              float* g_l, float* g_g, pph_stream_t stream) {
    using namespace pph;
    PPH_REQUIRE(dlogits && Wl && dmin_l && g_l && (Pg == 0 || (Wg && dmin_g && g_g)), PPH_EINVAL,
                "pph_logits_bwd: null pointer");
    PPH_REQUIRE(B >= 0 && P >= 1 && Pg >= 0 && C >= 1, PPH_EINVAL, "pph_logits_bwd: bad dims");
    if (B == 0) return 0;
    if (option(kOptLogitsBwd) != 1 && (size_t)kLbfTB * C * sizeof(float) <= 48 * 1024) {      // default: exact FP32 FMA
        const int nbl = ceil_div(P, kLbfThreads), nbg = Pg > 0 ? ceil_div(Pg, kLbfThreads) : 0;
        launch_k(logits_bwd_fma_kernel, dim3(nbl + nbg, ceil_div(B, kLbfTB)), dim3(kLbfThreads), sizeof(float) * kLbfTB * C,
                 as_stream(stream), dlogits, dlogits_g, dlogits_l, Wl, Wg, dmin_l, dmin_g, B, P, Pg, C, nbl, global_coe, act_fn,
                 eps, g_l, g_g);
        return launch_status("pph_logits_bwd");
    }
    const int Plpad = ceil_div(P, kTgBM) * kTgBM;
    LbAOp a{Wl, Wg, P, Plpad, Pg, C};
    LbBOp b{dlogits, dlogits_g, dlogits_l, B, C, Plpad, global_coe};
    LbEpi e{dmin_l, dmin_g, g_l, g_g, B, P, Plpad, Pg, act_fn, eps};
    const int N = ceil_div(B, 2) * 2;           // the kernel walks columns in pairs
    return launch_tcgemm(Plpad + Pg, N, C, tcgemm_pick_bn(N), 1, a, b, e, as_stream(stream), "pph_logits_bwd(tcgen05)");
}

extern "C" int pph_last_layer_wgrad(const float* dlogits, const float* dlogits_g, const float* dlogits_l,
                                    const float* act_l, const float* act_g, int B, int P, int Pg, int C, float global_coe,
                                    float* dWl, float* dWg, pph_stream_t stream) {
    using namespace pph;
    PPH_REQUIRE(B >= 1 && P >= 1 && Pg >= 0 && C >= 1, PPH_EINVAL, "pph_last_layer_wgrad: bad dims");
    if (Pg == 0) dWg = nullptr;                  // no global layer: nothing to write
    PPH_REQUIRE((!dWl && !dWg) || dlogits, PPH_EINVAL, "pph_last_layer_wgrad: null pointer (dlogits)");
    PPH_REQUIRE(!dWl || act_l, PPH_EINVAL, "pph_last_layer_wgrad: null pointer (act_l for dWl)");
    PPH_REQUIRE(!dWg || act_g, PPH_EINVAL, "pph_last_layer_wgrad: null pointer (act_g for dWg)");
    if (!dWl && !dWg) return 0;
    const int nl = dWl ? (dWg ? ceil_div(P, kGemmBN) * kGemmBN : P) : 0;
    const int ng = dWg ? Pg : 0;
    LwAOp a{dlogits, dlogits_g, dlogits_l, C, nl, global_coe};
    LwBOp b{act_l, act_g, P, Pg, ng, nl};
    LwEpi e{dWl, dWg, P, Pg, ng, nl};
    // maximum shared-memory carve-out, as every kernel of the training step asks for (pph_common.cuh, opt_in_smem): this
    // launch runs on a branch beside the step's co-resident kernels
    const cudaError_t err = opt_in_smem(sgemm_kernel<false, LwAOp, LwBOp, LwEpi>, 0);
    PPH_REQUIRE(err == cudaSuccess, (int)err, "pph_last_layer_wgrad: %s", cudaGetErrorString(err));
    launch_sgemm<false>(C, nl + ng, B, 1, a, b, e, as_stream(stream));
    return launch_status("pph_last_layer_wgrad");
}
