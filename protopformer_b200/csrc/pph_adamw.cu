// Fused AdamW for the head's parameter groups (SURVEY.md 8(f) next #3): one launch updates every trainable head
// tensor straight from the (all-reduced) flat gradient buffer.  Replaces, for the head's groups,
//   tools/create_optimizer.py:31-39  split_weights: add_on_layers (lr 3e-3, weight_decay 1e-3),
//                                    prototype_vectors / prototype_vectors_global (lr 3e-3, weight_decay args: 0.05)
//   tools/create_optimizer.py:92     optim.AdamW(parameters, weight_decay=..., eps=1e-8)   (torch decoupled AdamW)
//   tools/engine_proto.py:76-78      loss_scaler(...) -> optimizer.step()
// torch.optim.AdamW (single-tensor path) per element:
//   p *= 1 - lr * wd;  m += (g - m) * (1 - b1);  v = v * b2 + g * g * (1 - b2);
//   p -= (lr / (1 - b1^t)) * m / (sqrt(v) / sqrt(1 - b2^t) + eps)
// The step count t and the per-group (lr, weight_decay) live in DEVICE memory so that the launch can be replayed
// inside a CUDA graph while the schedule (timm cosine, main.py:402) changes the learning rates between replays.
// HBM bound: 16 B read + 12 B written per element (22.5 MB per step at the CUB shape, 805 k elements).
#include <math.h>

#include "pph_common.cuh"

namespace pph {

constexpr int kAdamMaxSeg = 8;
constexpr int kAdamThreads = 256;
constexpr int kAdamPerThread = 8;

struct AdamSegs {
    float* p[kAdamMaxSeg];
    const float* g[kAdamMaxSeg];
    float* m[kAdamMaxSeg];
    float* v[kAdamMaxSeg];
    long long n[kAdamMaxSeg];
    int block_start[kAdamMaxSeg + 1];
    int group[kAdamMaxSeg];
    int n_seg;
};

__global__ void __launch_bounds__(kAdamThreads)
adamw_kernel(const AdamSegs segs, const float* __restrict__ hyper, double beta1d, double beta2d, float eps,
             float grad_scale, int* __restrict__ step_state) {
    __shared__ float s_step_size, s_bc2_sqrt, s_decay;
    __shared__ int s_t;
    int sg = 0;
    while (sg + 1 < segs.n_seg && (int)blockIdx.x >= segs.block_start[sg + 1]) ++sg;
    if (threadIdx.x == 0) {
        const int t = *reinterpret_cast<volatile int*>(step_state) + 1;          // this update's step count
        const float lr = hyper[2 * segs.group[sg]], wd = hyper[2 * segs.group[sg] + 1];
        // bias corrections in double, as torch does in Python floats
        const double bc1 = 1.0 - pow(beta1d, (double)t), bc2 = 1.0 - pow(beta2d, (double)t);
        s_step_size = (float)((double)lr / bc1);
        s_bc2_sqrt = (float)sqrt(bc2);
        s_decay = (float)(1.0 - (double)lr * (double)wd);
        s_t = t;
    }
    __syncthreads();
    const float step_size = s_step_size, bc2_sqrt = s_bc2_sqrt, decay = s_decay;
    // scalars exactly as torch forms them: Python doubles (1 - beta) rounded once to fp32
    const float beta2 = (float)beta2d, w1 = (float)(1.0 - beta1d), w2 = (float)(1.0 - beta2d);
    float* __restrict__ P = segs.p[sg];
    const float* __restrict__ G = segs.g[sg];
    float* __restrict__ Mo = segs.m[sg];
    float* __restrict__ V = segs.v[sg];
    const long long n = segs.n[sg];
    const long long base = (long long)(blockIdx.x - segs.block_start[sg]) * (kAdamThreads * kAdamPerThread);
    float p[kAdamPerThread], g[kAdamPerThread], m[kAdamPerThread], v[kAdamPerThread];
#pragma unroll
    for (int i = 0; i < kAdamPerThread; ++i) {
        const long long e = base + i * kAdamThreads + threadIdx.x;
        if (e < n) { p[i] = P[e]; g[i] = G[e] * grad_scale; m[i] = Mo[e]; v[i] = V[e]; }
    }
#pragma unroll
    for (int i = 0; i < kAdamPerThread; ++i) {
        const long long e = base + i * kAdamThreads + threadIdx.x;
        if (e < n) {
            const float pd = p[i] * decay;
            const float mn = m[i] + w1 * (g[i] - m[i]);                 // lerp_(grad, 1 - beta1)
            const float vn = v[i] * beta2 + (w2 * g[i]) * g[i];         // mul_(beta2).addcmul_(grad, grad, 1 - beta2)
            const float denom = sqrtf(vn) / bc2_sqrt + eps;
            P[e] = pd + ((-step_size) * mn) / denom;                    // addcdiv_(exp_avg, denom, value=-step_size)
            Mo[e] = mn;
            V[e] = vn;
        }
    }
    // the last CTA to finish publishes the new step count (every CTA has read the old one before taking a ticket)
    __shared__ unsigned int s_ticket;
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) s_ticket = atomicAdd(reinterpret_cast<unsigned int*>(step_state + 1), 1u);
    __syncthreads();
    if (s_ticket == gridDim.x - 1 && threadIdx.x == 0) {
        step_state[0] = s_t;
        step_state[1] = 0;
    }
}

}  // namespace pph

extern "C" int pph_adamw_step(int n_seg, float* const* params, const float* const* grads, float* const* exp_avg,
                              float* const* exp_avg_sq, const long long* numel, const int* group,
                              const float* hyper, double beta1, double beta2, float eps, float grad_scale,
                              int* step_state, pph_stream_t stream) {
    using namespace pph;
    PPH_REQUIRE(params && grads && exp_avg && exp_avg_sq && numel && group && hyper && step_state, PPH_EINVAL,
                "pph_adamw_step: null pointer");
    PPH_REQUIRE(n_seg >= 1 && n_seg <= kAdamMaxSeg, PPH_EUNSUP, "pph_adamw_step: 1 <= n_seg <= %d (n_seg=%d)",
                kAdamMaxSeg, n_seg);
    PPH_REQUIRE(beta1 >= 0.0 && beta1 < 1.0 && beta2 >= 0.0 && beta2 < 1.0 && eps >= 0.f, PPH_EINVAL,
                "pph_adamw_step: bad betas / eps");
    AdamSegs s;
    s.n_seg = n_seg;
    int blocks = 0;
    for (int i = 0; i < kAdamMaxSeg; ++i) {
        if (i < n_seg) {
            PPH_REQUIRE(params[i] && grads[i] && exp_avg[i] && exp_avg_sq[i] && numel[i] >= 0 && group[i] >= 0 &&
                            group[i] < kAdamMaxSeg,
                        PPH_EINVAL, "pph_adamw_step: bad segment %d", i);
            s.p[i] = params[i]; s.g[i] = grads[i]; s.m[i] = exp_avg[i]; s.v[i] = exp_avg_sq[i];
            s.n[i] = numel[i]; s.group[i] = group[i];
            s.block_start[i] = blocks;
            blocks += (int)((numel[i] + kAdamThreads * kAdamPerThread - 1) / (kAdamThreads * kAdamPerThread));
        } else {
            s.p[i] = nullptr; s.g[i] = nullptr; s.m[i] = nullptr; s.v[i] = nullptr; s.n[i] = 0; s.group[i] = 0;
            s.block_start[i] = blocks;
        }
    }
    s.block_start[kAdamMaxSeg] = blocks;
    PPH_REQUIRE(blocks >= 1, PPH_EINVAL, "pph_adamw_step: nothing to update");
    launch_k(adamw_kernel, dim3(blocks), dim3(kAdamThreads), (size_t)0, as_stream(stream), s, hyper, beta1, beta2, eps,
             grad_scale, step_state);
    return launch_status("pph_adamw_step");
}
