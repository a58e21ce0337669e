// Loss tail of the training step (SURVEY.md 8(f) next #3, the part adjacent to the head): cross-entropy on the
// logits (engine_proto.py:51, criterion = CrossEntropyLoss, main.py:390), the weighted sum with the two PPC losses
// (engine_proto.py:61-64) and d(loss)/d(logits), in one launch and without a host round trip.
//   ce      = mean_b (logsumexp(logits[b,:]) - logits[b,label_b])
//   total   = ce + cov_coe * ppc[0] + mean_coe * ppc[1]
//   dlogits = (softmax(logits[b,:]) - onehot(label_b)) / B * upstream
// One warp per image; the per-image losses are summed in image order by the last CTA (deterministic).
#include <math.h>

#include "pph_common.cuh"

namespace pph {

__global__ void __launch_bounds__(256)
loss_tail_kernel(const float* __restrict__ logits, const int64_t* __restrict__ labels, const float* __restrict__ ppc,
                 float cov_coe, float mean_coe, float upstream, int B, int C, float* partial, unsigned int* counter,
                 float* __restrict__ out, float* __restrict__ dlogits) {
    const int b = blockIdx.x * 8 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    __shared__ unsigned int s_ticket;
    if (b < B) {
        const float* row = logits + (size_t)b * C;
        float mx = -INFINITY;
        for (int c = lane; c < C; c += 32) mx = fmaxf(mx, __ldg(row + c));
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
        float se = 0.f;
        for (int c = lane; c < C; c += 32) se += expf(__ldg(row + c) - mx);
        se = warp_sum(se);
        long y = labels[b];
        if (y < 0) y = 0;
        if (y >= C) y = C - 1;
        const float lse = logf(se) + mx;
        if (dlogits) {
            const float s = upstream / (float)B;
            for (int c = lane; c < C; c += 32) {
                const float p = expf(__ldg(row + c) - mx) / se;
                dlogits[(size_t)b * C + c] = (p - (c == (int)y ? 1.0f : 0.0f)) * s;
            }
        }
        if (lane == 0) partial[b] = lse - __ldg(row + y);
    }
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) s_ticket = atomicAdd(counter, 1u);
    __syncthreads();
    if (s_ticket == gridDim.x - 1 && threadIdx.x == 0) {
        __threadfence();
        float ce = 0.f;
        for (int i = 0; i < B; ++i) ce += __ldcg(partial + i);
        ce /= (float)B;
        const float cov = ppc ? __ldg(ppc) : 0.f, mean = ppc ? __ldg(ppc + 1) : 0.f;
        out[0] = ce + cov_coe * cov + mean_coe * mean;
        out[1] = ce;
        out[2] = cov;
        out[3] = mean;
        *counter = 0u;
    }
}

// total = ce + cov_coe * ppc[0] + mean_coe * ppc[1] from a cross-entropy computed WITHOUT the PPC terms: lets the loss
// tail (and with it the whole last-layer backward) start before the PPC loss has finished on its own stream.
__global__ void loss_combine_kernel(const float* __restrict__ ce_losses, const float* __restrict__ ppc, float cov_coe,
                                    float mean_coe, float* __restrict__ out) {
    if (threadIdx.x == 0 && blockIdx.x == 0) {
        const float ce = ce_losses[1], cov = ppc ? ppc[0] : 0.f, mean = ppc ? ppc[1] : 0.f;
        out[0] = ce + cov_coe * cov + mean_coe * mean;
        out[1] = ce;
        out[2] = cov;
        out[3] = mean;
    }
}

}  // namespace pph

extern "C" int pph_loss_combine(const float* ce_losses, const float* ppc_losses, float cov_coe, float mean_coe,
                                float* out_losses, pph_stream_t stream) {
    using namespace pph;
    PPH_REQUIRE(ce_losses && out_losses, PPH_EINVAL, "pph_loss_combine: null pointer");
    launch_k(loss_combine_kernel, dim3(1), dim3(32), (size_t)0, as_stream(stream), ce_losses, ppc_losses, cov_coe, mean_coe,
             out_losses);
    return launch_status("pph_loss_combine");
}

extern "C" int pph_loss_tail(const float* logits, const int64_t* labels, const float* ppc_losses,
                             float cov_coe, float mean_coe, float upstream, int B, int C,
                             float* partial, uint32_t* counter, float* out_losses, float* dlogits,
                             pph_stream_t stream) {
    using namespace pph;
    PPH_REQUIRE(logits && labels && partial && counter && out_losses, PPH_EINVAL, "pph_loss_tail: null pointer");
    PPH_REQUIRE(B >= 1 && C >= 1, PPH_EINVAL, "pph_loss_tail: bad dims B=%d C=%d", B, C);
    launch_k(loss_tail_kernel, dim3(ceil_div(B, 8)), dim3(256), (size_t)(0), as_stream(stream), logits, labels, ppc_losses, cov_coe, mean_coe, upstream, B, C, partial, counter, out_losses, dlogits);
    return launch_status("pph_loss_tail");
}
