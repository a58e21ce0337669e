// Class-row activation maps on the original token grid (SURVEY.md 8(f) next #4): what the interpretability /
// visualisation tools extract from the materialised (B,P,h,w) map, without materialising it.  Replaces
//   eval_interpretability.py:195-203   push_forward -> gather of the m prototypes of each image's label
//   eval_interpretability.py:214-225   scatter of the h*w activations to the side x side grid of ALL tokens (zeros
//                                      where a token was pruned); main_visualize.py:343-388 does the same per image
// For image b with label y: rows p = y*m .. y*m+m-1; maps[b, q, idx[b,k]] = act(relu(|z_k|^2 + (|p|^2 - 2 z_k.p)))
// (the association of protopformer.py:214-216), every other grid cell 0.
// One CTA per image: 648 KB/image of map traffic become m*N*4 = 7.8 KB; latency bound (eval-time tool path).
#include <math.h>
#include <stdlib.h>

#include "pph_common.cuh"

namespace pph {

constexpr int kCmThreads = 256;

__global__ void __launch_bounds__(kCmThreads)
class_maps_kernel(const float* __restrict__ Zs, const float* __restrict__ z2s, const float* __restrict__ Pl,
                  const float* __restrict__ p2l, const int32_t* __restrict__ idx, const int64_t* __restrict__ labels,
                  int K, int D, int P, int m, int N, int act_fn, float eps, float* __restrict__ maps) {
    const int b = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    float* out = maps + (size_t)b * m * N;
    for (int i = tid; i < m * N; i += kCmThreads) out[i] = 0.0f;
    __syncthreads();                                   // the scatter below must land on the cleared grid
    long y = labels[b];
    const int C = P / m;
    if (y < 0) y = 0;
    if (y >= C) y = C - 1;
    // warp = one (prototype q, token k) pair: lane-strided dot product over D, fixed shuffle tree
    for (int pair = warp; pair < m * K; pair += kCmThreads / 32) {
        const int q = pair / K, k = pair - q * K;
        const int p = (int)y * m + q;
        const float* z = Zs + ((size_t)b * K + k) * D;
        const float* pr = Pl + (size_t)p * D;
        float s = 0.f;
        for (int d = lane; d < D; d += 32) s = fmaf(z[d], pr[d], s);
        s = warp_sum(s);
        if (lane == 0) {
            const float dist = relu_keep_nan(z2s[(size_t)b * K + k] + (p2l[p] - 2.0f * s));
            const int n = idx[(size_t)b * K + k];
            if (n >= 0 && n < N) out[(size_t)q * N + n] = act_of_dist(dist, act_fn, eps);
        }
    }
}

}  // namespace pph

extern "C" int pph_class_maps(const float* Zs, const float* z2s, const float* Pl, const float* p2l,
                              const int32_t* idx32, const int64_t* labels, int B, int K, int D, int P, int m, int N,
                              int act_fn, float eps, float* maps, pph_stream_t stream) {
    using namespace pph;
    PPH_REQUIRE(Zs && z2s && Pl && p2l && idx32 && labels && maps, PPH_EINVAL, "pph_class_maps: null pointer");
    PPH_REQUIRE(B >= 0 && K >= 1 && D >= 1 && m >= 1 && P >= m && P % m == 0 && N >= K, PPH_EINVAL,
                "pph_class_maps: bad dims B=%d K=%d D=%d P=%d m=%d N=%d", B, K, D, P, m, N);
    PPH_REQUIRE(act_fn == PPH_ACT_LOG || act_fn == PPH_ACT_LINEAR, PPH_EINVAL, "pph_class_maps: act_fn %d", act_fn);
    if (B == 0) return 0;
    launch_k(class_maps_kernel, dim3(B), dim3(kCmThreads), (size_t)0, as_stream(stream), Zs, z2s, Pl, p2l, idx32, labels,
             K, D, P, m, N, act_fn, eps, maps);
    return launch_status("pph_class_maps");
}
