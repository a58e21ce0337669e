// (a1) Foreground-token selection: head-mean of the CLS-attention scores + per-image top-K, emitted as an
// ascending index list.  Replaces topk -> sort of protopformer.py:157-158 (and its copies at :273-274 and
// tools/deit_models_attn.py:229-230).
//
// One CTA of 128 threads per image.  Rank by counting (SURVEY.md 8(d)(ii)): token n is selected iff fewer than
// K tokens beat it (strict total order: larger score first, lower index first on equal scores), so the selected
// set is emitted directly in ascending token order with ballot/popc prefixes -- no sort, no (value,index) pairs.
// HBM traffic: H*N*4 B read + K*4 (+K*8) B written per image; the kernel is latency bound (DESIGN.md).
#include <math.h>

#include "pph_common.cuh"

namespace pph {

constexpr int kSelThreads = 128;
constexpr int kSelMaxN = 1024;

__global__ void __launch_bounds__(kSelThreads)
select_topk_kernel(const float* __restrict__ scores, int H, int N, int K,
                   int32_t* __restrict__ idx32, int64_t* __restrict__ idx64) {
    __shared__ __align__(16) float s[kSelMaxN];
    __shared__ int warp_cnt[kSelThreads / 32];
    const int b = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const float* sc = scores + (size_t)b * H * N;
    const int Npad = (N + 3) & ~3;
    for (int n = tid; n < Npad; n += kSelThreads) {
        float v = -INFINITY;
        if (n < N) {
            float a = sc[n];
            for (int h = 1; h < H; ++h) a += sc[(size_t)h * N + n];
            v = H > 1 ? a / (float)H : a;      // torch.mean = sum / count
            if (v != v) v = INFINITY;          // NaN ranks first (torch.topk); with the index tie-break: a total order
        }
        s[n] = v;
    }
    __syncthreads();
    int base = 0;
    for (int n0 = 0; n0 < N; n0 += kSelThreads) {      // uniform trip count
        const int n = n0 + tid;
        bool sel = false;
        if (n < N) {
            const float v = s[n];
            const int rank = rank_by_count(reinterpret_cast<const float4*>(s), n, Npad, v);
            sel = rank < K;
        }
        const unsigned m = __ballot_sync(0xffffffffu, sel);
        if (lane == 0) warp_cnt[warp] = __popc(m);
        __syncthreads();
        int off = base;
        for (int w = 0; w < warp; ++w) off += warp_cnt[w];
        int total = 0;
        for (int w = 0; w < kSelThreads / 32; ++w) total += warp_cnt[w];
        if (sel) {
            const int pos = off + __popc(m & ((1u << lane) - 1u));
            if (pos < K) {                     // a total order selects exactly K; the guard keeps a bug inside the row
                idx32[(size_t)b * K + pos] = n;
                if (idx64) idx64[(size_t)b * K + pos] = n;
            }
        }
        base += total;
        __syncthreads();
    }
}

}  // namespace pph

extern "C" int pph_select_topk(const float* scores, int B, int H, int N, int K,
                               int32_t* idx32, int64_t* idx64, pph_stream_t stream) {
    PPH_REQUIRE(scores && idx32, PPH_EINVAL, "pph_select_topk: null pointer");
    PPH_REQUIRE(B >= 0 && H >= 1 && N >= 1 && K >= 1 && K <= N, PPH_EINVAL,
                "pph_select_topk: bad dims B=%d H=%d N=%d K=%d", B, H, N, K);
    PPH_REQUIRE(N <= pph::kSelMaxN, PPH_EUNSUP, "pph_select_topk: N=%d > %d", N, pph::kSelMaxN);
    if (B == 0) return 0;
    pph::launch_k(pph::select_topk_kernel, dim3(B), dim3(pph::kSelThreads), (size_t)(0), pph::as_stream(stream), scores, H, N, K, idx32, idx64);
    return pph::launch_status("pph_select_topk");
}
