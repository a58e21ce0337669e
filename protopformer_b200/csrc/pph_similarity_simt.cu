// (a3-a5) PPH_MODE_FP32_FMA: squared-L2 distances + similarity + max over tokens on the CUDA cores in FP32 FMA.
// This is the exact-precision mode of pph_similarity_fwd and the only one that materialises the (B,P,K) maps
// (eval aux `distances`, protopformer.py:301; push_forward `proto_acts`, :344).  The throughput path is the
// tcgen05 kernel in pph_similarity_tc.cu.
//
// d[b,p,k] = relu(z2[b,k] + (p2[p] - 2 * <Z[b,k,:], P[p,:]>))      (association of protopformer.py:214-216)
#include <math.h>

#include "pph_common.cuh"
#include "pph_sgemm.cuh"

namespace pph {

constexpr int kSimTok = 96, kSimProt = 64, kSimBK = 16, kSimThreads = 256;

__global__ void __launch_bounds__(kSimThreads)
similarity_local_simt_kernel(const float* __restrict__ Zs, const float* __restrict__ z2s,
                             const float* __restrict__ Pl, const float* __restrict__ p2l,
                             int K, int D, int P, int act_fn, float eps,
                             float* __restrict__ dmin, int32_t* __restrict__ argmin, float* __restrict__ act,
                             float* __restrict__ dist_map, float* __restrict__ act_map) {
    __shared__ __align__(16) float Zt[kSimBK][kSimTok + 4];
    __shared__ __align__(16) float Pt[kSimBK][kSimProt + 4];
    const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
    const int b = blockIdx.y, p0 = blockIdx.x * kSimProt;
    const float* Zb = Zs + (size_t)b * K * D;

    float best[4];
    int best_k[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) { best[j] = INFINITY; best_k[j] = 0x7fffffff; }

    for (int kc = 0; kc < K; kc += kSimTok) {
        float acc[6][4];
#pragma unroll
        for (int i = 0; i < 6; ++i)
#pragma unroll
            for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;
        for (int c0 = 0; c0 < D; c0 += kSimBK) {
            const int c = tid & 15, r = tid >> 4;
#pragma unroll
            for (int i = 0; i < 6; ++i) {
                const int t = kc + r + 16 * i;
                Zt[c][r + 16 * i] = (t < K && c0 + c < D) ? __ldg(Zb + (size_t)t * D + c0 + c) : 0.f;
            }
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                const int p = p0 + r + 16 * i;
                Pt[c][r + 16 * i] = (p < P && c0 + c < D) ? __ldg(Pl + (size_t)p * D + c0 + c) : 0.f;
            }
            __syncthreads();
#pragma unroll
            for (int cc = 0; cc < kSimBK; ++cc) {
                const float4 pv4 = *reinterpret_cast<const float4*>(&Pt[cc][ty * 4]);
                const float pv[4] = {pv4.x, pv4.y, pv4.z, pv4.w};
#pragma unroll
                for (int i = 0; i < 6; ++i) {
                    const float z = Zt[cc][tx + 16 * i];
#pragma unroll
                    for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(z, pv[j], acc[i][j]);
                }
            }
            __syncthreads();
        }
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int p = p0 + ty * 4 + j;
            if (p >= P) continue;
            const float p2 = __ldg(p2l + p);
#pragma unroll
            for (int i = 0; i < 6; ++i) {
                const int k = kc + tx + 16 * i;
                if (k >= K) continue;
                const float d = relu_keep_nan(__ldg(z2s + (size_t)b * K + k) + fmaf(-2.0f, acc[i][j], p2));
                if (dist_map) dist_map[((size_t)b * P + p) * K + k] = d;
                if (act_map) act_map[((size_t)b * P + p) * K + k] = act_of_dist(d, act_fn, eps);
                if (d < best[j]) { best[j] = d; best_k[j] = k; }   // ascending k within a thread: lowest index wins
            }
        }
    }
    // reduce (d, k) lexicographically over the 16 lanes that share a prototype group
#pragma unroll
    for (int j = 0; j < 4; ++j) {
#pragma unroll
        for (int o = 8; o > 0; o >>= 1) {
            const float od = __shfl_xor_sync(0xffffffffu, best[j], o);
            const int ok = __shfl_xor_sync(0xffffffffu, best_k[j], o);
            if (od < best[j] || (od == best[j] && ok < best_k[j])) { best[j] = od; best_k[j] = ok; }
        }
        const int p = p0 + ty * 4 + j;
        if (tx == 0 && p < P) {
            dmin[(size_t)b * P + p] = best[j];
            argmin[(size_t)b * P + p] = best_k[j] == 0x7fffffff ? 0 : best_k[j];   // all distances +inf / NaN: a valid row
            act[(size_t)b * P + p] = act_of_dist(best[j], act_fn, eps);
        }
    }
}

struct GlobalSimEpi {   // CLS token vs global prototypes: one "token" per image, no pooling
    const float *z2c, *p2g;
    float *dmin_g, *act_g;
    int Pg, act_fn;
    float eps;
    __device__ __forceinline__ void operator()(int b, int p, float acc, float) const {
        const float d = relu_keep_nan(__ldg(z2c + b) + fmaf(-2.0f, acc, __ldg(p2g + p)));
        dmin_g[(size_t)b * Pg + p] = d;
        act_g[(size_t)b * Pg + p] = act_of_dist(d, act_fn, eps);
    }
};

int similarity_fwd_simt(int act_fn, float eps, int B, int K, int D, int P, int Pg,
                        const float* Zs, const float* Zc, const float* z2s, const float* z2c,
                        const float* Pl, const float* Pgl, const float* p2l, const float* p2g,
                        float* dmin_l, int32_t* argmin_l, float* act_l, float* dmin_g, float* act_g,
                        float* dist_map, float* act_map, cudaStream_t st) {
    if (P > 0) {
        dim3 grid(ceil_div(P, kSimProt), B);
        launch_k(similarity_local_simt_kernel, dim3(grid), dim3(kSimThreads), (size_t)(0), st, Zs, z2s, Pl, p2l, K, D, P, act_fn, eps, dmin_l, argmin_l, act_l, dist_map, act_map);
        int rc = launch_status("pph_similarity_fwd(fp32 local)");
        if (rc) return rc;
    }
    if (Pg > 0) {
        StridedOp<true> a{Zc, B, D, 1};
        StridedOp<true> bop{Pgl, Pg, D, 1};
        GlobalSimEpi epi{z2c, p2g, dmin_g, act_g, Pg, act_fn, eps};
        launch_sgemm<false>(B, Pg, D, 1, a, bop, epi, st);
        int rc = launch_status("pph_similarity_fwd(fp32 global)");
        if (rc) return rc;
    }
    return 0;
}

}  // namespace pph
