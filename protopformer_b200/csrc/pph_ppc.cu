// (a7) PPC (prototypical part concentration) loss, forward and backward.  Replaces PPNet.get_PPC_loss + batch_cov
// (protopformer.py:249-288): ~25 ATen launches, a third topk+sort, a (B*m,196,2) grid repeat and a bmm of
// B*m*196 2x1*1x2 outer products collapse to one CTA per image.
//
// Per image b with label y, for the m prototypes p_j = y*m + j (restatement verified in SURVEY.md 8(d)(iii)):
//   d[j,k]  = relu(z2[b,k] + (p2[p_j] - 2 <Z[b,k], P[p_j]>))      recomputed in fp32 (the reference gathers it)
//   w[j,k]  = act(d[j,k]);  pos_k = (idx[b,k] / side, idx[b,k] % side);  S_j = sum_k w
//   mu_j    = sum_k w pos_k / S_j;   V_j = sum_k w (pos_k - mu_j)^2 / S_j   (per coordinate);  var_j = V_j N/(N-1)
//   L_cov   = mean_{b,j} relu((var_r + var_c)/2 - cov_thresh)
//   L_mean  = mean_{b,i,j} relu(mean_thresh - |mu_i - mu_j|) [i != j]     (diagonal zeros stay in the denominator)
//
// Layout: the image's K token rows are staged once in shared memory (row stride D+4 floats: 128-bit reads by
// consecutive tokens hit distinct bank groups), the m label-class prototype rows next to them; thread = (token,
// prototype group) for the distance slice, warp = prototype for the statistics.  HBM/L2 traffic per image:
// K*D*4 + m*D*4 + K*4 B in, m*K*4 + m*32 B out -- latency bound; all global loads are 128-bit and coalesced.
#include <math.h>

#include "pph_common.cuh"

namespace pph {

constexpr int kPpcThreads = 256;
constexpr int kPpcMaxDV = 16;     // D <= 512

__device__ __forceinline__ float block_sum_256(float v, float* red) {
    v = warp_sum(v);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    __syncthreads();
    if (lane == 0) red[warp] = v;
    __syncthreads();
    float s = 0.f;
#pragma unroll
    for (int w = 0; w < kPpcThreads / 32; ++w) s += red[w];
    return s;
}

struct PpcSmem {
    float *Prow, *Zt, *dsl, *wbuf, *st;
    int zstride;
};

__device__ __forceinline__ PpcSmem ppc_carve(float* sm, int m, int D, int K, int kc) {
    PpcSmem s;
    s.zstride = D + 4;
    s.Prow = sm;                                 // [m][D]
    s.Zt = s.Prow + m * D;                       // [kc][D+4]
    s.dsl = s.Zt + (size_t)kc * s.zstride;       // [m][K]  distances (fwd) / d loss / d distance (bwd)
    s.wbuf = s.dsl + m * K;                      // [m][K]  activations
    s.st = s.wbuf + m * K;                       // [m][8]
    return s;
}

static size_t ppc_smem_bytes(int m, int D, int K, int kc) {
    return sizeof(float) * ((size_t)m * D + (size_t)kc * (D + 4) + 2 * (size_t)m * K + 8 * (size_t)m);
}

// stage token rows [k0, k0+n) of image b into shared memory (float4, coalesced).  Thread = (row lane, float4 column);
// 8 independent loads are in flight per thread before the first shared store (one L2 latency per 8 rows).
__device__ __forceinline__ void ppc_stage_tokens(const float* __restrict__ Zb, float* Zt, int zstride, int D, int k0,
                                                 int n) {
    const int d4 = D >> 2;                              // <= 128
    const int rpp = kPpcThreads / d4;                   // rows per pass
    const int c = threadIdx.x % d4, r0 = threadIdx.x / d4;
    if (r0 >= rpp) return;
    for (int rb = r0; rb < n; rb += 8 * rpp) {
        float4 v[8];
#pragma unroll
        for (int u = 0; u < 8; ++u) {
            const int r = rb + u * rpp;
            if (r < n) v[u] = __ldg(reinterpret_cast<const float4*>(Zb + (size_t)(k0 + r) * D) + c);
        }
#pragma unroll
        for (int u = 0; u < 8; ++u) {
            const int r = rb + u * rpp;
            if (r < n) *reinterpret_cast<float4*>(Zt + (size_t)r * zstride + 4 * c) = v[u];
        }
    }
}

__global__ void __launch_bounds__(kPpcThreads)
ppc_fwd_kernel(const float* __restrict__ Zs, const float* __restrict__ z2s, const float* __restrict__ Pl,
               const float* __restrict__ p2l, const int32_t* __restrict__ idx, const int64_t* __restrict__ labels,
               int B, int K, int D, int P, int m, int N, int side, int kc, int act_fn, float eps,
               float cov_thresh, float mean_thresh,
               float* __restrict__ dslice, float* __restrict__ stats, float* partial, unsigned int* counter,
               float* __restrict__ losses) {
    extern __shared__ __align__(16) float sm[];
    const PpcSmem s = ppc_carve(sm, m, D, K, kc);
    __shared__ float red[kPpcThreads / 32];
    const int b = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nwarp = kPpcThreads / 32;
    long y = labels[b];
    if (y < 0) y = 0;
    if (y * m + m > P) y = P / m - 1;                 // out-of-range labels are clamped (the reference would raise)
    const int prow0 = (int)y * m;
    for (int i = tid; i < m * D / 4; i += kPpcThreads)
        reinterpret_cast<float4*>(s.Prow)[i] = __ldg(reinterpret_cast<const float4*>(Pl + (size_t)prow0 * D) + i);
    const float* Zb = Zs + (size_t)b * K * D;

    // distance slice: thread = (token, prototype group jg of JG); 128-bit shared reads, fp32 FMA
    const int JG = kc * 3 <= kPpcThreads ? 3 : (kc * 2 <= kPpcThreads ? 2 : 1);
    for (int k0 = 0; k0 < K; k0 += kc) {
        const int n = min(kc, K - k0);
        __syncthreads();
        ppc_stage_tokens(Zb, s.Zt, s.zstride, D, k0, n);
        __syncthreads();
        for (int t = tid; t < n * JG; t += kPpcThreads) {
            const int r = t % n, jg = t / n;
            const float4* zr = reinterpret_cast<const float4*>(s.Zt + (size_t)r * s.zstride);
            const float zz = __ldg(z2s + (size_t)b * K + k0 + r);
            for (int j = jg; j < m; j += JG) {
                const float4* pr = reinterpret_cast<const float4*>(s.Prow + (size_t)j * D);
                float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
#pragma unroll 4
                for (int c = 0; c < D / 4; ++c) {
                    const float4 z = zr[c], p = pr[c];
                    a0 = fmaf(z.x, p.x, a0); a1 = fmaf(z.y, p.y, a1); a2 = fmaf(z.z, p.z, a2); a3 = fmaf(z.w, p.w, a3);
                }
                const float dot = (a0 + a1) + (a2 + a3);
                const float d = relu_keep_nan(zz + fmaf(-2.0f, dot, __ldg(p2l + prow0 + j)));
                s.dsl[j * K + k0 + r] = d;
                s.wbuf[j * K + k0 + r] = act_of_dist(d, act_fn, eps);
                dslice[((size_t)b * m + j) * K + k0 + r] = d;
            }
        }
    }
    __syncthreads();

    // weighted mean / variance of the grid positions: one warp per prototype
    float cov_sum = 0.f;    // meaningful on lane 0 of each warp
    for (int j = warp; j < m; j += nwarp) {
        float S = 0.f, Sr = 0.f, Sc = 0.f;
        for (int k = lane; k < K; k += 32) {
            const float w = s.wbuf[j * K + k];
            const int n = __ldg(idx + (size_t)b * K + k);
            S += w;
            Sr = fmaf(w, (float)(n / side), Sr);
            Sc = fmaf(w, (float)(n % side), Sc);
        }
        S = warp_sum(S); Sr = warp_sum(Sr); Sc = warp_sum(Sc);
        const float mr = Sr / S, mc = Sc / S;
        float Vr = 0.f, Vc = 0.f;
        for (int k = lane; k < K; k += 32) {
            const float w = s.wbuf[j * K + k];
            const int n = __ldg(idx + (size_t)b * K + k);
            const float dr = (float)(n / side) - mr, dc = (float)(n % side) - mc;
            Vr = fmaf(w, dr * dr, Vr);
            Vc = fmaf(w, dc * dc, Vc);
        }
        Vr = warp_sum(Vr) / S;
        Vc = warp_sum(Vc) / S;
        const float scale = (float)N / (float)(N - 1);
        const float pre = (Vr * scale + Vc * scale) * 0.5f - cov_thresh;
        if (lane == 0) {
            float* st = s.st + j * 8;
            st[0] = S; st[1] = mr; st[2] = mc; st[3] = Vr; st[4] = Vc; st[5] = pre; st[6] = 0.f; st[7] = 0.f;
            cov_sum += relu_keep_nan(pre);
        }
    }
    const float cov_img = block_sum_256(lane == 0 ? cov_sum : 0.f, red);   // includes the barrier that publishes st[]
    for (int i = tid; i < m * 8; i += kPpcThreads) stats[(size_t)b * m * 8 + i] = s.st[i];

    float mean_sum = 0.f;
    for (int t = tid; t < m * m; t += kPpcThreads) {
        const int i = t / m, j = t - i * m;
        if (i != j) {
            const float dr = s.st[i * 8 + 1] - s.st[j * 8 + 1], dc = s.st[i * 8 + 2] - s.st[j * 8 + 2];
            mean_sum += relu_keep_nan(mean_thresh - sqrtf(dr * dr + dc * dc));
        }
    }
    const float mean_img = block_sum_256(mean_sum, red);

    // deterministic final sum: the last CTA to finish adds the per-image partials in image order
    if (tid == 0) {
        partial[2 * b] = cov_img;
        partial[2 * b + 1] = mean_img;
        __threadfence();
        const unsigned int ticket = atomicAdd(counter, 1u);
        if (ticket == (unsigned int)(B - 1)) {
            __threadfence();
            float c = 0.f, sacc = 0.f;
            for (int i = 0; i < B; ++i) {
                c += __ldcg(partial + 2 * i);
                sacc += __ldcg(partial + 2 * i + 1);
            }
            losses[0] = c / ((float)B * (float)m);
            losses[1] = sacc / ((float)B * (float)m * (float)m);
            *counter = 0u;          // ready for the next launch / graph replay
        }
    }
}

// backward.  accumulate = 0: dZs rows are overwritten, dP is expected zero-filled (atomicAdd).
//            accumulate = 1: the PPC contribution is ADDED to dZs (one CTA owns its token rows: plain
//                            read-modify-write) and atomically added to dP -- the caller has already written the
//                            similarity gradients there.
// Grid = (image, chunk of kPpcBwdTok tokens): many small CTAs instead of one serial CTA per image (latency bound).
constexpr int kPpcBwdTok = 16, kPpcBwdThreads = 128;

template <int DV>
__global__ void __launch_bounds__(kPpcBwdThreads)
ppc_bwd_kernel(const float* __restrict__ Zs, const float* __restrict__ Pl, const int32_t* __restrict__ idx,
               const int64_t* __restrict__ labels, const float* __restrict__ dslice, const float* __restrict__ stats,
               const float* __restrict__ g_losses, float g_scale_cov, float g_scale_mean,
               int B, int K, int D, int P, int m, int N, int side,
               int act_fn, float eps, float mean_thresh, int accumulate, float* __restrict__ dZs,
               float* __restrict__ dP) {
    extern __shared__ __align__(16) float sm[];
    float* Prow = sm;                         // [m][D]
    float* Zt = Prow + m * D;                 // [kPpcBwdTok][D]
    float* dd = Zt + kPpcBwdTok * D;          // [m][kPpcBwdTok]
    float* st = dd + m * kPpcBwdTok;          // [m][8]
    const int b = blockIdx.x, k0 = blockIdx.y * kPpcBwdTok, n = min(kPpcBwdTok, K - k0);
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nwarp = kPpcBwdThreads / 32;
    long y = labels[b];
    if (y < 0) y = 0;
    if (y * m + m > P) y = P / m - 1;
    const int prow0 = (int)y * m;
    for (int i = tid; i < m * D / 4; i += kPpcBwdThreads)
        reinterpret_cast<float4*>(Prow)[i] = __ldg(reinterpret_cast<const float4*>(Pl + (size_t)prow0 * D) + i);
    for (int i = tid; i < n * D / 4; i += kPpcBwdThreads)
        reinterpret_cast<float4*>(Zt)[i] = __ldg(reinterpret_cast<const float4*>(Zs + ((size_t)b * K + k0) * D) + i);
    for (int i = tid; i < m * 8; i += kPpcBwdThreads) st[i] = __ldg(stats + (size_t)b * m * 8 + i);
    __syncthreads();
    const float up_cov = g_losses ? __ldg(g_losses) * g_scale_cov : g_scale_cov;
    const float up_mean = g_losses ? __ldg(g_losses + 1) * g_scale_mean : g_scale_mean;
    const float g_cov = up_cov / ((float)B * (float)m);
    const float g_mean = up_mean / ((float)B * (float)m * (float)m);
    // d loss / d mu_i from the pairwise term (both (i,j) and (j,i) depend on mu_i)
    if (tid < m) {
        const int i = tid;
        float gr = 0.f, gcn = 0.f;
        for (int j = 0; j < m; ++j) {
            if (j == i) continue;
            const float dr = st[i * 8 + 1] - st[j * 8 + 1], dc = st[i * 8 + 2] - st[j * 8 + 2];
            const float dist = sqrtf(dr * dr + dc * dc);
            if (mean_thresh - dist > 0.0f && dist > 0.0f) {
                gr -= 2.0f * g_mean * dr / dist;
                gcn -= 2.0f * g_mean * dc / dist;
            }
        }
        st[i * 8 + 6] = gr;
        st[i * 8 + 7] = gcn;
    }
    __syncthreads();
    const float scale = (float)N / (float)(N - 1);
    for (int t = tid; t < m * n; t += kPpcBwdThreads) {
        const int j = t / n, r = t - j * n;
        const float S = st[j * 8], mr = st[j * 8 + 1], mc = st[j * 8 + 2], Vr = st[j * 8 + 3], Vc = st[j * 8 + 4];
        const float dV = st[j * 8 + 5] > 0.0f ? 0.5f * g_cov * scale : 0.0f;
        const int tok = __ldg(idx + (size_t)b * K + k0 + r);
        const float dr = (float)(tok / side) - mr, dc = (float)(tok % side) - mc;
        const float dw = (dV * ((dr * dr - Vr) + (dc * dc - Vc)) + st[j * 8 + 6] * dr + st[j * 8 + 7] * dc) / S;
        const float d = __ldg(dslice + ((size_t)b * m + j) * K + k0 + r);
        dd[j * kPpcBwdTok + r] = 2.0f * dw * dact_of_dist(d, act_fn, eps);      // factor 2 of d|z-p|^2 folded in
    }
    __syncthreads();
    // token gradient rows: one warp per token, dZ[b,k,:] (+)= sum_j dd[j,k] (Z[b,k,:] - P_j)
    for (int r = warp; r < n; r += nwarp) {
        float z[DV], acc[DV];
#pragma unroll
        for (int i = 0; i < DV; ++i) {
            z[i] = (i * 32 + lane < D) ? Zt[r * D + i * 32 + lane] : 0.f;
            acc[i] = 0.f;
        }
        for (int j = 0; j < m; ++j) {
            const float c2 = dd[j * kPpcBwdTok + r];
#pragma unroll
            for (int i = 0; i < DV; ++i)
                if (i * 32 + lane < D) acc[i] = fmaf(c2, z[i] - Prow[j * D + i * 32 + lane], acc[i]);
        }
        float* out = dZs + ((size_t)b * K + k0 + r) * D;
#pragma unroll
        for (int i = 0; i < DV; ++i)
            if (i * 32 + lane < D) out[i * 32 + lane] = accumulate ? out[i * 32 + lane] + acc[i] : acc[i];
    }
    // prototype gradient rows: one warp per label-class prototype, dP_j += sum_k dd[j,k] (P_j - Z[b,k,:])
    for (int j = warp; j < m; j += nwarp) {
        float pj[DV], acc[DV];
#pragma unroll
        for (int i = 0; i < DV; ++i) {
            pj[i] = (i * 32 + lane < D) ? Prow[j * D + i * 32 + lane] : 0.f;
            acc[i] = 0.f;
        }
        for (int r = 0; r < n; ++r) {
            const float c2 = dd[j * kPpcBwdTok + r];
#pragma unroll
            for (int i = 0; i < DV; ++i)
                if (i * 32 + lane < D) acc[i] = fmaf(c2, pj[i] - Zt[r * D + i * 32 + lane], acc[i]);
        }
#pragma unroll
        for (int i = 0; i < DV; ++i)
            if (i * 32 + lane < D) atomicAdd(dP + (size_t)(prow0 + j) * D + i * 32 + lane, acc[i]);
    }
}

template <int DV>
static int launch_ppc_bwd(dim3 grid, size_t smem, cudaStream_t st, const float* Zs, const float* Pl,
                          const int32_t* idx32, const int64_t* labels, const float* dslice, const float* stats,
                          const float* g_losses, float gs_cov, float gs_mean, int B, int K, int D, int P, int m, int N,
                          int side, int act_fn, float eps, float mean_thresh, int accumulate, float* dZs, float* dP) {
    if (smem > 48 * 1024) {
        cudaError_t e = opt_in_smem(ppc_bwd_kernel<DV>, (int)smem);
        if (e != cudaSuccess) { set_error("pph_ppc_bwd: %s", cudaGetErrorString(e)); return (int)e; }
    }
    launch_k(ppc_bwd_kernel<DV>, dim3(grid), dim3(kPpcBwdThreads), (size_t)(smem), st, Zs, Pl, idx32, labels, dslice, stats, g_losses, gs_cov, gs_mean, B, K, D, P, m, N, side, act_fn, eps, mean_thresh, accumulate, dZs, dP);
    return launch_status("pph_ppc_bwd");
}

static int ppc_check(int B, int K, int D, int P, int m, int N, int* side, int* kc, size_t* smem) {
    PPH_REQUIRE(B >= 0 && K >= 1 && D >= 4 && D % 4 == 0 && D <= 32 * kPpcMaxDV && m >= 1 && P >= m && N >= 2,
                PPH_EINVAL, "pph_ppc: bad dims B=%d K=%d D=%d P=%d m=%d N=%d (D must be a multiple of 4, <= 512)", B,
                K, D, P, m, N);
    int s = (int)lrint(sqrt((double)N));
    PPH_REQUIRE(s * s == N, PPH_EINVAL, "pph_ppc: N=%d is not a perfect square", N);
    *side = s;
    // token chunk that fits ~200 KB of shared memory next to the prototype rows and the two (m,K) slices
    int c = K;
    while (c > 1 && ppc_smem_bytes(m, D, K, c) > 200 * 1024) c = (c + 1) / 2;
    PPH_REQUIRE(ppc_smem_bytes(m, D, K, c) <= 200 * 1024, PPH_EUNSUP, "pph_ppc: m*D / m*K too large for shared memory");
    *kc = c;
    *smem = ppc_smem_bytes(m, D, K, c);
    return 0;
}

}  // namespace pph

extern "C" int pph_ppc_fwd(const float* Zs, const float* z2s, const float* Pl, const float* p2l,
                           const int32_t* idx32, const int64_t* labels,
                           int B, int K, int D, int P, int m, int N, int act_fn, float eps,
                           float cov_thresh, float mean_thresh,
                           float* dslice, float* stats, float* partial, uint32_t* counter, float* losses,
                           pph_stream_t stream) {
    using namespace pph;
    PPH_REQUIRE(Zs && z2s && Pl && p2l && idx32 && labels && dslice && stats && partial && counter && losses,
                PPH_EINVAL, "pph_ppc_fwd: null pointer");
    int side = 0, kc = 0;
    size_t smem = 0;
    int rc = ppc_check(B, K, D, P, m, N, &side, &kc, &smem);
    if (rc) return rc;
    if (B == 0) return 0;
    if (smem > 48 * 1024) {
        cudaError_t e = opt_in_smem(ppc_fwd_kernel, (int)smem);
        if (e != cudaSuccess) { set_error("pph_ppc_fwd: %s", cudaGetErrorString(e)); return (int)e; }
    }
    launch_k(ppc_fwd_kernel, dim3(B), dim3(kPpcThreads), (size_t)(smem), as_stream(stream), Zs, z2s, Pl, p2l, idx32, labels, B, K, D, P, m, N, side, kc, act_fn, eps, cov_thresh, mean_thresh, dslice, stats, partial, counter, losses);
    return launch_status("pph_ppc_fwd");
}

extern "C" int pph_ppc_bwd(const float* Zs, const float* Pl, const int32_t* idx32, const int64_t* labels,
                           const float* dslice, const float* stats, const float* g_losses,
                           float g_scale_cov, float g_scale_mean,
                           int B, int K, int D, int P, int m, int N, int act_fn, float eps,
                           float cov_thresh, float mean_thresh, int accumulate, float* dZs, float* dP,
                           pph_stream_t stream) {
    using namespace pph;
    (void)cov_thresh;
    PPH_REQUIRE(Zs && Pl && idx32 && labels && dslice && stats && dZs && dP, PPH_EINVAL, "pph_ppc_bwd: null pointer");
    int side = 0, kc = 0;
    size_t smem_fwd = 0;
    int rc = ppc_check(B, K, D, P, m, N, &side, &kc, &smem_fwd);
    if (rc) return rc;
    if (B == 0) return 0;
    const size_t smem = sizeof(float) * ((size_t)m * D + (size_t)kPpcBwdTok * D + (size_t)m * kPpcBwdTok + 8 * (size_t)m);
    PPH_REQUIRE(smem <= 200 * 1024, PPH_EUNSUP, "pph_ppc_bwd: m*D too large for shared memory");
    dim3 grid(B, ceil_div(K, kPpcBwdTok));
    cudaStream_t st = as_stream(stream);
    const int dv = ceil_div(D, 32);
#define PPH_PPC_BWD(DV) launch_ppc_bwd<DV>(grid, smem, st, Zs, Pl, idx32, labels, dslice, stats, g_losses, g_scale_cov, \
                                           g_scale_mean, B, K, D, P, m, N, side, act_fn, eps, mean_thresh, accumulate, dZs, dP)
    if (dv <= 2) return PPH_PPC_BWD(2);
    if (dv <= 6) return PPH_PPC_BWD(6);
    if (dv <= 12) return PPH_PPC_BWD(12);
    return PPH_PPC_BWD(16);
#undef PPH_PPC_BWD
}
