// (a8, part 2) Backward of max-pool + log-similarity + squared-L2 distance in its argmin-routed (sparse) form,
// SURVEY.md 8(d)(iv).  Autograd of protopformer.py:201-247 would mirror ~10 passes over the (B,P,K) map; here the
// upstream gradient is one scalar g[b,p] placed at token argmin[b,p]:
//   dPl[p,:]   = 2 (Pl[p,:] sum_b g[b,p] - sum_b g[b,p] Zs[b,argmin[b,p],:])                      proto_grad_kernel
//   dZs[b,k,:] = 2 (Zs[b,k,:] sum_{p in bin(b,k)} g[b,p] - sum_{p in bin(b,k)} g[b,p] Pl[p,:])     token_grad_kernel
//   dPg, dZc   : same with one token per image (dense)                               proto_grad_kernel / cls_grad_kernel
// Byte-bound on L2: every (b,p) pair moves one D-float row twice (2*B*P*D*4 B = 197 MB at the CUB shape, B = 64).
// The gather kernels are one warp per output row with 8 independent 128B-line row loads in flight per lane group.
//   bin_tokens_kernel : per image, stable counting sort of the prototypes by argmin token (one warp, match.any) ->
//                       deterministic bins, so every gradient row is summed in a fixed order (bit-reproducible).
#include "pph_common.cuh"
#include "pph_bins.cuh"
#include "pph_step2.cuh"

namespace pph {

__global__ void __launch_bounds__(256)
bin_tokens_kernel(int4* __restrict__ item_desc, const int32_t* __restrict__ argmin_l, int K, int P, int32_t* __restrict__ bin_start,
                  int32_t* __restrict__ item_start, int32_t* __restrict__ bin_list) {
    extern __shared__ int smi[];
    bin_tokens_body<false>(blockIdx.x, argmin_l, K, P, bin_start, item_start, bin_list, smi, item_desc);
}

// Extras of the fused training step (pph_similarity_bwd_fused): per-image PPC prototype rows summed over the images of
// a class in image order (class lists from pph_head_mid), and token-side outputs written as the pre-activation gradient
// dpre = dZ * Z * (1 - Z) that pph_addon_bwd3 consumes.
struct BwdExtras {
    const float* dP_img;            // [B][m][D] or nullptr
    const int32_t *cls_start, *cls_order;
    int m, dpre_out;
};

// ---- gather kernels (templated on DV = ceil(D / 32) register slots per lane) ---------------------------------------
template <int DV, bool FULL>
__device__ __forceinline__ void
proto_grad_body(int vb, const float* __restrict__ g_l, const float* __restrict__ g_g, const int32_t* __restrict__ argmin_l,
                const float* __restrict__ Zs, const float* __restrict__ Zc, const float* __restrict__ Pl,
                const float* __restrict__ Pgl, int B, int K, int D, int P, int Pg, const float* __restrict__ add_dPl,
                float* __restrict__ dPl, float* __restrict__ dPg, const BwdExtras& ex) {
    const int row = vb * 8 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (row >= P + Pg) return;
    const bool global = row >= P;
    const int p = global ? row - P : row;
    const int np = global ? Pg : P;
    const float* g = global ? g_g : g_l;
    float acc[DV];
#pragma unroll
    for (int i = 0; i < DV; ++i) acc[i] = 0.f;
    float gsum = 0.f;
    for (int b0 = 0; b0 < B; b0 += 32) {
        const int bl = b0 + lane;
        const float gv = bl < B ? __ldg(g + (size_t)bl * np + p) : 0.f;
        const int av = (!global && bl < B) ? __ldg(argmin_l + (size_t)bl * P + p) : 0;
        const int cnt = min(32, B - b0);
        for (int t0 = 0; t0 < cnt; t0 += 8) {
            float gg[8];
            const float* zr[8];
#pragma unroll
            for (int u = 0; u < 8; ++u) {
                const int t = t0 + u;                                   // shuffles stay warp-uniform; masked by gg = 0
                gg[u] = __shfl_sync(0xffffffffu, gv, t & 31);
                const int aa = __shfl_sync(0xffffffffu, av, t & 31);
                const int bb = min(b0 + t, B - 1);
                if (t >= cnt) gg[u] = 0.f;
                zr[u] = global ? Zc + (size_t)bb * D : Zs + ((size_t)bb * K + aa) * D;
            }
            float v[8][DV];
#pragma unroll
            for (int u = 0; u < 8; ++u)
#pragma unroll
                for (int i = 0; i < DV; ++i) v[u][i] = (FULL || i * 32 + lane < D) ? __ldg(zr[u] + i * 32 + lane) : 0.f;
#pragma unroll
            for (int u = 0; u < 8; ++u) {
                gsum += gg[u];
#pragma unroll
                for (int i = 0; i < DV; ++i) acc[i] = fmaf(gg[u], v[u][i], acc[i]);
            }
        }
    }
    const float* pr = (global ? Pgl : Pl) + (size_t)p * D;
    float* out = (global ? dPg : dPl) + (size_t)p * D;
    const float* add = (!global && add_dPl) ? add_dPl + (size_t)p * D : nullptr;      // e.g. the PPC-loss contribution
    int c0 = 0, c1 = 0, jj = 0;
    if (!global && ex.dP_img) {
        const int cls = p / ex.m;
        jj = p - cls * ex.m;
        c0 = __ldg(ex.cls_start + cls);
        c1 = __ldg(ex.cls_start + cls + 1);
    }
#pragma unroll
    for (int i = 0; i < DV; ++i)
        if (FULL || i * 32 + lane < D) {
            float r = 2.0f * (__ldg(pr + i * 32 + lane) * gsum - acc[i]) + (add ? __ldg(add + i * 32 + lane) : 0.f);
            for (int c = c0; c < c1; ++c)          // PPC rows of this prototype's class, image order: deterministic
                r += __ldg(ex.dP_img + ((size_t)__ldg(ex.cls_order + c) * ex.m + jj) * D + i * 32 + lane);
            out[i * 32 + lane] = r;
        }
}

// One warp per work item = (image, token, chunk of <= kBinChunk bin entries).  Single-chunk bins write their row
// directly; multi-chunk bins (skewed argmin distributions put hundreds of prototypes on one token) write partials
// and the last warp to finish adds them in chunk order -> balanced AND deterministic.
template <int DV, bool FULL>
__device__ __forceinline__ void
token_grad_body(int vb, const float* __restrict__ g_l, const int4* __restrict__ item_desc, const int32_t* __restrict__ bin_list,
                const float* __restrict__ Zs, const float* __restrict__ Pl, int B, int K, int D, int P,
                int items_per_image, float* part, float* part_gsum, unsigned int* counters,
                const float* __restrict__ add_dZs, float* __restrict__ dZs, const BwdExtras& ex) {
    const int gw = vb * 8 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    const int b = gw / items_per_image, item = gw - b * items_per_image;
    if (b >= B) return;
    // one 16-byte descriptor per work item (written with the bins): token, entry range, chunk count | chunk << 16
    const int4 dsc = __ldg(item_desc + (size_t)b * items_per_image + item);
    if (dsc.x < 0) return;
    const int k = dsc.x, e0 = dsc.y, e1 = dsc.z, nchunks = dsc.w & 0xffff, chunk = dsc.w >> 16;
    const int32_t* list = bin_list + (size_t)b * P;
    const float* gb = g_l + (size_t)b * P;
    float acc[DV];
#pragma unroll
    for (int i = 0; i < DV; ++i) acc[i] = 0.f;
    float gsum = 0.f;
    {
        const int e = e0 + lane;
        const int pv = e < e1 ? __ldg(list + e) : 0;
        const float gv = e < e1 ? __ldg(gb + pv) : 0.f;
        const int cnt = max(0, e1 - e0);
        for (int t0 = 0; t0 < cnt; t0 += 8) {
            float gg[8];
            const float* pr[8];
#pragma unroll
            for (int u = 0; u < 8; ++u) {
                const int t = t0 + u;
                gg[u] = __shfl_sync(0xffffffffu, gv, t & 31);
                const int pp = __shfl_sync(0xffffffffu, pv, t & 31);
                if (t >= cnt) gg[u] = 0.f;
                pr[u] = Pl + (size_t)pp * D;
            }
            float v[8][DV];
#pragma unroll
            for (int u = 0; u < 8; ++u)
#pragma unroll
                for (int i = 0; i < DV; ++i) v[u][i] = (FULL || i * 32 + lane < D) ? __ldg(pr[u] + i * 32 + lane) : 0.f;
#pragma unroll
            for (int u = 0; u < 8; ++u) {
                gsum += gg[u];
#pragma unroll
                for (int i = 0; i < DV; ++i) acc[i] = fmaf(gg[u], v[u][i], acc[i]);
            }
        }
    }
    const size_t row = (size_t)b * K + k;
    const float* zr = Zs + row * D;
    float* out = dZs + row * D;
    const float* add = add_dZs ? add_dZs + row * D : nullptr;                          // e.g. the PPC-loss contribution
    if (nchunks == 1) {
#pragma unroll
        for (int i = 0; i < DV; ++i)
            if (FULL || i * 32 + lane < D) {
                const float z = __ldg(zr + i * 32 + lane);
                float r = 2.0f * (z * gsum - acc[i]) + (add ? __ldg(add + i * 32 + lane) : 0.f);
                if (ex.dpre_out) r *= z * (1.0f - z);
                out[i * 32 + lane] = r;
            }
        return;
    }
    const size_t slot = (size_t)b * items_per_image + item;                 // partial slot of this chunk
#pragma unroll
    for (int i = 0; i < DV; ++i)
        if (FULL || i * 32 + lane < D) part[slot * D + i * 32 + lane] = acc[i];
    if (lane == 0) part_gsum[slot] = gsum;
    __threadfence();
    __syncwarp();
    unsigned int ticket = 0;
    if (lane == 0) ticket = atomicAdd(counters + row, 1u);
    ticket = __shfl_sync(0xffffffffu, ticket, 0);
    if (ticket != (unsigned int)(nchunks - 1)) return;
    __threadfence();
    const size_t slot0 = slot - chunk;
    float tot[DV];
#pragma unroll
    for (int i = 0; i < DV; ++i) tot[i] = 0.f;
    float gt = 0.f;
    for (int c = 0; c < nchunks; ++c) {
        gt += __ldcg(part_gsum + slot0 + c);
#pragma unroll
        for (int i = 0; i < DV; ++i)
            if (FULL || i * 32 + lane < D) tot[i] += __ldcg(part + (slot0 + c) * D + i * 32 + lane);
    }
#pragma unroll
    for (int i = 0; i < DV; ++i)
        if (FULL || i * 32 + lane < D) {
            const float z = __ldg(zr + i * 32 + lane);
            float r = 2.0f * (z * gt - tot[i]) + (add ? __ldg(add + i * 32 + lane) : 0.f);
            if (ex.dpre_out) r *= z * (1.0f - z);
            out[i * 32 + lane] = r;
        }
    if (lane == 0) counters[row] = 0u;                                       // self-resetting (graph replay)
}

// CLS-token gradient: dZc[b,:] = 2 (Zc[b,:] sum_p g_g[b,p] - sum_p g_g[b,p] Pg[p,:]).  CTA = 8 images x a slice of
// the global prototypes (rows read once per CTA, coalesced), fixed-order two-level sum: per-slice partials in
// `part` [slices][B][D], then the last CTA of each image group adds the slices in order (deterministic).
constexpr int kClsTB = 8, kClsThreads = 256, kClsSlices = 16;
// The CLS slices are the long pole of the launch (token rows alone 15.9 us, prototype rows alone 17.1 us, token + CLS 29.3 us).
// Tried, measured, reverted: 32 slices of 64 rows with the final sum dealt to all threads (66 us), the dealt final sum alone
// (44.5 us), 2 images x 64 rows x 32 slices (38.9 us, more re-read rows) -- every restructuring of this body so far made the
// launch slower; a separate tensor-core product for dZc (a dense B x Pg x D GEMM) is the open item.
// Also tried: every slice CTA of an image group waits for the others and sums its share of the outputs (32 slices) -- the pair
// token + CLS drops to 23.1 us, but the waiting CTAs hold SM slots and the whole launch goes 32.1 -> 34.3 us; and the launch split
// into a high-priority token + CLS branch and a low-priority prototype branch under the add-on backward: the step's span moves by
// 136-139 vs 140 us, within run-to-run noise, because the add-on backward slows down by what the gather gains.

__device__ __forceinline__ void
cls_grad_body(int slice, int bgroup, int nslices, const float* __restrict__ g_g, const float* __restrict__ Zc,
              const float* __restrict__ Pgl, int B, int D, int Pg, int p_per_slice, float* part,
              unsigned int* counters, float* __restrict__ dZc, int dpre_out) {
    __shared__ __align__(16) float gs[64][kClsTB];      // [prototype][image]: two 128-bit broadcast reads per prototype
    __shared__ unsigned int s_ticket;
    const int tid = threadIdx.x, b0 = bgroup * kClsTB;
    const int pa = slice * p_per_slice, pb = min(Pg, pa + p_per_slice);
    float acc[kClsTB][2];           // D <= 512: each thread owns columns tid, tid + 256
    float gsum[kClsTB];
#pragma unroll
    for (int i = 0; i < kClsTB; ++i) { acc[i][0] = acc[i][1] = 0.f; gsum[i] = 0.f; }
    for (int p0 = pa; p0 < pb; p0 += 64) {
        __syncthreads();
        for (int i = tid; i < kClsTB * 64; i += kClsThreads) {
            const int bi = i >> 6, pp = p0 + (i & 63);
            gs[i & 63][bi] = (b0 + bi < B && pp < pb) ? __ldg(g_g + (size_t)(b0 + bi) * Pg + pp) : 0.f;
        }
        __syncthreads();
        const int n = min(64, pb - p0);
#pragma unroll 8
        for (int q = 0; q < n; ++q) {
            const float* pr = Pgl + (size_t)(p0 + q) * D;
            const float v0 = tid < D ? __ldg(pr + tid) : 0.f;
            const float v1 = tid + 256 < D ? __ldg(pr + tid + 256) : 0.f;
            const float4 ga = *reinterpret_cast<const float4*>(&gs[q][0]), gb2 = *reinterpret_cast<const float4*>(&gs[q][4]);
            const float gq8[8] = {ga.x, ga.y, ga.z, ga.w, gb2.x, gb2.y, gb2.z, gb2.w};
#pragma unroll
            for (int i = 0; i < kClsTB; ++i) {
                gsum[i] += gq8[i];
                acc[i][0] = fmaf(gq8[i], v0, acc[i][0]);
                acc[i][1] = fmaf(gq8[i], v1, acc[i][1]);
            }
        }
    }
    // partial of this slice: 2 (Zc * gsum - acc)
#pragma unroll
    for (int i = 0; i < kClsTB; ++i) {
        const int b = b0 + i;
        if (b >= B) continue;
#pragma unroll
        for (int h = 0; h < 2; ++h) {
            const int d = tid + 256 * h;
            if (d < D) part[((size_t)slice * B + b) * D + d] = 2.0f * (__ldg(Zc + (size_t)b * D + d) * gsum[i] - acc[i][h]);
        }
    }
    __threadfence();
    __syncthreads();
    if (tid == 0) s_ticket = atomicAdd(counters + bgroup, 1u);
    __syncthreads();
    if (s_ticket == (unsigned int)(nslices - 1)) {
        __threadfence();
        for (int i = 0; i < kClsTB; ++i) {
            const int b = b0 + i;
            if (b >= B) continue;
            for (int d = tid; d < D; d += kClsThreads) {
                float s = 0.f;
#pragma unroll 8
                for (int sl = 0; sl < nslices; ++sl) s += __ldcg(part + ((size_t)sl * B + b) * D + d);
                if (dpre_out) {
                    const float z = __ldg(Zc + (size_t)b * D + d);
                    s *= z * (1.0f - z);
                }
                dZc[(size_t)b * D + d] = s;
            }
        }
        if (tid == 0) counters[bgroup] = 0u;       // self-resetting (graph replay)
    }
}

// dPl[p,:] += sum over the images b of p's class (image order) of dP_img[b, p % m, :]: the PPC loss's prototype
// gradient, added after the similarity gradients were written (PPH_BWDF_PPCROWS).  One warp per prototype row.
__global__ void __launch_bounds__(256)
ppc_rows_add_kernel(const float* __restrict__ dP_img, const int32_t* __restrict__ cls_start,
                    const int32_t* __restrict__ cls_order, int P, int D, int m, float* __restrict__ dPl) {
    const int p = blockIdx.x * 8 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (p >= P) return;
    const int cls = p / m, jj = p - cls * m;
    const int c0 = __ldg(cls_start + cls), c1 = __ldg(cls_start + cls + 1);
    if (c0 >= c1) return;
    for (int d = lane; d < D; d += 32) {
        float r = dPl[(size_t)p * D + d];
        for (int c = c0; c < c1; ++c) r += __ldg(dP_img + ((size_t)__ldg(cls_order + c) * m + jj) * D + d);
        dPl[(size_t)p * D + d] = r;
    }
}

struct BwdWorkspace {
    int32_t *bin_start, *item_start, *bin_list;
    int4* item_desc;
    unsigned int *tok_counters, *cls_counters;
    float *tok_part, *tok_gsum, *cls_part;
    int items_per_image;
    size_t bytes;
};

static BwdWorkspace carve_ws(void* base, int B, int K, int D, int P, int Pg) {
    BwdWorkspace w;
    char* p = static_cast<char*>(base);
    size_t off = 0;
    auto take = [&](size_t n) { char* r = p ? p + off : nullptr; off += (n + 255) / 256 * 256; return r; };
    w.items_per_image = bin_items_per_image(K, P);
    // counters first: they are the part that must start zeroed
    w.tok_counters = reinterpret_cast<unsigned int*>(take(sizeof(int) * (size_t)B * K));
    w.cls_counters = reinterpret_cast<unsigned int*>(take(sizeof(int) * (size_t)((B + kClsTB - 1) / kClsTB + 1)));
    w.bin_start = reinterpret_cast<int32_t*>(take(sizeof(int) * (size_t)B * (K + 1)));
    w.item_start = reinterpret_cast<int32_t*>(take(sizeof(int) * (size_t)B * (K + 1)));
    w.bin_list = reinterpret_cast<int32_t*>(take(sizeof(int) * (size_t)B * P));
    w.item_desc = reinterpret_cast<int4*>(take(sizeof(int4) * (size_t)B * w.items_per_image));
    w.tok_part = reinterpret_cast<float*>(take(sizeof(float) * (size_t)B * w.items_per_image * D));
    w.tok_gsum = reinterpret_cast<float*>(take(sizeof(float) * (size_t)B * w.items_per_image));
    w.cls_part = reinterpret_cast<float*>(take(Pg > 0 ? sizeof(float) * (size_t)kClsSlices * B * D : 0));
    w.bytes = off + 256;
    return w;
}

// One launch for the three independent gradient pieces (CLS-token slices, prototype rows, token work items): their
// CTAs share the machine instead of running as three partially filled waves back to back.
// Measured (scripts/gather_parts.py, B = 64, CUB shape): token + CLS pieces alone 29.8 us, prototype rows alone 17.3 us, all
// three in one launch 33.9 us = 208 MB of L2 -> SM traffic (two 768-byte rows per (image, prototype) pair plus the CLS
// slices) at ~6 TB/s: the launch is L2-bandwidth bound.  Tried and rejected: token items first in block order (52 us: the CLS
// CTAs, the longest-running ones, must start first), shorter CLS slices (2 images x 64 rows x 32 slices: +37 MB of re-read
// prototype rows, 38.9 us).
template <int DV, bool FULL>
__global__ void __launch_bounds__(256, DV <= 6 ? 4 : 1)      // 64 registers at D <= 192: at 80 (one unroll pragma away) every piece slows by 25-40 %
sim_grads_kernel(const float* __restrict__ g_l, const float* __restrict__ g_g, const int32_t* __restrict__ argmin_l,
                 const int4* __restrict__ item_desc,
                 const int32_t* __restrict__ bin_list, const float* __restrict__ Zs, const float* __restrict__ Zc,
                 const float* __restrict__ Pl, const float* __restrict__ Pgl, int B, int K, int D, int P, int Pg,
                 int items_per_image, int n_cls, int n_slices, int p_per_slice, int n_proto,
                 float* tok_part, float* tok_gsum, unsigned int* tok_counters, float* cls_part,
                 unsigned int* cls_counters, const float* __restrict__ add_dZs, const float* __restrict__ add_dPl,
                 float* __restrict__ dZs, float* __restrict__ dZc, float* __restrict__ dPl, float* __restrict__ dPg,
                 const BwdExtras ex) {
    int vb = blockIdx.x;
    if (vb < n_cls) {
        cls_grad_body(vb % n_slices, vb / n_slices, n_slices, g_g, Zc, Pgl, B, D, Pg, p_per_slice, cls_part, cls_counters, dZc,
                      ex.dpre_out);
        return;
    }
    vb -= n_cls;
    if (vb < n_proto) {
        proto_grad_body<DV, FULL>(vb, g_l, g_g, argmin_l, Zs, Zc, Pl, Pgl, B, K, D, P, Pg, add_dPl, dPl, dPg, ex);
        return;
    }
    vb -= n_proto;
    token_grad_body<DV, FULL>(vb, g_l, item_desc, bin_list, Zs, Pl, B, K, D, P, items_per_image, tok_part,
                              tok_gsum, tok_counters, add_dZs, dZs, ex);
}

template <int DV, bool FULL>
static int launch_bwd(const float* g_l, const float* g_g, const int32_t* argmin_l, const BwdWorkspace& w,
                      const float* Zs, const float* Zc, const float* Pl, const float* Pgl,
                      int B, int K, int D, int P, int Pg, const float* add_dZs, const float* add_dPl,
                      float* dZs, float* dZc, float* dPl, float* dPg, cudaStream_t st, const BwdExtras& ex,
                      int roles = 3) {
    const int slices = kClsSlices;
    const int p_per_slice = Pg > 0 ? ceil_div(ceil_div(Pg, slices), 64) * 64 : 64;
    const int nsl = Pg > 0 ? ceil_div(Pg, p_per_slice) : 0;
    // roles: bit 0 token-side rows (dZs, dZc), bit 1 prototype rows (dPl, dPg) -- independent, may run as two launches
    const int n_cls = (roles & 1) ? nsl * ceil_div(B, kClsTB) : 0;
    const int n_proto = (roles & 2) ? ceil_div(P + Pg, 8) : 0;
    const int n_tok = (roles & 1) ? ceil_div(B * w.items_per_image, 8) : 0;
    launch_k(sim_grads_kernel<DV, FULL>, dim3(n_cls + n_proto + n_tok), dim3(256), (size_t)(0), st, g_l, g_g, argmin_l, w.item_desc, w.bin_list, Zs, Zc, Pl, Pgl, B, K, D, P, Pg, w.items_per_image, n_cls, nsl, p_per_slice, n_proto, w.tok_part, w.tok_gsum, w.tok_counters, w.cls_part, w.cls_counters, add_dZs, add_dPl, dZs, dZc, dPl, dPg, ex);
    return launch_status("pph_similarity_bwd(grads)");
}

}  // namespace pph

extern "C" int pph_similarity_bwd_ws_bytes(int B, int K, int D, int P, int Pg, long long* bytes) {
    using namespace pph;
    PPH_REQUIRE(bytes && B >= 0 && K >= 1 && D >= 1 && P >= 1 && Pg >= 0, PPH_EINVAL, "pph_similarity_bwd_ws_bytes: bad args");
    *bytes = (long long)carve_ws(nullptr, B > 0 ? B : 1, K, D, P, Pg).bytes;
    return 0;
}

extern "C" int pph_similarity_bwd(const float* g_l, const float* g_g, const int32_t* argmin_l,
                                  const float* Zs, const float* Zc, const float* Pl, const float* Pgl,
                                  int B, int K, int D, int P, int Pg, void* workspace, int parts,
                                  const float* add_dZs, const float* add_dPl,
                                  float* dZs, float* dZc, float* dPl, float* dPg, pph_stream_t stream) {
    using namespace pph;
    PPH_REQUIRE((parts & 3) != 0, PPH_EINVAL, "pph_similarity_bwd: parts must include PPH_BWD_BIN and/or PPH_BWD_GRADS");
    if (!(parts & PPH_BWD_GRADS)) {      // binning only: needs argmin and the workspace
        PPH_REQUIRE(argmin_l && workspace && B >= 1 && K >= 1 && P >= 1, PPH_EINVAL, "pph_similarity_bwd(bin): bad args");
        const size_t bs = sizeof(int) * ((size_t)8 * K + 2 * (size_t)(K + 1));
        PPH_REQUIRE(bs <= 48 * 1024, PPH_EUNSUP, "pph_similarity_bwd: K too large");
        const BwdWorkspace wb = carve_ws(workspace, B, K, D, P, Pg);
        launch_k(bin_tokens_kernel, dim3(B), dim3(256), (size_t)(bs), as_stream(stream), wb.item_desc, argmin_l, K, P, wb.bin_start, wb.item_start, wb.bin_list);
        return launch_status("pph_similarity_bwd(bin)");
    }
    PPH_REQUIRE(g_l && argmin_l && Zs && Pl && dZs && dPl, PPH_EINVAL, "pph_similarity_bwd: null local pointer");
    PPH_REQUIRE(Pg == 0 || (g_g && Zc && Pgl && dZc && dPg), PPH_EINVAL, "pph_similarity_bwd: null global pointer");
    PPH_REQUIRE(B >= 0 && K >= 1 && D >= 1 && D <= 512 && P >= 1 && Pg >= 0, PPH_EINVAL,
                "pph_similarity_bwd: bad dims B=%d K=%d D=%d P=%d Pg=%d", B, K, D, P, Pg);
    cudaStream_t st = as_stream(stream);
    if (B == 0) {
        cudaMemsetAsync(dPl, 0, sizeof(float) * (size_t)P * D, st);
        if (Pg > 0) cudaMemsetAsync(dPg, 0, sizeof(float) * (size_t)Pg * D, st);
        return launch_status("pph_similarity_bwd(empty)");
    }
    PPH_REQUIRE(workspace, PPH_EINVAL, "pph_similarity_bwd: null workspace (size it with pph_similarity_bwd_ws_bytes)");
    const size_t bin_smem = sizeof(int) * ((size_t)8 * K + 2 * (size_t)(K + 1));
    PPH_REQUIRE(bin_smem <= 48 * 1024, PPH_EUNSUP, "pph_similarity_bwd: K too large");
    const BwdWorkspace w = carve_ws(workspace, B, K, D, P, Pg);
    int rc = 0;
    if (parts & PPH_BWD_BIN) {
        launch_k(bin_tokens_kernel, dim3(B), dim3(256), (size_t)(bin_smem), st, w.item_desc, argmin_l, K, P, w.bin_start, w.item_start, w.bin_list);
        rc = launch_status("pph_similarity_bwd(bin)");
        if (rc) return rc;
    }
    const int dv = ceil_div(D, 32);
    const bool full = (D % 32 == 0);
    const BwdExtras ex{nullptr, nullptr, nullptr, 1, 0};
#define PPH_BWD(DV, FULL) launch_bwd<DV, FULL>(g_l, g_g, argmin_l, w, Zs, Zc, Pl, Pgl, B, K, D, P, Pg, add_dZs, add_dPl, dZs, dZc, dPl, dPg, st, ex)
    if (full && dv == 2) rc = PPH_BWD(2, true);
    else if (full && dv == 6) rc = PPH_BWD(6, true);
    else if (full && dv == 12) rc = PPH_BWD(12, true);
    else if (dv <= 2) rc = PPH_BWD(2, false);
    else if (dv <= 6) rc = PPH_BWD(6, false);
    else if (dv <= 12) rc = PPH_BWD(12, false);
    else rc = PPH_BWD(16, false);
#undef PPH_BWD
    return rc;
}

// Same gradient kernel inside the fused training step: the token bins and class lists come from pph_head_mid
// (step_workspace = the bwd_workspace given to it), `workspace` only provides this kernel's partial slots and counters.
extern "C" int pph_similarity_bwd_fused(int parts, const float* g_l, const float* g_g, const int32_t* argmin_l,
                                        const float* Zs, const float* Zc, const float* Pl, const float* Pgl,
                                        int B, int K, int D, int P, int Pg, int m, void* workspace, void* step_workspace,
                                        const float* add_dZs, const float* dP_img, int dpre_out,
                                        float* dZs, float* dZc, float* dPl, float* dPg, pph_stream_t stream) {
    using namespace pph;
    PPH_REQUIRE((parts & 7) != 0, PPH_EINVAL, "pph_similarity_bwd_fused: parts must name TOKENS (1), PROTOS (2), PPCROWS (4)");
    if (parts == 4) {          // only the PPC prototype rows, added onto dPl (after the launch that wrote dPl)
        PPH_REQUIRE(dP_img && dPl && step_workspace && m >= 1, PPH_EINVAL, "pph_similarity_bwd_fused(PPCROWS): null pointer");
        const Step2Bins bins4 = carve_bins(step_workspace, B, K, P);
        launch_k(ppc_rows_add_kernel, dim3(ceil_div(P, 8)), dim3(256), (size_t)0, as_stream(stream), dP_img, bins4.cls_start,
                 bins4.cls_order, P, D, m, dPl);
        return launch_status("pph_similarity_bwd_fused(ppc rows)");
    }
    PPH_REQUIRE(g_l && argmin_l && Zs && Pl && dZs && dPl && workspace && step_workspace, PPH_EINVAL,
                "pph_similarity_bwd_fused: null pointer");
    PPH_REQUIRE(Pg == 0 || (g_g && Zc && Pgl && dZc && dPg), PPH_EINVAL, "pph_similarity_bwd_fused: null global pointer");
    PPH_REQUIRE(B >= 1 && K >= 1 && D >= 1 && D <= 512 && P >= 1 && Pg >= 0 && m >= 1, PPH_EINVAL,
                "pph_similarity_bwd_fused: bad dims");
    BwdWorkspace w = carve_ws(workspace, B, K, D, P, Pg);
    const Step2Bins bins = carve_bins(step_workspace, B, K, P);
    w.bin_start = bins.bin_start; w.item_start = bins.item_start; w.bin_list = bins.bin_list;
    w.item_desc = bins.item_desc;
    const BwdExtras ex{dP_img, bins.cls_start, bins.cls_order, m, dpre_out};
    cudaStream_t st = as_stream(stream);
    const float* add_dPl = nullptr;
    const int dv = ceil_div(D, 32);
    const bool full = (D % 32 == 0);
#define PPH_BWD(DV, FULL) launch_bwd<DV, FULL>(g_l, g_g, argmin_l, w, Zs, Zc, Pl, Pgl, B, K, D, P, Pg, add_dZs, add_dPl, dZs, dZc, dPl, dPg, st, ex, parts & 3)
    if (full && dv == 2) return PPH_BWD(2, true);
    if (full && dv == 6) return PPH_BWD(6, true);
    if (full && dv == 12) return PPH_BWD(12, true);
    if (dv <= 2) return PPH_BWD(2, false);
    if (dv <= 6) return PPH_BWD(6, false);
    if (dv <= 12) return PPH_BWD(12, false);
    return PPH_BWD(16, false);
#undef PPH_BWD
}
