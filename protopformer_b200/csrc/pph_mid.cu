// The middle of the training step in ONE launch (judge item "fused head", SURVEY.md 8(d)/(f) next #3):
//
//   role LL  (blockIdx <  n_ll)            last layers + combine (protopformer.py:297-300, 314-316), cross-entropy and
//                                          d(loss)/d(logits) (engine_proto.py:51), last-layer backward collapsed with the
//                                          similarity derivative into g[b,p] (autograd of :228-244, :297-300)
//   role BIN (n_ll <= blockIdx < +n_bin)   token bins of the argmin-routed backward (pph_bins.cuh)
//   role PPC (the remaining n_ppc CTAs)    PPC loss forward AND backward (protopformer.py:249-288; the upstream
//                                          gradients of the two PPC terms are the constant loss coefficients of
//                                          engine_proto.py:61-64, so the backward needs nothing from the CE branch)
//
// Role LL is a three-phase split-K contraction over co-resident CTAs with two grid barriers:
//   phase 1  CTA (image tile of 64, prototype group s): partial logits over its 32-prototype slices -> part[s][b][c]
//   phase 2  CTA r < B: logits row = sum of the partials in a FIXED order (deterministic), log-sum-exp, dlogits
//            (also stored transposed for phase 3), per-image CE term; the batch mean is a fixed-order tree
//   phase 3  CTA (tile, s): g[b,p] = coef * (sum_c dlogits[b,c] W[c,p]) * act'(dmin[b,p]) for its slices, written as
//            g[b][p] (the token-gradient kernel gathers it through the bins) and as pairT[p][b] = (g, argmin) (the
//            prototype-gradient kernel walks it row by row).
// FP32 FMA throughout: 2 x 102 MFLOP at the CUB shape, far too skinny (64 x 200 outputs) for a tensor-core tile
// grid -- what matters here is that every SM has a CTA and that no intermediate leaves L2.
//
// Role LL has a second, class-sum form for last layers that hold the class-connection pattern of
// set_last_layer_incorrect_connection (protopformer.py:367-386: W[c,p] = a on the prototype's own class p / m, b
// elsewhere -- the frozen init of every run).  Then logit_c = b T + (a - b) s_c with s_c the sum of class c's m
// activations and T their total, and (dlogits W)[p] = b sum_c dlogits[c] + (a - b) dlogits[p / m]: O(B P) instead of
// O(B P C), one CTA per image, no grid barrier.  pph_last_layer_pattern checks both matrices on the device (every
// step, inside the graph: a host-side decision would go stale after W.data.copy_) and leaves its verdict at the start
// of the workspace; the launch reads it and runs the class-sum form only when both pass, the three phases otherwise.
#include <math.h>

#include <algorithm>

#include "pph_bins.cuh"
#include "pph_common.cuh"
#include "pph_step2.cuh"

namespace pph {

constexpr int kMidThreads = 256;
constexpr int kMidTB = 64;       // images per tile
constexpr int kMidPS = 32;       // prototypes per slice
constexpr int kMidAST = 68;      // row stride of the [*][64-image] shared tiles (16-byte aligned, 4 mod 32 banks)

// Verdict of pph_last_layer_pattern on one last layer (layout documented at PPH_LL_PATTERN_BYTES in protohead.h).
struct LLPattern {
    int ok;          // every entry is a on its own class and b elsewhere (exact float equality)
    float a, b;
    int unused;
};
// First bytes of the pph_head_mid workspace: the verdicts for Wl and Wg, then the check's own counters.  All zero at
// first use (ok = 0: the three-phase role); the launch that reads the verdicts clears `ok` again.
struct LLPatternWs {
    LLPattern rec[2];
    unsigned int bad, ticket;
};
static_assert(sizeof(LLPattern) * 2 == PPH_LL_PATTERN_BYTES, "protohead.h documents two 16-byte records");

struct MidArgs {
    int B, Bp, K, D, P, Pg, C, Cp, m, N, side;
    int tiles_b, S_l, S_g, nsl_l, nsl_g;
    int n_ll, n_bin, n_ppc, n_cls_cta;
    int have_ppc;                 // the step has a PPC role (in this launch or in a concurrent one)
    int ppc_dpre;                 // dZs_ppc is written as the pre-activation gradient dZ * Z * (1 - Z)
    float gc, eps, upstream, cov_thresh, mean_thresh, cov_coe, mean_coe;
    int act_fn, train;
    const float *act_l, *act_g, *dmin_l, *dmin_g;
    const int32_t* argmin_l;
    const float *Wl, *Wg;
    const int64_t* labels;
    float *logits, *logits_g, *logits_l, *losses, *dlogits, *g_l, *g_g;
    float* losses_mirror;              // optional second home of losses[0..3] (e.g. mapped pinned host memory), or nullptr
    float2* pairT;
    // workspace
    float *part, *dlT, *ce_part, *ppc_part, *ppc_losses;
    unsigned int* ctr;      // [0] barrier, [1] done, [2] fin, [3] ppc ticket, [4] class-sum LL ticket
    LLPatternWs* pattern;
    int32_t *bin_start, *item_start, *bin_list;
    int4* item_desc;
    int32_t *cls_id, *cls_start, *cls_item, *cls_order;
    // PPC role
    const float *Zs, *z2s, *Pl, *p2l;
    const int32_t* idx;
    float *dZs_ppc, *dP_img;
};

__device__ __forceinline__ float block_sum_any(float v, float* red, int nwarp) {
    v = warp_sum(v);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    __syncthreads();
    if (lane == 0) red[warp] = v;
    __syncthreads();
    float s = 0.f;
    for (int w = 0; w < nwarp; ++w) s += red[w];
    return s;
}

__device__ __forceinline__ float block_sum_mid(float v, float* red) {
    v = warp_sum(v);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    __syncthreads();
    if (lane == 0) red[warp] = v;
    __syncthreads();
    float s = 0.f;
#pragma unroll
    for (int w = 0; w < kMidThreads / 32; ++w) s += red[w];
    return s;
}

// total = ce + cov_coe * cov + mean_coe * mean (engine_proto.py:61-64): written by whichever role finishes second.
__device__ __forceinline__ void write_total(const MidArgs& a) {
    const float ce = __ldcg(a.losses + 1);
    const float cov = a.have_ppc ? __ldcg(a.ppc_losses) : 0.f, mean = a.have_ppc ? __ldcg(a.ppc_losses + 1) : 0.f;
    const float total = ce + a.cov_coe * cov + a.mean_coe * mean;
    a.losses[0] = total;
    a.losses[2] = cov;
    a.losses[3] = mean;
    if (a.losses_mirror) {      // the caller's copy of the result: one 16-byte store (over PCIe when it is host memory)
        *reinterpret_cast<float4*>(a.losses_mirror) = make_float4(total, ce, cov, mean);
        __threadfence_system();
    }
}
__device__ __forceinline__ void role_finished(const MidArgs& a) {      // one thread
    if (!a.have_ppc) {
        write_total(a);
        return;
    }
    __threadfence();
    if (atomicAdd(a.ctr + 2, 1u) == 1u) {
        __threadfence();
        write_total(a);
        a.ctr[2] = 0u;
    }
}

// ---------------------------------------------------------------------------------------------------------------
// role LL
// ---------------------------------------------------------------------------------------------------------------
// W slice, transposed on the way in: Ws[pl][c] = W[c][p0 + pl].  4-byte cp.async copies: a warp reads one 128-byte row
// segment and scatters it down a column of Ws (odd stride: conflict-free); all C copies of a thread are in flight at once.
__device__ __forceinline__ void stage_w(float* Ws, const float* __restrict__ W, int np, int p0, int C, int WST) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int pp = p0 + lane;
    float* dst = Ws + lane * WST;
    if (pp < np) {
        const float* src = W + pp;
        for (int c = warp; c < C; c += kMidThreads / 32) cp_async4(dst + c, src + (size_t)c * np);
    } else {
        for (int c = warp; c < C; c += kMidThreads / 32) dst[c] = 0.f;
    }
}

template <int CJ>
__device__ __forceinline__ void ll_role(const MidArgs& a, float* sm) {
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int cta = blockIdx.x;
    const int S = a.S_l + a.S_g;
    const int tb = cta / S, s = cta - tb * S;
    const bool glob = s >= a.S_l;
    const int sg = glob ? s - a.S_l : s;
    const int Sg = glob ? a.S_g : a.S_l;
    const int nsl = glob ? a.nsl_g : a.nsl_l;
    const int np = glob ? a.Pg : a.P;
    const float* act = glob ? a.act_g : a.act_l;
    const float* W = glob ? a.Wg : a.Wl;
    const int C = a.C, Cp = a.Cp, B = a.B;
    const int WST = C | 1;                          // odd row stride: transposed stores and column reads conflict-free
    float* Ws = sm;                                 // [kMidPS][WST]        W slice, Ws[pl][c] = W[c][p0 + pl]
    float* As = Ws + kMidPS * WST;                  // [kMidPS][kMidAST]    act tile, As[pl][bi]
    float* dls = As + kMidPS * kMidAST;             // [C][kMidAST]         dlogits tile (phase 3)
    float* red4 = dls + (size_t)C * kMidAST;        // [2][4][64] float4    phase-2 partial sums
    float* rowb = red4 + 2 * 4 * 64 * 4;            // [3][256]             logits_l, logits_g, logits of one image
    float* red = rowb + 3 * 256;                    // [8]
    const int b0 = tb * kMidTB;

    // ---- phase 1: partial logits of this CTA's slices ---------------------------------------------------------
    {
        float acc[8][CJ];
#pragma unroll
        for (int i = 0; i < 8; ++i)
#pragma unroll
            for (int j = 0; j < CJ; ++j) acc[i][j] = 0.f;
        for (int sl = sg; sl < nsl; sl += Sg) {
            const int p0 = sl * kMidPS;
            __syncthreads();
            stage_w(Ws, W, np, p0, C, WST);
            {   // act tile, transposed on the way in: As[pl][bi] = act[b0 + bi][p0 + pl]
                const int pl = lane, pp = p0 + pl;
                const float* src = act + (size_t)(b0 + warp) * np + pp;
#pragma unroll
                for (int u = 0; u < kMidTB / 8; ++u) {
                    const int bi = warp + 8 * u;
                    if (b0 + bi < B && pp < np) cp_async4(&As[pl * kMidAST + bi], src + (size_t)(8 * u) * np);
                    else As[pl * kMidAST + bi] = 0.f;
                }
            }
            cp_async_commit();
            cp_async_wait<0>();
            __syncthreads();
#pragma unroll 2
            for (int pl = 0; pl < kMidPS; ++pl) {
                const float4 a0 = *reinterpret_cast<const float4*>(&As[pl * kMidAST + warp * 8]);
                const float4 a1 = *reinterpret_cast<const float4*>(&As[pl * kMidAST + warp * 8 + 4]);
                const float av[8] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w};
                float wv[CJ];
#pragma unroll
                for (int j = 0; j < CJ; ++j) wv[j] = (lane + 32 * j < C) ? Ws[pl * WST + lane + 32 * j] : 0.f;
#pragma unroll
                for (int i = 0; i < 8; ++i)
#pragma unroll
                    for (int j = 0; j < CJ; ++j) acc[i][j] = fmaf(av[i], wv[j], acc[i][j]);
            }
        }
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            const int b = b0 + warp * 8 + i;
            if (b >= B) continue;
            float* pr = a.part + ((size_t)s * B + b) * Cp;
#pragma unroll
            for (int j = 0; j < CJ; ++j)
                if (lane + 32 * j < C) pr[lane + 32 * j] = acc[i][j];
        }
    }
    grid_barrier(a.ctr, (unsigned int)a.n_ll);

    // ---- phase 2: logits rows, cross-entropy, dlogits ---------------------------------------------------------
    {
        const int c4 = tid & 63, q = tid >> 6;
        float* rl = rowb;
        float* rg = rowb + 256;
        float* rt = rowb + 512;
        for (int r = cta; r < B; r += a.n_ll) {
            float4 sl4 = make_float4(0.f, 0.f, 0.f, 0.f), sg4 = sl4;
            if (c4 * 4 < Cp) {
                const float* base = a.part + (size_t)r * Cp + c4 * 4;
                const size_t plane = (size_t)B * Cp;
                for (int pl = q; pl < a.S_l; pl += 16) {          // 4 independent loads in flight per thread
                    float4 v[4];
#pragma unroll
                    for (int u = 0; u < 4; ++u)
                        v[u] = (pl + 4 * u < a.S_l) ? ldcg4(base + (size_t)(pl + 4 * u) * plane) : make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
                    for (int u = 0; u < 4; ++u) { sl4.x += v[u].x; sl4.y += v[u].y; sl4.z += v[u].z; sl4.w += v[u].w; }
                }
                for (int pl = q; pl < a.S_g; pl += 16) {
                    float4 v[4];
#pragma unroll
                    for (int u = 0; u < 4; ++u)
                        v[u] = (pl + 4 * u < a.S_g) ? ldcg4(base + (size_t)(a.S_l + pl + 4 * u) * plane) : make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
                    for (int u = 0; u < 4; ++u) { sg4.x += v[u].x; sg4.y += v[u].y; sg4.z += v[u].z; sg4.w += v[u].w; }
                }
            }
            reinterpret_cast<float4*>(red4)[q * 64 + c4] = sl4;
            reinterpret_cast<float4*>(red4)[256 + q * 64 + c4] = sg4;
            __syncthreads();
            if (tid < 64 && tid * 4 < Cp) {
                float4 l = reinterpret_cast<float4*>(red4)[tid], g = reinterpret_cast<float4*>(red4)[256 + tid];
#pragma unroll
                for (int qq = 1; qq < 4; ++qq) {
                    const float4 l2 = reinterpret_cast<float4*>(red4)[qq * 64 + tid];
                    const float4 g2 = reinterpret_cast<float4*>(red4)[256 + qq * 64 + tid];
                    l.x += l2.x; l.y += l2.y; l.z += l2.z; l.w += l2.w;
                    g.x += g2.x; g.y += g2.y; g.z += g2.z; g.w += g2.w;
                }
                const float lv[4] = {l.x, l.y, l.z, l.w}, gv[4] = {g.x, g.y, g.z, g.w};
#pragma unroll
                for (int e = 0; e < 4; ++e) {
                    const int c = tid * 4 + e;
                    if (c < C) {
                        const float t = a.gc * gv[e] + (1.0f - a.gc) * lv[e];
                        rl[c] = lv[e]; rg[c] = gv[e]; rt[c] = t;
                        a.logits_l[(size_t)r * C + c] = lv[e];
                        a.logits_g[(size_t)r * C + c] = gv[e];
                        a.logits[(size_t)r * C + c] = t;
                    }
                }
            }
            __syncthreads();
            if (warp == 0) {
                float mx = -INFINITY;
                for (int c = lane; c < C; c += 32) mx = fmaxf(mx, rt[c]);
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
                float se = 0.f;
                for (int c = lane; c < C; c += 32) se += expf(rt[c] - mx);
                se = warp_sum(se);
                long y = a.labels[r];
                if (y < 0) y = 0;
                if (y >= C) y = C - 1;
                const float lse = logf(se) + mx;
                if (a.train) {
                    const float sc = a.upstream / (float)B;
                    for (int c = lane; c < C; c += 32) {
                        const float p = expf(rt[c] - mx) / se;
                        const float dl = (p - (c == (int)y ? 1.0f : 0.0f)) * sc;
                        a.dlogits[(size_t)r * C + c] = dl;
                        a.dlT[(size_t)c * a.Bp + r] = dl;
                    }
                }
                if (lane == 0) a.ce_part[r] = lse - rt[y];
            }
            __syncthreads();
        }
    }
    grid_barrier(a.ctr, 2u * (unsigned int)a.n_ll);

    if (cta == 0) {        // batch mean of the per-image CE terms: fixed-order tree (deterministic)
        float v = 0.f;
        for (int i = tid; i < B; i += kMidThreads) v += __ldcg(a.ce_part + i);
        const float ce = block_sum_mid(v, red) / (float)B;
        if (tid == 0) {
            a.losses[1] = ce;
            role_finished(a);
        }
    }

    // ---- phase 3: g[b,p] = coef * (dlogits[b,:] . W[:,p]) * act'(dmin[b,p]) --------------------------------------
    if (a.train) {
        // dlogits tile of this image tile: rows of dlT are 64 contiguous floats (columns >= B of dlT stay zero: the
        // workspace starts zeroed and only columns < B are ever written)
        for (int i = tid; i < C * (kMidTB / 4); i += kMidThreads) {
            const int c = i >> 4, q = i & 15;
            cp_async16(&dls[c * kMidAST + q * 4], a.dlT + (size_t)c * a.Bp + b0 + q * 4);
        }
        cp_async_commit();
        const bool keepW = nsl <= Sg;            // one slice per CTA: Ws still holds it from phase 1
        const float coef = glob ? a.gc : 1.0f - a.gc;
        const float* dmin = glob ? a.dmin_g : a.dmin_l;
        float* gout = glob ? a.g_g : a.g_l;
        for (int sl = sg; sl < nsl; sl += Sg) {
            const int p0 = sl * kMidPS;
            if (!keepW) {
                __syncthreads();
                stage_w(Ws, W, np, p0, C, WST);
                cp_async_commit();
            }
            cp_async_wait<0>();
            __syncthreads();
            float g8[8];
#pragma unroll
            for (int i = 0; i < 8; ++i) g8[i] = 0.f;
#pragma unroll 4
            for (int c = 0; c < C; ++c) {
                const float4 d0 = *reinterpret_cast<const float4*>(&dls[c * kMidAST + warp * 8]);
                const float4 d1 = *reinterpret_cast<const float4*>(&dls[c * kMidAST + warp * 8 + 4]);
                const float w = Ws[lane * WST + c];
                g8[0] = fmaf(d0.x, w, g8[0]); g8[1] = fmaf(d0.y, w, g8[1]); g8[2] = fmaf(d0.z, w, g8[2]); g8[3] = fmaf(d0.w, w, g8[3]);
                g8[4] = fmaf(d1.x, w, g8[4]); g8[5] = fmaf(d1.y, w, g8[5]); g8[6] = fmaf(d1.z, w, g8[6]); g8[7] = fmaf(d1.w, w, g8[7]);
            }
            const int p = p0 + lane;
            if (p < np) {
                float2 pr[8];
#pragma unroll
                for (int i = 0; i < 8; ++i) {
                    const int b = b0 + warp * 8 + i;
                    float g = 0.f;
                    int am = 0;
                    if (b < B) {
                        const size_t o = (size_t)b * np + p;
                        g = coef * g8[i] * dact_of_dist(__ldg(dmin + o), a.act_fn, a.eps);
                        gout[o] = g;
                        am = glob ? a.K : __ldg(a.argmin_l + o);
                    }
                    pr[i] = make_float2(g, __int_as_float(am));
                }
                if (a.pairT) {          // only the staged backward (pph_similarity_bwd2) reads the transposed pairs
                    float4* dst = reinterpret_cast<float4*>(a.pairT + (size_t)(glob ? a.P + p : p) * a.Bp + b0 + warp * 8);
#pragma unroll
                    for (int i = 0; i < 4; ++i) dst[i] = make_float4(pr[2 * i].x, pr[2 * i].y, pr[2 * i + 1].x, pr[2 * i + 1].y);
                }
            }
        }
    }
    grid_finish(a.ctr, a.ctr + 1, (unsigned int)a.n_ll);
}

__device__ __forceinline__ float block_max_mid(float v, float* red) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    __syncthreads();
    if (lane == 0) red[warp] = v;
    __syncthreads();
    float s = red[0];
#pragma unroll
    for (int w = 1; w < kMidThreads / 32; ++w) s = fmaxf(s, red[w]);
    return s;
}

// g[b,p] of one branch in the class-sum form (and its pairT column when the staged backward wants it)
__device__ __forceinline__ void ll_class_grad(const MidArgs& a, int b, bool glob, const LLPattern& w, float Sdl,
                                              const float* dls) {
    const int np = glob ? a.Pg : a.P, m = np / a.C;
    const float coef = glob ? a.gc : 1.0f - a.gc;
    const float* dmin = glob ? a.dmin_g : a.dmin_l;
    float* gout = glob ? a.g_g : a.g_l;
    const float bS = w.b * Sdl, amb = w.a - w.b;
    const size_t row = (size_t)b * np;
    constexpr int U = 4;            // dmin loads in flight per thread before the first use
    for (int p0 = threadIdx.x; p0 < np; p0 += U * kMidThreads) {
        float d[U];
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const int p = p0 + u * kMidThreads;
            d[u] = p < np ? __ldg(dmin + row + p) : 0.f;
        }
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const int p = p0 + u * kMidThreads;
            if (p >= np) break;
            const float g = coef * fmaf(amb, dls[p / m], bS) * dact_of_dist(d[u], a.act_fn, a.eps);
            gout[row + p] = g;
            if (a.pairT)
                a.pairT[(size_t)(glob ? a.P + p : p) * a.Bp + b] =
                    make_float2(g, __int_as_float(glob ? a.K : __ldg(a.argmin_l + row + p)));
        }
    }
}

// role LL, class-sum form (both last layers passed pph_last_layer_pattern): LL CTA r takes images r, r + n_ll, ...; a
// thread owns one class (C <= 256).  Every sum runs in a fixed order (bit-identical replays).  The softmax and the
// cross-entropy are taken over the class-dependent part of the logits only, z_c = (1-gc)(a_l-b_l) s_l,c +
// gc (a_g-b_g) s_g,c: the b T terms are the same for every class and cancel, and at ~1e3 they would cost digits.
__device__ void ll_class_role(const MidArgs& a, const LLPattern& wl, const LLPattern& wg, float* sm) {
    const int tid = threadIdx.x, c = tid;
    const int B = a.B, C = a.C, ml = a.P / C, mg = a.Pg / C;
    float* dls = sm;                  // [256] dlogits of the image
    float* zs = dls + kMidThreads;    // [256] class-dependent logits
    float* red = zs + kMidThreads;    // [8]
    const float kl = (1.0f - a.gc) * (wl.a - wl.b), kg = a.gc * (wg.a - wg.b);
    for (int b = blockIdx.x; b < B; b += a.n_ll) {
        float sl = 0.f, sg = 0.f;
        if (c < C) {
            const float* rl = a.act_l + (size_t)b * a.P + (size_t)c * ml;
            const float* rg = a.act_g + (size_t)b * a.Pg + (size_t)c * mg;
            for (int j = 0; j < ml; ++j) sl += __ldg(rl + j);
            for (int j = 0; j < mg; ++j) sg += __ldg(rg + j);
        }
        const float Tl = block_sum_mid(sl, red), Tg = block_sum_mid(sg, red);
        const float z = c < C ? fmaf(kl, sl, kg * sg) : -INFINITY;
        zs[c] = z;
        if (c < C) {
            const float lv = fmaf(wl.a - wl.b, sl, wl.b * Tl), gv = fmaf(wg.a - wg.b, sg, wg.b * Tg);
            a.logits_l[(size_t)b * C + c] = lv;
            a.logits_g[(size_t)b * C + c] = gv;
            a.logits[(size_t)b * C + c] = a.gc * gv + (1.0f - a.gc) * lv;
        }
        const float mx = block_max_mid(z, red);       // its barriers also publish zs[]
        const float e = c < C ? expf(z - mx) : 0.f;
        const float se = block_sum_mid(e, red);
        long y = a.labels[b];
        if (y < 0) y = 0;
        if (y >= C) y = C - 1;
        if (tid == 0) a.ce_part[b] = logf(se) + mx - zs[y];
        if (a.train) {
            const float dl = c < C ? (e / se - (c == (int)y ? 1.0f : 0.0f)) * (a.upstream / (float)B) : 0.f;
            if (c < C) a.dlogits[(size_t)b * C + c] = dl;
            dls[c] = dl;
            const float Sdl = block_sum_mid(dl, red);      // its barriers also publish dls[]
            ll_class_grad(a, b, false, wl, Sdl, dls);
            ll_class_grad(a, b, true, wg, Sdl, dls);
        }
        __syncthreads();                                  // zs / dls / red are reused by the next image
    }
    if (a.train && a.pairT) {        // columns of the padded images are zeros, as the three-phase role writes them
        for (int b = a.B + blockIdx.x; b < a.Bp; b += a.n_ll)
            for (int p = tid; p < a.P + a.Pg; p += kMidThreads) a.pairT[(size_t)p * a.Bp + b] = make_float2(0.f, 0.f);
    }
    // every LL CTA takes the ticket (it read the verdicts first); the last one forms the batch mean of the CE terms in
    // the same fixed order as the three-phase role and clears the verdicts: the next launch without a fresh check
    // falls back to the general product
    __shared__ int last;
    __syncthreads();
    if (tid == 0) {
        __threadfence();
        last = atomicAdd(a.ctr + 4, 1u) == (unsigned int)a.n_ll - 1u;
        if (last) {
            __threadfence();
            a.pattern->rec[0].ok = 0;
            a.pattern->rec[1].ok = 0;
            a.ctr[4] = 0u;
        }
    }
    __syncthreads();
    if (last) {
        float v = 0.f;
        for (int i = tid; i < B; i += kMidThreads) v += __ldcg(a.ce_part + i);
        const float ce = block_sum_mid(v, red) / (float)B;
        if (tid == 0) {
            a.losses[1] = ce;
            role_finished(a);
        }
    }
}

// ---------------------------------------------------------------------------------------------------------------
// role PPC: forward (restatement of SURVEY.md 8(d)(iii), same arithmetic as pph_ppc.cu) + backward in one CTA per image
// ---------------------------------------------------------------------------------------------------------------
// `nsplit` CTAs share an image: each recomputes the (cheap) forward, CTA `part` takes every nsplit-th token row and
// work item of the backward, part 0 reports the losses.  Block size = blockDim.x (a multiple of 32, <= 1024).
__device__ __forceinline__ void ppc_role(const MidArgs& a, int b, int part, int nsplit, float* sm) {
    const int nthr = blockDim.x;
    const int K = a.K, D = a.D, m = a.m, B = a.B, side = a.side;
    const int zs = D + 4;
    float* Prow = sm;                     // [m][D]
    float* Zt = Prow + m * D;             // [K][D+4]
    float* dsl = Zt + (size_t)K * zs;     // [m][K] distances, later d loss / d distance
    float* wbuf = dsl + m * K;            // [m][K] activations
    float* st = wbuf + m * K;             // [m][8]
    float* red = st + m * 8;              // [32]
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nwarp = nthr >> 5;
    long y = a.labels[b];
    if (y < 0) y = 0;
    if (y * m + m > a.P) y = a.P / m - 1;
    const int prow0 = (int)y * m;
    for (int i = tid; i < m * D / 4; i += nthr) cp_async16(Prow + 4 * i, a.Pl + (size_t)prow0 * D + 4 * i);
    const float* Zb = a.Zs + (size_t)b * K * D;
    {
        const int d4 = D >> 2;
        for (int r = warp; r < K; r += nwarp)
            for (int c = lane; c < d4; c += 32) cp_async16(Zt + (size_t)r * zs + 4 * c, Zb + (size_t)r * D + 4 * c);
    }
    cp_async_commit();
    cp_async_wait<0>();
    __syncthreads();
    const int JG = K * m <= nthr ? m : (K * 5 <= nthr ? 5 : (K * 3 <= nthr ? 3 : (K * 2 <= nthr ? 2 : 1)));
    for (int t = tid; t < K * JG; t += nthr) {
        const int r = t % K, jg = t / K;
        const float4* zr = reinterpret_cast<const float4*>(Zt + (size_t)r * zs);
        const float zz = __ldg(a.z2s + (size_t)b * K + r);
        for (int j = jg; j < m; j += JG) {
            const float4* pr = reinterpret_cast<const float4*>(Prow + (size_t)j * D);
            float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
#pragma unroll 4
            for (int c = 0; c < D / 4; ++c) {
                const float4 z = zr[c], p = pr[c];
                a0 = fmaf(z.x, p.x, a0); a1 = fmaf(z.y, p.y, a1); a2 = fmaf(z.z, p.z, a2); a3 = fmaf(z.w, p.w, a3);
            }
            const float dot = (a0 + a1) + (a2 + a3);
            const float d = relu_keep_nan(zz + fmaf(-2.0f, dot, __ldg(a.p2l + prow0 + j)));
            dsl[j * K + r] = d;
            wbuf[j * K + r] = act_of_dist(d, a.act_fn, a.eps);
        }
    }
    __syncthreads();
    float cov_sum = 0.f;
    const float scale = (float)a.N / (float)(a.N - 1);
    for (int j = warp; j < m; j += nwarp) {
        float S = 0.f, Sr = 0.f, Sc = 0.f;
        for (int k = lane; k < K; k += 32) {
            const float w = wbuf[j * K + k];
            const int n = __ldg(a.idx + (size_t)b * K + k);
            S += w;
            Sr = fmaf(w, (float)(n / side), Sr);
            Sc = fmaf(w, (float)(n % side), Sc);
        }
        S = warp_sum(S); Sr = warp_sum(Sr); Sc = warp_sum(Sc);
        const float mr = Sr / S, mc = Sc / S;
        float Vr = 0.f, Vc = 0.f;
        for (int k = lane; k < K; k += 32) {
            const float w = wbuf[j * K + k];
            const int n = __ldg(a.idx + (size_t)b * K + k);
            const float dr = (float)(n / side) - mr, dc = (float)(n % side) - mc;
            Vr = fmaf(w, dr * dr, Vr);
            Vc = fmaf(w, dc * dc, Vc);
        }
        Vr = warp_sum(Vr) / S;
        Vc = warp_sum(Vc) / S;
        const float pre = (Vr * scale + Vc * scale) * 0.5f - a.cov_thresh;
        if (lane == 0) {
            float* s8 = st + j * 8;
            s8[0] = S; s8[1] = mr; s8[2] = mc; s8[3] = Vr; s8[4] = Vc; s8[5] = pre; s8[6] = 0.f; s8[7] = 0.f;
            cov_sum += relu_keep_nan(pre);
        }
    }
    const float cov_img = block_sum_any(lane == 0 ? cov_sum : 0.f, red, nwarp);     // its barriers also publish st[]
    float mean_sum = 0.f;
    for (int t = tid; t < m * m; t += nthr) {
        const int i = t / m, j = t - i * m;
        if (i != j) {
            const float dr = st[i * 8 + 1] - st[j * 8 + 1], dc = st[i * 8 + 2] - st[j * 8 + 2];
            mean_sum += relu_keep_nan(a.mean_thresh - sqrtf(dr * dr + dc * dc));
        }
    }
    const float mean_img = block_sum_any(mean_sum, red, nwarp);
    if (tid == 0 && part == 0) {        // deterministic batch sums: the last image CTA adds the partials in image order
        a.ppc_part[2 * b] = cov_img;
        a.ppc_part[2 * b + 1] = mean_img;
        __threadfence();
        if (atomicAdd(a.ctr + 3, 1u) == (unsigned int)(B - 1)) {
            __threadfence();
            float c = 0.f, sacc = 0.f;
            for (int i = 0; i < B; ++i) {
                c += __ldcg(a.ppc_part + 2 * i);
                sacc += __ldcg(a.ppc_part + 2 * i + 1);
            }
            a.ppc_losses[0] = c / ((float)B * (float)m);
            a.ppc_losses[1] = sacc / ((float)B * (float)m * (float)m);
            a.ctr[3] = 0u;
            role_finished(a);
        }
    }
    if (!a.train) return;

    // ---- backward (same arithmetic as ppc_bwd_kernel) -----------------------------------------------------------
    const float g_cov = a.cov_coe * a.upstream / ((float)B * (float)m);
    const float g_mean = a.mean_coe * a.upstream / ((float)B * (float)m * (float)m);
    if (tid < m) {
        const int i = tid;
        float gr = 0.f, gcn = 0.f;
        for (int j = 0; j < m; ++j) {
            if (j == i) continue;
            const float dr = st[i * 8 + 1] - st[j * 8 + 1], dc = st[i * 8 + 2] - st[j * 8 + 2];
            const float dist = sqrtf(dr * dr + dc * dc);
            if (a.mean_thresh - dist > 0.0f && dist > 0.0f) {
                gr -= 2.0f * g_mean * dr / dist;
                gcn -= 2.0f * g_mean * dc / dist;
            }
        }
        st[i * 8 + 6] = gr;
        st[i * 8 + 7] = gcn;
    }
    __syncthreads();
    for (int t = tid; t < m * K; t += nthr) {
        const int j = t / K, r = t - j * K;
        const float S = st[j * 8], mr = st[j * 8 + 1], mc = st[j * 8 + 2], Vr = st[j * 8 + 3], Vc = st[j * 8 + 4];
        const float dV = st[j * 8 + 5] > 0.0f ? 0.5f * g_cov * scale : 0.0f;
        const int tok = __ldg(a.idx + (size_t)b * K + r);
        const float dr = (float)(tok / side) - mr, dc = (float)(tok % side) - mc;
        const float dw = (dV * ((dr * dr - Vr) + (dc * dc - Vc)) + st[j * 8 + 6] * dr + st[j * 8 + 7] * dc) / S;
        const float d = dsl[j * K + r];
        dsl[j * K + r] = 2.0f * dw * dact_of_dist(d, a.act_fn, a.eps);        // factor 2 of d|z-p|^2 folded in
    }
    __syncthreads();
    // token rows: dZ[b,k,:] = Z[b,k,:] sum_j dd[j,k] - sum_j dd[j,k] P_j; one warp per token, a lane owns 4 features
    // of a 128-feature group (one broadcast read of dd and one 16-byte read of P_j per 4 FMAs)
    const int ngrp = (D + 127) >> 7;
    for (int r = warp * nsplit + part; r < K; r += nwarp * nsplit) {
        float S = 0.f;
        for (int j = 0; j < m; ++j) S += dsl[j * K + r];
        float* out = a.dZs_ppc + ((size_t)b * K + r) * D;
        for (int g = 0; g < ngrp; ++g) {
            const int d = g * 128 + lane * 4;
            if (d >= D) continue;
            const float4 z = *reinterpret_cast<const float4*>(Zt + (size_t)r * zs + d);
            float4 acc = make_float4(z.x * S, z.y * S, z.z * S, z.w * S);
#pragma unroll 2
            for (int j = 0; j < m; ++j) {
                const float c = -dsl[j * K + r];
                const float4 p = *reinterpret_cast<const float4*>(Prow + j * D + d);
                acc.x = fmaf(c, p.x, acc.x); acc.y = fmaf(c, p.y, acc.y); acc.z = fmaf(c, p.z, acc.z); acc.w = fmaf(c, p.w, acc.w);
            }
            if (a.ppc_dpre) {
                acc.x *= z.x * (1.0f - z.x); acc.y *= z.y * (1.0f - z.y); acc.z *= z.z * (1.0f - z.z); acc.w *= z.w * (1.0f - z.w);
            }
            *reinterpret_cast<float4*>(out + d) = acc;
        }
    }
    // prototype rows of THIS image (summed over the images of a class by the prototype-gradient kernel, in image
    // order: deterministic, unlike the atomics of pph_ppc_bwd): dP_img[b,j,:] = P_j sum_k dd[j,k] - sum_k dd[j,k] Z[b,k,:]
    for (int it = warp * nsplit + part; it < m * ngrp; it += nwarp * nsplit) {       // work item = (prototype, 128-feature group)
        const int j = it / ngrp, g = it - j * ngrp;
        const int d = g * 128 + lane * 4;
        if (d >= D) continue;
        float S = 0.f;
        float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll 4
        for (int r = 0; r < K; ++r) {
            const float c = dsl[j * K + r];
            const float4 z = *reinterpret_cast<const float4*>(Zt + (size_t)r * zs + d);
            S += c;
            acc.x = fmaf(c, z.x, acc.x); acc.y = fmaf(c, z.y, acc.y); acc.z = fmaf(c, z.z, acc.z); acc.w = fmaf(c, z.w, acc.w);
        }
        const float4 p = *reinterpret_cast<const float4*>(Prow + j * D + d);
        *reinterpret_cast<float4*>(a.dP_img + ((size_t)b * m + j) * D + d) =
            make_float4(p.x * S - acc.x, p.y * S - acc.y, p.z * S - acc.z, p.w * S - acc.w);
    }
}

template <int CJ>
__global__ void __launch_bounds__(kMidThreads)
head_mid_kernel(const MidArgs a) {
    pdl_sync();
    extern __shared__ __align__(16) float sm_mid[];
    const int bid = blockIdx.x;
    if (bid < a.n_ll) {
        // one decision for the whole grid: the verdicts were written by an earlier launch and change only in this
        // launch's last class-sum CTA, after every LL CTA has read them
        const LLPattern wl = a.pattern->rec[0], wg = a.pattern->rec[1];
        if (wl.ok && wg.ok) ll_class_role(a, wl, wg, sm_mid);
        else ll_role<CJ>(a, sm_mid);
    } else if (bid < a.n_ll + a.n_bin) {
        bin_tokens_body<false>(bid - a.n_ll, a.argmin_l, a.K, a.P, a.bin_start, a.item_start, a.bin_list,
                        reinterpret_cast<int*>(sm_mid), a.item_desc);
    } else if (bid < a.n_ll + a.n_bin + a.n_ppc) {
        ppc_role(a, bid - a.n_ll - a.n_bin, 0, 1, sm_mid);
    } else {
        // role CLS (one CTA): the images sorted by clamped label (stable counting sort: image order inside a class)
        const int n_cls = a.P / a.m;
        for (int b = threadIdx.x; b < a.B; b += kMidThreads) {
            long y = a.labels[b];
            if (y < 0) y = 0;
            if (y * a.m + a.m > a.P) y = a.P / a.m - 1;
            a.cls_id[b] = (int)y;
        }
        __threadfence();
        __syncthreads();
        bin_tokens_body<true>(0, a.cls_id, n_cls, a.B, a.cls_start, a.cls_item, a.cls_order, reinterpret_cast<int*>(sm_mid));
    }
}

// PPC role as its own launch (use_ppc = 3): two 512-thread CTAs per image
constexpr int kPpcSplit = 2, kPpcThreads = 512;
__global__ void __launch_bounds__(kPpcThreads)
head_ppc_kernel(const MidArgs a) {
    pdl_sync();
    extern __shared__ __align__(16) float sm_mid[];
    ppc_role(a, blockIdx.x / kPpcSplit, blockIdx.x % kPpcSplit, kPpcSplit, sm_mid);
}

struct MidPlan {
    int tiles_b, nsl_l, nsl_g, S_l, S_g, n_ll, Cp, Bp;
    size_t smem_ll, smem_ppc, smem_bin;
};

static MidPlan mid_plan(int B, int K, int D, int P, int Pg, int C, int m, int max_ctas) {
    MidPlan p;
    p.tiles_b = ceil_div(B, kMidTB);
    p.nsl_l = ceil_div(P, kMidPS);
    p.nsl_g = Pg > 0 ? ceil_div(Pg, kMidPS) : 0;
    p.Cp = (C + 3) & ~3;
    p.Bp = p.tiles_b * kMidTB;
    int budget = max_ctas / p.tiles_b;                 // prototype groups per image tile
    const int need = Pg > 0 ? 2 : 1;
    if (budget < need) budget = need;
    if (p.nsl_l + p.nsl_g <= budget) {
        p.S_l = p.nsl_l;
        p.S_g = p.nsl_g;
    } else if (Pg > 0) {
        p.S_l = (int)((long)budget * p.nsl_l / (p.nsl_l + p.nsl_g));
        if (p.S_l < 1) p.S_l = 1;
        if (p.S_l > budget - 1) p.S_l = budget - 1;
        p.S_g = budget - p.S_l;
        if (p.S_l > p.nsl_l) p.S_l = p.nsl_l;
        if (p.S_g > p.nsl_g) p.S_g = p.nsl_g;
    } else {
        p.S_l = budget < p.nsl_l ? budget : p.nsl_l;
        p.S_g = 0;
    }
    p.n_ll = p.tiles_b * (p.S_l + p.S_g);
    const int WST = C | 1;
    p.smem_ll = sizeof(float) * ((size_t)kMidPS * WST + (size_t)kMidPS * kMidAST + (size_t)C * kMidAST + 2 * 4 * 64 * 4 + 3 * 256 + 8);
    p.smem_ppc = sizeof(float) * ((size_t)m * D + (size_t)K * (D + 4) + 2 * (size_t)m * K + 8 * (size_t)m + 32);
    p.smem_bin = bin_tokens_smem_bytes(K);
    return p;
}

struct MidWs {
    LLPatternWs* pattern;
    unsigned int* ctr;
    float *part, *dlT, *ce_part, *ppc_part, *ppc_losses;
    size_t bytes;
};

static MidWs mid_carve(void* base, const MidPlan& p, int B) {
    MidWs w;
    char* q = static_cast<char*>(base);
    size_t off = 0;
    auto take = [&](size_t n) { char* r = q ? q + off : nullptr; off += (n + 255) / 256 * 256; return r; };
    // first: the part that must start zeroed (pph_last_layer_pattern finds its records at offset 0 without the plan)
    w.pattern = reinterpret_cast<LLPatternWs*>(take(sizeof(LLPatternWs)));
    w.ctr = reinterpret_cast<unsigned int*>(take(sizeof(int) * 8));
    w.ppc_losses = reinterpret_cast<float*>(take(sizeof(float) * 2));
    w.ce_part = reinterpret_cast<float*>(take(sizeof(float) * (size_t)B));
    w.ppc_part = reinterpret_cast<float*>(take(sizeof(float) * 2 * (size_t)B));
    w.dlT = reinterpret_cast<float*>(take(sizeof(float) * (size_t)p.Cp * p.Bp));
    w.part = reinterpret_cast<float*>(take(sizeof(float) * (size_t)(p.S_l + p.S_g) * B * p.Cp));
    w.bytes = off + 256;
    return w;
}

static int mid_max_ctas() {
    int n = pph_sm_count();
    return n > 0 ? n : 148;
}

// ---------------------------------------------------------------------------------------------------------------
// pph_last_layer_pattern: is W[c,p] == (p / m == c ? W[0,0] : W[1,0]) for every entry of a (C, n) matrix, m = n / C?
// ---------------------------------------------------------------------------------------------------------------
constexpr int kPatThreads = 256, kPatVecPerThread = 4;

// 1 if this thread's share of W holds an entry off the pattern.  vec4: n % 4 == 0 and W 16-byte aligned, so a float4
// never straddles two rows.
__device__ __forceinline__ unsigned int pattern_scan(const float* __restrict__ W, int C, int n, bool vec4) {
    if (n == 0) return 0u;
    if (n % C != 0) return 1u;
    const int m = n / C, total = C * n;
    const float a = __ldg(W), b = C > 1 ? __ldg(W + n) : a;
    const int t0 = blockIdx.x * blockDim.x + threadIdx.x, stride = gridDim.x * blockDim.x;
    bool bad = false;
    if (vec4) {
        const float4* W4 = reinterpret_cast<const float4*>(W);
#pragma unroll 4
        for (int i = t0; i < total / 4; i += stride) {
            const float4 v = __ldg(W4 + i);
            const int e = 4 * i, c = e / n, p = e - c * n;
            bad |= v.x != ((p / m == c) ? a : b);
            bad |= v.y != (((p + 1) / m == c) ? a : b);
            bad |= v.z != (((p + 2) / m == c) ? a : b);
            bad |= v.w != (((p + 3) / m == c) ? a : b);
        }
    } else {
#pragma unroll 4
        for (int e = t0; e < total; e += stride) {
            const int c = e / n, p = e - c * n;
            bad |= __ldg(W + e) != ((p / m == c) ? a : b);
        }
    }
    return bad ? 1u : 0u;
}

__device__ __forceinline__ LLPattern pattern_record(const float* W, int C, int n, bool bad) {
    LLPattern r;
    r.ok = !bad;
    r.a = n > 0 ? W[0] : 0.f;
    r.b = n > 0 ? (C > 1 ? W[n] : r.a) : 0.f;
    r.unused = 0;
    return r;
}

// Integer flags only: CTAs that saw a mismatch OR a bit into `bad`; the last CTA to take the ticket writes both
// verdicts and resets the counters (self-resetting under graph replay, no host sync).
__global__ void __launch_bounds__(kPatThreads)
last_layer_pattern_kernel(const float* __restrict__ Wl, int P, int vec_l, const float* __restrict__ Wg, int Pg, int vec_g,
                          int C, LLPatternWs* ws) {
    pdl_sync();
    const unsigned int bits = pattern_scan(Wl, C, P, vec_l) | (pattern_scan(Wg, C, Pg, vec_g) << 1);
    const int bad_l = __syncthreads_or(bits & 1u), bad_g = __syncthreads_or(bits & 2u);
    if (threadIdx.x != 0) return;
    if (bad_l || bad_g) atomicOr(&ws->bad, (bad_l ? 1u : 0u) | (bad_g ? 2u : 0u));
    __threadfence();
    if (atomicAdd(&ws->ticket, 1u) != gridDim.x - 1u) return;
    __threadfence();
    const unsigned int all = atomicExch(&ws->bad, 0u);
    ws->rec[0] = pattern_record(Wl, C, P, all & 1u);
    ws->rec[1] = pattern_record(Wg, C, Pg, all & 2u);
    ws->ticket = 0u;
}

}  // namespace pph

extern "C" int pph_last_layer_pattern(const float* Wl, int P, const float* Wg, int Pg, int C, void* workspace,
                                      pph_stream_t stream) {
    using namespace pph;
    PPH_REQUIRE(Wl && workspace && (Pg == 0 || Wg), PPH_EINVAL, "pph_last_layer_pattern: null pointer");
    PPH_REQUIRE(P >= 1 && Pg >= 0 && C >= 1, PPH_EINVAL, "pph_last_layer_pattern: bad dims");
    PPH_REQUIRE((long long)C * P < (1LL << 31) && (long long)C * Pg < (1LL << 31), PPH_EUNSUP,
                "pph_last_layer_pattern: C x P = %lld entries", (long long)C * (P > Pg ? P : Pg));
    auto vec4 = [](const float* W, int n) { return (n % 4 == 0 && (reinterpret_cast<uintptr_t>(W) & 15) == 0) ? 1 : 0; };
    const int vl = vec4(Wl, P), vg = vec4(Wg, Pg);
    const int per_cta = kPatThreads * kPatVecPerThread * 4;             // entries a CTA covers with one pass
    const int ctas = std::min(mid_max_ctas(), std::max(1, ceil_div(C * std::max(P, Pg), per_cta)));
    launch_k(last_layer_pattern_kernel, dim3(ctas), dim3(kPatThreads), 0, as_stream(stream), Wl, P, vl, Wg, Pg, vg, C,
             static_cast<LLPatternWs*>(workspace));
    return launch_status("pph_last_layer_pattern");
}

extern "C" int pph_head_mid_ws_bytes(int B, int K, int D, int P, int Pg, int C, int m, long long* bytes) {
    using namespace pph;
    PPH_REQUIRE(bytes && B >= 1 && K >= 1 && D >= 1 && P >= 1 && Pg >= 0 && C >= 1 && m >= 1, PPH_EINVAL,
                "pph_head_mid_ws_bytes: bad args");
    // sized for the largest plan any device can choose (plans with fewer CTAs have fewer partial planes)
    const MidPlan p = mid_plan(B, K, D, P, Pg, C, m, 1 << 20);
    *bytes = (long long)mid_carve(nullptr, p, B).bytes;
    return 0;
}

extern "C" int pph_head_mid(const float* act_l, const float* act_g, const float* dmin_l, const float* dmin_g,
                            const int32_t* argmin_l, const float* Wl, const float* Wg, const int64_t* labels,
                            int B, int K, int D, int P, int Pg, int C, int m, int N,
                            float global_coe, int act_fn, float eps, float upstream, int train,
                            int use_ppc, const float* Zs, const float* z2s, const float* Pl, const float* p2l,
                            const int32_t* idx32, float cov_thresh, float mean_thresh, float cov_coe, float mean_coe,
                            void* workspace, void* bwd_workspace,
                            float* logits, float* logits_g, float* logits_l, float* losses, float* dlogits,
                            float* g_l, float* g_g, float* pairT, float* dZs_ppc, float* dP_img,
                            float* losses_mirror, pph_stream_t stream) {
    using namespace pph;
    PPH_REQUIRE(act_l && dmin_l && Wl && labels && workspace && logits && logits_g && logits_l && losses, PPH_EINVAL,
                "pph_head_mid: null pointer");
    PPH_REQUIRE(Pg == 0 || (act_g && dmin_g && Wg), PPH_EINVAL, "pph_head_mid: null global-branch pointer");
    PPH_REQUIRE((reinterpret_cast<uintptr_t>(losses_mirror) & 15) == 0, PPH_EINVAL, "pph_head_mid: losses_mirror must be 16-byte aligned");
    PPH_REQUIRE(B >= 1 && K >= 1 && D >= 4 && P >= 1 && Pg >= 0 && C >= 1 && m >= 1 && N >= 2, PPH_EINVAL,
                "pph_head_mid: bad dims");
    PPH_REQUIRE(C <= 256, PPH_EUNSUP, "pph_head_mid: C=%d > 256 (use the modular entry points)", C);
    PPH_REQUIRE(!train || (argmin_l && dlogits && g_l && bwd_workspace && (Pg == 0 || g_g)), PPH_EINVAL,
                "pph_head_mid: null training pointer");
    PPH_REQUIRE(!use_ppc || (Zs && z2s && Pl && p2l && idx32 && (!train || (dZs_ppc && dP_img))), PPH_EINVAL,
                "pph_head_mid: null PPC pointer");
    const int max_ctas = mid_max_ctas();
    const MidPlan p = mid_plan(B, K, D, P, Pg, C, m, max_ctas);
    const MidWs w = mid_carve(workspace, p, B);
    MidArgs a;
    a.B = B; a.Bp = p.Bp; a.K = K; a.D = D; a.P = P; a.Pg = Pg; a.C = C; a.Cp = p.Cp; a.m = m; a.N = N;
    a.side = (int)lrint(sqrt((double)N));
    a.tiles_b = p.tiles_b; a.S_l = p.S_l; a.S_g = p.S_g; a.nsl_l = p.nsl_l; a.nsl_g = p.nsl_g;
    // use_ppc: 0 no PPC loss | 1 PPC role in this launch | 2 this launch runs everything BUT the PPC role, which a
    // concurrent launch (use_ppc = 3) of the same step runs: the second of the two to finish writes losses[0]
    a.ppc_dpre = (use_ppc & 4) ? 1 : 0;       // bit 2: dZs_ppc leaves as dpre (for pph_addon_bwd3's dpre_add_s)
    use_ppc &= 3;
    const bool have_ppc = use_ppc != 0, run_ll = use_ppc != 3, run_ppc = use_ppc == 1 || use_ppc == 3;
    a.have_ppc = have_ppc ? 1 : 0;
    a.n_ll = run_ll ? p.n_ll : 0;
    a.n_bin = (train && run_ll) ? B : 0;
    a.n_ppc = run_ppc ? B : 0;
    a.gc = global_coe; a.eps = eps; a.upstream = upstream; a.cov_thresh = cov_thresh; a.mean_thresh = mean_thresh;
    a.cov_coe = cov_coe; a.mean_coe = mean_coe; a.act_fn = act_fn; a.train = train;
    a.act_l = act_l; a.act_g = act_g; a.dmin_l = dmin_l; a.dmin_g = dmin_g; a.argmin_l = argmin_l;
    a.Wl = Wl; a.Wg = Wg; a.labels = labels;
    a.logits = logits; a.logits_g = logits_g; a.logits_l = logits_l; a.losses = losses; a.dlogits = dlogits;
    a.losses_mirror = losses_mirror;
    a.g_l = g_l; a.g_g = g_g; a.pairT = reinterpret_cast<float2*>(pairT);
    a.part = w.part; a.dlT = w.dlT; a.ce_part = w.ce_part; a.ppc_part = w.ppc_part; a.ppc_losses = w.ppc_losses;
    a.ctr = w.ctr;
    a.pattern = w.pattern;
    a.bin_start = a.item_start = a.bin_list = nullptr;
    a.item_desc = nullptr;
    a.cls_id = a.cls_start = a.cls_item = a.cls_order = nullptr;
    a.n_cls_cta = 0;
    if (train) {
        const Step2Bins bw = carve_bins(bwd_workspace, B, K, P);
        a.bin_start = bw.bin_start; a.item_start = bw.item_start; a.bin_list = bw.bin_list;
        a.item_desc = bw.item_desc;
        a.cls_id = bw.cls_id; a.cls_start = bw.cls_start; a.cls_item = bw.cls_item; a.cls_order = bw.cls_order;
        if (have_ppc && run_ll && bin_tokens_smem_bytes(P / m) <= 200 * 1024) a.n_cls_cta = 1;
    }
    a.Zs = Zs; a.z2s = z2s; a.Pl = Pl; a.p2l = p2l; a.idx = idx32; a.dZs_ppc = dZs_ppc; a.dP_img = dP_img;
    size_t smem = run_ll ? p.smem_ll : 0;
    if (a.n_bin && p.smem_bin > smem) smem = p.smem_bin;
    if (a.n_cls_cta && bin_tokens_smem_bytes(P / m) > smem) smem = bin_tokens_smem_bytes(P / m);
    if (have_ppc) {
        PPH_REQUIRE(D % 4 == 0 && a.side * a.side == N && P >= m && m <= kMidThreads, PPH_EINVAL, "pph_head_mid: bad PPC dims");
        PPH_REQUIRE(p.smem_ppc <= 200 * 1024, PPH_EUNSUP, "pph_head_mid: an image's K x D slice does not fit shared memory");
        if (run_ppc && p.smem_ppc > smem) smem = p.smem_ppc;
    }
    PPH_REQUIRE(smem <= 220 * 1024, PPH_EUNSUP, "pph_head_mid: shared memory %zu B", smem);
    // all LL CTAs must be co-resident (grid barriers): they come first in the grid and number <= SM count
    PPH_REQUIRE(p.n_ll <= max_ctas, PPH_EUNSUP, "pph_head_mid: B=%d needs %d co-resident CTAs (> %d SMs)", B, p.n_ll,
                max_ctas);
    if (use_ppc == 3) {        // PPC role alone: its own kernel, two 512-thread CTAs per image
        cudaError_t e = opt_in_smem(head_ppc_kernel, (int)p.smem_ppc);
        if (e != cudaSuccess) { set_error("pph_head_mid: %s", cudaGetErrorString(e)); return (int)e; }
        launch_k(head_ppc_kernel, dim3(B * kPpcSplit), dim3(kPpcThreads), p.smem_ppc, as_stream(stream), a);
        return launch_status("pph_head_mid(ppc)");
    }
    const int cj = ceil_div(C, 32);
    PPH_REQUIRE(!(have_ppc && train && run_ll) || a.n_cls_cta == 1, PPH_EUNSUP, "pph_head_mid: too many classes");

    const dim3 grid(a.n_ll + a.n_bin + a.n_ppc + a.n_cls_cta), block(kMidThreads);
    cudaStream_t st = as_stream(stream);
#define PPH_MID(CJ)                                                                                                   \
    do {                                                                                                              \
        cudaError_t e = opt_in_smem(head_mid_kernel<CJ>, (int)smem); \
        if (e != cudaSuccess) { set_error("pph_head_mid: %s", cudaGetErrorString(e)); return (int)e; }                \
        launch_k(head_mid_kernel<CJ>, grid, block, smem, st, a);                                                      \
    } while (0)
    if (cj <= 4) PPH_MID(4);
    else if (cj <= 7) PPH_MID(7);
    else PPH_MID(8);
#undef PPH_MID
    return launch_status("pph_head_mid");
}
