// (a8, part 2) second implementation of the argmin-routed backward of max-pool + similarity + squared-L2 distance
// (autograd of protopformer.py:201-247; restatement SURVEY.md 8(d)(iv)):
//   dPl[p,:]   = 2 (Pl[p,:] sum_b g[b,p] - sum_b g[b,p] Zs[b,argmin[b,p],:])      dPg[p,:] likewise with Zc[b,:]
//   dZs[b,k,:] = 2 (Zs[b,k,:] sum_{p in bin(b,k)} g[b,p] - sum_{p in bin(b,k)} g[b,p] Pl[p,:])
//   dZc[b,:]   = 2 (Zc[b,:] sum_p g_g[b,p] - sum_p g_g[b,p] Pg[p,:])
// The round-1 kernel (pph_similarity_bwd.cu) gathers one D-float row per (image, prototype) pair from L2, twice:
// 197 MB of L2 traffic for 16 MB of operands at the CUB shape, 33 us, latency bound.  Here the feature axis is cut into
// slices and the operand that is gathered FROM is staged in shared memory once per CTA, so the data-dependent reads
// are shared-memory reads and L2 only sees coalesced segments.  Three kernels (PPH_BWD2_* parts) that the caller runs
// on concurrent streams (they have different shared-memory footprints, so separate launches let CTAs of different
// kinds share an SM):
//   TOKENS  CTA = (16-float slice, image group): Pl[:, slice] resident (P x 64 B).  Per image the bin-sorted list of
//           (row offset, g) is cut into chunks of 16 entries -- one chunk per 4-lane group, so the work is balanced
//           however skewed the argmin distribution is; a chunk that crosses bin boundaries leaves one partial per
//           (chunk, bin) in shared memory at slot chunk + bin (unique, ordered), and a second pass adds the partials
//           of each bin in slot order: deterministic.  -> dZs rows (or dpre = dZ * Z * (1 - Z), see below)
//   PROTOS  CTA = (4-float slice, 512 prototypes): Zs/Zc[:, :, slice] of 64 images resident (84 KB: two CTAs per SM);
//           a lane owns two prototypes and walks their pairT rows = (g, token slot) per image.  -> dPl, dPg rows,
//           including the PPC rows of the prototype's class (added in image order from the class lists of pph_head_mid)
//   CLS     CTA = (16-float slice, 1/8 of the global prototypes): dense; a lane owns two images, every Pg row read
//           feeds all 64 images of the chunk; per-warp partials are added in warp order, the 8 prototype splits by the
//           last CTA to finish in split order.  -> dZc rows (or dpre)
// Every output element has one writer and a fixed summation order -> bit-reproducible, no atomics on data.
// dpre_out != 0: the token-side outputs are multiplied by Z (1 - Z) while they are written, i.e. they are the
// pre-activation gradients pph_addon_bwd2 consumes (saves that kernel a pass over Z and dZ).
#include "pph_common.cuh"
#include "pph_step2.cuh"

namespace pph {

constexpr int kG2DS = 16;            // floats per slice row (TOKENS, CLS)
constexpr int kG2CH = 16;            // entries per chunk (TOKENS)
constexpr int kG2TokThreads = 512;
constexpr int kG2ProThreads = 256;
constexpr int kG2ProPT = 512;        // prototypes per PROTOS CTA (8 warps x 32 lanes x 2)
constexpr int kG2ProMaxIB = 64;      // images resident per PROTOS chunk (fewer when K is large)
constexpr int kG2ClsThreads = 256;
constexpr int kG2ClsSplit = 8;       // prototype splits (CLS)
constexpr int kG2ClsIB = 64;         // images per CLS chunk (a lane owns two)

struct Grad2Args {
    int B, Bp, K, D, P, Pg, m;
    int NS, IA, nIG;                  // TOKENS: slices of 16, images per CTA, image groups
    int NS4, nPT, IB;                 // PROTOS: slices of 4, prototype tiles over [0, P + Pg), images per chunk (even)
    int psplit;                       // CLS: global prototypes per split
    int dpre_out;
    const float *g_l, *g_g;
    const float2* pairT;
    const int32_t *bin_start, *bin_list, *cls_start, *cls_order;
    const float *Zs, *Zc, *Pl, *Pgl;
    const float *add_dZs, *dP_img;
    float *dZs, *dZc, *dPl, *dPg;
    float* cls_part;                  // [NS][kG2ClsSplit][B][17]
    unsigned int* cls_cnt;            // [NS]
};

__device__ __forceinline__ float4 fma4(float s, float4 v, float4 a) {
    a.x = fmaf(s, v.x, a.x); a.y = fmaf(s, v.y, a.y); a.z = fmaf(s, v.z, a.z); a.w = fmaf(s, v.w, a.w);
    return a;
}
// shared-memory accessors on 32-bit shared-window addresses (keeps the inner loops free of 64-bit pointer arithmetic)
__device__ __forceinline__ float4 lds128(uint32_t addr) {
    float4 v;
    asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(addr));
    return v;
}
__device__ __forceinline__ float2 lds64(uint32_t addr) {
    float2 v;
    asm volatile("ld.shared.v2.f32 {%0, %1}, [%2];" : "=f"(v.x), "=f"(v.y) : "r"(addr));
    return v;
}
// final combine of a token-side row: 2 (z gs - acc) [+ add] [* z (1 - z)]
__device__ __forceinline__ float4 token_out(float4 z, float gs, float4 acc, const float4* add, bool dpre) {
    float4 r;
    r.x = 2.0f * (z.x * gs - acc.x); r.y = 2.0f * (z.y * gs - acc.y);
    r.z = 2.0f * (z.z * gs - acc.z); r.w = 2.0f * (z.w * gs - acc.w);
    if (add) { r.x += add->x; r.y += add->y; r.z += add->z; r.w += add->w; }
    if (dpre) { r.x *= z.x * (1.0f - z.x); r.y *= z.y * (1.0f - z.y); r.z *= z.z * (1.0f - z.z); r.w *= z.w * (1.0f - z.w); }
    return r;
}

// ---------------------------------------------------------------------------------------------------------------
// TOKENS
// ---------------------------------------------------------------------------------------------------------------
// The CTA's 16 warps form kG2TokGroups independent groups; each group walks its own images with private staging
// buffers and its own named barrier, so the exposed latencies of one group's phases (list gather -> barrier -> walk ->
// barrier -> final loads / stores) are covered by the other groups' work.
constexpr int kG2TokGroups = 2;
constexpr int kG2TokGT = kG2TokThreads / kG2TokGroups;        // threads per group

__device__ __forceinline__ void group_bar(int g) { asm volatile("bar.sync %0, %1;" ::"r"(g + 1), "n"(kG2TokGT) : "memory"); }

__global__ void __launch_bounds__(kG2TokThreads, 1)
grad2_tokens_kernel(const Grad2Args a) {
    extern __shared__ __align__(16) float sm_g2[];
    const int K = a.K, P = a.P, D = a.D;
    const int NC = (P + kG2CH - 1) / kG2CH;                 // chunks per image
    const int NSEG = NC + K;                                // partial slots: chunk + bin
    const int Pe = (P + 1) & ~1;
    // shared memory: Psl [P][16] | per group: sp [Pe] float2, seg [NSEG][20], bst [K+1], kc [NC]
    float* Psl = sm_g2;
    const size_t grp_floats = 2 * (size_t)Pe + (size_t)NSEG * 20 + (size_t)((K + 1 + NC + 3) & ~3);
    const int tid = threadIdx.x, g = tid / kG2TokGT, gt = tid - g * kG2TokGT;
    const int lane = tid & 31, gw = gt >> 5, grp = lane >> 2, dq = lane & 3;
    float* gbase = Psl + (size_t)P * kG2DS + (size_t)g * grp_floats;
    float2* sp = reinterpret_cast<float2*>(gbase);           // (row offset bits, g), bin order
    float* seg = gbase + 2 * (size_t)Pe;                     // float4 x 4 lanes + gs per slot
    int* bst = reinterpret_cast<int*>(seg + (size_t)NSEG * 20);
    int* kc = bst + (K + 1);                                 // bin of the first entry of each chunk
    const int sa = blockIdx.x % a.NS, ig = blockIdx.x / a.NS;
    const int c0 = sa * kG2DS;
    const int bA = ig * a.IA, bE = min(a.B, bA + a.IA);
    for (int i = tid; i < P * 4; i += kG2TokThreads)
        cp_async16(Psl + (i >> 2) * kG2DS + (i & 3) * 4, a.Pl + (size_t)(i >> 2) * D + c0 + (i & 3) * 4);
    cp_async_commit();
    cp_async_wait<0>();
    __syncthreads();
    const uint32_t psl_u = (uint32_t)__cvta_generic_to_shared(Psl) + dq * 16;
    const uint32_t sp_u = (uint32_t)__cvta_generic_to_shared(sp);
    const uint32_t seg_u = (uint32_t)__cvta_generic_to_shared(seg);
    constexpr int EPT = 4;                                   // list entries staged per thread and pass
    for (int b = bA + g; b < bE; b += kG2TokGroups) {
        // ---- stage this image's list: (prototype -> row offset, g) in bin order, and the bin offsets -------------
        {
            const int32_t* list = a.bin_list + (size_t)b * P;
            const float* gb = a.g_l + (size_t)b * P;
            for (int e0 = gt; e0 < P; e0 += EPT * kG2TokGT) {
                int p[EPT];
                float gv[EPT];
#pragma unroll
                for (int u = 0; u < EPT; ++u) p[u] = e0 + u * kG2TokGT < P ? __ldg(list + e0 + u * kG2TokGT) : 0;
#pragma unroll
                for (int u = 0; u < EPT; ++u) gv[u] = __ldg(gb + p[u]);
#pragma unroll
                for (int u = 0; u < EPT; ++u)
                    if (e0 + u * kG2TokGT < P) sp[e0 + u * kG2TokGT] = make_float2(__int_as_float(p[u] * (kG2DS * 4)), gv[u]);
            }
            for (int k = gt; k <= K; k += kG2TokGT) bst[k] = __ldg(a.bin_start + (size_t)b * (K + 1) + k);
        }
        group_bar(g);
        for (int c = gt; c < NC; c += kG2TokGT) {           // bin of entry c * CH: the last k with bst[k] <= e
            const int e = c * kG2CH;
            int lo = 0, hi = K - 1;
            while (lo < hi) {
                const int mid = (lo + hi + 1) >> 1;
                if (bst[mid] <= e) lo = mid; else hi = mid - 1;
            }
            kc[c] = lo;
        }
        group_bar(g);
        // ---- walk: one chunk per 4-lane sub-group -------------------------------------------------------------------
        for (int c = gw * 8 + grp; c < NC; c += (kG2TokGT / 32) * 8) {
            int e = c * kG2CH;
            const int e1 = min(P, e + kG2CH);
            int k = kc[c];
            while (e < e1) {
                const int send = min(e1, bst[k + 1]);
                float4 acc = make_float4(0.f, 0.f, 0.f, 0.f), acc2 = acc;
                float gs = 0.f, gs2 = 0.f;
                uint32_t pe = sp_u + (uint32_t)e * 8u;
                const uint32_t pend = sp_u + (uint32_t)send * 8u;
                for (; pe + 8u < pend; pe += 16u) {
                    const float2 q0 = lds64(pe), q1 = lds64(pe + 8u);
                    const float4 v0 = lds128(psl_u + (uint32_t)__float_as_int(q0.x));
                    const float4 v1 = lds128(psl_u + (uint32_t)__float_as_int(q1.x));
                    acc = fma4(q0.y, v0, acc);
                    acc2 = fma4(q1.y, v1, acc2);
                    gs += q0.y;
                    gs2 += q1.y;
                }
                if (pe < pend) {
                    const float2 q0 = lds64(pe);
                    const float4 v0 = lds128(psl_u + (uint32_t)__float_as_int(q0.x));
                    acc = fma4(q0.y, v0, acc);
                    gs += q0.y;
                }
                acc.x += acc2.x; acc.y += acc2.y; acc.z += acc2.z; acc.w += acc2.w;
                float* sg = seg + (size_t)(c + k) * 20;
                *reinterpret_cast<float4*>(sg + dq * 4) = acc;
                if (dq == 0) sg[16] = gs + gs2;
                e = send;
                if (e < e1) {
                    ++k;
                    while (bst[k + 1] <= e) ++k;              // skip empty bins
                }
            }
        }
        group_bar(g);
        // ---- second pass: bin totals in slot order, final combine, store ----------------------------------------------
        for (int t = gt; t < K * 4; t += kG2TokGT) {
            const int k = t >> 2, q = t & 3;
            const size_t o = ((size_t)b * K + k) * D + c0 + q * 4;
            const float4 z = __ldg(reinterpret_cast<const float4*>(a.Zs + o));      // in flight during the slot sums
            float4 ad;
            if (a.add_dZs) ad = __ldg(reinterpret_cast<const float4*>(a.add_dZs + o));
            const int e0 = bst[k], e1 = bst[k + 1];
            float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
            float gs = 0.f;
            if (e0 < e1) {
                const int clo = e0 / kG2CH, chi = (e1 - 1) / kG2CH;
                for (int c = clo; c <= chi; ++c) {
                    const float4 v = lds128(seg_u + (uint32_t)(c + k) * 80u + q * 16);
                    acc.x += v.x; acc.y += v.y; acc.z += v.z; acc.w += v.w;
                    gs += seg[(c + k) * 20 + 16];
                }
            }
            *reinterpret_cast<float4*>(a.dZs + o) = token_out(z, gs, acc, a.add_dZs ? &ad : nullptr, a.dpre_out != 0);
        }
        group_bar(g);
    }
}

// ---------------------------------------------------------------------------------------------------------------
// PROTOS
// ---------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kG2ProThreads)
grad2_protos_kernel(const Grad2Args a) {
    extern __shared__ __align__(16) float sm_g2[];
    const int K = a.K, D = a.D, B = a.B, P = a.P, R = K + 1;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int s4 = blockIdx.x % a.NS4, pt = blockIdx.x / a.NS4;
    const int c0 = s4 * 4;
    const int PA = P + a.Pg;
    float* Zsl = sm_g2;                                      // [IB][K+1][4]: row K of an image = its CLS feature
    int p0 = pt * kG2ProPT + warp * 64 + lane, p1 = p0 + 32;
    const bool ok0 = p0 < PA, ok1 = p1 < PA;
    if (!ok0) p0 = PA - 1;                                   // clamped duplicates compute in lockstep, are not stored
    if (!ok1) p1 = PA - 1;
    const float4* pr0 = reinterpret_cast<const float4*>(a.pairT + (size_t)p0 * a.Bp);
    const float4* pr1 = reinterpret_cast<const float4*>(a.pairT + (size_t)p1 * a.Bp);
    const uint32_t zsl_u = (uint32_t)__cvta_generic_to_shared(Zsl);
    float4 acc0 = make_float4(0.f, 0.f, 0.f, 0.f), acc1 = acc0;
    float gs0 = 0.f, gs1 = 0.f;
    const int last_pair = (a.Bp >> 1) - 1;
    for (int b0 = 0; b0 < B; b0 += a.IB) {
        const int n = min(a.IB, B - b0);
        __syncthreads();                                     // previous chunk's readers are done
        {
            const float* zs = a.Zs + (size_t)b0 * K * D + c0;
            const float* zc = a.Zc + (size_t)b0 * D + c0;
            float* dst = Zsl;
            for (int bi = 0; bi < n; ++bi, zs += (size_t)K * D, zc += D, dst += R * 4)
                for (int i = tid; i < R; i += kG2ProThreads) cp_async16(dst + i * 4, i < K ? zs + (size_t)i * D : zc);
        }
        cp_async_commit();
        float4 n0 = __ldg(pr0 + (b0 >> 1)), n1 = __ldg(pr1 + (b0 >> 1));
        cp_async_wait<0>();
        __syncthreads();
        uint32_t zb = zsl_u;
        const uint32_t rowpair = (uint32_t)(R * 16);
#pragma unroll 2
        for (int bi = 0; bi < n; bi += 2, zb += 2 * rowpair) {
            const float4 q0 = n0, q1 = n1;
            const int nx = min((b0 + bi + 2) >> 1, last_pair);          // clamped prefetch of the next image pair
            n0 = __ldg(pr0 + nx);
            n1 = __ldg(pr1 + nx);
            const float4 v00 = lds128(zb + (uint32_t)__float_as_int(q0.y) * 16u);
            const float4 v10 = lds128(zb + (uint32_t)__float_as_int(q1.y) * 16u);
            acc0 = fma4(q0.x, v00, acc0);
            acc1 = fma4(q1.x, v10, acc1);
            gs0 += q0.x;
            gs1 += q1.x;
            if (bi + 1 < n) {        // images >= B carry g = 0 but their rows are not staged: mask the second image
                const float4 v01 = lds128(zb + rowpair + (uint32_t)__float_as_int(q0.w) * 16u);
                const float4 v11 = lds128(zb + rowpair + (uint32_t)__float_as_int(q1.w) * 16u);
                acc0 = fma4(q0.z, v01, acc0);
                acc1 = fma4(q1.z, v11, acc1);
                gs0 += q0.z;
                gs1 += q1.z;
            }
        }
    }
#pragma unroll
    for (int j = 0; j < 2; ++j) {
        if (!(j ? ok1 : ok0)) continue;
        const int p = j ? p1 : p0;
        const float4 acc = j ? acc1 : acc0;
        const float gs = j ? gs1 : gs0;
        const bool glob = p >= P;
        const size_t o = (size_t)(glob ? p - P : p) * D + c0;
        const float4 base = __ldg(reinterpret_cast<const float4*>((glob ? a.Pgl : a.Pl) + o));
        float4 r;
        r.x = 2.0f * (base.x * gs - acc.x); r.y = 2.0f * (base.y * gs - acc.y);
        r.z = 2.0f * (base.z * gs - acc.z); r.w = 2.0f * (base.w * gs - acc.w);
        if (!glob && a.dP_img) {       // PPC rows of the images labelled with this prototype's class, in image order
            const int cls = p / a.m, jj = p - cls * a.m;
            const int i0 = __ldg(a.cls_start + cls), i1 = __ldg(a.cls_start + cls + 1);
            for (int i = i0; i < i1; ++i) {
                const int b = __ldg(a.cls_order + i);
                const float4 ad = __ldg(reinterpret_cast<const float4*>(a.dP_img + ((size_t)b * a.m + jj) * D + c0));
                r.x += ad.x; r.y += ad.y; r.z += ad.z; r.w += ad.w;
            }
        }
        *reinterpret_cast<float4*>((glob ? a.dPg : a.dPl) + o) = r;
    }
}

// ---------------------------------------------------------------------------------------------------------------
// CLS
// ---------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kG2ClsThreads)
grad2_cls_kernel(const Grad2Args a) {
    extern __shared__ __align__(16) float sm_g2[];
    const int D = a.D, Pg = a.Pg, B = a.B, P = a.P;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nwarp = kG2ClsThreads / 32;
    const int sc = blockIdx.x % a.NS, sp_ = blockIdx.x / a.NS;
    const int c0 = sc * kG2DS;
    const int pA = sp_ * a.psplit, pE = min(Pg, pA + a.psplit), np = max(0, pE - pA);
    float* Gsl = sm_g2;                                      // [psplit][16]
    float* red = Gsl + (size_t)a.psplit * kG2DS;             // [nwarp][64 images][17]
    __shared__ unsigned int s_ticket;
    for (int i = tid; i < np * 4; i += kG2ClsThreads)
        cp_async16(Gsl + (i >> 2) * kG2DS + (i & 3) * 4, a.Pgl + (size_t)(pA + (i >> 2)) * D + c0 + (i & 3) * 4);
    cp_async_commit();
    cp_async_wait<0>();
    __syncthreads();
    const uint32_t g_u = (uint32_t)__cvta_generic_to_shared(Gsl);
    const int per = (np + nwarp - 1) / nwarp;
    const int wA = min(np, warp * per), wE = min(np, wA + per);
    for (int b0 = 0; b0 < B; b0 += kG2ClsIB) {
        // a lane owns images b0 + 2 lane, + 1: one coalesced 16-byte read of pairT per prototype covers both
        float4 acc[2][4];
        float gs[2] = {0.f, 0.f};
#pragma unroll
        for (int j = 0; j < 2; ++j)
#pragma unroll
            for (int q = 0; q < 4; ++q) acc[j][q] = make_float4(0.f, 0.f, 0.f, 0.f);
        const float4* pr = reinterpret_cast<const float4*>(a.pairT + (size_t)(P + pA) * a.Bp + b0) + lane;
        const size_t pstride = (size_t)a.Bp >> 1;            // float4 per pairT row
#pragma unroll 4
        for (int p = wA; p < wE; ++p) {
            const float4 q = __ldg(pr + (size_t)p * pstride);
            const uint32_t row = g_u + (uint32_t)p * 64u;
#pragma unroll
            for (int qq = 0; qq < 4; ++qq) {
                const float4 v = lds128(row + qq * 16);
                acc[0][qq] = fma4(q.x, v, acc[0][qq]);
                acc[1][qq] = fma4(q.z, v, acc[1][qq]);
            }
            gs[0] += q.x;
            gs[1] += q.z;
        }
        __syncthreads();                                     // previous chunk's reduction has been read
#pragma unroll
        for (int j = 0; j < 2; ++j) {
            float* r = red + ((size_t)warp * kG2ClsIB + 2 * lane + j) * 17;
#pragma unroll
            for (int qq = 0; qq < 4; ++qq) {
                r[qq * 4 + 0] = acc[j][qq].x; r[qq * 4 + 1] = acc[j][qq].y; r[qq * 4 + 2] = acc[j][qq].z; r[qq * 4 + 3] = acc[j][qq].w;
            }
            r[16] = gs[j];
        }
        __syncthreads();
        // per-CTA partial of this prototype split: warps added in warp order
        const int n = min(kG2ClsIB, B - b0);
        for (int t = tid; t < n * 17; t += kG2ClsThreads) {
            float s = 0.f;
#pragma unroll
            for (int w = 0; w < kG2ClsThreads / 32; ++w) s += red[(size_t)w * kG2ClsIB * 17 + t];
            a.cls_part[(((size_t)sc * kG2ClsSplit + sp_) * B + b0) * 17 + t] = s;
        }
    }
    // the last split of this slice to finish adds the splits in split order and writes the rows
    __threadfence();
    __syncthreads();
    if (tid == 0) s_ticket = atomicAdd(a.cls_cnt + sc, 1u);
    __syncthreads();
    if (s_ticket != (unsigned int)(kG2ClsSplit - 1)) return;
    __threadfence();
    for (int t = tid; t < B * 4; t += kG2ClsThreads) {
        const int b = t >> 2, q = t & 3;
        float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
        float gs = 0.f;
        for (int s = 0; s < kG2ClsSplit; ++s) {
            const float* pp = a.cls_part + (((size_t)sc * kG2ClsSplit + s) * B + b) * 17;
            acc.x += __ldcg(pp + q * 4 + 0); acc.y += __ldcg(pp + q * 4 + 1);
            acc.z += __ldcg(pp + q * 4 + 2); acc.w += __ldcg(pp + q * 4 + 3);
            gs += __ldcg(pp + 16);
        }
        const size_t o = (size_t)b * D + c0 + q * 4;
        const float4 z = __ldg(reinterpret_cast<const float4*>(a.Zc + o));
        *reinterpret_cast<float4*>(a.dZc + o) = token_out(z, gs, acc, nullptr, a.dpre_out != 0);
    }
    if (tid == 0) a.cls_cnt[sc] = 0u;                        // self-resetting (graph replay)
}

static size_t g2_tok_smem(int K, int P) {
    const int NC = (P + kG2CH - 1) / kG2CH;
    const size_t grp = 2 * (size_t)((P + 1) & ~1) + (size_t)(NC + K) * 20 + (size_t)((K + 1 + NC + 3) & ~3);
    return sizeof(float) * ((size_t)P * kG2DS + kG2TokGroups * grp);
}
static int g2_pro_ib(int K) {
    int ib = (int)((size_t)100 * 1024 / ((size_t)(K + 1) * 16)) & ~1;
    return ib > kG2ProMaxIB ? kG2ProMaxIB : ib;
}
static size_t g2_pro_smem(int K) { return sizeof(float) * (size_t)g2_pro_ib(K) * (K + 1) * 4; }
static int g2_cls_psplit(int Pg) { return (Pg + kG2ClsSplit - 1) / kG2ClsSplit; }
static size_t g2_cls_smem(int Pg) {
    return sizeof(float) * ((size_t)g2_cls_psplit(Pg) * kG2DS + (size_t)(kG2ClsThreads / 32) * kG2ClsIB * 17);
}
static size_t g2_ws_bytes(int B, int K, int D, int P) {
    return carve_bins(nullptr, B, K, P).bytes + 256 + sizeof(float) * (size_t)(D / kG2DS) * kG2ClsSplit * B * 17 +
           sizeof(int) * (size_t)((D / kG2DS + 63) / 64 * 64 + 64);
}

}  // namespace pph

extern "C" int pph_similarity_bwd2_supported(int B, int K, int D, int P, int Pg) {
    using namespace pph;
    if (B < 1 || K < 1 || P < 1 || Pg < 0 || D < kG2DS || D % kG2DS != 0) return 0;
    return (g2_tok_smem(K, P) <= 220 * 1024 && g2_pro_ib(K) >= 2 && g2_cls_smem(Pg) <= 110 * 1024) ? 1 : 0;
}

extern "C" int pph_similarity_bwd2_ws_bytes(int B, int K, int D, int P, long long* bytes) {
    using namespace pph;
    PPH_REQUIRE(bytes && B >= 1 && K >= 1 && P >= 1 && D >= kG2DS, PPH_EINVAL, "pph_similarity_bwd2_ws_bytes: bad args");
    *bytes = (long long)g2_ws_bytes(B, K, D, P);
    return 0;
}

extern "C" int pph_similarity_bwd2(int parts, const float* g_l, const float* g_g, const float* pairT, void* bwd_workspace,
                                   const float* Zs, const float* Zc, const float* Pl, const float* Pgl,
                                   int B, int K, int D, int P, int Pg, int m,
                                   const float* add_dZs, const float* dP_img, int dpre_out,
                                   float* dZs, float* dZc, float* dPl, float* dPg, pph_stream_t stream) {
    using namespace pph;
    PPH_REQUIRE((parts & 7) != 0, PPH_EINVAL, "pph_similarity_bwd2: parts must name at least one of TOKENS|PROTOS|CLS");
    PPH_REQUIRE(g_l && pairT && bwd_workspace && Zs && Pl, PPH_EINVAL, "pph_similarity_bwd2: null pointer");
    PPH_REQUIRE(Pg == 0 || (g_g && Zc && Pgl), PPH_EINVAL, "pph_similarity_bwd2: null global pointer");
    PPH_REQUIRE(!dP_img || m >= 1, PPH_EINVAL, "pph_similarity_bwd2: dP_img needs m");
    PPH_REQUIRE(pph_similarity_bwd2_supported(B, K, D, P, Pg), PPH_EUNSUP,
                "pph_similarity_bwd2: shape B=%d K=%d D=%d P=%d Pg=%d (D %% 16, shared memory)", B, K, D, P, Pg);
    const Step2Bins bins = carve_bins(bwd_workspace, B, K, P);
    Grad2Args a;
    a.B = B; a.Bp = ceil_div(B, 64) * 64; a.K = K; a.D = D; a.P = P; a.Pg = Pg; a.m = m > 0 ? m : 1;
    a.NS = D / kG2DS;
    a.NS4 = D / 4;
    int sms = pph_sm_count();
    if (sms <= 0) sms = 148;
    a.IA = ceil_div(B * a.NS, sms);                  // one TOKENS CTA per SM
    if (a.IA < 1) a.IA = 1;
    a.nIG = ceil_div(B, a.IA);
    a.nPT = ceil_div(P + Pg, kG2ProPT);
    a.IB = g2_pro_ib(K);
    a.psplit = g2_cls_psplit(Pg);
    a.dpre_out = dpre_out;
    a.g_l = g_l; a.g_g = g_g; a.pairT = reinterpret_cast<const float2*>(pairT);
    a.bin_start = bins.bin_start; a.bin_list = bins.bin_list; a.cls_start = bins.cls_start; a.cls_order = bins.cls_order;
    a.Zs = Zs; a.Zc = Zc; a.Pl = Pl; a.Pgl = Pgl; a.add_dZs = add_dZs; a.dP_img = dP_img;
    a.dZs = dZs; a.dZc = dZc; a.dPl = dPl; a.dPg = dPg;
    char* extra = static_cast<char*>(bwd_workspace) + bins.bytes;
    a.cls_cnt = reinterpret_cast<unsigned int*>(extra);
    a.cls_part = reinterpret_cast<float*>(extra + sizeof(int) * (size_t)((a.NS + 63) / 64 * 64));
    cudaStream_t st = as_stream(stream);
    if (parts & PPH_BWD2_TOKENS) {
        PPH_REQUIRE(dZs, PPH_EINVAL, "pph_similarity_bwd2(TOKENS): null dZs");
        const size_t smem = g2_tok_smem(K, P);
        cudaError_t e = opt_in_smem(grad2_tokens_kernel, (int)smem);
        if (e != cudaSuccess) { set_error("pph_similarity_bwd2: %s", cudaGetErrorString(e)); return (int)e; }
        launch_k(grad2_tokens_kernel, dim3(a.NS * a.nIG), dim3(kG2TokThreads), smem, st, a);
        const int rc = launch_status("pph_similarity_bwd2(tokens)");
        if (rc) return rc;
    }
    if (parts & PPH_BWD2_PROTOS) {
        PPH_REQUIRE(dPl && (Pg == 0 || dPg), PPH_EINVAL, "pph_similarity_bwd2(PROTOS): null output");
        const size_t smem = g2_pro_smem(K);
        cudaError_t e = opt_in_smem(grad2_protos_kernel, (int)smem);
        if (e != cudaSuccess) { set_error("pph_similarity_bwd2: %s", cudaGetErrorString(e)); return (int)e; }
        launch_k(grad2_protos_kernel, dim3(a.NS4 * a.nPT), dim3(kG2ProThreads), smem, st, a);
        const int rc = launch_status("pph_similarity_bwd2(protos)");
        if (rc) return rc;
    }
    if ((parts & PPH_BWD2_CLS) && Pg > 0) {
        PPH_REQUIRE(dZc, PPH_EINVAL, "pph_similarity_bwd2(CLS): null dZc");
        const size_t smem = g2_cls_smem(Pg);
        cudaError_t e = opt_in_smem(grad2_cls_kernel, (int)smem);
        if (e != cudaSuccess) { set_error("pph_similarity_bwd2: %s", cudaGetErrorString(e)); return (int)e; }
        launch_k(grad2_cls_kernel, dim3(a.NS * kG2ClsSplit), dim3(kG2ClsThreads), smem, st, a);
        const int rc = launch_status("pph_similarity_bwd2(cls)");
        if (rc) return rc;
    }
    return 0;
}
