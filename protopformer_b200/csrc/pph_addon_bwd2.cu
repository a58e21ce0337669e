// (a8, part 3) backward of gather -> add-on layer -> sigmoid (autograd of protopformer.py:159-172) in ONE launch:
//   dpre = dZ * Z * (1 - Z)                        is the INPUT (pph_similarity_bwd2 writes it with dpre_out = 1), so both
//                                                  operand tiles are staged with plain cp.async copies
//   role X (blockIdx < nX)   dtokens[b, 1+idx[b,j], :] = dpre[r,:] Wa   (CLS row 0 likewise) for a tile of TR rows, and
//                            the zero fill of this CTA's share of the token rows that were not selected
//   role W (the rest)        dWa = dpre^T X_sel, dba = sum_r dpre: 64 x 64 output tiles x S row splits; every split
//                            writes its partial, the last split of a tile to finish adds the S partials in split order
//                            (deterministic: no atomics on data, one ticket counter per tile)
// Replaces the round-1 launches tcgemm<Dx...> || tcgemm<Wgrad...> -> wgrad_reduce_kernel (17 + 35 + 5 us at the CUB
// shape, tensor pipe < 3 % active): the two products are 2 x 193 MFLOP -- what they need is every SM busy with
// back-to-back FMAs, which is what this kernel provides (exact FP32, FP32-pipe bound: 20 k cycles per SM).
#include "pph_common.cuh"

namespace pph {

constexpr int kAbKC = 32;          // role X: rows of Wa per chunk
constexpr int kAbWT = 64;          // role W: output tile edge
constexpr int kAbRC = 32;          // role W: rows per chunk
constexpr int kAbWThreads = 256;

struct AddonBwdArgs {
    int B, N, Din, D, K, R;
    int TR, Dp, nchunks, threadsX, nX;     // role X plan
    int tilesO, tilesI, S, RS, nW;         // role W plan: S row splits of RS rows
    int want_dx, want_dw;
    const float *Wa, *dpre_s, *dpre_c;
    const void* tokens;                    // [B, 1+N, Din] of the kernel's token type (float or bf16)
    const int32_t* idx;
    float *dWa, *dba;
    void* dtokens;                         // same type as tokens
    float *part, *partb;                   // [S][D][Din], [S][D]
    unsigned int* cnt;                     // [tilesO * tilesI]
};

__device__ __forceinline__ void row_of(int r, int K, int& b, int& j) {
    b = r / (K + 1);
    j = r - b * (K + 1);
}

// address of dpre(r, col): selected-token rows live in dpre_s [B,K,D], the CLS row of an image in dpre_c [B,D]
__device__ __forceinline__ const float* dpre_ptr(const AddonBwdArgs& a, int r, int col) {
    int b, j;
    row_of(r, a.K, b, j);
    return (j < a.K ? a.dpre_s + ((size_t)b * a.K + j) * a.D : a.dpre_c + (size_t)b * a.D) + col;
}

// ---- role X ----------------------------------------------------------------------------------------------------
template <class T>
__device__ __forceinline__ void addon_bwd_x(const AddonBwdArgs& a, float* sm) {
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nthr = a.threadsX, nwarp = nthr >> 5;
    const int K = a.K, N = a.N, Din = a.Din, D = a.D, TR = a.TR, Dp = a.Dp;
    const int r0 = blockIdx.x * TR, nrow = min(TR, a.R - r0);
    float* Ds = sm;                                   // [TR][Dp]     dpre rows
    float* Wt = Ds + (size_t)TR * Dp;                  // [2][kAbKC][Din]
    const int d4 = Dp >> 2;
    for (int rl = warp; rl < TR; rl += nwarp) {                  // one warp per row: no division in the copy loop
        const float* src = rl < nrow ? dpre_ptr(a, r0 + rl, 0) : nullptr;
        for (int q = lane; q < d4; q += 32) {
            float* dst = Ds + (size_t)rl * Dp + q * 4;
            if (src && q * 4 < D) cp_async16(dst, src + q * 4);
            else *reinterpret_cast<float4*>(dst) = make_float4(0.f, 0.f, 0.f, 0.f);
        }
    }
    const int i4 = Din >> 2;
    auto issue = [&](int ch, int buf) {
        float* dst = Wt + (size_t)buf * kAbKC * Din;
        for (int ol = warp; ol < kAbKC; ol += nwarp) {
            const int o = ch * kAbKC + ol;
            for (int q = lane; q < i4; q += 32) {
                if (o < D) cp_async16(dst + (size_t)ol * Din + q * 4, a.Wa + (size_t)o * Din + q * 4);
                else *reinterpret_cast<float4*>(dst + (size_t)ol * Din + q * 4) = make_float4(0.f, 0.f, 0.f, 0.f);
            }
        }
        cp_async_commit();
    };
    const int CG = Din >> 3;
    const int ncomp = (TR >> 2) * CG;
    const bool comp = tid < ncomp;
    const int rg = tid / CG, cg = tid - rg * CG;
    float acc[4][8];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 8; ++j) acc[i][j] = 0.f;
    issue(0, 0);
    for (int ch = 0; ch < a.nchunks; ++ch) {
        if (ch + 1 < a.nchunks) {
            issue(ch + 1, (ch + 1) & 1);
            cp_async_wait<1>();
        } else {
            cp_async_wait<0>();
        }
        __syncthreads();
        if (comp) {
            const float* xr = Ds + (size_t)(rg * 4) * Dp + ch * kAbKC;
            const float* wb = Wt + (size_t)(ch & 1) * kAbKC * Din;
            const float* w0 = wb + cg * 4;
            const float* w1 = wb + (Din >> 1) + cg * 4;
#pragma unroll 2
            for (int kk = 0; kk < kAbKC; kk += 4) {
                float4 xv[4];
#pragma unroll
                for (int i = 0; i < 4; ++i) xv[i] = *reinterpret_cast<const float4*>(xr + (size_t)i * Dp + kk);
#pragma unroll
                for (int e = 0; e < 4; ++e) {
                    const float4 b0 = *reinterpret_cast<const float4*>(w0 + (size_t)(kk + e) * Din);
                    const float4 b1 = *reinterpret_cast<const float4*>(w1 + (size_t)(kk + e) * Din);
                    const float bv[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
#pragma unroll
                    for (int i = 0; i < 4; ++i) {
                        const float xa = e == 0 ? xv[i].x : (e == 1 ? xv[i].y : (e == 2 ? xv[i].z : xv[i].w));
#pragma unroll
                        for (int j = 0; j < 8; ++j) acc[i][j] = fmaf(xa, bv[j], acc[i][j]);
                    }
                }
            }
        }
        __syncthreads();
    }
    if (comp) {
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const int rl = rg * 4 + i;
            if (rl >= nrow) continue;
            int b, j;
            row_of(r0 + rl, K, b, j);
            const int tok = j < K ? 1 + __ldg(a.idx + (size_t)b * K + j) : 0;
            T* dst = static_cast<T*>(a.dtokens) + ((size_t)b * (1 + N) + tok) * Din;
#pragma unroll
            for (int h = 0; h < 2; ++h)
                st4_tok(dst + h * (Din >> 1) + cg * 4,
                        make_float4(acc[i][h * 4], acc[i][h * 4 + 1], acc[i][h * 4 + 2], acc[i][h * 4 + 3]));
        }
    }
    // zero fill of the token rows nobody selected: this CTA's share of the B * (1 + N) rows, one warp per row
    const long rows_all = (long)a.B * (1 + N);
    const long per = (rows_all + a.nX - 1) / a.nX;
    const long za = (long)blockIdx.x * per, zb = min(rows_all, za + per);
    for (long row = za + warp; row < zb; row += nwarp) {
        const int b = (int)(row / (1 + N)), t = (int)(row - (long)b * (1 + N));
        if (t == 0) continue;                                    // the CLS row always carries a gradient
        bool hit = false;
        for (int k = lane; k < K; k += 32) hit |= (__ldg(a.idx + (size_t)b * K + k) == t - 1);
        if (__any_sync(0xffffffffu, hit)) continue;
        float4* dst = reinterpret_cast<float4*>(static_cast<T*>(a.dtokens) + (size_t)row * Din);
        const int row16 = Din * (int)sizeof(T) / 16;                   // 16-byte words per row (Din % 8 == 0)
        for (int c = lane; c < row16; c += 32) dst[c] = make_float4(0.f, 0.f, 0.f, 0.f);
    }
}

// ---- role W ----------------------------------------------------------------------------------------------------
// barrier of the 256 threads that run role W (the launch may have more threads per CTA: role X sizes it)
__device__ __forceinline__ void bar_w() { asm volatile("bar.sync 1, 256;" ::: "memory"); }

template <class T>
__device__ __forceinline__ void addon_bwd_w(const AddonBwdArgs& a, int vb, float* sm) {
    const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
    const int K = a.K, N = a.N, Din = a.Din, D = a.D;
    const int tiles = a.tilesO * a.tilesI;
    const int tile = vb % tiles, s = vb / tiles;
    const int to = tile / a.tilesI, ti = tile - to * a.tilesI;
    const int o0 = to * kAbWT, i0 = ti * kAbWT;
    float* As = sm;                                    // [2][kAbRC][64]   dpre rows, columns o0..o0+63
    float* Xs = As + 2 * kAbRC * kAbWT;                // [2][kAbRC][64]   gathered token rows, columns i0..i0+63
    __shared__ unsigned int s_ticket;
    const int rA = s * a.RS, rE = min(a.R, rA + a.RS);
    const int nch = rA < rE ? (rE - rA + kAbRC - 1) / kAbRC : 0;
    float acc[4][4];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;
    float bsum[4] = {0.f, 0.f, 0.f, 0.f};
    // stage chunk ch into buffer buf: both operand tiles are plain copies (gathered token rows, dpre rows)
    const int lr = tid >> 4, lq = tid & 15;            // (row, float4 column) of this thread's two staging elements
    auto issue = [&](int ch, int buf) {
#pragma unroll
        for (int u = 0; u < 2; ++u) {
            const int rl = lr + 16 * u, r = rA + ch * kAbRC + rl;
            float* dx = Xs + ((size_t)buf * kAbRC + rl) * kAbWT + lq * 4;
            float* da = As + ((size_t)buf * kAbRC + rl) * kAbWT + lq * 4;
            if (r < rE) {
                int b, j;
                row_of(r, K, b, j);
                if (i0 + lq * 4 < Din) {
                    const int tok = j < K ? 1 + __ldg(a.idx + (size_t)b * K + j) : 0;
                    const T* src = static_cast<const T*>(a.tokens) + ((size_t)b * (1 + N) + tok) * Din + i0 + lq * 4;
                    if constexpr (sizeof(T) == 4) cp_async16(dx, src);
                    else *reinterpret_cast<float4*>(dx) = ldg4_tok(src);     // bf16: widened on the way in
                } else {
                    *reinterpret_cast<float4*>(dx) = make_float4(0.f, 0.f, 0.f, 0.f);
                }
                if (o0 + lq * 4 < D)
                    cp_async16(da, (j < K ? a.dpre_s + ((size_t)b * K + j) * D : a.dpre_c + (size_t)b * D) + o0 + lq * 4);
                else
                    *reinterpret_cast<float4*>(da) = make_float4(0.f, 0.f, 0.f, 0.f);
            } else {
                *reinterpret_cast<float4*>(dx) = make_float4(0.f, 0.f, 0.f, 0.f);
                *reinterpret_cast<float4*>(da) = make_float4(0.f, 0.f, 0.f, 0.f);
            }
        }
        cp_async_commit();
    };
    if (nch > 0) issue(0, 0);
    for (int ch = 0; ch < nch; ++ch) {
        const int buf = ch & 1;
        if (ch + 1 < nch) {
            issue(ch + 1, buf ^ 1);
            cp_async_wait<1>();
        } else {
            cp_async_wait<0>();
        }
        bar_w();
        const float* Ab = As + (size_t)buf * kAbRC * kAbWT + ty * 4;
        const float* Xb = Xs + (size_t)buf * kAbRC * kAbWT + tx * 4;
#pragma unroll 8
        for (int r = 0; r < kAbRC; ++r) {
            const float4 aa = *reinterpret_cast<const float4*>(Ab + r * kAbWT);
            const float4 xx = *reinterpret_cast<const float4*>(Xb + r * kAbWT);
            const float a4[4] = {aa.x, aa.y, aa.z, aa.w}, x4[4] = {xx.x, xx.y, xx.z, xx.w};
#pragma unroll
            for (int i = 0; i < 4; ++i) {
                bsum[i] += a4[i];
#pragma unroll
                for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(a4[i], x4[j], acc[i][j]);
            }
        }
        bar_w();                                       // buffer buf is free for the copies of chunk ch + 2
    }
    // partial of this split
    float* part = a.part + (size_t)s * D * Din;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const int o = o0 + ty * 4 + i;
        if (o < D && i0 + tx * 4 < Din)
            *reinterpret_cast<float4*>(part + (size_t)o * Din + i0 + tx * 4) = make_float4(acc[i][0], acc[i][1], acc[i][2], acc[i][3]);
        if (ti == 0 && tx == 0 && o < D) a.partb[(size_t)s * D + o] = bsum[i];
    }
    __threadfence();
    bar_w();
    if (tid == 0) s_ticket = atomicAdd(a.cnt + tile, 1u);
    bar_w();
    if (s_ticket != (unsigned int)(a.S - 1)) return;
    __threadfence();
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const int o = o0 + ty * 4 + i;
        if (o >= D) continue;
        if (i0 + tx * 4 < Din) {
            float4 t = make_float4(0.f, 0.f, 0.f, 0.f);
            for (int q = 0; q < a.S; ++q) {
                const float4 v = ldcg4(a.part + ((size_t)q * D + o) * Din + i0 + tx * 4);
                t.x += v.x; t.y += v.y; t.z += v.z; t.w += v.w;
            }
            *reinterpret_cast<float4*>(a.dWa + (size_t)o * Din + i0 + tx * 4) = t;
        }
        if (ti == 0 && tx == 0) {
            float t = 0.f;
            for (int q = 0; q < a.S; ++q) t += __ldcg(a.partb + (size_t)q * D + o);
            a.dba[o] = t;
        }
    }
    if (tid == 0) a.cnt[tile] = 0u;                   // self-resetting (graph replay)
}

template <int MAXT, class T>
__global__ void __launch_bounds__(MAXT, 1)
addon_bwd2_kernel(const AddonBwdArgs a) {
    extern __shared__ __align__(16) float sm_ab[];
    if ((int)blockIdx.x < a.nX) {
        addon_bwd_x<T>(a, sm_ab);
    } else {
        if ((int)threadIdx.x < kAbWThreads) addon_bwd_w<T>(a, blockIdx.x - a.nX, sm_ab);
    }
}

struct AddonBwdPlan {
    int TR, Dp, nchunks, threadsX, nX, tilesO, tilesI, S, RS, nW, threads;
    size_t smem, ws_bytes;
};

static bool addon_bwd_plan(int B, int N, int Din, int D, int K, int sms, AddonBwdPlan* out) {
    AddonBwdPlan p;
    const int R = B * (K + 1);
    int tr = (ceil_div(R, sms) + 3) & ~3;
    if (tr < 32) tr = 32;
    if (tr > 48) tr = 48;
    p.TR = tr;
    p.Dp = ceil_div(D, kAbKC) * kAbKC;
    p.nchunks = p.Dp / kAbKC;
    int thr = (tr / 4) * (Din / 8);
    thr = (thr + 31) & ~31;
    if (thr < kAbWThreads) thr = kAbWThreads;         // role W needs 256 threads
    p.threadsX = thr;
    p.threads = thr;
    if (thr > 640) return false;
    p.nX = ceil_div(R, tr);
    p.tilesO = ceil_div(D, kAbWT);
    p.tilesI = ceil_div(Din, kAbWT);
    const int tiles = p.tilesO * p.tilesI;
    int S = sms / tiles;
    if (S < 1) S = 1;
    if (S > 64) S = 64;
    const int maxS = ceil_div(R, kAbRC);
    if (S > maxS) S = maxS;
    p.RS = ceil_div(ceil_div(R, S), kAbRC) * kAbRC;
    p.S = ceil_div(R, p.RS);
    p.nW = tiles * p.S;
    const size_t sx = sizeof(float) * ((size_t)tr * p.Dp + 2 * (size_t)kAbKC * Din);
    const size_t sw = sizeof(float) * 4 * (size_t)kAbRC * kAbWT;
    p.smem = sx > sw ? sx : sw;
    if (p.smem > 200 * 1024) return false;
    p.ws_bytes = 256 + sizeof(int) * (size_t)((tiles + 63) / 64 * 64) +
                 sizeof(float) * ((size_t)p.S * D * Din + (size_t)p.S * D + 64);
    *out = p;
    return true;
}

}  // namespace pph

extern "C" int pph_addon_bwd2_supported(int B, int N, int Din, int D, int K) {
    using namespace pph;
    if (B < 1 || N < 1 || K < 1 || K > N || Din < 8 || Din % 8 != 0 || D < 4 || D % 4 != 0) return 0;
    AddonBwdPlan p;
    return addon_bwd_plan(B, N, Din, D, K, 148, &p) ? 1 : 0;
}

extern "C" int pph_addon_bwd2_ws_bytes(int B, int N, int Din, int D, int K, long long* bytes) {
    using namespace pph;
    PPH_REQUIRE(bytes, PPH_EINVAL, "pph_addon_bwd2_ws_bytes: null pointer");
    PPH_REQUIRE(pph_addon_bwd2_supported(B, N, Din, D, K), PPH_EUNSUP, "pph_addon_bwd2_ws_bytes: unsupported shape");
    // sized for the largest split count any device can choose (S <= 64)
    AddonBwdPlan p;
    addon_bwd_plan(B, N, Din, D, K, 1 << 16, &p);
    *bytes = (long long)p.ws_bytes;
    return 0;
}

namespace pph {

template <class T>
static int addon_bwd2_impl(const char* name, int parts, const T* tokens, const int32_t* idx32, const float* Wa,
                           const float* dpre_s, const float* dpre_c,
                           int B, int N, int Din, int D, int K, void* workspace,
                           float* dWa, float* dba, T* dtokens, pph_stream_t stream) {
    PPH_REQUIRE((parts & 3) != 0, PPH_EINVAL, "%s: parts must name WGRAD and/or DGRAD", name);
    PPH_REQUIRE(tokens && idx32 && Wa && dpre_s && dpre_c && workspace, PPH_EINVAL, "%s: null pointer", name);
    PPH_REQUIRE(!(parts & PPH_ADDON_WGRAD) || (dWa && dba), PPH_EINVAL, "%s(WGRAD): null output", name);
    PPH_REQUIRE(!(parts & PPH_ADDON_DGRAD) || dtokens, PPH_EINVAL, "%s(DGRAD): null dtokens", name);
    PPH_REQUIRE(sizeof(T) == 4 || Din % 8 == 0, PPH_EINVAL, "%s: bf16 tokens need Din %% 8 == 0 (Din=%d)", name, Din);
    PPH_REQUIRE(pph_addon_bwd2_supported(B, N, Din, D, K), PPH_EUNSUP, "%s: unsupported shape", name);
    int sms = pph_sm_count();
    if (sms <= 0) sms = 148;
    AddonBwdPlan p;
    PPH_REQUIRE(addon_bwd_plan(B, N, Din, D, K, sms, &p), PPH_EUNSUP, "%s: no plan", name);
    AddonBwdArgs a;
    a.B = B; a.N = N; a.Din = Din; a.D = D; a.K = K; a.R = B * (K + 1);
    a.TR = p.TR; a.Dp = p.Dp; a.nchunks = p.nchunks; a.threadsX = p.threadsX;
    a.nX = (parts & PPH_ADDON_DGRAD) ? p.nX : 0;
    a.tilesO = p.tilesO; a.tilesI = p.tilesI; a.S = p.S; a.RS = p.RS;
    a.nW = (parts & PPH_ADDON_WGRAD) ? p.nW : 0;
    a.want_dx = a.nX ? 1 : 0; a.want_dw = a.nW ? 1 : 0;
    a.tokens = tokens; a.Wa = Wa; a.dpre_s = dpre_s; a.dpre_c = dpre_c; a.idx = idx32;
    a.dWa = dWa; a.dba = dba; a.dtokens = dtokens;
    char* w = static_cast<char*>(workspace);
    const int tiles = p.tilesO * p.tilesI;
    a.cnt = reinterpret_cast<unsigned int*>(w);
    size_t off = 256 + sizeof(int) * (size_t)((tiles + 63) / 64 * 64);
    off = (off + 255) / 256 * 256;
    a.part = reinterpret_cast<float*>(w + off);
    a.partb = a.part + (size_t)p.S * D * Din;
    auto k_small = addon_bwd2_kernel<256, T>;
    auto k_large = addon_bwd2_kernel<640, T>;
    auto kern = p.threads <= 256 ? k_small : k_large;
    cudaError_t e = opt_in_smem(kern, (int)p.smem);
    if (e != cudaSuccess) { set_error("%s: %s", name, cudaGetErrorString(e)); return (int)e; }
    launch_k(kern, dim3(a.nX + a.nW), dim3(p.threads), p.smem, as_stream(stream), a);
    return launch_status(name);
}

}  // namespace pph

extern "C" int pph_addon_bwd2(int parts, const float* tokens, const int32_t* idx32, const float* Wa,
                              const float* dpre_s, const float* dpre_c,
                              int B, int N, int Din, int D, int K, void* workspace,
                              float* dWa, float* dba, float* dtokens, pph_stream_t stream) {
    return pph::addon_bwd2_impl("pph_addon_bwd2", parts, tokens, idx32, Wa, dpre_s, dpre_c, B, N, Din, D, K, workspace, dWa,
                                dba, dtokens, stream);
}

extern "C" int pph_addon_bwd2_bf16tok(int parts, const uint16_t* tokens, const int32_t* idx32, const float* Wa,
                                      const float* dpre_s, const float* dpre_c,
                                      int B, int N, int Din, int D, int K, void* workspace,
                                      float* dWa, float* dba, uint16_t* dtokens, pph_stream_t stream) {
    return pph::addon_bwd2_impl("pph_addon_bwd2_bf16tok", parts, tokens, idx32, Wa, dpre_s, dpre_c, B, N, Din, D, K,
                                workspace, dWa, dba, dtokens, stream);
}
