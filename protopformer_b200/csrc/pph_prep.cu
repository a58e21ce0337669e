// Head of the training / inference step in ONE launch: foreground-token selection, gather, 'regular' add-on layer
// (1x1 conv == per-token linear map) + sigmoid, the centred bf16 hi/lo operands and the three norm flavours the
// tcgen05 similarity kernel consumes, and -- spread over the same CTAs -- the operand split of both prototype
// tensors.  Replaces protopformer.py:156-172 (+ the p2 term of :207-208) and the round-1 launches select_topk ->
// tcgemm<Fwd...> || split_rows x2.
//
// Rows r in [0, B*(K+1)): b = r / (K+1), j = r % (K+1); j < K: selected patch token idx[b,j] -> Zs[b,j,:];
// j == K: CLS token -> Zc[b,:].  One CTA = TR consecutive rows x all D outputs:
//   1. every image the tile touches is ranked by counting (the rule of pph_select.cu: larger score first, lower index
//      on ties, NaN counts as +inf like torch.topk) -> ascending index list in shared memory; the CTA that owns row
//      j = 0 of an image publishes idx32[b,:] (and idx64);
//   2. the TR source token rows are gathered with 16-byte cp.async copies (768 B rows at the CUB shape);
//   3. exact FP32 FMA contraction against Wa, streamed through shared memory in k-chunks that are transposed on the
//      way in (register double buffer: chunk i+1 is in flight while chunk i is multiplied); thread = 4 rows x 8 columns;
//   4. epilogue: bias, sigmoid, fp32 + centred bf16 hi/lo stores, row norms by a fixed-order shared-memory sum.
// 387 MFLOP at the CUB shape, B = 64: FP32-pipe bound (10.4 k cycles per SM at 128 FMA/clk), one CTA per SM.
#include <math.h>

#include "pph_common.cuh"

namespace pph {

constexpr int kPrepMaxN = 1024;

struct PrepArgs {
    int B, H, N, Din, D, K, R;         // R = B * (K + 1)
    int TR, KC, nchunks, Dinp;         // rows per CTA, k-chunk, number of chunks, Din padded to a multiple of KC
    int max_img;                       // images one tile can touch
    int threads;
    float center;
    const float *scores, *Wa, *ba;
    const void* tokens;                // [B, 1+N, Din] of the kernel's token type (float or bf16)
    int32_t* idx32;
    int64_t* idx64;
    float *Zs, *Zc, *z2s, *z2c, *z2s_ctr, *z2c_ctr, *z2s_hi, *z2c_hi;
    uint16_t *Zs_hi, *Zs_lo, *Zc_hi, *Zc_lo;
    // prototype operand split: two tensors, rows dealt out over the CTAs
    const float* V[2];
    int VR[2];
    uint16_t *Vhi[2], *Vlo[2];
    float *V2[2], *V2ctr[2], *V2hi[2];
};

__device__ __forceinline__ void split_row(const float* __restrict__ v, int D, float center, uint16_t* hi, uint16_t* lo,
                                          float* v2, float* v2_ctr, float* v2_hi, int lane) {
    float s = 0.f, sh = 0.f, sc = 0.f;
    for (int c = lane; c < D; c += 32) {
        const float x = __ldg(v + c);
        const float xc = x - center;
        const uint16_t hb = bf16_bits(xc);
        const float hf = bf16_to_float(hb);
        if (hi) hi[c] = hb;
        if (lo) lo[c] = bf16_bits(xc - hf);
        s = fmaf(x, x, s);
        sc = fmaf(xc, xc, sc);
        sh = fmaf(hf, hf, sh);
    }
    s = warp_sum(s);
    sc = warp_sum(sc);
    sh = warp_sum(sh);
    if (lane == 0) {
        if (v2) *v2 = s;
        if (v2_ctr) *v2_ctr = sc;
        if (v2_hi) *v2_hi = sh;
    }
}

template <int MAXT, int LD, class T>
__global__ void __launch_bounds__(MAXT, 1)
head_prep_kernel(const PrepArgs a) {
    extern __shared__ __align__(16) float sm_prep[];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nthr = a.threads, nwarp = nthr >> 5;
    const int K = a.K, N = a.N, Din = a.Din, D = a.D, TR = a.TR, KC = a.KC;
    const int r0 = blockIdx.x * TR;
    const int nrow = min(TR, a.R - r0);
    const int bF = r0 / (K + 1), bL = (r0 + nrow - 1) / (K + 1);
    // shared-memory carve-up
    float* Xs = sm_prep;                                   // [TR][Dinp]
    float* Wt = Xs + (size_t)TR * a.Dinp;                   // [KC][D]   transposed chunk of Wa
    float* sc = Wt + (size_t)KC * D;                        // [Npad]    one image's fused scores
    float* nrm = sc + ((N + 3) & ~3);                       // [3][TR][D/8]
    int* sel = reinterpret_cast<int*>(nrm + 3 * (size_t)TR * (D / 8));   // [max_img][K]
    int* wcnt = sel + (size_t)a.max_img * K;                // [32]

    // ---- 0. this CTA's share of the prototype operand split (independent work, overlaps the loads below) ----------
    {
        const int total = a.VR[0] + a.VR[1];
        const int per = (total + gridDim.x - 1) / gridDim.x;
        const int lo = blockIdx.x * per, hi = min(total, lo + per);
        for (int row = lo + warp; row < hi; row += nwarp) {
            const int t = row >= a.VR[0] ? 1 : 0;
            const int rr = row - (t ? a.VR[0] : 0);
            split_row(a.V[t] + (size_t)rr * D, D, a.center, a.Vhi[t] ? a.Vhi[t] + (size_t)rr * D : nullptr,
                      a.Vlo[t] ? a.Vlo[t] + (size_t)rr * D : nullptr, a.V2[t] ? a.V2[t] + rr : nullptr,
                      a.V2ctr[t] ? a.V2ctr[t] + rr : nullptr, a.V2hi[t] ? a.V2hi[t] + rr : nullptr, lane);
        }
    }

    // ---- 1. selection of every image this tile touches --------------------------------------------------------------
    const int Npad = (N + 3) & ~3;
    for (int b = bF; b <= bL; ++b) {
        const float* sg = a.scores + (size_t)b * a.H * N;
        __syncthreads();
        for (int n = tid; n < Npad; n += nthr) {
            float v = -INFINITY;
            if (n < N) {
                float s = sg[n];
                for (int h = 1; h < a.H; ++h) s += sg[(size_t)h * N + n];
                v = a.H > 1 ? s / (float)a.H : s;          // torch.mean = sum / count
                if (v != v) v = INFINITY;                   // NaN ranks first (torch.topk), ties by index: a total order
            }
            sc[n] = v;
        }
        __syncthreads();
        int* out = sel + (size_t)(b - bF) * K;
        const bool publish = (b * (K + 1) >= r0);           // row j = 0 of image b lies in this tile
        int base = 0;
        for (int n0 = 0; n0 < N; n0 += nthr) {              // uniform trip count
            const int n = n0 + tid;
            bool s_ = false;
            if (n < N) {
                const float v = sc[n];
                int rank = 0;
                const float4* s4 = reinterpret_cast<const float4*>(sc);
                for (int j = 0; j < Npad; j += 4) {
                    const float4 q = s4[j >> 2];
                    rank += (q.x > v) || (q.x == v && j + 0 < n);
                    rank += (q.y > v) || (q.y == v && j + 1 < n);
                    rank += (q.z > v) || (q.z == v && j + 2 < n);
                    rank += (q.w > v) || (q.w == v && j + 3 < n);
                }
                s_ = rank < K;
            }
            const unsigned mk = __ballot_sync(0xffffffffu, s_);
            if (lane == 0) wcnt[warp] = __popc(mk);
            __syncthreads();
            int off = base, total = 0;
            for (int w = 0; w < nwarp; ++w) {
                const int c = wcnt[w];
                if (w < warp) off += c;
                total += c;
            }
            if (s_) {
                const int pos = off + __popc(mk & ((1u << lane) - 1u));
                if (pos < K) {
                    out[pos] = n;
                    if (publish) {
                        a.idx32[(size_t)b * K + pos] = n;
                        if (a.idx64) a.idx64[(size_t)b * K + pos] = n;
                    }
                }
            }
            base += total;
            __syncthreads();
        }
    }
    __syncthreads();

    // ---- 2. gather the source rows (zero rows past the end / zero padding of the k axis); bf16 rows are widened to
    //         fp32 on the way in (a register round trip instead of cp.async) ------------------------------------------
    {
        const T* tokens = static_cast<const T*>(a.tokens);
        const int c4 = a.Dinp >> 2;
        for (int i = tid; i < TR * c4; i += nthr) {
            const int rl = i / c4, q = i - rl * c4;
            float* dst = Xs + (size_t)rl * a.Dinp + q * 4;
            if (rl < nrow && q * 4 < Din) {
                const int r = r0 + rl;
                const int b = r / (K + 1), j = r - b * (K + 1);
                const int tok = j < K ? 1 + sel[(size_t)(b - bF) * K + j] : 0;
                const T* srcp = tokens + ((size_t)b * (1 + N) + tok) * Din + q * 4;
                if constexpr (sizeof(T) == 4) cp_async16(dst, srcp);
                else *reinterpret_cast<float4*>(dst) = ldg4_tok(srcp);
            } else {
                *reinterpret_cast<float4*>(dst) = make_float4(0.f, 0.f, 0.f, 0.f);
            }
        }
        cp_async_commit();
    }

    // ---- 3. contraction --------------------------------------------------------------------------------------------
    const int CG = D >> 3;                       // column groups: thread columns = {h * D/2 + cg*4 + e}
    const int ncomp = (TR >> 2) * CG;            // compute threads
    const bool comp = tid < ncomp;
    const int rg = tid / CG, cg = tid - rg * CG;
    float acc[4][8];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 8; ++j) acc[i][j] = 0.f;
    // W chunk loader: element group g = (o, i4): float4 Wa[o][k0 + 4*i4 .. +3] -> Wt[4*i4 + e][o]; consecutive threads
    // take consecutive o, so the transposed stores are conflict-free
    const int groups = (KC >> 2) * D;
    constexpr int kMaxLd = LD;
    float4 wreg[kMaxLd];
    auto load_chunk = [&](int ch) {
        const int k0 = ch * KC;
#pragma unroll
        for (int u = 0; u < kMaxLd; ++u) {
            const int g = tid + u * nthr;
            wreg[u] = make_float4(0.f, 0.f, 0.f, 0.f);
            if (g < groups) {
                const int o = g % D, i4 = g / D;
                const int k = k0 + 4 * i4;
                if (k < Din) wreg[u] = __ldg(reinterpret_cast<const float4*>(a.Wa + (size_t)o * Din + k));
            }
        }
    };
    auto store_chunk = [&]() {
#pragma unroll
        for (int u = 0; u < kMaxLd; ++u) {
            const int g = tid + u * nthr;
            if (g < groups) {
                const int o = g % D, i4 = g / D;
                Wt[(size_t)(4 * i4 + 0) * D + o] = wreg[u].x;
                Wt[(size_t)(4 * i4 + 1) * D + o] = wreg[u].y;
                Wt[(size_t)(4 * i4 + 2) * D + o] = wreg[u].z;
                Wt[(size_t)(4 * i4 + 3) * D + o] = wreg[u].w;
            }
        }
    };
    load_chunk(0);
    cp_async_wait<0>();
    for (int ch = 0; ch < a.nchunks; ++ch) {
        __syncthreads();                        // previous chunk's readers done (and, first time, Xs visible)
        store_chunk();
        __syncthreads();
        if (ch + 1 < a.nchunks) load_chunk(ch + 1);
        if (comp) {
            const float* xr = Xs + (size_t)(rg * 4) * a.Dinp + ch * KC;
            const float* w0 = Wt + cg * 4;
            const float* w1 = Wt + (D >> 1) + cg * 4;
#pragma unroll 2
            for (int kk = 0; kk < KC; kk += 4) {
                float4 xv[4];
#pragma unroll
                for (int i = 0; i < 4; ++i) xv[i] = *reinterpret_cast<const float4*>(xr + (size_t)i * a.Dinp + kk);
#pragma unroll
                for (int e = 0; e < 4; ++e) {
                    const float4 b0 = *reinterpret_cast<const float4*>(w0 + (size_t)(kk + e) * D);
                    const float4 b1 = *reinterpret_cast<const float4*>(w1 + (size_t)(kk + e) * D);
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
    }

    // ---- 4. epilogue -----------------------------------------------------------------------------------------------
    float* nq = nrm;                                  // |z|^2
    float* nc = nrm + (size_t)TR * CG;                // |z - center|^2
    float* nh = nc + (size_t)TR * CG;                 // |bf16(z - center)|^2
    if (comp) {
        float bia[8];
#pragma unroll
        for (int h = 0; h < 2; ++h) {
            const float4 t = __ldg(reinterpret_cast<const float4*>(a.ba + h * (D >> 1) + cg * 4));
            bia[h * 4 + 0] = t.x; bia[h * 4 + 1] = t.y; bia[h * 4 + 2] = t.z; bia[h * 4 + 3] = t.w;
        }
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const int rl = rg * 4 + i;
            float s = 0.f, sctr = 0.f, shi = 0.f;
            float z[8];
            uint16_t hb[8], lb[8];
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                const float pre = acc[i][j] + bia[j];
                z[j] = 1.0f / (1.0f + expf(-pre));
                const float zc = z[j] - a.center;       // tensor-core operands are centred (translation-invariant distance)
                hb[j] = bf16_bits(zc);
                const float hf = bf16_to_float(hb[j]);
                lb[j] = bf16_bits(zc - hf);
                s = fmaf(z[j], z[j], s);
                sctr = fmaf(zc, zc, sctr);
                shi = fmaf(hf, hf, shi);
            }
            nq[rl * CG + cg] = s;
            nc[rl * CG + cg] = sctr;
            nh[rl * CG + cg] = shi;
            if (rl < nrow) {
                const int r = r0 + rl;
                const int b = r / (K + 1), j = r - b * (K + 1);
                const bool cls = j == K;
                const size_t o = cls ? (size_t)b * D : ((size_t)b * K + j) * D;
                float* zf = (cls ? a.Zc : a.Zs) + o;
                uint16_t* zh = cls ? a.Zc_hi : a.Zs_hi;
                uint16_t* zl = cls ? a.Zc_lo : a.Zs_lo;
#pragma unroll
                for (int h = 0; h < 2; ++h) {
                    const int col = h * (D >> 1) + cg * 4;
                    *reinterpret_cast<float4*>(zf + col) = make_float4(z[h * 4], z[h * 4 + 1], z[h * 4 + 2], z[h * 4 + 3]);
                    if (zh) {
                        const uint32_t w0_ = (uint32_t)hb[h * 4] | ((uint32_t)hb[h * 4 + 1] << 16);
                        const uint32_t w1_ = (uint32_t)hb[h * 4 + 2] | ((uint32_t)hb[h * 4 + 3] << 16);
                        *reinterpret_cast<uint2*>(zh + o + col) = make_uint2(w0_, w1_);
                    }
                    if (zl) {
                        const uint32_t w0_ = (uint32_t)lb[h * 4] | ((uint32_t)lb[h * 4 + 1] << 16);
                        const uint32_t w1_ = (uint32_t)lb[h * 4 + 2] | ((uint32_t)lb[h * 4 + 3] << 16);
                        *reinterpret_cast<uint2*>(zl + o + col) = make_uint2(w0_, w1_);
                    }
                }
            }
        }
    }
    __syncthreads();
    for (int t = tid; t < 3 * nrow; t += nthr) {          // fixed-order row sums of the per-thread partial norms
        const int which = t / nrow, rl = t - which * nrow;
        const float* src = nrm + ((size_t)which * TR + rl) * CG;
        float s = 0.f;
        for (int c = 0; c < CG; ++c) s += src[c];
        const int r = r0 + rl;
        const int b = r / (K + 1), j = r - b * (K + 1);
        float* dst;
        if (j < K) dst = which == 0 ? a.z2s : (which == 1 ? a.z2s_ctr : a.z2s_hi);
        else dst = which == 0 ? a.z2c : (which == 1 ? a.z2c_ctr : a.z2c_hi);
        if (dst) dst[j < K ? (size_t)b * K + j : (size_t)b] = s;
    }
}

struct PrepPlan {
    int TR, KC, nchunks, Dinp, max_img, threads, grid;
    size_t smem;
};

static bool prep_plan(int B, int N, int Din, int D, int K, int sms, PrepPlan* out) {
    const int R = B * (K + 1);
    int pref = (ceil_div(R, sms) + 3) & ~3;
    if (pref < 32) pref = 32;
    if (pref > 48) pref = 48;
    const int cand[6] = {pref, 48, 44, 40, 36, 32};
    for (int ci = 0; ci < 6; ++ci) {
        PrepPlan p;
        const int tr = cand[ci];
        p.TR = tr;
        p.KC = 32;
        p.Dinp = ceil_div(Din, p.KC) * p.KC;
        p.nchunks = p.Dinp / p.KC;
        p.max_img = (tr + K) / (K + 1) + 1;
        int thr = (tr / 4) * (D / 8);
        thr = (thr + 31) & ~31;
        if (thr < 128) thr = 128;
        p.threads = thr;
        p.smem = sizeof(float) * ((size_t)tr * p.Dinp + (size_t)p.KC * D + (size_t)((N + 3) & ~3) +
                                  3 * (size_t)tr * (D / 8)) + sizeof(int) * ((size_t)p.max_img * K + 32);
        const int groups = (p.KC / 4) * D;
        const bool ok = (thr <= 256 && ceil_div(groups, thr) <= 8) || (thr > 256 && thr <= 640 && ceil_div(groups, thr) <= 6);
        if (!ok || p.smem > 200 * 1024) continue;
        p.grid = ceil_div(R, p.TR);
        *out = p;
        return true;
    }
    return false;
}

}  // namespace pph

extern "C" int pph_head_prep_supported(int B, int N, int Din, int D, int K) {
    using namespace pph;
    if (B < 1 || N < 1 || N > kPrepMaxN || K < 1 || K > N || Din < 4 || Din % 4 != 0 || D < 8 || D % 8 != 0) return 0;
    PrepPlan p;
    return prep_plan(B, N, Din, D, K, 148, &p) ? 1 : 0;
}

namespace pph {

template <class T>
static int head_prep_impl(const char* name, const float* scores, const T* tokens, const float* Wa, const float* ba,
                          int B, int H, int N, int Din, int D, int K, float center,
                          int32_t* idx32, int64_t* idx64,
                          float* Zs, float* Zc, float* z2s, float* z2c, float* z2s_ctr, float* z2c_ctr,
                          float* z2s_hi, float* z2c_hi, uint16_t* Zs_hi, uint16_t* Zs_lo, uint16_t* Zc_hi,
                          uint16_t* Zc_lo,
                          const float* Pl, int P, uint16_t* Pl_hi, uint16_t* Pl_lo, float* p2l, float* p2l_ctr,
                          float* p2l_hi,
                          const float* Pgl, int Pg, uint16_t* Pg_hi, uint16_t* Pg_lo, float* p2g, float* p2g_ctr,
                          float* p2g_hi, pph_stream_t stream) {
    PPH_REQUIRE(scores && tokens && Wa && ba && idx32 && Zs && Zc && z2s && z2c, PPH_EINVAL, "%s: null pointer", name);
    PPH_REQUIRE(H >= 1 && (P == 0 || Pl) && (Pg == 0 || Pgl) && P >= 0 && Pg >= 0, PPH_EINVAL, "%s: bad args", name);
    PPH_REQUIRE(sizeof(T) == 4 || Din % 8 == 0, PPH_EINVAL, "%s: bf16 tokens need Din %% 8 == 0 (Din=%d)", name, Din);
    PPH_REQUIRE(pph_head_prep_supported(B, N, Din, D, K), PPH_EUNSUP,
                "%s: shape B=%d N=%d Din=%d D=%d K=%d (Din %% 4, D %% 8, N <= 1024)", name, B, N, Din, D, K);
    int sms = pph_sm_count();
    if (sms <= 0) sms = 148;
    PrepPlan p;
    PPH_REQUIRE(prep_plan(B, N, Din, D, K, sms, &p), PPH_EUNSUP, "%s: no plan", name);
    PrepArgs a;
    a.B = B; a.H = H; a.N = N; a.Din = Din; a.D = D; a.K = K; a.R = B * (K + 1);
    a.TR = p.TR; a.KC = p.KC; a.nchunks = p.nchunks; a.Dinp = p.Dinp; a.max_img = p.max_img; a.threads = p.threads;
    a.center = center;
    a.scores = scores; a.tokens = tokens; a.Wa = Wa; a.ba = ba; a.idx32 = idx32; a.idx64 = idx64;
    a.Zs = Zs; a.Zc = Zc; a.z2s = z2s; a.z2c = z2c; a.z2s_ctr = z2s_ctr; a.z2c_ctr = z2c_ctr; a.z2s_hi = z2s_hi;
    a.z2c_hi = z2c_hi; a.Zs_hi = Zs_hi; a.Zs_lo = Zs_lo; a.Zc_hi = Zc_hi; a.Zc_lo = Zc_lo;
    a.V[0] = Pl; a.VR[0] = Pl ? P : 0; a.Vhi[0] = Pl_hi; a.Vlo[0] = Pl_lo; a.V2[0] = p2l; a.V2ctr[0] = p2l_ctr; a.V2hi[0] = p2l_hi;
    a.V[1] = Pgl; a.VR[1] = Pgl ? Pg : 0; a.Vhi[1] = Pg_hi; a.Vlo[1] = Pg_lo; a.V2[1] = p2g; a.V2ctr[1] = p2g_ctr; a.V2hi[1] = p2g_hi;
    auto k_small = head_prep_kernel<256, 8, T>;
    auto k_large = head_prep_kernel<640, 6, T>;
    auto kern = p.threads <= 256 ? k_small : k_large;
    cudaError_t e = opt_in_smem(kern, (int)p.smem);
    if (e != cudaSuccess) { set_error("%s: %s", name, cudaGetErrorString(e)); return (int)e; }
    launch_k(kern, dim3(p.grid), dim3(p.threads), p.smem, as_stream(stream), a);
    return launch_status(name);
}

}  // namespace pph

extern "C" int pph_head_prep(const float* scores, const float* tokens, const float* Wa, const float* ba,
                             int B, int H, int N, int Din, int D, int K, float center,
                             int32_t* idx32, int64_t* idx64,
                             float* Zs, float* Zc, float* z2s, float* z2c, float* z2s_ctr, float* z2c_ctr,
                             float* z2s_hi, float* z2c_hi, uint16_t* Zs_hi, uint16_t* Zs_lo, uint16_t* Zc_hi,
                             uint16_t* Zc_lo,
                             const float* Pl, int P, uint16_t* Pl_hi, uint16_t* Pl_lo, float* p2l, float* p2l_ctr,
                             float* p2l_hi,
                             const float* Pgl, int Pg, uint16_t* Pg_hi, uint16_t* Pg_lo, float* p2g, float* p2g_ctr,
                             float* p2g_hi, pph_stream_t stream) {
    return pph::head_prep_impl("pph_head_prep", scores, tokens, Wa, ba, B, H, N, Din, D, K, center, idx32, idx64, Zs, Zc, z2s,
                               z2c, z2s_ctr, z2c_ctr, z2s_hi, z2c_hi, Zs_hi, Zs_lo, Zc_hi, Zc_lo, Pl, P, Pl_hi, Pl_lo, p2l,
                               p2l_ctr, p2l_hi, Pgl, Pg, Pg_hi, Pg_lo, p2g, p2g_ctr, p2g_hi, stream);
}

extern "C" int pph_head_prep_bf16tok(const float* scores, const uint16_t* tokens, const float* Wa, const float* ba,
                                     int B, int H, int N, int Din, int D, int K, float center,
                                     int32_t* idx32, int64_t* idx64,
                                     float* Zs, float* Zc, float* z2s, float* z2c, float* z2s_ctr, float* z2c_ctr,
                                     float* z2s_hi, float* z2c_hi, uint16_t* Zs_hi, uint16_t* Zs_lo, uint16_t* Zc_hi,
                                     uint16_t* Zc_lo,
                                     const float* Pl, int P, uint16_t* Pl_hi, uint16_t* Pl_lo, float* p2l, float* p2l_ctr,
                                     float* p2l_hi,
                                     const float* Pgl, int Pg, uint16_t* Pg_hi, uint16_t* Pg_lo, float* p2g, float* p2g_ctr,
                                     float* p2g_hi, pph_stream_t stream) {
    return pph::head_prep_impl("pph_head_prep_bf16tok", scores, tokens, Wa, ba, B, H, N, Din, D, K, center, idx32, idx64, Zs,
                               Zc, z2s, z2c, z2s_ctr, z2c_ctr, z2s_hi, z2c_hi, Zs_hi, Zs_lo, Zc_hi, Zc_lo, Pl, P, Pl_hi,
                               Pl_lo, p2l, p2l_ctr, p2l_hi, Pgl, Pg, Pg_hi, Pg_lo, p2g, p2g_ctr, p2g_hi, stream);
}
