// The three add-on layer products of the training step on the single-shot tcgen05 kernel (pph_tcshot.cuh):
//   pph_addon_fwd2   Z = sigmoid(X_sel Wa^T + ba) (+ centred bf16 hi/lo operands and norms), protopformer.py:159-172
//   pph_addon_bwd3   dX = dpre Wa (scattered to the token rows) | dWa = dpre^T X_sel, dba = sum dpre
// where dpre = dZ * Z * (1 - Z) arrives precomputed from pph_similarity_bwd2 (dpre_out = 1).
// Same functors and the same 3-term bf16 split as pph_addon.cu; what changes is the launch shape: one 128 x BN tile
// per CTA with its whole k range resident (82 CTAs for the two row-tiled products, 112 for the weight gradient at the
// CUB shape instead of 41-82), no per-k-block round trips, and the split-k partials of the weight gradient reduced by
// all CTAs behind one grid barrier instead of a second launch.
#include "pph_addon_ops.cuh"
#include "pph_common.cuh"
#include "pph_tcshot.cuh"

namespace pph {

// ---- forward: column tiles live in different CTAs, so the row norms are completed by the LAST column tile of a row
// tile to finish (ticket), adding the per-tile partials in tile order: deterministic -----------------------------------
struct FwdEpi2 : FwdEpi {
    float* npart;            // [column tiles][Rpad][4]
    unsigned int* cnt;       // [row tiles], zero before first use, self-resetting
    int Rpad;
    __device__ __forceinline__ void finish(State& s, int r, int row_local, int cgroup, float* scratch, bool valid) const {
        __shared__ unsigned int s_ticket;
        if (cgroup > 0) {
            float* p = scratch + row_local * 16 + (cgroup - 1) * 3;
            p[0] = s.sq; p[1] = s.sq_ctr; p[2] = s.sq_hi;
        }
        __syncthreads();
        if (cgroup == 0 && valid) {
            float a = s.sq, c = s.sq_ctr, h = s.sq_hi;
#pragma unroll
            for (int g = 0; g < kTsWarps / 4 - 1; ++g) {
                const float* p = scratch + row_local * 16 + g * 3;
                a += p[0]; c += p[1]; h += p[2];
            }
            float* q = npart + ((size_t)blockIdx.y * Rpad + r) * 4;
            q[0] = a; q[1] = c; q[2] = h;
        }
        __threadfence();
        __syncthreads();
        if (threadIdx.x == 0) s_ticket = atomicAdd(cnt + blockIdx.x, 1u);
        __syncthreads();
        if (s_ticket != gridDim.y - 1) return;
        __threadfence();
        if (cgroup == 0 && valid) {
            float a = 0.f, c = 0.f, h = 0.f;
            for (unsigned int t = 0; t < gridDim.y; ++t) {
                const float* q = npart + ((size_t)t * Rpad + r) * 4;
                a += __ldcg(q); c += __ldcg(q + 1); h += __ldcg(q + 2);
            }
            const int b = r / (K + 1), j = r - b * (K + 1);
            if (j < K) {
                const size_t o = (size_t)b * K + j;
                z2s[o] = a;
                if (z2s_ctr) z2s_ctr[o] = c;
                if (z2s_hi) z2s_hi[o] = h;
            } else {
                z2c[b] = a;
                if (z2c_ctr) z2c_ctr[b] = c;
                if (z2c_hi) z2c_hi[b] = h;
            }
        }
        if (threadIdx.x == 0) cnt[blockIdx.x] = 0u;
    }
};

// ---- backward operands: dpre is an input here ---------------------------------------------------------------------------
struct PreRowOp {   // (row = r, k = d): dpre rows (+ the PPC loss's share add_s on the selected-token rows), contiguous along d
    static constexpr bool kContigK = true;
    const float *dpre_s, *dpre_c, *add_s;
    int K, D, R;
    __device__ __forceinline__ void load8(int r, int d0, float (&v)[8]) const {
        if (r >= R || d0 >= D) { zero8(v); return; }
        const int b = r / (K + 1), j = r - b * (K + 1);
        ld8((j < K ? dpre_s + ((size_t)b * K + j) * D : dpre_c + (size_t)b * D) + d0, v);
        if (add_s && j < K) {
            float w[8];
            ld8(add_s + ((size_t)b * K + j) * D + d0, w);
#pragma unroll
            for (int i = 0; i < 8; ++i) v[i] += w[i];
        }
    }
};
struct PreColOp {   // (row = d, k = r): the same matrix, transposed access (consecutive lanes = consecutive d)
    static constexpr bool kContigK = false;
    const float *dpre_s, *dpre_c, *add_s;
    int K, D, R;
    __device__ __forceinline__ void load8(int d, int r0, float (&v)[8]) const {
        if (d >= D) { zero8(v); return; }
        int b = r0 / (K + 1), j = r0 - b * (K + 1);
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            float x = 0.f;
            if (r0 + i < R) {
                if (j < K) {
                    const size_t o = ((size_t)b * K + j) * D + d;
                    x = __ldg(dpre_s + o);
                    if (add_s) x += __ldg(add_s + o);
                } else {
                    x = __ldg(dpre_c + (size_t)b * D + d);
                }
            }
            v[i] = x;
            if (++j > K) { j = 0; ++b; }
        }
    }
};
// quad variants of the transposed operands (see pph_tcshot.cuh): 128-bit loads along the rows
__device__ __forceinline__ float4 ldg4(const float* p) { return __ldg(reinterpret_cast<const float4*>(p)); }
struct PreColQOp : PreColOp {       // (rows d..d+3, k = r0..r0+7); D % 4 == 0
    static constexpr bool kQuad = true;
    __device__ __forceinline__ void load8x4(int d, int r0, float (&v)[4][8]) const {
        int b = r0 / (K + 1), j = r0 - b * (K + 1);
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            float4 x = make_float4(0.f, 0.f, 0.f, 0.f);
            if (r0 + i < R && d < D) {
                if (j < K) {
                    const size_t o = ((size_t)b * K + j) * D + d;
                    x = ldg4(dpre_s + o);
                    if (add_s) {
                        const float4 y = ldg4(add_s + o);
                        x.x += y.x; x.y += y.y; x.z += y.z; x.w += y.w;
                    }
                } else {
                    x = ldg4(dpre_c + (size_t)b * D + d);
                }
            }
            v[0][i] = x.x; v[1][i] = x.y; v[2][i] = x.z; v[3][i] = x.w;
            if (++j > K) { j = 0; ++b; }
        }
    }
};
template <class T>
struct XselColQOp : XselColOp<T> {  // (rows din..din+3, k = r0..r0+7); Din % 4 == 0; row Din = the all-ones column
    static constexpr bool kQuad = true;
    __device__ __forceinline__ void load8x4(int din, int r0, float (&v)[4][8]) const {
        const RowSrc& src = this->src;
        const int K = src.K;
        int b = r0 / (K + 1), j = r0 - b * (K + 1);
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            float4 x = make_float4(0.f, 0.f, 0.f, 0.f);
            if (r0 + i < src.R) {
                if (din < src.Din) {
                    const int tok = j < K ? 1 + __ldg(src.idx + (size_t)b * K + j) : 0;
                    x = ldg4_tok(this->tokens + ((size_t)b * (1 + src.N) + tok) * src.Din + din);
                } else if (din == src.Din) {
                    x.x = 1.0f;
                }
            }
            v[0][i] = x.x; v[1][i] = x.y; v[2][i] = x.z; v[3][i] = x.w;
            if (++j > K) { j = 0; ++b; }
        }
    }
};
struct WaTQOp : WaTOp {             // (rows din..din+3, k = d0..d0+7): Wa[d, din]; Din % 4 == 0
    static constexpr bool kQuad = true;
    __device__ __forceinline__ void load8x4(int din, int d0, float (&v)[4][8]) const {
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            float4 x = make_float4(0.f, 0.f, 0.f, 0.f);
            if (din < Din && d0 + i < D) x = ldg4(Wa + (size_t)(d0 + i) * Din + din);
            v[0][i] = x.x; v[1][i] = x.y; v[2][i] = x.z; v[3][i] = x.w;
        }
    }
};

struct WgradEpi2 {      // split-k partial tiles [split][D][ldn] + in-kernel reduction behind the grid barrier
    static constexpr bool kDirect = false;
    static constexpr bool kGridReduce = true;
    float *part, *dWa, *dba;
    int D, Din, ldn, splits;
    struct State { int dummy; };
    __device__ __forceinline__ void init(State& s) const { s.dummy = 0; }
    __device__ __forceinline__ void row_ptrs(int d, void* (&p)[3]) const { p[0] = part + ((size_t)blockIdx.z * D + d) * ldn; }
    __device__ __forceinline__ void transform(State&, int, int, uint32_t (&)[32]) const {}
    __device__ __forceinline__ void store2(void* const* p, int n, float v0, float v1) const {
        *reinterpret_cast<float2*>(static_cast<float*>(p[0]) + n) = make_float2(v0, v1);
    }
    __device__ __forceinline__ void finish(State&, int, int, int, float*, bool) const {}
    // dWa[d,din] = sum_s part[s][d][din];  dba[d] = sum_s part[s][d][Din]   (split order: deterministic)
    __device__ __forceinline__ void reduce(int cta, int n_ctas, int tid, int nthreads) const {
        const int total = D * (Din + 1);
        for (int i = cta * nthreads + tid; i < total; i += n_ctas * nthreads) {
            const int d = i / (Din + 1), n = i - d * (Din + 1);
            const float* src = part + (size_t)d * ldn + n;
            float s = 0.f;
            int sp = 0;
            for (; sp + 8 <= splits; sp += 8) {        // eight loads in flight, added in split order
                float v[8];
#pragma unroll
                for (int u = 0; u < 8; ++u) v[u] = __ldcg(src + (size_t)(sp + u) * D * ldn);
#pragma unroll
                for (int u = 0; u < 8; ++u) s += v[u];
            }
            for (; sp < splits; ++sp) s += __ldcg(src + (size_t)sp * D * ldn);
            if (n < Din) dWa[(size_t)d * Din + n] = s; else dba[d] = s;
        }
    }
};

struct Tc2Plan {
    bool fwd_ok, dx_ok, w_ok;
    int bn_fwd, bn_dx, bn_w, ldn, w_splits, w_ctas;
    size_t ws_bytes;
};

static Tc2Plan tc2_plan(int B, int Din, int D, int K, int sms) {
    Tc2Plan p{};
    const int R = B * (K + 1);
    auto pick = [](int n) {          // two column tiles when that keeps BN <= 128, multiples of 16
        int tiles = ceil_div(n, kTsMaxBN);
        if (tiles < 2 && n > 32) tiles = 2;
        return ceil_div(ceil_div(n, tiles), 16) * 16;
    };
    const bool dims = Din % 8 == 0 && D % 8 == 0 && Din >= 16 && D >= 16;
    p.bn_fwd = pick(D);
    p.bn_dx = pick(Din);
    p.fwd_ok = dims && Din <= kTsMaxKB * kTsBK;                 // k = Din resident
    p.dx_ok = dims && D <= kTsMaxKB * kTsBK;                    // k = D resident
    p.ldn = ceil_div(Din + 1, 4) * 4;
    p.bn_w = pick(Din + 1);
    p.w_splits = ceil_div(R, kTsMaxKB * kTsBK);
    p.w_ctas = ceil_div(D, kTsBM) * ceil_div(Din + 1, p.bn_w) * p.w_splits;
    p.w_ok = dims && p.w_ctas <= sms;
    p.ws_bytes = 256 + sizeof(int) * 1024 + sizeof(float) * ((size_t)4 * 4 * (ceil_div(R, kTsBM) * kTsBM) +
                                                             (size_t)p.w_splits * D * p.ldn + 64);
    return p;
}

struct Tc2Ws {
    unsigned int *sync_ctr, *fwd_cnt;
    float *npart, *wpart;
};
static Tc2Ws tc2_carve(void* base, int R) {
    Tc2Ws w;
    char* q = static_cast<char*>(base);
    w.sync_ctr = reinterpret_cast<unsigned int*>(q);                 // [2]   (+ padding)
    w.fwd_cnt = reinterpret_cast<unsigned int*>(q + 64);             // [row tiles] <= 1008
    w.npart = reinterpret_cast<float*>(q + 256 + sizeof(int) * 1024);
    w.wpart = w.npart + (size_t)4 * 4 * (ceil_div(R, kTsBM) * kTsBM);
    return w;
}

static int tc2_sms() {
    const int n = pph_sm_count();
    return n > 0 ? n : 148;
}

}  // namespace pph

extern "C" int pph_addon_tc2_supported(int B, int N, int Din, int D, int K) {
    using namespace pph;
    if (B < 1 || N < 1 || K < 1 || K > N || B * (K + 1) > 1008 * kTsBM) return 0;
    const Tc2Plan p = tc2_plan(B, Din, D, K, 148);
    const bool sel_ok = p.fwd_ok && N <= 256 && FwdSelAOp<float>::words(N, K) <= 128 * 16;
    return (p.fwd_ok ? 1 : 0) | (p.dx_ok ? 2 : 0) | (p.w_ok ? 4 : 0) | (sel_ok ? 8 : 0);
}

extern "C" int pph_addon_tc2_ws_bytes(int B, int N, int Din, int D, int K, long long* bytes) {
    using namespace pph;
    (void)N;
    PPH_REQUIRE(bytes && B >= 1 && Din >= 1 && D >= 1 && K >= 1, PPH_EINVAL, "pph_addon_tc2_ws_bytes: bad args");
    *bytes = (long long)tc2_plan(B, Din, D, K, 148).ws_bytes;
    return 0;
}

namespace pph {

template <class T>
static int addon_fwd2_impl(const char* name, const T* tokens, const int32_t* idx32, const float* Wa, const float* ba,
                           int B, int N, int Din, int D, int K,
                           float* Zs, float* Zc, float* z2s, float* z2c,
                           float center, float* z2s_ctr, float* z2c_ctr, float* z2s_hi, float* z2c_hi,
                           uint16_t* Zs_hi, uint16_t* Zs_lo, uint16_t* Zc_hi, uint16_t* Zc_lo,
                           void* workspace, pph_stream_t stream) {
    PPH_REQUIRE(tokens && idx32 && Wa && ba && Zs && Zc && z2s && z2c && workspace, PPH_EINVAL, "%s: null pointer", name);
    PPH_REQUIRE(B >= 1 && N >= 1 && K >= 1 && K <= N, PPH_EINVAL, "%s: bad dims", name);
    PPH_REQUIRE(sizeof(T) == 4 || Din % 8 == 0, PPH_EINVAL, "%s: bf16 tokens need Din %% 8 == 0 (Din=%d)", name, Din);
    const Tc2Plan p = tc2_plan(B, Din, D, K, tc2_sms());
    PPH_REQUIRE(p.fwd_ok && B * (K + 1) <= 1008 * kTsBM, PPH_EUNSUP, "%s: Din=%d D=%d outside the single-shot kernel", name, Din, D);
    const int R = B * (K + 1);
    const Tc2Ws w = tc2_carve(workspace, R);
    RowSrc src{idx32, B, N, Din, K, R};
    FwdAOp<T> a{tokens, src};
    FwdBOp b{Wa, D, Din};
    FwdEpi2 e;
    static_cast<FwdEpi&>(e) = FwdEpi{ba, Zs, Zc, z2s, z2c, z2s_ctr, z2c_ctr, z2s_hi, z2c_hi, Zs_hi, Zs_lo, Zc_hi, Zc_lo, center, K, D};
    e.npart = w.npart; e.cnt = w.fwd_cnt; e.Rpad = ceil_div(R, kTsBM) * kTsBM;
    return launch_tcshot(R, D, Din, p.bn_fwd, ceil_div(Din, kTsBK) * kTsBK, w.sync_ctr, a, b, e, as_stream(stream),
                         "pph_addon_fwd2(tcgen05 single shot)");
}

template <class T>
static int select_addon_fwd_impl(const char* name, const float* scores, int H, const T* tokens, const float* Wa,
                                 const float* ba, int B, int N, int Din, int D, int K, int32_t* idx32,
                                 float* Zs, float* Zc, float* z2s, float* z2c,
                                 float center, float* z2s_ctr, float* z2c_ctr, float* z2s_hi, float* z2c_hi,
                                 uint16_t* Zs_hi, uint16_t* Zs_lo, uint16_t* Zc_hi, uint16_t* Zc_lo,
                                 void* workspace, pph_stream_t stream) {
    PPH_REQUIRE(scores && tokens && idx32 && Wa && ba && Zs && Zc && z2s && z2c && workspace, PPH_EINVAL,
                "%s: null pointer", name);
    PPH_REQUIRE(B >= 1 && H >= 1 && N >= 1 && K >= 1 && K <= N, PPH_EINVAL, "%s: bad dims", name);
    PPH_REQUIRE(sizeof(T) == 4 || Din % 8 == 0, PPH_EINVAL, "%s: bf16 tokens need Din %% 8 == 0 (Din=%d)", name, Din);
    const Tc2Plan p = tc2_plan(B, Din, D, K, tc2_sms());
    PPH_REQUIRE(p.fwd_ok && B * (K + 1) <= 1008 * kTsBM && N <= 256 && FwdSelAOp<T>::words(N, K) <= 128 * 16, PPH_EUNSUP,
                "%s: N=%d K=%d Din=%d D=%d outside the fused selection + add-on kernel", name, N, K, Din, D);
    const int R = B * (K + 1);
    const Tc2Ws w = tc2_carve(workspace, R);
    FwdSelAOp<T> a{tokens, scores, idx32, B, N, Din, K, R, H};
    FwdBOp b{Wa, D, Din};
    FwdEpi2 e;
    static_cast<FwdEpi&>(e) = FwdEpi{ba, Zs, Zc, z2s, z2c, z2s_ctr, z2c_ctr, z2s_hi, z2c_hi, Zs_hi, Zs_lo, Zc_hi, Zc_lo, center, K, D};
    e.npart = w.npart; e.cnt = w.fwd_cnt; e.Rpad = ceil_div(R, kTsBM) * kTsBM;
    return launch_tcshot(R, D, Din, p.bn_fwd, ceil_div(Din, kTsBK) * kTsBK, w.sync_ctr, a, b, e, as_stream(stream),
                         "pph_select_addon_fwd(tcgen05 single shot)");
}

template <class T>
static int addon_bwd3_impl(const char* name, int parts, const T* tokens, const int32_t* idx32, const float* Wa,
                           const float* dpre_s, const float* dpre_c, const float* dpre_add_s,
                           int B, int N, int Din, int D, int K, void* workspace,
                           float* dWa, float* dba, T* dtokens, pph_stream_t stream) {
    PPH_REQUIRE((parts & 3) != 0, PPH_EINVAL, "%s: parts must name WGRAD and/or DGRAD", name);
    PPH_REQUIRE(tokens && idx32 && Wa && dpre_s && dpre_c && workspace, PPH_EINVAL, "%s: null pointer", name);
    PPH_REQUIRE(B >= 1 && N >= 1 && K >= 1 && K <= N, PPH_EINVAL, "%s: bad dims", name);
    PPH_REQUIRE(sizeof(T) == 4 || Din % 8 == 0, PPH_EINVAL, "%s: bf16 tokens need Din %% 8 == 0 (Din=%d)", name, Din);
    const Tc2Plan p = tc2_plan(B, Din, D, K, tc2_sms());
    const int R = B * (K + 1);
    const Tc2Ws w = tc2_carve(workspace, R);
    cudaStream_t st = as_stream(stream);
    RowSrc src{idx32, B, N, Din, K, R};
    if (parts & PPH_ADDON_WGRAD) {
        PPH_REQUIRE(dWa && dba, PPH_EINVAL, "%s(WGRAD): null output", name);
        PPH_REQUIRE(p.w_ok, PPH_EUNSUP, "%s(WGRAD): %d CTAs for B=%d K=%d Din=%d D=%d", name, p.w_ctas, B, K, Din, D);
        PreColQOp a;
        static_cast<PreColOp&>(a) = PreColOp{dpre_s, dpre_c, dpre_add_s, K, D, R};
        XselColQOp<T> b;
        static_cast<XselColOp<T>&>(b) = XselColOp<T>{tokens, src};
        WgradEpi2 e{w.wpart, dWa, dba, D, Din, p.ldn, p.w_splits};
        const int rc = launch_tcshot(D, Din + 1, R, p.bn_w, kTsMaxKB * kTsBK, w.sync_ctr, a, b, e, st,
                                     "pph_addon_bwd3(wgrad tcgen05 single shot)");
        if (rc) return rc;
    }
    if (parts & PPH_ADDON_DGRAD) {
        PPH_REQUIRE(dtokens, PPH_EINVAL, "%s(DGRAD): null dtokens", name);
        PPH_REQUIRE(p.dx_ok, PPH_EUNSUP, "%s(DGRAD): D=%d outside the single-shot kernel", name, D);
        PreRowOp a{dpre_s, dpre_c, dpre_add_s, K, D, R};
        WaTQOp b;
        static_cast<WaTOp&>(b) = WaTOp{Wa, D, Din};
        DxTcEpi<T> e{dtokens, src};
        const int rc = launch_tcshot(R, Din, D, p.bn_dx, ceil_div(D, kTsBK) * kTsBK, w.sync_ctr, a, b, e, st,
                                     "pph_addon_bwd3(dgrad tcgen05 single shot)");
        if (rc) return rc;
    }
    return 0;
}

}  // namespace pph

extern "C" int pph_addon_fwd2(const float* tokens, const int32_t* idx32, const float* Wa, const float* ba,
                              int B, int N, int Din, int D, int K,
                              float* Zs, float* Zc, float* z2s, float* z2c,
                              float center, float* z2s_ctr, float* z2c_ctr, float* z2s_hi, float* z2c_hi,
                              uint16_t* Zs_hi, uint16_t* Zs_lo, uint16_t* Zc_hi, uint16_t* Zc_lo,
                              void* workspace, pph_stream_t stream) {
    return pph::addon_fwd2_impl("pph_addon_fwd2", tokens, idx32, Wa, ba, B, N, Din, D, K, Zs, Zc, z2s, z2c, center, z2s_ctr,
                                z2c_ctr, z2s_hi, z2c_hi, Zs_hi, Zs_lo, Zc_hi, Zc_lo, workspace, stream);
}

extern "C" int pph_addon_fwd2_bf16tok(const uint16_t* tokens, const int32_t* idx32, const float* Wa, const float* ba,
                                      int B, int N, int Din, int D, int K,
                                      float* Zs, float* Zc, float* z2s, float* z2c,
                                      float center, float* z2s_ctr, float* z2c_ctr, float* z2s_hi, float* z2c_hi,
                                      uint16_t* Zs_hi, uint16_t* Zs_lo, uint16_t* Zc_hi, uint16_t* Zc_lo,
                                      void* workspace, pph_stream_t stream) {
    return pph::addon_fwd2_impl("pph_addon_fwd2_bf16tok", tokens, idx32, Wa, ba, B, N, Din, D, K, Zs, Zc, z2s, z2c, center,
                                z2s_ctr, z2c_ctr, z2s_hi, z2c_hi, Zs_hi, Zs_lo, Zc_hi, Zc_lo, workspace, stream);
}

extern "C" int pph_select_addon_fwd(const float* scores, int H, const float* tokens, const float* Wa, const float* ba,
                                    int B, int N, int Din, int D, int K, int32_t* idx32,
                                    float* Zs, float* Zc, float* z2s, float* z2c,
                                    float center, float* z2s_ctr, float* z2c_ctr, float* z2s_hi, float* z2c_hi,
                                    uint16_t* Zs_hi, uint16_t* Zs_lo, uint16_t* Zc_hi, uint16_t* Zc_lo,
                                    void* workspace, pph_stream_t stream) {
    return pph::select_addon_fwd_impl("pph_select_addon_fwd", scores, H, tokens, Wa, ba, B, N, Din, D, K, idx32, Zs, Zc, z2s,
                                      z2c, center, z2s_ctr, z2c_ctr, z2s_hi, z2c_hi, Zs_hi, Zs_lo, Zc_hi, Zc_lo, workspace,
                                      stream);
}

extern "C" int pph_select_addon_fwd_bf16tok(const float* scores, int H, const uint16_t* tokens, const float* Wa,
                                            const float* ba, int B, int N, int Din, int D, int K, int32_t* idx32,
                                            float* Zs, float* Zc, float* z2s, float* z2c,
                                            float center, float* z2s_ctr, float* z2c_ctr, float* z2s_hi, float* z2c_hi,
                                            uint16_t* Zs_hi, uint16_t* Zs_lo, uint16_t* Zc_hi, uint16_t* Zc_lo,
                                            void* workspace, pph_stream_t stream) {
    return pph::select_addon_fwd_impl("pph_select_addon_fwd_bf16tok", scores, H, tokens, Wa, ba, B, N, Din, D, K, idx32, Zs,
                                      Zc, z2s, z2c, center, z2s_ctr, z2c_ctr, z2s_hi, z2c_hi, Zs_hi, Zs_lo, Zc_hi, Zc_lo,
                                      workspace, stream);
}

extern "C" int pph_addon_bwd3(int parts, const float* tokens, const int32_t* idx32, const float* Wa,
                              const float* dpre_s, const float* dpre_c, const float* dpre_add_s,
                              int B, int N, int Din, int D, int K, void* workspace,
                              float* dWa, float* dba, float* dtokens, pph_stream_t stream) {
    return pph::addon_bwd3_impl("pph_addon_bwd3", parts, tokens, idx32, Wa, dpre_s, dpre_c, dpre_add_s, B, N, Din, D, K,
                                workspace, dWa, dba, dtokens, stream);
}

extern "C" int pph_addon_bwd3_bf16tok(int parts, const uint16_t* tokens, const int32_t* idx32, const float* Wa,
                                      const float* dpre_s, const float* dpre_c, const float* dpre_add_s,
                                      int B, int N, int Din, int D, int K, void* workspace,
                                      float* dWa, float* dba, uint16_t* dtokens, pph_stream_t stream) {
    return pph::addon_bwd3_impl("pph_addon_bwd3_bf16tok", parts, tokens, idx32, Wa, dpre_s, dpre_c, dpre_add_s, B, N, Din, D,
                                K, workspace, dWa, dba, dtokens, stream);
}
