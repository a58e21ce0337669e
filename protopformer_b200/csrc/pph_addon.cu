// (a2) gather of the selected tokens + 'regular' add-on layer (1x1 conv == per-token linear map) + sigmoid,
// its backward, and the bf16 hi/lo operand split used by the tensor-core similarity kernel.
// Replaces protopformer.py:159-172 (forward) and the autograd of those lines (backward).
//
// Row numbering used throughout: r in [0, B*(K+1)), b = r / (K+1), j = r % (K+1);
//   j <  K : selected patch token  -> source row 1 + idx[b,j] of tokens[b], output Zs[b,j,:]
//   j == K : CLS token             -> source row 0,                         output Zc[b,:]
#include "pph_common.cuh"
#include "pph_sgemm.cuh"
#include "pph_tcgemm.cuh"
#include "pph_addon_ops.cuh"

namespace pph {

// ---------------------------------------------------------------------------------------------------------------
// forward: one CTA = 32 gathered rows x all D outputs (192-wide chunks), FP32 FMA, fused bias + sigmoid + norms
// ---------------------------------------------------------------------------------------------------------------
constexpr int kAddBM = 32, kAddBN = 192, kAddBK = 16, kAddThreads = 256;

template <class T>
__global__ void __launch_bounds__(kAddThreads)
addon_fwd_kernel(const T* __restrict__ tokens, const int32_t* __restrict__ idx, const float* __restrict__ Wa,
                 const float* __restrict__ ba, int B, int N, int Din, int D, int K,
                 float* __restrict__ Zs, float* __restrict__ Zc, float* __restrict__ z2s, float* __restrict__ z2c,
                 float center, float* __restrict__ z2s_ctr, float* __restrict__ z2c_ctr,
                 float* __restrict__ z2s_hi, float* __restrict__ z2c_hi,
                 uint16_t* __restrict__ Zs_hi, uint16_t* __restrict__ Zs_lo,
                 uint16_t* __restrict__ Zc_hi, uint16_t* __restrict__ Zc_lo) {
    __shared__ __align__(16) float As[kAddBK][kAddBM + 4];
    __shared__ __align__(16) float Ws[kAddBK][kAddBN + 4];
    __shared__ long src_off[kAddBM];    // element offset of the source token row, -1 = row out of range
    __shared__ long dst_off[kAddBM];    // element offset of the output row inside Zs (>=0) or -(1 + b) for Zc[b]
    const int tid = threadIdx.x, tx = tid & 31, ty = tid >> 5;
    const int R = B * (K + 1), r0 = blockIdx.x * kAddBM;
    if (tid < kAddBM) {
        const int r = r0 + tid;
        long so = -1, dof = 0;
        if (r < R) {
            const int b = r / (K + 1), j = r - b * (K + 1);
            const int tok = j < K ? 1 + idx[(size_t)b * K + j] : 0;
            so = ((long)b * (1 + N) + tok) * Din;
            dof = j < K ? ((long)b * K + j) * D : -(long)(1 + b);
        }
        src_off[tid] = so;
        dst_off[tid] = dof;
    }
    __syncthreads();

    float sq[4] = {0.f, 0.f, 0.f, 0.f}, sq_hi[4] = {0.f, 0.f, 0.f, 0.f}, sq_ctr[4] = {0.f, 0.f, 0.f, 0.f};
    for (int nc = 0; nc < D; nc += kAddBN) {
        float acc[4][6];
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
            for (int j = 0; j < 6; ++j) acc[i][j] = 0.f;
        for (int k0 = 0; k0 < Din; k0 += kAddBK) {
            {   // A tile: 16 k x 32 rows
                const int k = tid & 15, r = tid >> 4;
#pragma unroll
                for (int i = 0; i < 2; ++i) {
                    const int row = r + 16 * i;
                    const long so = src_off[row];
                    As[k][row] = (so >= 0 && k0 + k < Din) ? ldg_tok(tokens + so + k0 + k) : 0.f;
                }
                // W tile: 16 k x 192 n   (Wa is [D, Din], k contiguous)
#pragma unroll
                for (int i = 0; i < 12; ++i) {
                    const int n = r + 16 * i;
                    Ws[k][n] = (nc + n < D && k0 + k < Din) ? __ldg(Wa + (size_t)(nc + n) * Din + k0 + k) : 0.f;
                }
            }
            __syncthreads();
#pragma unroll
            for (int kk = 0; kk < kAddBK; ++kk) {
                const float4 a = *reinterpret_cast<const float4*>(&As[kk][ty * 4]);
                const float av[4] = {a.x, a.y, a.z, a.w};
                float bv[6];
#pragma unroll
                for (int j = 0; j < 6; ++j) bv[j] = Ws[kk][tx + 32 * j];
#pragma unroll
                for (int i = 0; i < 4; ++i)
#pragma unroll
                    for (int j = 0; j < 6; ++j) acc[i][j] = fmaf(av[i], bv[j], acc[i][j]);
            }
            __syncthreads();
        }
        // epilogue of this 192-wide chunk: bias + sigmoid, fp32 + bf16 hi/lo stores, running row norms
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const int row = ty * 4 + i;
            if (src_off[row] < 0) continue;
            const long dof = dst_off[row];
#pragma unroll
            for (int j = 0; j < 6; ++j) {
                const int n = nc + tx + 32 * j;
                if (n >= D) continue;
                const float pre = acc[i][j] + __ldg(ba + n);
                const float z = 1.0f / (1.0f + expf(-pre));
                const float zc = z - center;          // tensor-core operands are centred (translation-invariant distance)
                const uint16_t hb = bf16_bits(zc);
                const float hf = bf16_to_float(hb);
                const uint16_t lb = bf16_bits(zc - hf);
                sq[i] = fmaf(z, z, sq[i]);
                sq_ctr[i] = fmaf(zc, zc, sq_ctr[i]);
                sq_hi[i] = fmaf(hf, hf, sq_hi[i]);
                if (dof >= 0) {
                    Zs[dof + n] = z;
                    if (Zs_hi) Zs_hi[dof + n] = hb;
                    if (Zs_lo) Zs_lo[dof + n] = lb;
                } else {
                    const long o = (-dof - 1) * (long)D + n;
                    Zc[o] = z;
                    if (Zc_hi) Zc_hi[o] = hb;
                    if (Zc_lo) Zc_lo[o] = lb;
                }
            }
        }
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const float s = warp_sum(sq[i]), sh = warp_sum(sq_hi[i]), sc = warp_sum(sq_ctr[i]);   // a warp owns its 4 rows
        const int row = ty * 4 + i;
        if (tx == 0 && src_off[row] >= 0) {
            const long dof = dst_off[row];
            if (dof >= 0) {
                z2s[dof / D] = s;
                if (z2s_ctr) z2s_ctr[dof / D] = sc;
                if (z2s_hi) z2s_hi[dof / D] = sh;
            } else {
                z2c[-dof - 1] = s;
                if (z2c_ctr) z2c_ctr[-dof - 1] = sc;
                if (z2c_hi) z2c_hi[-dof - 1] = sh;
            }
        }
    }
}

// ---------------------------------------------------------------------------------------------------------------
// operand split: V [R,D] fp32 -> hi/lo bf16, |V|^2 (fp32 operand and rounded-operand flavours). One warp per row.
// ---------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
split_rows_kernel(const float* __restrict__ V, int R, int D, float center, uint16_t* __restrict__ hi,
                  uint16_t* __restrict__ lo, float* __restrict__ v2, float* __restrict__ v2_ctr,
                  float* __restrict__ v2_hi) {
    const int row = blockIdx.x * 8 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (row >= R) return;
    const float* v = V + (size_t)row * D;
    float s = 0.f, sh = 0.f, sc = 0.f;
    for (int c = lane; c < D; c += 32) {
        const float x = __ldg(v + c);
        const float xc = x - center;
        const uint16_t hb = bf16_bits(xc);
        const float hf = bf16_to_float(hb);
        if (hi) hi[(size_t)row * D + c] = hb;
        if (lo) lo[(size_t)row * D + c] = bf16_bits(xc - hf);
        s = fmaf(x, x, s);
        sc = fmaf(xc, xc, sc);
        sh = fmaf(hf, hf, sh);
    }
    s = warp_sum(s);
    sc = warp_sum(sc);
    sh = warp_sum(sh);
    if (lane == 0) {
        if (v2) v2[row] = s;
        if (v2_ctr) v2_ctr[row] = sc;
        if (v2_hi) v2_hi[row] = sh;
    }
}

// ---------------------------------------------------------------------------------------------------------------
// backward operands (evaluated on the fly inside the tile loader of the generic FP32 GEMM)
// ---------------------------------------------------------------------------------------------------------------
struct RowMap {
    int B, K, D;
    __device__ __forceinline__ long z_off(int r, bool& is_cls) const {   // offset into Zs (or Zc when is_cls)
        const int b = r / (K + 1), j = r - b * (K + 1);
        is_cls = (j == K);
        return is_cls ? (long)b * D : ((long)b * K + j) * D;
    }
};

// dpre(r, d) = dZ * Z * (1 - Z).   TRANSPOSED=false: operand rows are r, k runs over d (contiguous);
// TRANSPOSED=true: operand rows are d, k runs over r.
template <bool TRANSPOSED>
struct DpreOp {
    static constexpr bool kContigK = !TRANSPOSED;
    const float *Zs, *Zc, *dZs, *dZc;
    RowMap map;
    int R;
    __device__ __forceinline__ float operator()(int row, int k) const {
        const int r = TRANSPOSED ? k : row, d = TRANSPOSED ? row : k;
        if (r >= R || d >= map.D) return 0.f;
        bool cls;
        const long o = map.z_off(r, cls) + d;
        const float z = cls ? __ldg(Zc + o) : __ldg(Zs + o);
        const float g = cls ? __ldg(dZc + o) : __ldg(dZs + o);
        return g * z * (1.0f - z);
    }
};

// gathered source token rows as a (row = din, k = r) operand
template <class T>
struct XselOp {
    static constexpr bool kContigK = false;
    const T* tokens;
    const int32_t* idx;
    int B, N, Din, K, R;
    __device__ __forceinline__ float operator()(int din, int r) const {
        if (r >= R || din >= Din) return 0.f;
        const int b = r / (K + 1), j = r - b * (K + 1);
        const int tok = j < K ? 1 + __ldg(idx + (size_t)b * K + j) : 0;
        return ldg_tok(tokens + ((size_t)b * (1 + N) + tok) * Din + din);
    }
};

struct WgradEpi {   // split-K accumulation of dWa and dba
    float *dWa, *dba;
    int Din;
    __device__ __forceinline__ void operator()(int m, int n, float acc, float rs) const {
        atomicAdd(dWa + (size_t)m * Din + n, acc);
        if (n == 0) atomicAdd(dba + m, rs);
    }
};

template <class T>
struct DxEpi {      // scatter of the token gradient rows
    T* dtokens;
    const int32_t* idx;
    int N, Din, K;
    __device__ __forceinline__ void operator()(int r, int n, float acc, float) const {
        const int b = r / (K + 1), j = r - b * (K + 1);
        const int tok = j < K ? 1 + __ldg(idx + (size_t)b * K + j) : 0;
        st_tok(dtokens + ((size_t)b * (1 + N) + tok) * Din + n, acc);
    }
};


// ---------------------------------------------------------------------------------------------------------------
// tensor-core path (tcgen05, bf16x3, operands prepared in-kernel: pph_tcgemm.cuh).  Used when Din % 8 == 0 and
// D % 8 == 0; the CUDA-core kernels above remain for other shapes.
// ---------------------------------------------------------------------------------------------------------------
// dWa[d,din] = sum_s part[s][d][din];  dba[d] = sum_s part[s][d][Din]     (fixed order: deterministic)
__global__ void __launch_bounds__(256)
wgrad_reduce_kernel(const float* __restrict__ part, int splits, int D, int Din, int ldn, float* __restrict__ dWa,
                    float* __restrict__ dba) {
    const int i = blockIdx.x * 256 + threadIdx.x;
    if (i >= D * (Din + 1)) return;
    const int d = i / (Din + 1), n = i - d * (Din + 1);
    float s = 0.f;
    for (int sp = 0; sp < splits; ++sp) s += __ldg(part + ((size_t)sp * D + d) * ldn + n);
    if (n < Din) dWa[(size_t)d * Din + n] = s; else dba[d] = s;
}

static bool addon_tc_ok(int Din, int D) { return Din % 8 == 0 && D % 8 == 0 && Din >= 8 && D >= 16; }
static int wgrad_splits(int R) { int s = ceil_div(R, 2 * kTgBK); return s < 1 ? 1 : (s > 64 ? 64 : s); }

template <class T>
static int addon_fwd_impl(const char* name, const T* tokens, const int32_t* idx32, const float* Wa, const float* ba,
                          int B, int N, int Din, int D, int K,
                          float* Zs, float* Zc, float* z2s, float* z2c,
                          float center, float* z2s_ctr, float* z2c_ctr, float* z2s_hi, float* z2c_hi,
                          uint16_t* Zs_hi, uint16_t* Zs_lo, uint16_t* Zc_hi, uint16_t* Zc_lo,
                          pph_stream_t stream) {
    PPH_REQUIRE(tokens && idx32 && Wa && ba && Zs && Zc && z2s && z2c, PPH_EINVAL, "%s: null pointer", name);
    PPH_REQUIRE(B >= 0 && N >= 1 && Din >= 1 && D >= 1 && K >= 1 && K <= N, PPH_EINVAL,
                "%s: bad dims B=%d N=%d Din=%d D=%d K=%d", name, B, N, Din, D, K);
    PPH_REQUIRE(sizeof(T) == 4 || Din % 8 == 0, PPH_EINVAL, "%s: bf16 tokens need Din %% 8 == 0 (Din=%d)", name, Din);
    if (B == 0) return 0;
    const int R = B * (K + 1);
    if (addon_tc_ok(Din, D)) {
        RowSrc src{idx32, B, N, Din, K, R};
        FwdAOp<T> a{tokens, src};
        FwdBOp b{Wa, D, Din};
        FwdEpi e{ba, Zs, Zc, z2s, z2c, z2s_ctr, z2c_ctr, z2s_hi, z2c_hi, Zs_hi, Zs_lo, Zc_hi, Zc_lo, center, K, D};
        return launch_tcgemm(R, D, Din, tcgemm_pick_bn(D), 1, a, b, e, as_stream(stream), "pph_addon_fwd(tcgen05)");
    }
    launch_k(addon_fwd_kernel<T>, dim3(ceil_div(R, kAddBM)), dim3(kAddThreads), (size_t)(0), as_stream(stream), tokens, idx32, Wa, ba, B, N, Din, D, K, Zs, Zc, z2s, z2c, center, z2s_ctr, z2c_ctr, z2s_hi, z2c_hi, Zs_hi, Zs_lo, Zc_hi, Zc_lo);
    return launch_status(name);
}

template <class T>
static int addon_bwd_impl(const char* name, const T* tokens, const int32_t* idx32, const float* Wa,
                          const float* Zs, const float* Zc, const float* dZs, const float* dZc,
                          int B, int N, int Din, int D, int K, void* workspace, int parts,
                          float* dWa, float* dba, T* dtokens, pph_stream_t stream) {
    PPH_REQUIRE((parts & 3) != 0, PPH_EINVAL, "%s: parts must include PPH_ADDON_WGRAD and/or PPH_ADDON_DGRAD", name);
    if (!(parts & PPH_ADDON_DGRAD)) dtokens = nullptr;
    const bool want_w = (parts & PPH_ADDON_WGRAD) != 0;
    PPH_REQUIRE(tokens && idx32 && Wa && Zs && Zc && dZs && dZc && (!want_w || (dWa && dba)), PPH_EINVAL,
                "%s: null pointer", name);
    PPH_REQUIRE(B >= 0 && N >= 1 && Din >= 1 && D >= 1 && K >= 1 && K <= N, PPH_EINVAL,
                "%s: bad dims B=%d N=%d Din=%d D=%d K=%d", name, B, N, Din, D, K);
    PPH_REQUIRE(sizeof(T) == 4 || Din % 8 == 0, PPH_EINVAL, "%s: bf16 tokens need Din %% 8 == 0 (Din=%d)", name, Din);
    cudaStream_t st = as_stream(stream);
    const bool tc = addon_tc_ok(Din, D) && B > 0;
    cudaError_t e = cudaSuccess;
    if (!tc && want_w) {
        e = cudaMemsetAsync(dWa, 0, sizeof(float) * (size_t)D * Din, st);
        if (e == cudaSuccess) e = cudaMemsetAsync(dba, 0, sizeof(float) * (size_t)D, st);
    }
    if (e == cudaSuccess && dtokens)
        e = cudaMemsetAsync(dtokens, 0, sizeof(T) * (size_t)B * (1 + N) * Din, st);
    if (e != cudaSuccess) {
        set_error("%s: memset: %s", name, cudaGetErrorString(e));
        return (int)e;
    }
    if (B == 0) return 0;
    const int R = B * (K + 1);
    if (tc) {
        PPH_REQUIRE(workspace || !want_w, PPH_EINVAL, "%s: null workspace (size it with pph_addon_bwd_ws_bytes)", name);
        RowSrc src{idx32, B, N, Din, K, R};
        if (want_w) {   // dWa / dba: [D x (Din+1)] = dpre^T [D x R] * [Xsel | 1]^T, split over r, partials + ordered reduction
            const int ldn = ceil_div(Din + 1, 4) * 4;
            int splits = wgrad_splits(R);
            const int k_per_split = ceil_div(ceil_div(R, splits), kTgBK) * kTgBK;
            splits = ceil_div(R, k_per_split);
            float* part = static_cast<float*>(workspace);
            DpreColOp a{Zs, Zc, dZs, dZc, K, D, R};
            XselColOp<T> b{tokens, src};
            WgradPartEpi epi{part, D, ldn};
            int rc = launch_tcgemm(D, ldn, R, tcgemm_pick_bn(ldn), splits, a, b, epi, st, "pph_addon_bwd(wgrad tcgen05)");
            if (rc) return rc;
            launch_k(wgrad_reduce_kernel, dim3(ceil_div(D * (Din + 1), 256)), dim3(256), (size_t)(0), st, part, splits, D, Din, ldn, dWa, dba);
            rc = launch_status("pph_addon_bwd(wgrad reduce)");
            if (rc) return rc;
        }
        if (dtokens) {   // dX [R x Din] = dpre [R x D] * Wa [D x Din]
            DpreRowOp a{Zs, Zc, dZs, dZc, K, D, R};
            WaTOp b{Wa, D, Din};
            DxTcEpi<T> epi{dtokens, src};
            int rc = launch_tcgemm(R, Din, D, tcgemm_pick_bn(Din), 1, a, b, epi, st, "pph_addon_bwd(dgrad tcgen05)");
            if (rc) return rc;
        }
        return 0;
    }
    RowMap map{B, K, D};
    if (want_w) {   // dWa[d, din] = sum_r dpre[r,d] * X[r,din];  dba[d] = sum_r dpre[r,d]   (split over r)
        DpreOp<true> a{Zs, Zc, dZs, dZc, map, R};
        XselOp<T> b{tokens, idx32, B, N, Din, K, R};
        WgradEpi epi{dWa, dba, Din};
        const int tiles = ceil_div(D, kGemmBM) * ceil_div(Din, kGemmBN);
        int splits = ceil_div(2 * 148, tiles);
        launch_sgemm<true>(D, Din, R, splits, a, b, epi, st);
        int rc = launch_status("pph_addon_bwd(wgrad)");
        if (rc) return rc;
    }
    if (dtokens) {   // dX[r, din] = sum_d dpre[r,d] * Wa[d,din]  -> scattered into the zero-filled token gradient
        DpreOp<false> a{Zs, Zc, dZs, dZc, map, R};
        StridedOp<false> b{Wa, Din, 1, Din};       // (row = din, k = d) -> Wa[d*Din + din]
        DxEpi<T> epi{dtokens, idx32, N, Din, K};
        launch_sgemm<false>(R, Din, D, 1, a, b, epi, st);
        int rc = launch_status("pph_addon_bwd(dgrad)");
        if (rc) return rc;
    }
    return 0;
}

}  // namespace pph

extern "C" int pph_addon_fwd(const float* tokens, const int32_t* idx32, const float* Wa, const float* ba,
                             int B, int N, int Din, int D, int K,
                             float* Zs, float* Zc, float* z2s, float* z2c,
                             float center, float* z2s_ctr, float* z2c_ctr, float* z2s_hi, float* z2c_hi,
                             uint16_t* Zs_hi, uint16_t* Zs_lo, uint16_t* Zc_hi, uint16_t* Zc_lo,
                             pph_stream_t stream) {
    return pph::addon_fwd_impl("pph_addon_fwd", tokens, idx32, Wa, ba, B, N, Din, D, K, Zs, Zc, z2s, z2c, center, z2s_ctr,
                               z2c_ctr, z2s_hi, z2c_hi, Zs_hi, Zs_lo, Zc_hi, Zc_lo, stream);
}

extern "C" int pph_addon_fwd_bf16tok(const uint16_t* tokens, const int32_t* idx32, const float* Wa, const float* ba,
                                     int B, int N, int Din, int D, int K,
                                     float* Zs, float* Zc, float* z2s, float* z2c,
                                     float center, float* z2s_ctr, float* z2c_ctr, float* z2s_hi, float* z2c_hi,
                                     uint16_t* Zs_hi, uint16_t* Zs_lo, uint16_t* Zc_hi, uint16_t* Zc_lo,
                                     pph_stream_t stream) {
    return pph::addon_fwd_impl("pph_addon_fwd_bf16tok", tokens, idx32, Wa, ba, B, N, Din, D, K, Zs, Zc, z2s, z2c, center,
                               z2s_ctr, z2c_ctr, z2s_hi, z2c_hi, Zs_hi, Zs_lo, Zc_hi, Zc_lo, stream);
}

extern "C" int pph_split_rows(const float* V, int R, int D, float center, uint16_t* hi, uint16_t* lo, float* v2,
                              float* v2_ctr, float* v2_hi, pph_stream_t stream) {
    PPH_REQUIRE(V, PPH_EINVAL, "pph_split_rows: null pointer");
    PPH_REQUIRE(R >= 0 && D >= 1, PPH_EINVAL, "pph_split_rows: bad dims R=%d D=%d", R, D);
    if (R == 0) return 0;
    pph::launch_k(pph::split_rows_kernel, dim3(pph::ceil_div(R, 8)), dim3(256), (size_t)(0), pph::as_stream(stream), V, R, D, center, hi, lo, v2, v2_ctr, v2_hi);
    return pph::launch_status("pph_split_rows");
}

#ifdef PPH_DEBUG_STAMPS
// development aid (only in -DPPH_DEBUG_STAMPS builds): phase timestamps (ns) of CTA 0 of the last tcgemm launch
extern "C" int pph_debug_read(long long* out32) {
    cudaError_t e = cudaMemcpyFromSymbol(out32, pph::g_dbg_ts, sizeof(long long) * 32);
    return e == cudaSuccess ? 0 : (int)e;
}
#endif

extern "C" int pph_addon_bwd_ws_bytes(int B, int N, int Din, int D, int K, long long* bytes) {
    using namespace pph;
    PPH_REQUIRE(bytes && B >= 0 && Din >= 1 && D >= 1 && K >= 1, PPH_EINVAL, "pph_addon_bwd_ws_bytes: bad args");
    (void)N;
    const int ldn = ceil_div(Din + 1, 4) * 4;
    *bytes = addon_tc_ok(Din, D) ? (long long)sizeof(float) * wgrad_splits(B * (K + 1)) * D * ldn + 256 : 256;
    return 0;
}

extern "C" int pph_addon_bwd(const float* tokens, const int32_t* idx32, const float* Wa,
                             const float* Zs, const float* Zc, const float* dZs, const float* dZc,
                             int B, int N, int Din, int D, int K, void* workspace, int parts,
                             float* dWa, float* dba, float* dtokens, pph_stream_t stream) {
    return pph::addon_bwd_impl("pph_addon_bwd", tokens, idx32, Wa, Zs, Zc, dZs, dZc, B, N, Din, D, K, workspace, parts, dWa,
                               dba, dtokens, stream);
}

extern "C" int pph_addon_bwd_bf16tok(const uint16_t* tokens, const int32_t* idx32, const float* Wa,
                                     const float* Zs, const float* Zc, const float* dZs, const float* dZc,
                                     int B, int N, int Din, int D, int K, void* workspace, int parts,
                                     float* dWa, float* dba, uint16_t* dtokens, pph_stream_t stream) {
    return pph::addon_bwd_impl("pph_addon_bwd_bf16tok", tokens, idx32, Wa, Zs, Zc, dZs, dZc, B, N, Din, D, K, workspace,
                               parts, dWa, dba, dtokens, stream);
}
