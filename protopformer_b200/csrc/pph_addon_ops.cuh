// Operand and epilogue functors of the add-on layer products on tcgen05 (shared by pph_addon.cu -- pph_tcgemm.cuh
// kernel -- and pph_addon_tc2.cu -- pph_tcshot.cuh kernel).  Row numbering: r in [0, B*(K+1)), b = r / (K+1),
// j = r % (K+1); j < K: selected patch token idx[b,j], j == K: the CLS token.
#pragma once

#include "pph_common.cuh"
#include "pph_tcgemm.cuh"

namespace pph {

struct RowSrc {     // r -> element offset of the source token row
    const int32_t* idx;
    int B, N, Din, K, R;
    __device__ __forceinline__ long operator()(int r) const {
        const int b = r / (K + 1), j = r - b * (K + 1);
        const int tok = j < K ? 1 + __ldg(idx + (size_t)b * K + j) : 0;
        return ((long)b * (1 + N) + tok) * Din;
    }
};

__device__ __forceinline__ void ld8(const float* p, float (&v)[8]) {
    const float4 a = __ldg(reinterpret_cast<const float4*>(p)), b = __ldg(reinterpret_cast<const float4*>(p) + 1);
    v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w; v[4] = b.x; v[5] = b.y; v[6] = b.z; v[7] = b.w;
}
__device__ __forceinline__ void ld8(const uint16_t* p, float (&v)[8]) {     // eight bf16 tokens values: one 16-byte load
    const uint4 q = __ldg(reinterpret_cast<const uint4*>(p));
    const uint32_t w[4] = {q.x, q.y, q.z, q.w};
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        v[2 * i] = __uint_as_float(w[i] << 16);
        v[2 * i + 1] = __uint_as_float(w[i] & 0xffff0000u);
    }
}
__device__ __forceinline__ void zero8(float (&v)[8]) {
#pragma unroll
    for (int i = 0; i < 8; ++i) v[i] = 0.f;
}

// ---- forward: Z = sigmoid(Xsel Wa^T + ba) --------------------------------------------------------------------------
template <class T>   // token element type: float or bf16 (uint16_t), here and in every token operand / epilogue below
struct FwdAOp {     // (row = r, k = din): gathered token rows
    static constexpr bool kContigK = true;
    const T* tokens;
    RowSrc src;
    __device__ __forceinline__ void load8(int r, int k0, float (&v)[8]) const {
        if (r < src.R && k0 < src.Din) ld8(tokens + src(r) + k0, v); else zero8(v);
    }
};
// Gathered token rows with the SELECTION done by the kernel that consumes it (protopformer.py:157-166 in one launch): every
// CTA ranks the CLS-attention scores of the (<= 4) images its 128-row tile touches -- rank by counting with the same
// total order as select_topk_kernel (larger score first, lower index on ties, NaN first) -- and keeps the ascending index
// lists in shared memory; the CTAs of the first column tile also write them to idx_out for the kernels downstream.
template <class T>
struct FwdSelAOp {
    static constexpr bool kContigK = true;
    static constexpr bool kSelect = true;
    const T* tokens;
    const float* scores;       // [B, H, N]
    int32_t* idx_out;          // [B, K]
    int B, N, Din, K, R, H;
    __host__ __device__ static int images_per_tile(int K) { return 127 / (K + 1) + 2; }
    __host__ __device__ static int words(int N, int K) { return images_per_tile(K) * (((N + 3) & ~3) + 8 + K); }
    __device__ __forceinline__ void prologue(int m0, int* smi, bool write_out) const {
        const int tid = threadIdx.x, lane = tid & 31, nthr = blockDim.x;
        const int b_lo = m0 / (K + 1), b_hi = min(m0 + 127, R - 1) / (K + 1), n_here = b_hi - b_lo + 1;
        const int nimg = images_per_tile(K), Np = (N + 3) & ~3, N32 = (N + 31) & ~31;
        float* sc = reinterpret_cast<float*>(smi);            // [nimg][Np]  fused scores (-inf padding)
        int* cnt = smi + nimg * Np;                           // [nimg][8]   selected tokens per 32-token group
        int* sidx = cnt + nimg * 8;                           // [nimg][K]   ascending selected tokens
        for (int w = tid; w < n_here * Np; w += nthr) {
            const int i = w / Np, n = w - i * Np;
            float v = -INFINITY;
            if (n < N) {
                const float* row = scores + (size_t)(b_lo + i) * H * N;
                float a = row[n];
                for (int h = 1; h < H; ++h) a += row[(size_t)h * N + n];
                v = H > 1 ? a / (float)H : a;
                if (v != v) v = INFINITY;
            }
            sc[i * Np + n] = v;
        }
        __syncthreads();
        const int items = n_here * N32;                       // warp-aligned: 32-token groups never straddle images
        bool sel[2] = {false, false};
        unsigned mask[2] = {0u, 0u};
#pragma unroll
        for (int p = 0; p < 2; ++p) {
            const int w = tid + p * nthr;
            if (w < items) {
                const int i = w / N32, n = w - i * N32;
                if (n < N) {
                    const float v = sc[i * Np + n];
                    const int rank = rank_by_count(reinterpret_cast<const float4*>(sc + i * Np), n, Np, v);
                    sel[p] = rank < K;
                }
                mask[p] = __ballot_sync(0xffffffffu, sel[p]);
                if (lane == 0) cnt[i * 8 + (n >> 5)] = __popc(mask[p]);
            }
        }
        __syncthreads();
#pragma unroll
        for (int p = 0; p < 2; ++p) {
            const int w = tid + p * nthr;
            if (w < items && sel[p]) {
                const int i = w / N32, n = w - i * N32;
                int pos = __popc(mask[p] & ((1u << lane) - 1u));
                for (int g = 0; g < (n >> 5); ++g) pos += cnt[i * 8 + g];
                if (pos < K) {
                    sidx[i * K + pos] = n;
                    if (write_out) idx_out[(size_t)(b_lo + i) * K + pos] = n;
                }
            }
        }
    }
    __device__ __forceinline__ void load8(int r, int k0, float (&v)[8], int m0, const int* smi) const {
        if (r < R && k0 < Din) {
            const int b = r / (K + 1), j = r - b * (K + 1);
            const int nimg = images_per_tile(K), Np = (N + 3) & ~3;
            const int* sidx = smi + nimg * (Np + 8);
            const int tok = j < K ? 1 + sidx[(b - m0 / (K + 1)) * K + j] : 0;
            ld8(tokens + ((long)b * (1 + N) + tok) * Din + k0, v);
        } else {
            zero8(v);
        }
    }
};
struct FwdBOp {     // (row = n, k = din): Wa[n, din]
    static constexpr bool kContigK = true;
    const float* Wa;
    int D, Din;
    __device__ __forceinline__ void load8(int n, int k0, float (&v)[8]) const {
        if (n < D && k0 < Din) ld8(Wa + (size_t)n * Din + k0, v); else zero8(v);
    }
};
struct FwdEpi {
    static constexpr bool kDirect = false;
    static constexpr bool kGridReduce = false;
    const float* ba;
    float *Zs, *Zc, *z2s, *z2c, *z2s_ctr, *z2c_ctr, *z2s_hi, *z2c_hi;
    uint16_t *Zs_hi, *Zs_lo, *Zc_hi, *Zc_lo;
    float center;
    int K, D;
    struct State { float sq, sq_ctr, sq_hi; };
    __device__ __forceinline__ void init(State& s) const { s.sq = s.sq_ctr = s.sq_hi = 0.f; }
    __device__ __forceinline__ void row_ptrs(int r, void* (&p)[3]) const {
        const int b = r / (K + 1), j = r - b * (K + 1);
        if (j < K) {
            const size_t o = ((size_t)b * K + j) * D;
            p[0] = Zs + o; p[1] = Zs_hi ? Zs_hi + o : nullptr; p[2] = Zs_lo ? Zs_lo + o : nullptr;
        } else {
            const size_t o = (size_t)b * D;
            p[0] = Zc + o; p[1] = Zc_hi ? Zc_hi + o : nullptr; p[2] = Zc_lo ? Zc_lo + o : nullptr;
        }
    }
    __device__ __forceinline__ void transform(State& s, int, int n0, uint32_t (&acc)[32]) const {
#pragma unroll
        for (int i = 0; i < 32; i += 2) {
            if (n0 + i < D) {          // D is even: columns come in pairs (packed bf16 conversion, F2FP not F2F)
                const float2 bb = __ldg(reinterpret_cast<const float2*>(ba + n0 + i));
                const float z0 = __fdividef(1.0f, 1.0f + __expf(-(__uint_as_float(acc[i]) + bb.x)));
                const float z1 = __fdividef(1.0f, 1.0f + __expf(-(__uint_as_float(acc[i + 1]) + bb.y)));
                const float c0 = z0 - center, c1 = z1 - center;
                const __nv_bfloat162 h = __floats2bfloat162_rn(c0, c1);
                const uint32_t hb = *reinterpret_cast<const uint32_t*>(&h);
                const float h0 = __uint_as_float(hb << 16), h1 = __uint_as_float(hb & 0xffff0000u);
                s.sq = fmaf(z0, z0, fmaf(z1, z1, s.sq));
                s.sq_ctr = fmaf(c0, c0, fmaf(c1, c1, s.sq_ctr));
                s.sq_hi = fmaf(h0, h0, fmaf(h1, h1, s.sq_hi));
                acc[i] = __float_as_uint(z0);
                acc[i + 1] = __float_as_uint(z1);
            }
        }
    }
    __device__ __forceinline__ void store2(void* const* p, int n, float z0, float z1) const {
        uint32_t hi, lo;
        tg_split2(z0 - center, z1 - center, hi, lo);      // tensor-core operands are centred
        *reinterpret_cast<float2*>(static_cast<float*>(p[0]) + n) = make_float2(z0, z1);
        if (p[1]) *reinterpret_cast<uint32_t*>(static_cast<uint16_t*>(p[1]) + n) = hi;
        if (p[2]) *reinterpret_cast<uint32_t*>(static_cast<uint16_t*>(p[2]) + n) = lo;
    }
    __device__ __forceinline__ void finish(State& s, int r, int row_local, int cgroup, float* scratch, bool valid) const {
        if (cgroup > 0) {
            float* p = scratch + row_local * 16 + (cgroup - 1) * 3;
            p[0] = s.sq; p[1] = s.sq_ctr; p[2] = s.sq_hi;
        }
        __syncthreads();
        if (cgroup == 0 && valid) {
            float a = s.sq, c = s.sq_ctr, h = s.sq_hi;
#pragma unroll
            for (int g = 0; g < kTgWarps / 4 - 1; ++g) {
                const float* p = scratch + row_local * 16 + g * 3;
                a += p[0]; c += p[1]; h += p[2];
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
    }
};

// ---- backward operands ------------------------------------------------------------------------------------------------
struct DpreRowOp {  // (row = r, k = d): dpre = dZ * Z * (1 - Z), contiguous along d
    static constexpr bool kContigK = true;
    const float *Zs, *Zc, *dZs, *dZc;
    int K, D, R;
    __device__ __forceinline__ void load8(int r, int d0, float (&v)[8]) const {
        if (r >= R || d0 >= D) { zero8(v); return; }
        const int b = r / (K + 1), j = r - b * (K + 1);
        const bool cls = (j == K);
        const size_t o = (cls ? (size_t)b * D : ((size_t)b * K + j) * D) + d0;
        float z[8], g[8];
        ld8((cls ? Zc : Zs) + o, z);
        ld8((cls ? dZc : dZs) + o, g);
#pragma unroll
        for (int i = 0; i < 8; ++i) v[i] = g[i] * z[i] * (1.0f - z[i]);
    }
};
struct DpreColOp {  // (row = d, k = r): the same matrix, transposed access (consecutive lanes = consecutive d)
    static constexpr bool kContigK = false;
    const float *Zs, *Zc, *dZs, *dZc;
    int K, D, R;
    __device__ __forceinline__ void load8(int d, int r0, float (&v)[8]) const {
        if (d >= D) { zero8(v); return; }
        int b = r0 / (K + 1), j = r0 - b * (K + 1);
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            float val = 0.f;
            if (r0 + i < R) {
                const bool cls = (j == K);
                const size_t o = (cls ? (size_t)b * D : ((size_t)b * K + j) * D) + d;
                const float z = __ldg((cls ? Zc : Zs) + o), g = __ldg((cls ? dZc : dZs) + o);
                val = g * z * (1.0f - z);
            }
            v[i] = val;
            if (++j > K) { j = 0; ++b; }
        }
    }
};
struct WaTOp {      // (row = din, k = d): Wa[d, din]
    static constexpr bool kContigK = false;
    const float* Wa;
    int D, Din;
    __device__ __forceinline__ void load8(int din, int d0, float (&v)[8]) const {
#pragma unroll
        for (int i = 0; i < 8; ++i) v[i] = (din < Din && d0 + i < D) ? __ldg(Wa + (size_t)(d0 + i) * Din + din) : 0.f;
    }
};
template <class T>
struct XselColOp {  // (row = din, k = r): gathered token rows transposed; row Din is the all-ones column (-> dba)
    static constexpr bool kContigK = false;
    const T* tokens;
    RowSrc src;
    __device__ __forceinline__ void load8(int din, int r0, float (&v)[8]) const {
        const int K = src.K;
        int b = r0 / (K + 1), j = r0 - b * (K + 1);
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            float val = 0.f;
            if (r0 + i < src.R) {
                if (din < src.Din) {
                    const int tok = j < K ? 1 + __ldg(src.idx + (size_t)b * K + j) : 0;
                    val = ldg_tok(tokens + ((size_t)b * (1 + src.N) + tok) * src.Din + din);
                } else if (din == src.Din) {
                    val = 1.0f;
                }
            }
            v[i] = val;
            if (++j > K) { j = 0; ++b; }
        }
    }
};
template <class T>
struct DxTcEpi {    // scatter rows of dX into the (zero-filled) token gradient
    static constexpr bool kDirect = false;
    static constexpr bool kGridReduce = false;
    T* dtokens;
    RowSrc src;
    struct State { int dummy; };
    __device__ __forceinline__ void init(State& s) const { s.dummy = 0; }
    __device__ __forceinline__ void row_ptrs(int r, void* (&p)[3]) const { p[0] = dtokens + src(r); }
    __device__ __forceinline__ void transform(State&, int, int, uint32_t (&)[32]) const {}
    __device__ __forceinline__ void store2(void* const* p, int n, float v0, float v1) const {
        st2_tok(static_cast<T*>(p[0]) + n, v0, v1);
    }
    __device__ __forceinline__ void finish(State&, int, int, int, float*, bool) const {}
};
struct WgradPartEpi {   // per-split partial tile [split][D][ldn]
    static constexpr bool kDirect = false;
    static constexpr bool kGridReduce = false;
    float* part;
    int D, ldn;
    struct State { int dummy; };
    __device__ __forceinline__ void init(State& s) const { s.dummy = 0; }
    __device__ __forceinline__ void row_ptrs(int d, void* (&p)[3]) const { p[0] = part + ((size_t)blockIdx.y * D + d) * ldn; }
    __device__ __forceinline__ void transform(State&, int, int, uint32_t (&)[32]) const {}
    __device__ __forceinline__ void store2(void* const* p, int n, float v0, float v1) const {
        *reinterpret_cast<float2*>(static_cast<float*>(p[0]) + n) = make_float2(v0, v1);
    }
    __device__ __forceinline__ void finish(State&, int, int, int, float*, bool) const {}
};

}  // namespace pph
