// Attention rollout -> CLS-row token score (SURVEY.md 8(f) next #1): the producer of `cls_token_attn`, the score the
// prototype head's foreground selection consumes.  Replaces, per reserve layer,
//   tools/deit_models_attn.py:99-124  attn_rollout   (head mean, discard of the int(T*T*0.9) smallest entries by
//                                     topk + scatter_, (A + 0.2 I) / 1.2, row normalisation, L batched T^3 matmuls)
//   tools/deit_models_attn.py:226     cls_token_attn = attn_rollout[:, 0, 1:]
// Only row 0 of the product is consumed, so the matmul chain collapses to L vector-matrix products walked from the
// last layer to the first, and after the discard only ~10 % of every matrix is non-zero.  Two kernels:
//
//  rollout_prepare2_kernel  (HBM bound: reads every attention tensor exactly once, H*T*T*4 B per (layer, image))
//    persistent CTAs, one (layer, image) tile at a time: stream the H head maps, fuse them into a T x T fp32 tile in
//    shared memory (155 KB at T = 197), find the EXACT k-th smallest entry with a radix select on the
//    order-preserving integer image of the floats (shared-memory histograms), zero the k smallest (ties at the
//    threshold: lowest flat index first), add the identity, normalise the rows, and write the surviving entries as a
//    column-compressed sparse matrix (<= T*T - k + T entries: ~25 KB instead of 155 KB).
//  rollout_chain2_kernel    (latency bound, tiny: the sparse matrices are L2 resident)
//    one CTA per image: v = e_0 (or a caller-supplied start row, the CaiT variant cait_models_attn.py:255-259);
//    for l = L-1 .. 0: v <- v @ a_l as a gather over the columns' entry lists (fixed summation order ->
//    bit-reproducible); scores[b, :] = v[1:] (or all of v).  When a layer's entry list does not fit in shared memory
//    (small discard ratios at T = 197), rollout_chain_kernel walks it from global memory instead.
#include <cuda_fp16.h>
#include <math.h>
#include <stdio.h>
#include <stdlib.h>

#include "pph_common.cuh"

namespace pph {

constexpr int kRoThreads = 1024;
constexpr int kRoMaxLayers = 32;
constexpr int kRoMaxT = 224;              // T*T*4 B must fit in shared memory beside the scratch
constexpr int kRoChainThreads = 512;

// Attention maps of element type E: float, __nv_bfloat16 or __half.  Every bf16 and fp16 value is exact in fp32, so
// a half-precision map is widened at its load and nothing after the load changes: the results equal, bit for bit,
// those of the fp32 maps holding the widened values.
template <class E>
struct RoLayers {
    const E* p[kRoMaxLayers];
};
__device__ __forceinline__ float ro_f32(float x) { return x; }
__device__ __forceinline__ float ro_f32(__nv_bfloat16 x) { return __bfloat162float(x); }
__device__ __forceinline__ float ro_f32(__half x) { return __half2float(x); }

struct RoWorkspace {
    int32_t* col_ptr;      // [L*B][T+1]
    float* ent_val;        // [L*B][cap]
    uint16_t* ent_row;     // [L*B][cap]
    int cap;
};

static inline int rollout_cap(int T, int k_discard) { return ((T * T - k_discard + T) + 7) & ~7; }

static RoWorkspace rollout_carve(void* ws, int L, int B, int T, int k_discard) {
    RoWorkspace w;
    w.cap = rollout_cap(T, k_discard);
    uint8_t* p = reinterpret_cast<uint8_t*>(ws);
    const size_t tiles = (size_t)L * B;
    w.col_ptr = reinterpret_cast<int32_t*>(p);
    p += ((tiles * (T + 1) * 4 + 255) / 256) * 256;
    w.ent_val = reinterpret_cast<float*>(p);
    p += ((tiles * w.cap * 4 + 255) / 256) * 256;
    w.ent_row = reinterpret_cast<uint16_t*>(p);
    return w;
}

static long long rollout_ws_bytes(int L, int B, int T, int k_discard) {
    const size_t tiles = (size_t)L * B;
    const int cap = rollout_cap(T, k_discard);
    return (long long)(((tiles * (T + 1) * 4 + 255) / 256) * 256 + ((tiles * cap * 4 + 255) / 256) * 256 +
                       ((tiles * cap * 2 + 255) / 256) * 256);
}

// order-preserving map float -> uint32 (a < b  <=>  key(a) < key(b); -0 is folded onto +0 first)
__device__ __forceinline__ uint32_t ro_key(float x) {
    const uint32_t b = __float_as_uint(x + 0.0f);
    return (b & 0x80000000u) ? ~b : (b | 0x80000000u);
}

// Step 1 of the prepare kernels for half-precision maps (E = __nv_bfloat16 / __half): stream the H head maps of one
// (layer, image) tile and fuse them into M exactly as the fp32 loop does (fp32 arithmetic, heads in order 0..H-1, the
// mean as sum / H).  A thread holds 16 elements (8 fp32 registers' worth of 4-byte words) per head: the fp32 loop's
// 32*H bytes in flight without its register count, which the 64-register budget of a 1024-thread CTA cannot grow.
// Words: a per-(image, head) slab starts at element (b*H + h)*T*T, odd for odd T*T, so a slab is only 2-byte aligned
// and the heads fused in one register can have different alignments.  Each slab is read as the 4-byte words of its
// own alignment (word j holds elements 2j - odd and 2j + 1 - odd); on an odd slab the element pair of a thread is the
// upper half of its word and the lower half of the next lane's, fetched by one shuffle.  Warp w covers element pairs
// [256 w, 256 w + 256) of a 16384-element chunk, lane-major per step i, so lane 31's next word is lane 0's word of step
// i + 1, and of step 8 for i = 7 (one more word, loaded by lane 0).  A word is loaded when it holds an element of the
// slab; being 4-byte aligned, it never crosses an allocation granule.
__device__ __forceinline__ float ro_lo(uint32_t w, __nv_bfloat16) { return __uint_as_float(w << 16); }
__device__ __forceinline__ float ro_hi(uint32_t w, __nv_bfloat16) { return __uint_as_float(w & 0xffff0000u); }
__device__ __forceinline__ float ro_lo(uint32_t w, __half) { return __low2float(*reinterpret_cast<const __half2*>(&w)); }
__device__ __forceinline__ float ro_hi(uint32_t w, __half) { return __high2float(*reinterpret_cast<const __half2*>(&w)); }

template <int HT, class E>
__device__ __forceinline__ void ro_stream_fuse_half(const E* A, int n, int Hh, int head_fusion, float* M) {
    static_assert(sizeof(E) == 2, "half-precision maps");
    constexpr int kChunk = 16 * kRoThreads;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (int e0 = 0; e0 < n; e0 += kChunk) {
        const int j0 = (e0 >> 1) + warp * 256 + lane;          // word of step i: j0 + 32 i
        float s[16];
#pragma unroll (HT > 0 ? HT : 1)                                   // runtime H: no unrolling (64-register budget)
        for (int h = 0; h < Hh; ++h) {
            const E* S = A + (size_t)h * n;
            const int odd = (int)((reinterpret_cast<uintptr_t>(S) >> 1) & 1);      // uniform over the CTA
            const uint32_t* W = reinterpret_cast<const uint32_t*>(S - odd);
            uint32_t w[8];
#pragma unroll
            for (int i = 0; i < 8; ++i) {
                const int j = j0 + 32 * i;
                w[i] = 2 * j - odd < n ? __ldcs(W + j) : 0u;
            }
            if (odd) {
                const int j8 = j0 + 256;                                 // lane 0: the word after the warp's range
                const uint32_t w8 = lane == 0 && 2 * j8 - 1 < n ? __ldcs(W + j8) : 0u;
#pragma unroll
                for (int i = 0; i < 8; ++i) {
                    const uint32_t nb = __shfl_sync(0xffffffffu, lane == 0 ? (i < 7 ? w[i + 1] : w8) : w[i], (lane + 1) & 31);
                    w[i] = __byte_perm(w[i], nb, 0x5432);               // (upper half of w[i], lower half of nb)
                }
            }
#pragma unroll
            for (int i = 0; i < 8; ++i) {
                const float x0 = ro_lo(w[i], E()), x1 = ro_hi(w[i], E());
                if (h == 0) {
                    s[2 * i] = x0;
                    s[2 * i + 1] = x1;
                } else if (head_fusion == 0) {
                    s[2 * i] += x0;
                    s[2 * i + 1] += x1;
                } else if (head_fusion == 1) {
                    s[2 * i] = fmaxf(s[2 * i], x0);
                    s[2 * i + 1] = fmaxf(s[2 * i + 1], x1);
                } else {
                    s[2 * i] = fminf(s[2 * i], x0);
                    s[2 * i + 1] = fminf(s[2 * i + 1], x1);
                }
            }
        }
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            const int e = 2 * (j0 + 32 * i);
            const float a = head_fusion == 0 ? s[2 * i] / (float)Hh : s[2 * i];
            const float c = head_fusion == 0 ? s[2 * i + 1] / (float)Hh : s[2 * i + 1];
            if (e + 1 < n) {
                *reinterpret_cast<float2*>(M + e) = make_float2(a, c);      // e even: 8-byte aligned
            } else if (e < n) {
                M[e] = a;
            }
        }
    }
}

// exclusive scan of one value per thread over the whole CTA (kRoThreads threads); `wsum` = 32 ints of scratch
__device__ __forceinline__ int block_excl_scan(int v, int* wsum, int& total) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    int incl = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const int t = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += t;
    }
    if (lane == 31) wsum[warp] = incl;
    __syncthreads();
    if (warp == 0) {
        const int w = wsum[lane];
        int wi = w;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int t = __shfl_up_sync(0xffffffffu, wi, o);
            if (lane >= o) wi += t;
        }
        wsum[lane] = wi - w;                     // exclusive warp offsets
        if (lane == 31) wsum[32] = wi;           // grand total
    }
    __syncthreads();
    total = wsum[32];
    const int r = wsum[warp] + incl - v;
    __syncthreads();                             // wsum may be reused by the caller
    return r;
}

// Fused foreground-token selection (protopformer.py:157-158 / deit_models_attn.py:229-230) on the finished score row:
// rank by counting over the W scores in shared memory (larger score first, lower index first on ties -- the rule of
// pph_select_topk), emitted in ascending token order.  All kRoChainThreads threads call it; W <= kRoChainThreads.
__device__ __forceinline__ void ro_emit_topk(const float* sc, int W, int K, int32_t* __restrict__ idx32,
                                             int64_t* __restrict__ idx64, int* wcnt) {
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    bool sel = false;
    if (tid < W) {
        float v = sc[tid];
        if (v != v) v = INFINITY;          // NaN ranks first (torch.topk); with the index tie-break: a total order
        int rank = 0;
        for (int j = 0; j < W; ++j) {
            float q = sc[j];
            if (q != q) q = INFINITY;
            rank += (q > v) || (q == v && j < tid);
        }
        sel = rank < K;
    }
    const unsigned m = __ballot_sync(0xffffffffu, sel);
    if (lane == 0) wcnt[warp] = __popc(m);
    __syncthreads();
    if (sel) {
        int off = 0;
        for (int w = 0; w < warp; ++w) off += wcnt[w];
        const int pos = off + __popc(m & ((1u << lane) - 1u));
        if (pos < K) {
            idx32[pos] = tid;
            if (idx64) idx64[pos] = tid;
        }
    }
}

__global__ void __launch_bounds__(kRoChainThreads)
rollout_chain_kernel(int L, int B, int T, int cap, const int32_t* __restrict__ col_ptr,
                     const float* __restrict__ ent_val, const uint16_t* __restrict__ ent_row,
                     const float* __restrict__ v0, int drop_first, float* __restrict__ scores, int K,
                      int32_t* __restrict__ idx32, int64_t* __restrict__ idx64) {
    __shared__ int wcnt[kRoChainThreads / 32];
    __shared__ float v[2][kRoMaxT];
    const int b = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    for (int j = tid; j < T; j += kRoChainThreads) v[0][j] = v0 ? v0[(size_t)b * T + j] : (j == 0 ? 1.0f : 0.0f);
    __syncthreads();
    int cur = 0;
    for (int l = L - 1; l >= 0; --l) {
        const size_t tile = (size_t)l * B + b;
        const int32_t* cp = col_ptr + tile * (T + 1);
        const float* ev = ent_val + tile * cap;
        const uint16_t* er = ent_row + tile * cap;
        for (int j = warp; j < T; j += kRoChainThreads / 32) {
            const int beg = cp[j], end = cp[j + 1];
            float s = 0.f;
            for (int e = beg + lane; e < end; e += 32) s = fmaf(v[cur][er[e]], ev[e], s);
            s = warp_sum(s);
            if (lane == 0) v[cur ^ 1][j] = s;
        }
        __syncthreads();
        cur ^= 1;
    }
    const int W = T - drop_first;
    for (int j = tid; j < W; j += kRoChainThreads) {
        const float sc = v[cur][j + drop_first];
        scores[(size_t)b * W + j] = sc;
        v[cur ^ 1][j] = sc;                              // the other buffer is free: score row for the selection
    }
    if (K > 0) {
        __syncthreads();
        ro_emit_topk(v[cur ^ 1], W, K, idx32 + (size_t)b * K, idx64 ? idx64 + (size_t)b * K : nullptr, wcnt);
    }
}


// ---------------------------------------------------------------------------------------------------------------
// Why the prepare kernel looks the way it does.  ncu on a first version (profiles/r1b_ncu_rollout_v1.txt): 449 us for
// 328 MB = 9 % of HBM, 13 k instructions per warp per tile, ADU (vote / match / shared atomics) and XU (IEEE divisions)
// pipes busiest -- instruction bound, not memory bound.  Hence:
//   * radix select in 3 passes of 11/11/10 bits with plain shared-memory atomics on a 2048-bin histogram: an 8-bit
//     first digit put ~40 % of all entries into ONE bin (same exponent), so even warp-aggregated atomics serialised on
//     one address; with 11 bits the hottest bin holds a few percent and no vote / match is needed;
//   * zero entries (90 % after the discard) skip both divisions of the normalisation;
//   * the chain kernel stages each layer's sparse matrix in shared memory with coalesced loads and walks one column
//     per THREAD (independent sequential sums) instead of one dependent global-load chain per warp and column.
// The two chain kernels sum a column in different fixed orders (rollout_chain_kernel lane-strided then by shuffle
// tree, rollout_chain2_kernel in row order): each is reproducible, and which one runs depends on the shape alone.
// ---------------------------------------------------------------------------------------------------------------
constexpr int kRo2Bins = 2048;

template <int HT, class E>
__global__ void __launch_bounds__(kRoThreads, 1)
rollout_prepare2_kernel(const RoLayers<E> layers, int L, int B, int H, int T, int k_discard, int head_fusion,
                        float identity_w, int cap, int32_t* __restrict__ col_ptr, float* __restrict__ ent_val,
                        uint16_t* __restrict__ ent_row) {
    extern __shared__ __align__(16) uint8_t ro_smem[];
    const int n = T * T;
    float* M = reinterpret_cast<float*>(ro_smem);                            // [T*T]
    uint32_t* hist = reinterpret_cast<uint32_t*>(M + ((n + 3) & ~3));        // [2048]
    int* cnt = reinterpret_cast<int*>(hist + kRo2Bins);                      // [1024]
    int* wsum = cnt + kRoThreads;                                            // [33]
    __shared__ uint32_t s_prefix, s_cnt;
    __shared__ int s_krem;

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int Hh = HT > 0 ? HT : H;
    const int seg = min(5, kRoThreads / T);
    const int rps = (T + seg - 1) / seg;

    for (int tile = blockIdx.x; tile < L * B; tile += gridDim.x) {
        const int l = tile / B, b = tile - l * B;
        // ---- 1. stream the H head maps once, fuse (deit_models_attn.py:102-107); 8 x H loads in flight per thread ----
        const E* A = layers.p[l] + (size_t)b * Hh * n;
        if constexpr (sizeof(E) == 2) {
            ro_stream_fuse_half<HT>(A, n, Hh, head_fusion, M);
        } else {
            for (int e0 = 0; e0 < n; e0 += 8 * kRoThreads) {
                float s[8];
#pragma unroll
                for (int i = 0; i < 8; ++i) {
                    const int e = e0 + i * kRoThreads + tid;
                    s[i] = e < n ? __ldcs(A + e) : 0.0f;
                }
#pragma unroll
                for (int h = 1; h < Hh; ++h) {
                    float t[8];
#pragma unroll
                    for (int i = 0; i < 8; ++i) {
                        const int e = e0 + i * kRoThreads + tid;
                        t[i] = e < n ? __ldcs(A + (size_t)h * n + e) : 0.0f;
                    }
#pragma unroll
                    for (int i = 0; i < 8; ++i)
                        s[i] = head_fusion == 0 ? s[i] + t[i] : head_fusion == 1 ? fmaxf(s[i], t[i]) : fminf(s[i], t[i]);
                }
#pragma unroll
                for (int i = 0; i < 8; ++i) {
                    const int e = e0 + i * kRoThreads + tid;
                    if (e < n) M[e] = head_fusion == 0 ? s[i] / (float)Hh : s[i];
                }
            }
        }
        __syncthreads();
        // (tried: prefetch.global.L2 of this CTA's next tile here, while HBM is idle -- measured 260.6 -> 290.0 us, rejected)

        // ---- 2. exact k-th smallest: radix select, digits of 11 / 11 / 10 bits, MSB first ----
        uint32_t prefix = 0, eq_total = 0;
        int krem = k_discard < n ? k_discard : n;
        if (krem > 0) {
#pragma unroll 1
            for (int pass = 0; pass < 3; ++pass) {
                const int shift = pass == 0 ? 21 : pass == 1 ? 10 : 0;
                const uint32_t dmask = pass == 2 ? 0x3FFu : 0x7FFu;
                const uint32_t himask = pass == 0 ? 0u : pass == 1 ? 0xFFE00000u : 0xFFFFFC00u;
                hist[tid] = 0;
                hist[tid + kRoThreads] = 0;
                __syncthreads();
                for (int e = tid; e < n; e += kRoThreads) {
                    const uint32_t key = ro_key(M[e]);
                    if ((key & himask) == prefix) atomicAdd(&hist[(key >> shift) & dmask], 1u);
                }
                __syncthreads();
                // bin holding the krem-th active entry: thread = 2 consecutive bins, exclusive scan over the CTA
                const uint32_t c0 = hist[2 * tid], c1 = hist[2 * tid + 1];
                int total;
                const int excl = block_excl_scan((int)(c0 + c1), wsum, total);
                if (excl < krem && krem <= excl + (int)(c0 + c1)) {            // exactly one thread
                    const bool first = krem <= excl + (int)c0;
                    s_prefix = prefix | ((uint32_t)(2 * tid + (first ? 0 : 1)) << shift);
                    s_krem = first ? krem - excl : krem - excl - (int)c0;
                    s_cnt = first ? c0 : c1;
                }
                __syncthreads();
                prefix = s_prefix;
                krem = s_krem;
                eq_total = s_cnt;
                __syncthreads();
            }
            // ---- 3. discard ----
            const bool all_equal_go = (uint32_t)krem == eq_total;
            for (int e = tid; e < n; e += kRoThreads) {
                const uint32_t key = ro_key(M[e]);
                if (key < prefix || (all_equal_go && key == prefix)) M[e] = 0.0f;
            }
            __syncthreads();
            if (!all_equal_go && warp == 0) {                                   // rare: a tie straddles the threshold
                int seen = 0;
                for (int e0 = 0; e0 < n && seen < krem; e0 += 32) {
                    const int e = e0 + lane;
                    const bool eq = e < n && ro_key(M[e]) == prefix;
                    const unsigned m = __ballot_sync(0xffffffffu, eq);
                    if (eq && seen + __popc(m & ((1u << lane) - 1u)) < krem) M[e] = 0.0f;
                    seen += __popc(m);
                }
            }
            __syncthreads();
        }

        // ---- 4. a = (A + w I) / (1 + w), rows normalised; zero off-diagonal entries stay zero without arithmetic ----
        // (both column loops unrolled by 4: left rolled, the DeiT-Ti B = 64 rollout took 295 instead of 284 us, B200 at 1000 W)
        const float den = 1.0f + identity_w;
        for (int r = warp; r < T; r += kRoThreads / 32) {
            float* row = M + r * T;
            float s = 0.f;
#pragma unroll 4
            for (int j = lane; j < T; j += 32) {
                const float x = row[j];
                if (x != 0.0f || j == r) {
                    const float a = (x + (j == r ? identity_w : 0.0f)) / den;
                    row[j] = a;
                    s += a;
                }
            }
            s = warp_sum(s);
#pragma unroll 4
            for (int j = lane; j < T; j += 32) {
                const float a = row[j];
                if (a != 0.0f) row[j] = a / s;
            }
        }
        __syncthreads();

        // ---- 5. column-compressed sparse output: thread = (row segment sg, column j), entries ordered by (j, row) ----
        const bool worker = tid < seg * T;
        const int sg = tid / T, j = tid - sg * T;
        const int r0 = sg * rps, r1 = min(T, r0 + rps);
        int mine = 0;
        if (worker)
            for (int r = r0; r < r1; ++r) mine += (M[r * T + j] != 0.0f);
        cnt[tid] = 0;
        __syncthreads();
        if (worker) cnt[j * seg + sg] = mine;
        __syncthreads();
        int total;
        const int excl = block_excl_scan(cnt[tid], wsum, total);
        cnt[tid] = excl;
        __syncthreads();
        int32_t* cp = col_ptr + (size_t)tile * (T + 1);
        if (worker) {
            int o = cnt[j * seg + sg];
            if (sg == 0) cp[j] = o;
            float* ev = ent_val + (size_t)tile * cap;
            uint16_t* er = ent_row + (size_t)tile * cap;
            for (int r = r0; r < r1; ++r) {
                const float a = M[r * T + j];
                if (a != 0.0f && o < cap) {
                    ev[o] = a;
                    er[o] = (uint16_t)r;
                    ++o;
                }
            }
        }
        if (tid == 0) cp[T] = total < cap ? total : cap;
        __syncthreads();
    }
}

// chain, v2: the layer's sparse matrix is staged in shared memory (coalesced), then thread = column.
__global__ void __launch_bounds__(kRoChainThreads)
rollout_chain2_kernel(int L, int B, int T, int cap, const int32_t* __restrict__ col_ptr,
                      const float* __restrict__ ent_val, const uint16_t* __restrict__ ent_row,
                      const float* __restrict__ v0, int drop_first, float* __restrict__ scores, int K,
                      int32_t* __restrict__ idx32, int64_t* __restrict__ idx64) {
    __shared__ int wcnt[kRoChainThreads / 32];
    extern __shared__ __align__(16) uint8_t ch_smem[];
    float* sval = reinterpret_cast<float*>(ch_smem);                          // [cap]
    int* scp = reinterpret_cast<int*>(sval + cap);                            // [T+1]
    uint16_t* srow = reinterpret_cast<uint16_t*>(scp + T + 1);                // [cap]
    __shared__ float v[2][kRoMaxT];
    const int b = blockIdx.x, tid = threadIdx.x;
    for (int j = tid; j < T; j += kRoChainThreads) v[0][j] = v0 ? v0[(size_t)b * T + j] : (j == 0 ? 1.0f : 0.0f);
    int cur = 0;
    for (int l = L - 1; l >= 0; --l) {
        const size_t tile = (size_t)l * B + b;
        const int32_t* cp = col_ptr + tile * (T + 1);
        const float* ev = ent_val + tile * cap;
        const uint16_t* er = ent_row + tile * cap;
        __syncthreads();                                  // previous layer's readers are done with the stage
        for (int j = tid; j <= T; j += kRoChainThreads) scp[j] = cp[j];
        __syncthreads();
        const int total = scp[T];
        for (int e = tid; e < total; e += kRoChainThreads) {
            sval[e] = ev[e];
            srow[e] = er[e];
        }
        __syncthreads();
        for (int j = tid; j < T; j += kRoChainThreads) {
            const int beg = scp[j], end = scp[j + 1];
            float s = 0.f;
            for (int e = beg; e < end; ++e) s = fmaf(v[cur][srow[e]], sval[e], s);
            v[cur ^ 1][j] = s;
        }
        cur ^= 1;
    }
    __syncthreads();
    const int W = T - drop_first;
    for (int j = tid; j < W; j += kRoChainThreads) {
        const float sc = v[cur][j + drop_first];
        scores[(size_t)b * W + j] = sc;
        v[cur ^ 1][j] = sc;                              // the other buffer is free: score row for the selection
    }
    if (K > 0) {
        __syncthreads();
        ro_emit_topk(v[cur ^ 1], W, K, idx32 + (size_t)b * K, idx64 ? idx64 + (size_t)b * K : nullptr, wcnt);
    }
}


// CaiT start row (cait_models_attn.py:223-259): the class-attention maps (B,H,1,Tc) of the token-only blocks go
// through the same per-layer processing (head fusion, discard of the int(Tc*ratio) smallest entries, + w on the
// CLS column -- `I[:1]` --, row normalisation); the mean over those layers without the CLS column is the row that
// multiplies the patch-layer product.  One CTA per image, thread = entry; the discard is a rank count (stable: among
// equal values the lowest index is discarded first).
constexpr int kRoClsThreads = 256;

template <class E>
__global__ void __launch_bounds__(kRoClsThreads)
rollout_cls_rows_kernel(const RoLayers<E> layers, int n_cls, int B, int H, int Tc, int k_discard, int head_fusion,
                        float identity_w, float* __restrict__ v0) {
    __shared__ float x[kRoClsThreads], acc[kRoClsThreads], wred[kRoClsThreads / 32];
    const int b = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    acc[tid] = 0.0f;
    for (int c = 0; c < n_cls; ++c) {
        const E* A = layers.p[c] + (size_t)b * H * Tc;
        float s = 0.0f;
        if (tid < Tc) {
            s = ro_f32(A[tid]);
            for (int h = 1; h < H; ++h) {
                const float t = ro_f32(A[(size_t)h * Tc + tid]);
                s = head_fusion == 0 ? s + t : head_fusion == 1 ? fmaxf(s, t) : fminf(s, t);
            }
            if (head_fusion == 0) s = s / (float)H;
        }
        __syncthreads();                      // previous layer's readers of x[] are done
        x[tid] = s;
        __syncthreads();
        float a = 0.0f;
        if (tid < Tc) {
            int rank = 0;
            for (int j = 0; j < Tc; ++j) rank += (x[j] < s) || (x[j] == s && j < tid);
            const float kept = rank < k_discard ? 0.0f : s;
            a = (kept + (tid == 0 ? identity_w : 0.0f)) / (1.0f + identity_w);
        }
        float part = warp_sum(a);
        if (lane == 0) wred[warp] = part;
        __syncthreads();
        float tot = 0.0f;
        for (int w = 0; w < kRoClsThreads / 32; ++w) tot += wred[w];
        if (tid < Tc) acc[tid] += a / tot;
    }
    if (tid >= 1 && tid < Tc) v0[(size_t)b * (Tc - 1) + tid - 1] = acc[tid] / (float)n_cls;
}
}  // namespace pph

extern "C" int pph_rollout_ws_bytes(int L, int B, int T, int k_discard, long long* bytes) {
    using namespace pph;
    PPH_REQUIRE(bytes && L >= 1 && B >= 0 && T >= 1 && k_discard >= 0, PPH_EINVAL, "pph_rollout_ws_bytes: bad arguments");
    *bytes = rollout_ws_bytes(L, B, T, k_discard < T * T ? k_discard : T * T);
    return 0;
}

namespace pph {

// pph_rollout_scores and its half-precision-map twins: `fn` names the entry point in error messages
template <class E>
static int rollout_scores_impl(const char* fn, const E* const* attn_layers, int L, int B, int H, int T, int k_discard,
                               int head_fusion, float identity_w, const float* v0, int drop_first, void* workspace,
                               float* scores, int K, int32_t* idx32, int64_t* idx64, pph_stream_t stream) {
    PPH_REQUIRE(attn_layers && workspace && scores, PPH_EINVAL, "%s: null pointer", fn);
    PPH_REQUIRE(L >= 1 && L <= kRoMaxLayers, PPH_EUNSUP, "%s: 1 <= L <= %d (L=%d)", fn, kRoMaxLayers, L);
    PPH_REQUIRE(B >= 0 && H >= 1 && T >= 2 && k_discard >= 0 && (drop_first == 0 || drop_first == 1), PPH_EINVAL,
                "%s: bad dims B=%d H=%d T=%d k=%d", fn, B, H, T, k_discard);
    PPH_REQUIRE(T <= kRoMaxT, PPH_EUNSUP, "%s: T=%d > %d (the fused map must fit in shared memory)", fn, T, kRoMaxT);
    PPH_REQUIRE(head_fusion >= 0 && head_fusion <= 2, PPH_EINVAL, "%s: head_fusion %d", fn, head_fusion);
    PPH_REQUIRE(K == 0 || (K >= 1 && K <= T - drop_first && idx32), PPH_EINVAL,
                "%s: fused selection needs 1 <= K <= %d and idx32 (K=%d)", fn, T - drop_first, K);
    if (B == 0) return 0;
    if (k_discard > T * T) k_discard = T * T;
    RoLayers<E> layers;
    for (int l = 0; l < kRoMaxLayers; ++l) layers.p[l] = l < L ? attn_layers[l] : nullptr;
    for (int l = 0; l < L; ++l) PPH_REQUIRE(layers.p[l], PPH_EINVAL, "%s: layer %d is null", fn, l);
    const RoWorkspace w = rollout_carve(workspace, L, B, T, k_discard);
    const int n = T * T;
    char what_prep[96], what_chain[96];
    snprintf(what_prep, sizeof what_prep, "%s(prepare)", fn);
    snprintf(what_chain, sizeof what_chain, "%s(chain)", fn);
    // the fused map of the largest T fits: kRoMaxT^2 * 4 + scratch <= the 220 KB opted in below
    static_assert((size_t)kRoMaxT * kRoMaxT * 4 + kRo2Bins * 4 + (kRoThreads + 40) * 4 <= 220 * 1024, "kRoMaxT");
    const size_t smem = (size_t)((n + 3) & ~3) * 4 + kRo2Bins * 4 + (kRoThreads + 40) * 4;
    int sms = pph_sm_count();            // per call: the current device may differ between calls
    if (sms <= 0) sms = 148;
    const int tiles = L * B;
    cudaStream_t st = as_stream(stream);
    const dim3 grid(tiles < sms ? tiles : sms);
    auto go = [&](auto kern) -> int {
        cudaError_t e = opt_in_smem(kern, 220 * 1024);
        if (e != cudaSuccess) { set_error("%s: cudaFuncSetAttribute: %s", fn, cudaGetErrorString(e)); return (int)e; }
        launch_k(kern, grid, dim3(kRoThreads), smem, st, layers, L, B, H, T, k_discard, head_fusion, identity_w, w.cap,
                 w.col_ptr, w.ent_val, w.ent_row);
        return launch_status(what_prep);
    };
    // head counts of the reference's backbones: DeiT-Ti 3, CaiT-XXS 4, DeiT-S 6 (deit_models_attn.py:288,303)
    const int rc = H == 3 ? go(rollout_prepare2_kernel<3, E>) : H == 4 ? go(rollout_prepare2_kernel<4, E>)
                   : H == 6 ? go(rollout_prepare2_kernel<6, E>) : go(rollout_prepare2_kernel<0, E>);
    if (rc) return rc;
    // the staged chain needs the layer's entry list in shared memory (cap * 6 B): small discard ratios at large T
    // (T = 197 below a ratio of about 0.3) walk it from global memory instead
    const size_t csmem = (size_t)w.cap * 4 + (size_t)(T + 1) * 4 + (size_t)w.cap * 2 + 16;
    if (csmem <= 160 * 1024) {
        cudaError_t e = opt_in_smem(rollout_chain2_kernel, 160 * 1024);
        if (e != cudaSuccess) { set_error("%s: cudaFuncSetAttribute: %s", fn, cudaGetErrorString(e)); return (int)e; }
        launch_k(rollout_chain2_kernel, dim3(B), dim3(kRoChainThreads), csmem, st, L, B, T, w.cap, w.col_ptr, w.ent_val,
                 w.ent_row, v0, drop_first, scores, K, idx32, idx64);
    } else {
        launch_k(rollout_chain_kernel, dim3(B), dim3(kRoChainThreads), (size_t)0, st, L, B, T, w.cap, w.col_ptr,
                 w.ent_val, w.ent_row, v0, drop_first, scores, K, idx32, idx64);
    }
    return launch_status(what_chain);
}

template <class E>
static int rollout_cls_rows_impl(const char* fn, const E* const* cls_layers, int n_cls, int B, int H, int Tc,
                                 int k_discard, int head_fusion, float identity_w, float* v0, pph_stream_t stream) {
    PPH_REQUIRE(cls_layers && v0, PPH_EINVAL, "%s: null pointer", fn);
    PPH_REQUIRE(n_cls >= 1 && n_cls <= kRoMaxLayers, PPH_EUNSUP, "%s: 1 <= n_cls <= %d", fn, kRoMaxLayers);
    PPH_REQUIRE(B >= 0 && H >= 1 && Tc >= 2 && k_discard >= 0, PPH_EINVAL, "%s: bad dims", fn);
    PPH_REQUIRE(Tc <= kRoClsThreads, PPH_EUNSUP, "%s: Tc=%d > %d", fn, Tc, kRoClsThreads);
    PPH_REQUIRE(head_fusion >= 0 && head_fusion <= 2, PPH_EINVAL, "%s: head_fusion %d", fn, head_fusion);
    if (B == 0) return 0;
    RoLayers<E> layers;
    for (int l = 0; l < kRoMaxLayers; ++l) layers.p[l] = l < n_cls ? cls_layers[l] : nullptr;
    for (int l = 0; l < n_cls; ++l) PPH_REQUIRE(layers.p[l], PPH_EINVAL, "%s: layer %d is null", fn, l);
    launch_k(rollout_cls_rows_kernel<E>, dim3(B), dim3(kRoClsThreads), (size_t)0, as_stream(stream), layers, n_cls, B,
             H, Tc, k_discard, head_fusion, identity_w, v0);
    return launch_status(fn);
}
}  // namespace pph

extern "C" int pph_rollout_scores(const float* const* attn_layers, int L, int B, int H, int T, int k_discard,
                                  int head_fusion, float identity_w, const float* v0, int drop_first, void* workspace,
                                  float* scores, int K, int32_t* idx32, int64_t* idx64, pph_stream_t stream) {
    return pph::rollout_scores_impl("pph_rollout_scores", attn_layers, L, B, H, T, k_discard, head_fusion, identity_w,
                                    v0, drop_first, workspace, scores, K, idx32, idx64, stream);
}

extern "C" int pph_rollout_scores_bf16attn(const uint16_t* const* attn_layers, int L, int B, int H, int T,
                                           int k_discard, int head_fusion, float identity_w, const float* v0,
                                           int drop_first, void* workspace, float* scores, int K, int32_t* idx32,
                                           int64_t* idx64, pph_stream_t stream) {
    return pph::rollout_scores_impl("pph_rollout_scores_bf16attn",
                                    reinterpret_cast<const __nv_bfloat16* const*>(attn_layers), L, B, H, T, k_discard,
                                    head_fusion, identity_w, v0, drop_first, workspace, scores, K, idx32, idx64, stream);
}

extern "C" int pph_rollout_scores_f16attn(const uint16_t* const* attn_layers, int L, int B, int H, int T,
                                          int k_discard, int head_fusion, float identity_w, const float* v0,
                                          int drop_first, void* workspace, float* scores, int K, int32_t* idx32,
                                          int64_t* idx64, pph_stream_t stream) {
    return pph::rollout_scores_impl("pph_rollout_scores_f16attn", reinterpret_cast<const __half* const*>(attn_layers),
                                    L, B, H, T, k_discard, head_fusion, identity_w, v0, drop_first, workspace, scores,
                                    K, idx32, idx64, stream);
}

extern "C" int pph_rollout_cls_rows(const float* const* cls_layers, int n_cls, int B, int H, int Tc, int k_discard,
                                    int head_fusion, float identity_w, float* v0, pph_stream_t stream) {
    return pph::rollout_cls_rows_impl("pph_rollout_cls_rows", cls_layers, n_cls, B, H, Tc, k_discard, head_fusion,
                                      identity_w, v0, stream);
}

extern "C" int pph_rollout_cls_rows_bf16attn(const uint16_t* const* cls_layers, int n_cls, int B, int H, int Tc,
                                             int k_discard, int head_fusion, float identity_w, float* v0,
                                             pph_stream_t stream) {
    return pph::rollout_cls_rows_impl("pph_rollout_cls_rows_bf16attn",
                                      reinterpret_cast<const __nv_bfloat16* const*>(cls_layers), n_cls, B, H, Tc,
                                      k_discard, head_fusion, identity_w, v0, stream);
}

extern "C" int pph_rollout_cls_rows_f16attn(const uint16_t* const* cls_layers, int n_cls, int B, int H, int Tc,
                                            int k_discard, int head_fusion, float identity_w, float* v0,
                                            pph_stream_t stream) {
    return pph::rollout_cls_rows_impl("pph_rollout_cls_rows_f16attn", reinterpret_cast<const __half* const*>(cls_layers),
                                      n_cls, B, H, Tc, k_discard, head_fusion, identity_w, v0, stream);
}
