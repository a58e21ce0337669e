// (a3-a5) Fused normalise + similarity + max-pool kernel on the 5th-gen tensor cores (PPH_MODE_BF16X3 / PPH_MODE_BF16).
// Replaces the two conv2d + ~10 elementwise passes + max_pool2d of protopformer.py:201-247 with ONE persistent
// kernel; the (B,P,K) distance map lives only in TMEM and never touches HBM.
//
//   tile (local)  : 128 prototypes (UMMA M, TMEM lanes) x G images * K tokens (UMMA N <= 256, TMEM columns)
//                   A = prototype rows [128 x D] bf16 K-major, B = token rows [G*K x D] bf16 K-major (Zs is [B*K, D],
//                   so G consecutive images are one contiguous TMA box), accumulated over D in 64-wide k-blocks.
//   tile (global) : 128 global prototypes x up to 256 images (one CLS token each).
//   precision     : BF16X3 runs three k-passes into the same accumulator, P_lo*Z_hi + P_hi*Z_lo + P_hi*Z_hi
//                   (small terms first), which restores ~16 mantissa bits per operand; BF16 runs P_hi*Z_hi only.
//   epilogue      : thread = prototype (TMEM lane), walks its row with tcgen05.ld: d = z2[col] - 2*acc, running
//                   min/argmin per image, then + p2, relu, log((d+1)/(d+eps)); writes dmin/argmin/act [B,P].
//
// Warp roles (384 threads, 1 CTA / SM, persistent over tiles):
//   warp 0 TMA producer | warp 1 MMA issuer | warp 2 TMEM allocator | warp 3 idle
//   warps 4-7 epilogue group 0 (even tiles of this CTA) | warps 8-11 epilogue group 1 (odd tiles)
// Pipelines: 4-stage smem ring (full/empty mbarriers, TMA complete_tx / tcgen05.commit) and a 2-stage TMEM
// accumulator ring (2 x 256 columns; tmem_full by tcgen05.commit, tmem_empty by the epilogue warps), so the
// epilogue of tile i overlaps the MMAs of tile i+1 and the other group's epilogue of tile i-1.
#include <math.h>
#include <stdlib.h>

#include "pph_common.cuh"
#include "pph_tc_ptx.cuh"

namespace pph {

constexpr int kTcThreads = 384;
constexpr int kTcStages = 4;
constexpr int kTcBlockM = 128;
constexpr int kTcBlockK = 64;                               // bf16 elements per k-block = one 128B swizzle row
constexpr int kTcMaxN = 256;
constexpr int kTcABytes = kTcBlockM * kTcBlockK * 2;        // 16 KB
constexpr int kTcBBytes = kTcMaxN * kTcBlockK * 2;          // 32 KB
constexpr int kTcStageBytes = kTcABytes + kTcBBytes;
constexpr int kTcSmemBytes = 1024 /*align slack*/ + kTcStages * kTcStageBytes + 2 * kTcMaxN * 4 /*x2*/ + 256 /*bars*/;

struct TcParams {
    int B, K, D, P, Pg;
    int G;                    // images per local tile
    int MT_l, NG_l;           // local tiles: prototype tiles x image groups
    int MT_g, NB_g;           // global tiles: prototype tiles x image chunks (256 images)
    int n_local, n_tiles;
    int umma_n_l, umma_n_g;   // UMMA N (multiple of 16)
    int gN;                   // images per global tile (<= 256)
    int box_rows_l, box_rows_g;
    int act_fn;
    float eps;
    const float *z2s, *z2c, *p2l, *p2g;
    float *dmin_l, *act_l, *dmin_g, *act_g;
    int32_t* argmin_l;
};

struct TcTile {
    bool is_global;
    int mt;        // prototype tile
    int grp;       // image group (local) or image chunk (global)
};

__host__ __device__ __forceinline__ TcTile tc_decode(const TcParams& prm, int tile) {
    TcTile t;
    if (tile < prm.n_local) {
        t.is_global = false;
        t.grp = tile / prm.MT_l;
        t.mt = tile - t.grp * prm.MT_l;
    } else {
        const int u = tile - prm.n_local;
        t.is_global = true;
        t.grp = u / prm.MT_g;
        t.mt = u - t.grp * prm.MT_g;
    }
    return t;
}

__device__ __forceinline__ void named_bar_sync(int id, int nthreads) {
    asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}

__device__ __forceinline__ float4 lds_f4(uint32_t saddr) {
    float4 v;
    asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(saddr));
    return v;
}

// Local tile, compile-time token count, latency-tolerant form.  The straightforward running
// (min, argmin) scan is ONE dependent compare->select chain of K links per image (~10 cycles per link with 1-2
// epilogue warps per scheduler: ncu put the 128 x 243 tile at ~4.3 k cycles, 3x the MMA time of the bf16 mode).
// Here every image keeps four independent (min, argmin) chains over the token slots k = 0,1,2,3 (mod 4), merged at the
// image boundary with the lowest-index tie rule, and the tcgen05.ld of chunk i+1 is in flight while chunk i is
// scanned.  Results are identical to the sequential scan (lowest k among equal minima).
template <int KT>
__device__ __forceinline__ void tc_epilogue_local_ilp(const TcParams& prm, const TcTile& t, uint32_t taddr,
                                                      uint32_t x2_saddr, int quarter, int lane) {
    static_assert(KT >= 4, "four chains need four token slots");
    constexpr int GS = kTcMaxN / KT, TC = GS * KT, NCH = (TC + 31) / 32;
    const int p = t.mt * kTcBlockM + quarter * 32 + lane;
    const bool pv = p < prm.P;
    const float p2 = pv ? __ldg(prm.p2l + p) : 0.f;
    const int b0 = t.grp * prm.G;
    float best[4];
    int bk[4];
    uint32_t va[32], vb[32];
    ptx::tmem_ld_32x32(taddr, va);
    ptx::tmem_ld_wait(va);
#pragma unroll
    for (int ch = 0; ch < NCH; ++ch) {
        uint32_t(&cur)[32] = (ch & 1) ? vb : va;
        uint32_t(&nxt)[32] = (ch & 1) ? va : vb;
        if (ch + 1 < NCH) ptx::tmem_ld_32x32(taddr + (ch + 1) * 32, nxt);
        float4 xq[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) xq[i] = lds_f4(x2_saddr + (uint32_t)(ch * 8 + i) * 16u);
#pragma unroll
        for (int j = 0; j < 32; ++j) {
            const int col = ch * 32 + j;
            if (col < TC) {
                const int k = col % KT, g = col / KT, c = k & 3;
                const float4 q = xq[j >> 2];
                const float xx = (j & 3) == 0 ? q.x : (j & 3) == 1 ? q.y : (j & 3) == 2 ? q.z : q.w;
                const float d = fmaf(-2.0f, __uint_as_float(cur[j]), xx);
                if (k < 4) { best[c] = d; bk[c] = k; }
                else if (d < best[c]) { best[c] = d; bk[c] = k; }
                if (k == KT - 1) {
                    float bb = best[0];
                    int kk = bk[0];
#pragma unroll
                    for (int cc = 1; cc < 4; ++cc)
                        if (best[cc] < bb || (best[cc] == bb && bk[cc] < kk)) { bb = best[cc]; kk = bk[cc]; }
                    const int b = b0 + g;
                    if (pv && b < prm.B) {
                        const float dd = relu_keep_nan(bb + p2);
                        const size_t o = (size_t)b * prm.P + p;
                        prm.dmin_l[o] = dd;
                        prm.argmin_l[o] = kk;
                        prm.act_l[o] = act_of_dist(dd, prm.act_fn, prm.eps);
                    }
                }
            }
        }
        if (ch + 1 < NCH) ptx::tmem_ld_wait(nxt);
    }
}

// Drain one accumulator tile: thread = prototype row (TMEM lane), walks its columns with tcgen05.ld.
template <int KT>
__device__ __forceinline__ void tc_epilogue_tile(const TcParams& prm, const TcTile& t, uint32_t taddr, const float* x2,
                                                 int quarter, int lane) {
    if constexpr (KT >= 4) {
        if (!t.is_global) {
            tc_epilogue_local_ilp<KT>(prm, t, taddr, ptx::smem_u32(x2), quarter, lane);
            return;
        }
    }
    const int p = t.mt * kTcBlockM + quarter * 32 + lane;
    if (!t.is_global) {
        const bool pv = p < prm.P;
        const float p2 = pv ? __ldg(prm.p2l + p) : 0.f;
        const int b0 = t.grp * prm.G;
        auto store = [&](int g, float best, int bk) {
            const int b = b0 + g;
            if (pv && b < prm.B) {
                const float d = relu_keep_nan(best + p2);
                const size_t o = (size_t)b * prm.P + p;
                prm.dmin_l[o] = d;
                prm.argmin_l[o] = bk;
                prm.act_l[o] = act_of_dist(d, prm.act_fn, prm.eps);
            }
        };
        float best = INFINITY;
        int bk = 0;
        const int Kc = prm.K;
        const int gcnt = min(prm.G, prm.B - b0);
        const int ncols = gcnt * Kc;
        int g = 0, k = 0;
        for (int c0 = 0; c0 < ncols; c0 += 32) {
            uint32_t v[32];
            ptx::tmem_ld_32x32(taddr + c0, v);
            ptx::tmem_ld_wait(v);
#pragma unroll
            for (int j = 0; j < 32; ++j) {
                if (c0 + j < ncols) {
                    const float d = fmaf(-2.0f, __uint_as_float(v[j]), x2[c0 + j]);
                    if (d < best) { best = d; bk = k; }
                    if (++k == Kc) {
                        store(g, best, bk);
                        ++g; k = 0; best = INFINITY; bk = 0;
                    }
                }
            }
        }
    } else {
        const bool pv = p < prm.Pg;
        const float p2 = pv ? __ldg(prm.p2g + p) : 0.f;
        const int b0 = t.grp * prm.gN;
        const int ncols = min(prm.B - b0, prm.gN);
        for (int c0 = 0; c0 < ncols; c0 += 32) {
            uint32_t v[32];
            ptx::tmem_ld_32x32(taddr + c0, v);
            ptx::tmem_ld_wait(v);
#pragma unroll
            for (int j = 0; j < 32; ++j) {
                if (c0 + j < ncols && pv) {
                    const float d = relu_keep_nan(fmaf(-2.0f, __uint_as_float(v[j]), x2[c0 + j]) + p2);
                    const size_t o = (size_t)(b0 + c0 + j) * prm.Pg + p;
                    prm.dmin_g[o] = d;
                    prm.act_g[o] = act_of_dist(d, prm.act_fn, prm.eps);
                }
            }
        }
    }
}

template <int NTERMS, int KT>
__global__ void __launch_bounds__(kTcThreads, 1)
similarity_tc_kernel(const __grid_constant__ CUtensorMap tmAl_hi, const __grid_constant__ CUtensorMap tmAl_lo,
                     const __grid_constant__ CUtensorMap tmBl_hi, const __grid_constant__ CUtensorMap tmBl_lo,
                     const __grid_constant__ CUtensorMap tmAg_hi, const __grid_constant__ CUtensorMap tmAg_lo,
                     const __grid_constant__ CUtensorMap tmBg_hi, const __grid_constant__ CUtensorMap tmBg_lo,
                     const TcParams prm) {
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
    uint8_t* ring = smem;
    float* x2s = reinterpret_cast<float*>(smem + kTcStages * kTcStageBytes);          // [2][256]
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem + kTcStages * kTcStageBytes + 2 * kTcMaxN * 4);
    uint64_t* full = bars;                      // [kTcStages]
    uint64_t* empty = bars + kTcStages;         // [kTcStages]
    uint64_t* tmem_full = bars + 2 * kTcStages; // [2]
    uint64_t* tmem_empty = tmem_full + 2;       // [2]
    uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(tmem_empty + 2);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int kblocks = prm.D / kTcBlockK;      // per term

    if (warp == 0 && lane == 0) {
        ptx::prefetch_tmap(&tmAl_hi);
        ptx::prefetch_tmap(&tmBl_hi);
        if (NTERMS == 3) { ptx::prefetch_tmap(&tmAl_lo); ptx::prefetch_tmap(&tmBl_lo); }
    }
    if (warp == 1 && lane == 0) {
        for (int s = 0; s < kTcStages; ++s) { ptx::mbar_init(&full[s], 1); ptx::mbar_init(&empty[s], 1); }
        for (int s = 0; s < 2; ++s) { ptx::mbar_init(&tmem_full[s], 1); ptx::mbar_init(&tmem_empty[s], 4); }
        ptx::fence_mbar_init();
    }
    if (warp == 2) ptx::tmem_alloc(tmem_ptr, 512);
    ptx::tc_fence_before();
    __syncthreads();
    ptx::tc_fence_after();
    const uint32_t tmem_base = *tmem_ptr;

    if (warp == 0) {
        // ===================== TMA producer =====================
        int stage = 0;
        uint32_t phase = 0;
        for (int tile = blockIdx.x; tile < prm.n_tiles; tile += gridDim.x) {
            const TcTile t = tc_decode(prm, tile);
            const int rowA = t.mt * kTcBlockM;
            const int rowB = t.is_global ? t.grp * prm.gN : t.grp * prm.G * prm.K;
            const uint32_t bytes = kTcABytes + (uint32_t)(t.is_global ? prm.box_rows_g : prm.box_rows_l) * kTcBlockK * 2;
#pragma unroll 1
            for (int term = 0; term < NTERMS; ++term) {
                // BF16X3 pass order: (A_lo,B_hi), (A_hi,B_lo), (A_hi,B_hi); BF16: (A_hi,B_hi)
                const bool a_lo = (NTERMS == 3) && term == 0;
                const bool b_lo = (NTERMS == 3) && term == 1;
                const CUtensorMap* ma = t.is_global ? (a_lo ? &tmAg_lo : &tmAg_hi) : (a_lo ? &tmAl_lo : &tmAl_hi);
                const CUtensorMap* mb = t.is_global ? (b_lo ? &tmBg_lo : &tmBg_hi) : (b_lo ? &tmBl_lo : &tmBl_hi);
#pragma unroll 1
                for (int kb = 0; kb < kblocks; ++kb) {
                    if (lane == 0) {
                        ptx::mbar_wait(&empty[stage], phase ^ 1u);
                        ptx::mbar_expect_tx(&full[stage], bytes);
                        uint8_t* sA = ring + stage * kTcStageBytes;
                        ptx::tma_load_2d(sA, ma, &full[stage], kb * kTcBlockK, rowA);
                        ptx::tma_load_2d(sA + kTcABytes, mb, &full[stage], kb * kTcBlockK, rowB);
                    }
                    __syncwarp();
                    if (++stage == kTcStages) { stage = 0; phase ^= 1u; }
                }
            }
        }
    } else if (warp == 1) {
        // ===================== MMA issuer =====================
        int stage = 0;
        uint32_t phase = 0;
        int it = 0;
        const uint32_t idesc_l = ptx::umma_idesc_bf16(kTcBlockM, prm.umma_n_l);
        const uint32_t idesc_g = ptx::umma_idesc_bf16(kTcBlockM, prm.umma_n_g);
        for (int tile = blockIdx.x; tile < prm.n_tiles; tile += gridDim.x, ++it) {
            const TcTile t = tc_decode(prm, tile);
            const int acc = it & 1;
            const uint32_t acc_phase = (uint32_t)(it >> 1) & 1u;
            const uint32_t idesc = t.is_global ? idesc_g : idesc_l;
            const uint32_t d_tmem = tmem_base + (uint32_t)acc * kTcMaxN;
            if (lane == 0) ptx::mbar_wait(&tmem_empty[acc], acc_phase ^ 1u);   // epilogue drained this accumulator
            __syncwarp();
            ptx::tc_fence_after();
            const int nkb = NTERMS * kblocks;
#pragma unroll 1
            for (int kbt = 0; kbt < nkb; ++kbt) {
                if (lane == 0) {
                    ptx::mbar_wait(&full[stage], phase);
                    ptx::tc_fence_after();
                    const uint32_t a_base = ptx::smem_u32(ring + stage * kTcStageBytes);
                    const uint32_t b_base = a_base + kTcABytes;
#pragma unroll
                    for (int kk = 0; kk < kTcBlockK / 16; ++kk) {
                        ptx::mma_bf16_ss(d_tmem, ptx::umma_desc_k_sw128(a_base + kk * 32),
                                         ptx::umma_desc_k_sw128(b_base + kk * 32), idesc, (uint32_t)((kbt | kk) != 0));
                    }
                    ptx::mma_commit(&empty[stage]);                       // smem slot reusable once these MMAs retire
                    if (kbt == nkb - 1) ptx::mma_commit(&tmem_full[acc]);  // accumulator complete
                }
                __syncwarp();
                if (++stage == kTcStages) { stage = 0; phase ^= 1u; }
            }
        }
    } else if (warp >= 4) {
        // ===================== epilogue =====================
        const int grp_id = (warp - 4) >> 2;          // which accumulator stage this warp drains
        const int quarter = warp & 3;                // TMEM lane quarter this warp may read
        const int gtid = threadIdx.x - 128 - grp_id * 128;   // 0..127 inside the group
        float* x2 = x2s + grp_id * kTcMaxN;
        int it = 0;
        for (int tile = blockIdx.x; tile < prm.n_tiles; tile += gridDim.x, ++it) {
            if ((it & 1) != grp_id) continue;
            const TcTile t = tc_decode(prm, tile);
            const uint32_t acc_phase = (uint32_t)(it >> 1) & 1u;
            // stage the token norms of this tile's columns (overlaps the MMAs of this tile)
            named_bar_sync(1 + grp_id, 128);
            if (!t.is_global) {
                const long r0 = (long)t.grp * prm.G * prm.K, rmax = (long)prm.B * prm.K;
                for (int c = gtid; c < kTcMaxN; c += 128) x2[c] = (r0 + c < rmax) ? __ldg(prm.z2s + r0 + c) : 0.f;
            } else {
                const int b0 = t.grp * prm.gN;
                for (int c = gtid; c < kTcMaxN; c += 128) x2[c] = (b0 + c < prm.B) ? __ldg(prm.z2c + b0 + c) : 0.f;
            }
            named_bar_sync(1 + grp_id, 128);
            const uint32_t taddr = tmem_base + (uint32_t)grp_id * kTcMaxN + ((uint32_t)(quarter * 32) << 16);

            ptx::mbar_wait(&tmem_full[grp_id], acc_phase);
            ptx::tc_fence_after();
            tc_epilogue_tile<KT>(prm, t, taddr, x2, quarter, lane);
            ptx::tc_fence_before();
            __syncwarp();
            if (lane == 0) ptx::mbar_arrive(&tmem_empty[grp_id]);
        }
    }
    ptx::tc_fence_before();
    __syncthreads();
    if (warp == 2) {
        ptx::tc_fence_after();
        ptx::tmem_dealloc(tmem_base, 512);
    }
}

// ---------------------------------------------------------------------------------------------------------------
// v2: prototype tile resident in shared memory.
// The v1 kernel above re-streams both operands for every (tile, term): 423 KB of L2->SM traffic per 128x243 tile in
// BF16X3 mode, 156 MB per B=64 launch -- it is L2-bandwidth bound (ncu: tensor pipe 22 % of elapsed), not MMA bound.
// Here a CTA keeps ONE prototype tile (hi and lo, all of D) in shared memory for its whole life and walks the image
// groups assigned to it, streaming only the token operand, whose hi and lo k-blocks are loaded once per k-block and
// shared by the three MMA terms: 186 KB per tile (2.3x less).  Used whenever the resident tile leaves room for >= 2
// pipeline stages (D <= 192 in BF16X3, D <= 384 in BF16); larger D falls back to v1.
//   CTA c < n_local_ctas : prototype tile c % MT_l, image groups c / MT_l, + lanes_l, ...
//   remaining CTAs       : global prototype tiles, round robin (each reloads its resident tile per phase)
// ---------------------------------------------------------------------------------------------------------------
constexpr int kTc2MaxStages = 6;
constexpr int kTc2MaxKBlocks = 8;                           // D <= 512

struct Tc2Job {
    bool is_global;
    int mt, t_begin, t_step, t_end;
};

__host__ __device__ __forceinline__ bool tc2_phase(const TcParams& prm, int cta, int p, int lanes_l, int n_local_ctas, int grid,
                                          Tc2Job& j) {
    int q = p;
    if (cta < n_local_ctas) {
        if (p == 0) {
            j.is_global = false;
            j.mt = cta % prm.MT_l;
            j.t_begin = cta / prm.MT_l;
            j.t_step = lanes_l;
            j.t_end = prm.NG_l;
            return true;
        }
        q = p - 1;
    }
    // global prototype tiles are dealt from the END of the grid: first to the CTAs without a local job, then to the
    // highest local lanes (the ones with the fewest image groups when NG_l % lanes_l != 0)
    const int mt = (grid - 1 - cta) + q * grid;
    if (mt >= prm.MT_g) return false;
    j.is_global = true;
    j.mt = mt;
    j.t_begin = 0;
    j.t_step = 1;
    j.t_end = prm.NB_g;
    return true;
}

template <int NTERMS, int KT>
__global__ void __launch_bounds__(kTcThreads, 1)
similarity_tc2_kernel(const __grid_constant__ CUtensorMap tmAl_hi, const __grid_constant__ CUtensorMap tmAl_lo,
                      const __grid_constant__ CUtensorMap tmBl_hi, const __grid_constant__ CUtensorMap tmBl_lo,
                      const __grid_constant__ CUtensorMap tmAg_hi, const __grid_constant__ CUtensorMap tmAg_lo,
                      const __grid_constant__ CUtensorMap tmBg_hi, const __grid_constant__ CUtensorMap tmBg_lo,
                      const TcParams prm, int lanes_l, int n_local_ctas, int stages, int b_tile_bytes) {
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
    constexpr int NOPS = NTERMS == 3 ? 2 : 1;                 // hi (+ lo) copies of each operand
    const int kblocks = prm.D / kTcBlockK;
    const int a_bytes = NOPS * kblocks * kTcABytes;
    const int stage_bytes = NOPS * b_tile_bytes;
    uint8_t* a_res = smem;                                    // [NOPS][kblocks][128 x 64 bf16]
    uint8_t* ring = smem + a_bytes;                           // [stages][NOPS][b_tile_bytes]
    float* x2s = reinterpret_cast<float*>(ring + (size_t)stages * stage_bytes);          // [2][256]
    uint64_t* bars = reinterpret_cast<uint64_t*>(reinterpret_cast<uint8_t*>(x2s) + 2 * kTcMaxN * 4);
    uint64_t* full = bars;                                    // [kTc2MaxStages]
    uint64_t* empty = bars + kTc2MaxStages;                   // [kTc2MaxStages]
    uint64_t* tmem_full = bars + 2 * kTc2MaxStages;           // [2]
    uint64_t* tmem_empty = tmem_full + 2;                     // [2]
    uint64_t* a_full = tmem_empty + 2;                        // [kTc2MaxKBlocks] one per k-block of the resident tile
    uint64_t* a_empty = a_full + kTc2MaxKBlocks;              // [1]
    uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(a_empty + 1);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, cta = blockIdx.x, grid = gridDim.x;

    if (warp == 0 && lane == 0) {
        ptx::prefetch_tmap(&tmAl_hi);
        ptx::prefetch_tmap(&tmBl_hi);
        if (NTERMS == 3) { ptx::prefetch_tmap(&tmAl_lo); ptx::prefetch_tmap(&tmBl_lo); }
    }
    if (warp == 1 && lane == 0) {
        for (int s = 0; s < kTc2MaxStages; ++s) { ptx::mbar_init(&full[s], 1); ptx::mbar_init(&empty[s], 1); }
        for (int s = 0; s < 2; ++s) { ptx::mbar_init(&tmem_full[s], 1); ptx::mbar_init(&tmem_empty[s], 4); }
        for (int kb = 0; kb < kTc2MaxKBlocks; ++kb) ptx::mbar_init(&a_full[kb], 1);
        ptx::mbar_init(a_empty, 1);
        ptx::fence_mbar_init();
    }
    if (warp == 2) ptx::tmem_alloc(tmem_ptr, 512);
    ptx::tc_fence_before();
    __syncthreads();
    ptx::tc_fence_after();
    const uint32_t tmem_base = *tmem_ptr;

    if (warp == 0) {
        // ===================== TMA producer =====================
        int stage = 0;
        uint32_t phase = 0;
        Tc2Job job;
        for (int p = 0; tc2_phase(prm, cta, p, lanes_l, n_local_ctas, grid, job); ++p) {
            // the resident prototype tile is loaded k-block by k-block, interleaved with the first tile's token
            // k-blocks, each k-block on its own barrier: the first MMAs start after 1/kblocks of the tile has landed
            if (lane == 0 && p > 0) ptx::mbar_wait(a_empty, (uint32_t)(p - 1) & 1u);   // MMAs of the previous job retired
            __syncwarp();
            const uint32_t bytes = (uint32_t)NOPS * (uint32_t)(job.is_global ? prm.box_rows_g : prm.box_rows_l) * kTcBlockK * 2;
            for (int t = job.t_begin; t < job.t_end; t += job.t_step) {
                const int rowB = job.is_global ? t * prm.gN : t * prm.G * prm.K;
#pragma unroll 1
                for (int kb = 0; kb < kblocks; ++kb) {
                    if (lane == 0) {
                        if (t == job.t_begin) {
                            ptx::mbar_expect_tx(&a_full[kb], (uint32_t)(NOPS * kTcABytes));
                            for (int op = 0; op < NOPS; ++op) {
                                const CUtensorMap* ma =
                                    job.is_global ? (op ? &tmAg_lo : &tmAg_hi) : (op ? &tmAl_lo : &tmAl_hi);
                                ptx::tma_load_2d(a_res + (size_t)(op * kblocks + kb) * kTcABytes, ma, &a_full[kb],
                                                 kb * kTcBlockK, job.mt * kTcBlockM);
                            }
                        }
                        ptx::mbar_wait(&empty[stage], phase ^ 1u);
                        ptx::mbar_expect_tx(&full[stage], bytes);
                        uint8_t* sB = ring + (size_t)stage * stage_bytes;
                        ptx::tma_load_2d(sB, job.is_global ? &tmBg_hi : &tmBl_hi, &full[stage], kb * kTcBlockK, rowB);
                        if (NTERMS == 3)
                            ptx::tma_load_2d(sB + b_tile_bytes, job.is_global ? &tmBg_lo : &tmBl_lo, &full[stage],
                                             kb * kTcBlockK, rowB);
                    }
                    __syncwarp();
                    if (++stage == stages) { stage = 0; phase ^= 1u; }
                }
            }
        }
    } else if (warp == 1) {
        // ===================== MMA issuer =====================
        int stage = 0;
        uint32_t phase = 0;
        int it = 0;
        const uint32_t idesc_l = ptx::umma_idesc_bf16(kTcBlockM, prm.umma_n_l);
        const uint32_t idesc_g = ptx::umma_idesc_bf16(kTcBlockM, prm.umma_n_g);
        const uint32_t a_base = ptx::smem_u32(a_res);
        Tc2Job job;
        for (int p = 0; tc2_phase(prm, cta, p, lanes_l, n_local_ctas, grid, job); ++p) {
            const uint32_t idesc = job.is_global ? idesc_g : idesc_l;
            for (int t = job.t_begin; t < job.t_end; t += job.t_step, ++it) {
                const int acc = it & 1;
                const uint32_t acc_phase = (uint32_t)(it >> 1) & 1u;
                const uint32_t d_tmem = tmem_base + (uint32_t)acc * kTcMaxN;
                if (lane == 0) ptx::mbar_wait(&tmem_empty[acc], acc_phase ^ 1u);
                __syncwarp();
                ptx::tc_fence_after();
                const bool last_tile = (t + job.t_step >= job.t_end);
#pragma unroll 1
                for (int kb = 0; kb < kblocks; ++kb) {
                    if (lane == 0) {
                        if (t == job.t_begin) ptx::mbar_wait(&a_full[kb], (uint32_t)p & 1u);   // resident k-block landed
                        ptx::mbar_wait(&full[stage], phase);
                        ptx::tc_fence_after();
                        const uint32_t b_hi = ptx::smem_u32(ring + (size_t)stage * stage_bytes);
                        const uint32_t b_lo = b_hi + (uint32_t)b_tile_bytes;
                        const uint32_t a_hi = a_base + (uint32_t)kb * kTcABytes;
                        const uint32_t a_lo = a_base + (uint32_t)(kblocks + kb) * kTcABytes;
#pragma unroll
                        for (int kk = 0; kk < kTcBlockK / 16; ++kk) {
                            const uint32_t o = kk * 32;
                            if (NTERMS == 3) {
                                ptx::mma_bf16_ss(d_tmem, ptx::umma_desc_k_sw128(a_lo + o), ptx::umma_desc_k_sw128(b_hi + o),
                                                 idesc, (uint32_t)((kb | kk) != 0));
                                ptx::mma_bf16_ss(d_tmem, ptx::umma_desc_k_sw128(a_hi + o), ptx::umma_desc_k_sw128(b_lo + o),
                                                 idesc, 1u);
                                ptx::mma_bf16_ss(d_tmem, ptx::umma_desc_k_sw128(a_hi + o), ptx::umma_desc_k_sw128(b_hi + o),
                                                 idesc, 1u);
                            } else {
                                ptx::mma_bf16_ss(d_tmem, ptx::umma_desc_k_sw128(a_hi + o), ptx::umma_desc_k_sw128(b_hi + o),
                                                 idesc, (uint32_t)((kb | kk) != 0));
                            }
                        }
                        ptx::mma_commit(&empty[stage]);
                        if (kb == kblocks - 1) {
                            ptx::mma_commit(&tmem_full[acc]);
                            if (last_tile) ptx::mma_commit(a_empty);            // resident tile may be replaced
                        }
                    }
                    __syncwarp();
                    if (++stage == stages) { stage = 0; phase ^= 1u; }
                }
            }
        }
    } else if (warp >= 4) {
        // ===================== epilogue =====================
        const int grp_id = (warp - 4) >> 2;
        const int quarter = warp & 3;
        const int gtid = threadIdx.x - 128 - grp_id * 128;
        float* x2 = x2s + grp_id * kTcMaxN;
        int it = 0;
        Tc2Job job;
        for (int p = 0; tc2_phase(prm, cta, p, lanes_l, n_local_ctas, grid, job); ++p) {
            for (int tt = job.t_begin; tt < job.t_end; tt += job.t_step, ++it) {
                if ((it & 1) != grp_id) continue;
                TcTile t;
                t.is_global = job.is_global; t.mt = job.mt; t.grp = tt;
                const uint32_t acc_phase = (uint32_t)(it >> 1) & 1u;
                named_bar_sync(1 + grp_id, 128);
                if (!t.is_global) {
                    const long r0 = (long)t.grp * prm.G * prm.K, rmax = (long)prm.B * prm.K;
                    for (int c = gtid; c < kTcMaxN; c += 128) x2[c] = (r0 + c < rmax) ? __ldg(prm.z2s + r0 + c) : 0.f;
                } else {
                    const int b0 = t.grp * prm.gN;
                    for (int c = gtid; c < kTcMaxN; c += 128) x2[c] = (b0 + c < prm.B) ? __ldg(prm.z2c + b0 + c) : 0.f;
                }
                named_bar_sync(1 + grp_id, 128);
                const uint32_t taddr = tmem_base + (uint32_t)grp_id * kTcMaxN + ((uint32_t)(quarter * 32) << 16);
                ptx::mbar_wait(&tmem_full[grp_id], acc_phase);
                ptx::tc_fence_after();
                tc_epilogue_tile<KT>(prm, t, taddr, x2, quarter, lane);
                ptx::tc_fence_before();
                __syncwarp();
                if (lane == 0) ptx::mbar_arrive(&tmem_empty[grp_id]);
            }
        }
    }
    ptx::tc_fence_before();
    __syncthreads();
    if (warp == 2) {
        ptx::tc_fence_after();
        ptx::tmem_dealloc(tmem_base, 512);
    }
}

// ---------------------------------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn get_encode_fn() {
    static EncodeTiledFn fn = nullptr;
    if (fn) return fn;
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    cudaError_t e = cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q);
    if (e != cudaSuccess || q != cudaDriverEntryPointSuccess || !p) {
        (void)cudaGetLastError();
        return nullptr;
    }
    fn = reinterpret_cast<EncodeTiledFn>(p);
    return fn;
}

// bf16 matrix [rows, D] row-major -> 2-D tiled map, box {64 elements, box_rows}, 128B swizzle, OOB rows read as 0.
// A tensor map depends only on (base pointer, rows, D, box_rows): the eager drop-in path calls this entry point every
// step on the same operand buffers, so the encoded maps are kept in a small per-thread cache (SURVEY.md 8(b): "cached
// tensor maps"); a hit costs a 64-byte copy instead of a driver call.
struct MapKey {
    const void* base;
    int rows, D, box_rows;
};
constexpr int kMapCache = 32;
static thread_local MapKey g_map_key[kMapCache];
static thread_local CUtensorMap g_map_val[kMapCache];
static thread_local int g_map_n = 0, g_map_next = 0;

static int make_map_uncached(CUtensorMap* m, const uint16_t* base, int rows, int D, int box_rows);

static int make_map(CUtensorMap* m, const uint16_t* base, int rows, int D, int box_rows) {
    for (int i = 0; i < g_map_n; ++i) {
        const MapKey& k = g_map_key[i];
        if (k.base == base && k.rows == rows && k.D == D && k.box_rows == box_rows) {
            *m = g_map_val[i];
            return 0;
        }
    }
    const int rc = make_map_uncached(m, base, rows, D, box_rows);
    if (rc) return rc;
    const int slot = g_map_n < kMapCache ? g_map_n++ : (g_map_next++ % kMapCache);
    g_map_key[slot] = MapKey{base, rows, D, box_rows};
    g_map_val[slot] = *m;
    return 0;
}

static int make_map_uncached(CUtensorMap* m, const uint16_t* base, int rows, int D, int box_rows) {
    EncodeTiledFn fn = get_encode_fn();
    if (!fn) { set_error("cuTensorMapEncodeTiled entry point unavailable"); return PPH_EDRIVER; }
    cuuint64_t gdim[2] = {(cuuint64_t)D, (cuuint64_t)rows};
    cuuint64_t gstr[1] = {(cuuint64_t)D * 2};
    cuuint32_t box[2] = {(cuuint32_t)kTcBlockK, (cuuint32_t)box_rows};
    cuuint32_t estr[2] = {1, 1};
    CUresult r = fn(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<uint16_t*>(base), gdim, gstr, box, estr,
                    CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                    CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) {
        set_error("cuTensorMapEncodeTiled failed: CUresult %d (rows=%d D=%d box_rows=%d ptr=%p)", (int)r, rows, D,
                  box_rows, (const void*)base);
        return PPH_EDRIVER;
    }
    return 0;
}

constexpr int kTcSmemLimit = 232448;     // 227 KB opt-in maximum per CTA on sm_100

struct Tc2Plan {
    bool ok;
    int stages, b_tile_bytes, lanes_l, n_local_ctas, grid, smem;
};

static Tc2Plan plan_tc2(const TcParams& prm, int nterms, int sms) {
    Tc2Plan pl{};
    const int nops = nterms == 3 ? 2 : 1;
    const int kblocks = prm.D / kTcBlockK;
    const int a_bytes = nops * kblocks * kTcABytes;
    const int rows = prm.box_rows_l > prm.box_rows_g ? prm.box_rows_l : prm.box_rows_g;
    pl.b_tile_bytes = ceil_div(rows * kTcBlockK * 2, 1024) * 1024;
    const int stage_bytes = nops * pl.b_tile_bytes;
    const int fixed = 1024 + a_bytes + 2 * kTcMaxN * 4 + 512;
    int stages = (kTcSmemLimit - fixed) / stage_bytes;
    if (stages > kTc2MaxStages) stages = kTc2MaxStages;
    pl.stages = stages;
    pl.ok = stages >= 2 && kblocks <= kTc2MaxKBlocks;
    pl.smem = fixed + stages * stage_bytes;
    // one CTA per global prototype tile beside the local CTAs (lanes = image-group walkers per prototype tile).
    // Measured on B200 (profiles/r1b_sim_plan_ab.txt): giving the local walkers all 148 SMs and dealing the global
    // tiles out as second jobs (9 lanes instead of 8 at the CUB shape) is 1.5-1.7x SLOWER at every batch size, so
    // the dedicated plan stays.
    const int avail = sms - (prm.MT_g <= sms / 4 ? prm.MT_g : sms / 4);
    int lanes = avail / prm.MT_l;
    if (lanes < 1) lanes = 1;
    if (lanes > prm.NG_l) lanes = prm.NG_l;
    pl.lanes_l = lanes;
    pl.n_local_ctas = prm.MT_l * lanes;
    int grid = pl.n_local_ctas + prm.MT_g;
    if (grid > sms) grid = sms;
    if (grid < pl.n_local_ctas) grid = pl.n_local_ctas;
    pl.grid = grid;
    return pl;
}

// Shape-dependent part of the launch: tile counts, UMMA / TMA box sizes, global-branch chunking and the CTA plan.
// Host-only logic, shared by the launcher and by pph_similarity_plan (which lets the CPU test suite check that every
// tile of every shape is visited exactly once).
static void tc_shape_plan(bool x3, int B, int K, int D, int P, int Pg, int sms, TcParams& prm, Tc2Plan& pl) {
    prm.B = B; prm.K = K; prm.D = D; prm.P = P; prm.Pg = Pg;
    prm.G = kTcMaxN / K;
    prm.MT_l = ceil_div(P, kTcBlockM);
    prm.NG_l = ceil_div(B, prm.G);
    prm.MT_g = Pg > 0 ? ceil_div(Pg, kTcBlockM) : 0;
    prm.n_local = prm.MT_l * prm.NG_l;
    prm.box_rows_l = prm.G * K;
    prm.umma_n_l = ceil_div(prm.box_rows_l, 16) * 16;
    auto set_global_chunk = [&](int gN) {            // images per global tile
        prm.gN = gN;
        prm.NB_g = Pg > 0 ? ceil_div(B, gN) : 0;
        prm.n_tiles = prm.n_local + prm.MT_g * prm.NB_g;
        prm.umma_n_g = ceil_div(B < gN ? B : gN, 16) * 16;
        prm.box_rows_g = prm.umma_n_g;
    };
    set_global_chunk(kTcMaxN);
    // resident-prototype kernel (v2) whenever >= 2 token stages fit beside the resident tile; a 256-image global tile
    // is what breaks that for BF16X3 at D = 192, so large batches chunk the global branch by 128 images instead
    pl = plan_tc2(prm, x3 ? 3 : 1, sms);
    if (!pl.ok && B > 128) {
        set_global_chunk(128);
        pl = plan_tc2(prm, x3 ? 3 : 1, sms);
        if (!pl.ok) set_global_chunk(kTcMaxN);
    }
}

template <int NTERMS, int KT>
static int launch_tc2(const CUtensorMap* maps, const TcParams& prm, const Tc2Plan& pl, cudaStream_t st) {
    auto kern = similarity_tc2_kernel<NTERMS, KT>;
    {   // per call, not cached in a static: the attribute is per device and setting it is cheap
        cudaError_t e = opt_in_smem(kern, kTcSmemLimit);
        if (e != cudaSuccess) { set_error("cudaFuncSetAttribute: %s", cudaGetErrorString(e)); return (int)e; }
    }
    launch_k(kern, dim3(pl.grid), dim3(kTcThreads), (size_t)(pl.smem), st, maps[0], maps[1], maps[2], maps[3], maps[4], maps[5], maps[6], maps[7], prm, pl.lanes_l, pl.n_local_ctas, pl.stages, pl.b_tile_bytes);
    return launch_status("pph_similarity_fwd(tcgen05, resident prototypes)");
}

template <int NTERMS, int KT>
static int launch_tc(const CUtensorMap* maps, const TcParams& prm, int grid, cudaStream_t st) {
    auto kern = similarity_tc_kernel<NTERMS, KT>;
    {
        cudaError_t e = opt_in_smem(kern, kTcSmemBytes);
        if (e != cudaSuccess) { set_error("cudaFuncSetAttribute: %s", cudaGetErrorString(e)); return (int)e; }
    }
    launch_k(kern, dim3(grid), dim3(kTcThreads), (size_t)(kTcSmemBytes), st, maps[0], maps[1], maps[2], maps[3], maps[4], maps[5], maps[6], maps[7], prm);
    return launch_status("pph_similarity_fwd(tcgen05)");
}

int similarity_fwd_tc(int mode, int act_fn, float eps, int B, int K, int D, int P, int Pg,
                      const float* z2s, const float* z2c,
                      const uint16_t* Zs_hi, const uint16_t* Zs_lo, const uint16_t* Zc_hi, const uint16_t* Zc_lo,
                      const float* p2l, const float* p2g,
                      const uint16_t* Pl_hi, const uint16_t* Pl_lo, const uint16_t* Pg_hi, const uint16_t* Pg_lo,
                      float* dmin_l, int32_t* argmin_l, float* act_l, float* dmin_g, float* act_g, cudaStream_t st) {
    const bool x3 = (mode == PPH_MODE_BF16X3);
    PPH_REQUIRE(D % kTcBlockK == 0 && D >= 64 && D <= 512, PPH_EUNSUP,
                "tcgen05 similarity needs D %% 64 == 0 and 64 <= D <= 512 (D=%d)", D);
    PPH_REQUIRE(K >= 1 && K <= kTcMaxN, PPH_EUNSUP, "tcgen05 similarity needs 1 <= K <= 256 (K=%d)", K);
    PPH_REQUIRE(P >= 1 && Zs_hi && Pl_hi && z2s && p2l && dmin_l && argmin_l && act_l, PPH_EINVAL,
                "tcgen05 similarity: null local operand");
    PPH_REQUIRE(!x3 || (Zs_lo && Pl_lo), PPH_EINVAL, "PPH_MODE_BF16X3 needs the lo operands");
    PPH_REQUIRE(Pg == 0 || (Zc_hi && Pg_hi && z2c && p2g && dmin_g && act_g && (!x3 || (Zc_lo && Pg_lo))), PPH_EINVAL,
                "tcgen05 similarity: null global operand");

    int sms = pph_sm_count();
    if (sms <= 0) sms = 148;
    TcParams prm;
    Tc2Plan pl;
    tc_shape_plan(x3, B, K, D, P, Pg, sms, prm, pl);
    prm.act_fn = act_fn; prm.eps = eps;
    prm.z2s = z2s; prm.z2c = z2c; prm.p2l = p2l; prm.p2g = p2g;
    prm.dmin_l = dmin_l; prm.act_l = act_l; prm.dmin_g = dmin_g; prm.act_g = act_g; prm.argmin_l = argmin_l;

    CUtensorMap maps[8];
    int rc;
    if ((rc = make_map(&maps[0], Pl_hi, P, D, kTcBlockM))) return rc;
    if ((rc = make_map(&maps[1], x3 ? Pl_lo : Pl_hi, P, D, kTcBlockM))) return rc;
    if ((rc = make_map(&maps[2], Zs_hi, B * K, D, prm.box_rows_l))) return rc;
    if ((rc = make_map(&maps[3], x3 ? Zs_lo : Zs_hi, B * K, D, prm.box_rows_l))) return rc;
    if (Pg > 0) {
        if ((rc = make_map(&maps[4], Pg_hi, Pg, D, kTcBlockM))) return rc;
        if ((rc = make_map(&maps[5], x3 ? Pg_lo : Pg_hi, Pg, D, kTcBlockM))) return rc;
        if ((rc = make_map(&maps[6], Zc_hi, B, D, prm.box_rows_g))) return rc;
        if ((rc = make_map(&maps[7], x3 ? Zc_lo : Zc_hi, B, D, prm.box_rows_g))) return rc;
    } else {
        for (int i = 4; i < 8; ++i) maps[i] = maps[i - 4];
    }
    const int grid = prm.n_tiles < sms ? prm.n_tiles : sms;
    // compile-time token counts: every K of the BASELINE sweep (49..196 squares) gets an epilogue whose image
    // boundaries are static; any other K takes the generic epilogue (KT = 0)
#define PPH_TC_DISPATCH(KT)                                                                          \
    do {                                                                                             \
        if (pl.ok) return x3 ? launch_tc2<3, KT>(maps, prm, pl, st) : launch_tc2<1, KT>(maps, prm, pl, st); \
        return x3 ? launch_tc<3, KT>(maps, prm, grid, st) : launch_tc<1, KT>(maps, prm, grid, st);   \
    } while (0)
    switch (K) {
        case 49: PPH_TC_DISPATCH(49);
        case 64: PPH_TC_DISPATCH(64);
        case 81: PPH_TC_DISPATCH(81);
        case 100: PPH_TC_DISPATCH(100);
        case 121: PPH_TC_DISPATCH(121);
        case 144: PPH_TC_DISPATCH(144);
        case 169: PPH_TC_DISPATCH(169);
        case 196: PPH_TC_DISPATCH(196);
        default: PPH_TC_DISPATCH(0);
    }
#undef PPH_TC_DISPATCH
}

// Host-side view of the launch plan (no device access, no launch): see include/protohead.h.
int similarity_plan(int mode, int B, int K, int D, int P, int Pg, int sms, int* out, int* coverage) {
    if (sms <= 0) sms = 148;
    const bool x3 = (mode == PPH_MODE_BF16X3);
    TcParams prm;
    Tc2Plan pl;
    tc_shape_plan(x3, B, K, D, P, Pg, sms, prm, pl);
    const int grid_v1 = prm.n_tiles < sms ? prm.n_tiles : sms;
    if (out) {
        const int v[16] = {pl.ok ? 1 : 0, pl.ok ? pl.grid : grid_v1, pl.lanes_l, pl.n_local_ctas, pl.stages, pl.b_tile_bytes,
                           pl.ok ? pl.smem : kTcSmemBytes, prm.gN, prm.MT_l, prm.NG_l, prm.MT_g, prm.NB_g, prm.G,
                           prm.umma_n_l, prm.umma_n_g, prm.n_tiles};
        for (int i = 0; i < 16; ++i) out[i] = v[i];
    }
    if (coverage) {
        if (pl.ok) {
            for (int cta = 0; cta < pl.grid; ++cta) {
                Tc2Job job;
                for (int p = 0; tc2_phase(prm, cta, p, pl.lanes_l, pl.n_local_ctas, pl.grid, job); ++p)
                    for (int t = job.t_begin; t < job.t_end; t += job.t_step)
                        coverage[job.is_global ? prm.n_local + t * prm.MT_g + job.mt : t * prm.MT_l + job.mt] += 1;
            }
        } else {
            for (int cta = 0; cta < grid_v1; ++cta)
                for (int tile = cta; tile < prm.n_tiles; tile += grid_v1) {
                    const TcTile t = tc_decode(prm, tile);
                    coverage[t.is_global ? prm.n_local + t.grp * prm.MT_g + t.mt : t.grp * prm.MT_l + t.mt] += 1;
                }
        }
    }
    return 0;
}

}  // namespace pph
