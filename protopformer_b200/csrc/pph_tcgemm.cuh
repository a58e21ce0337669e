// Small-GEMM kernel on tcgen05 with in-kernel operand preparation ("manual fill"):
//
//   C[m,n] = sum_k A(m,k) * B(n,k)       A, B: fp32 functors (gathers, transposes, on-the-fly elementwise math)
//
// The producers evaluate the functors 8 consecutive k at a time, split every value into bf16 hi + lo
// (hi = rn(v), lo = rn(v - hi)) and store both into shared memory in the UMMA canonical K-major SWIZZLE_128B layout
// (row r of a 64-element k-block at r*128 B, its 16-byte chunk c at position c ^ (r & 7)) -- what TMA would have
// written had the operand existed in HBM as bf16.  One thread then issues the three bf16 passes
// A_lo*B_hi + A_hi*B_lo + A_hi*B_hi into one fp32 TMEM accumulator (fp32-grade product, see pph_similarity_tc.cu).
// This removes every "convert / transpose / gather into a staging buffer" pre-pass the add-on layer GEMMs would
// otherwise need in front of a TMA-fed kernel.
//
// CTA = 128 output rows (UMMA M = 128) x all N columns in tiles of BN <= 256, one k-split (blockIdx.y); 512 threads:
// all 16 warps fill (two shared-memory stages: the fill of k-block i+1 overlaps the MMAs of k-block i), thread 0
// issues the MMAs, all 16 warps drain TMEM (warp w: lane quarter w & 3, column group w >> 2).  The epilogue
// transforms its 32 accumulators per row in registers (thread = row), then transposes them through shared memory so
// that global stores are row-contiguous (lane = column): 32 lanes write one 128-byte line per instruction.
#pragma once

#include "pph_common.cuh"
#include "pph_tc_ptx.cuh"

namespace pph {

// phase timestamps (globaltimer ns) of CTA 0 of the most recent tcgemm launch: development aid, compiled in only with
// -DPPH_DEBUG_STAMPS (then read back through pph_debug_read); the shipped library carries neither
#ifdef PPH_DEBUG_STAMPS
static __device__ long long g_dbg_ts[32];   // one copy per translation unit (the add-on kernels live in pph_addon.cu)
__device__ __forceinline__ void dbg_stamp(int slot) {
    if (blockIdx.x == 0 && blockIdx.y == 0 && threadIdx.x == 0 && slot < 32) {
        long long t;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
        g_dbg_ts[slot] = t;
    }
}
#else
__device__ __forceinline__ void dbg_stamp(int) {}
#endif

constexpr int kTgThreads = 512;
constexpr int kTgWarps = kTgThreads / 32;
constexpr int kTgBM = 128;
constexpr int kTgBK = 64;
constexpr int kTgMaxBN = 256;

__host__ __device__ inline size_t tcgemm_stage_bytes(int BN) { return (size_t)2 * (kTgBM + BN) * kTgBK * 2; }
inline size_t tcgemm_smem_bytes(int BN) { return 1024 + 2 * tcgemm_stage_bytes(BN) + 128 * 16 * 4 + 128 * 3 * 8 + 256; }

// (v0, v1) -> packed bf16x2 hi word and bf16x2 lo word (cvt.rn.bf16x2.f32: one instruction per pair)
__device__ __forceinline__ void tg_split2(float v0, float v1, uint32_t& hi, uint32_t& lo) {
    const __nv_bfloat162 h = __floats2bfloat162_rn(v0, v1);
    hi = *reinterpret_cast<const uint32_t*>(&h);
    const float r0 = v0 - __uint_as_float(hi << 16), r1 = v1 - __uint_as_float(hi & 0xffff0000u);
    const __nv_bfloat162 l = __floats2bfloat162_rn(r0, r1);
    lo = *reinterpret_cast<const uint32_t*>(&l);
}

__device__ __forceinline__ void tg_store_split8(uint8_t* hi_tile, uint8_t* lo_tile, int row, int c, const float (&v)[8]) {
    uint32_t h[4], l[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) tg_split2(v[2 * i], v[2 * i + 1], h[i], l[i]);
    const int off = row * 128 + ((c ^ (row & 7)) << 4);
    *reinterpret_cast<uint4*>(hi_tile + off) = make_uint4(h[0], h[1], h[2], h[3]);
    *reinterpret_cast<uint4*>(lo_tile + off) = make_uint4(l[0], l[1], l[2], l[3]);
}

// Operand functor contract:
//   static constexpr bool kContigK;                              // memory-contiguous along k (else along rows)
//   __device__ void load8(int row, int k0, float (&v)[8]) const; // values (row, k0..k0+7); zeros outside the operand
// Epilogue functor contract:
//   struct State;  __device__ void init(State&) const;
//   __device__ void row_ptrs(int m, void* (&p)[3]) const;                      // up to 3 output row base pointers
//   __device__ void transform(State&, int m, int n0, uint32_t (&acc)[32]) const;  // thread = row m, in place
//   __device__ void store2(void* const* p, int n, float v0, float v1) const;   // columns n, n+1 (n even), coalesced
//   __device__ void finish(State&, int m, int row_local, int cgroup, float* scratch, bool valid) const;
//   static constexpr bool kDirect;   // true: transform() stores its own results (thread = row), no transposed store phase
template <class AOp, class BOp, class Epi>
__global__ void __launch_bounds__(kTgThreads, 1)
tcgemm_kernel(int M, int N, int Kd, int BN, int k_per_split, AOp a_op, BOp b_op, Epi epi) {
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
    const size_t stage_bytes = tcgemm_stage_bytes(BN);
    const int a_bytes = kTgBM * kTgBK * 2, b_bytes = BN * kTgBK * 2;
    float* scratch = reinterpret_cast<float*>(smem + 2 * stage_bytes);                        // [128][16]
    void** rowptr = reinterpret_cast<void**>(smem + 2 * stage_bytes + 128 * 16 * 4);          // [128][3]
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem + 2 * stage_bytes + 128 * 16 * 4 + 128 * 3 * 8);
    uint64_t* empty = bars;            // [2]
    uint64_t* acc_done = bars + 2;     // [1]
    uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(bars + 3);

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int m0 = blockIdx.x * kTgBM;
    const int kz0 = blockIdx.y * k_per_split, kz1 = min(Kd, kz0 + k_per_split);

    dbg_stamp(0);
    if (tid == 0) {
        ptx::mbar_init(&empty[0], 1);
        ptx::mbar_init(&empty[1], 1);
        ptx::mbar_init(acc_done, 1);
        ptx::fence_mbar_init();
    }
    if (warp == 1) ptx::tmem_alloc(tmem_ptr, 256);
    if (tid >= 128 && tid < 256) {
        void* p3[3] = {nullptr, nullptr, nullptr};
        if (m0 + tid - 128 < M) epi.row_ptrs(m0 + tid - 128, p3);
        rowptr[(tid - 128) * 3 + 0] = p3[0]; rowptr[(tid - 128) * 3 + 1] = p3[1]; rowptr[(tid - 128) * 3 + 2] = p3[2];
    }
    ptx::tc_fence_before();
    __syncthreads();
    ptx::tc_fence_after();
    const uint32_t tmem_base = *tmem_ptr;
    const uint32_t idesc = ptx::umma_idesc_bf16(kTgBM, BN);
    dbg_stamp(1);

    typename Epi::State st;
    epi.init(st);
    const int quarter = warp & 3, cgroup = warp >> 2;
    const int m_row = m0 + quarter * 32 + lane;
    float* tstage = reinterpret_cast<float*>(smem) + warp * (32 * 34);     // per-warp transpose tile (stages are idle then)
    int fill = 0;                                   // k-blocks filled so far (stage = fill & 1)
    int ntile = 0;
    // A values of the NEXT k-block are fetched one iteration ahead (its rows are usually the HBM-latency operand)
    float va[2][8];
    auto load_a = [&](int kb) {
#pragma unroll
        for (int i = 0; i < 2; ++i) {
            const int g = tid + i * kTgThreads;
            const int row = AOp::kContigK ? (g >> 3) : (g & (kTgBM - 1));
            const int c = AOp::kContigK ? (g & 7) : (g >> 7);
            a_op.load8(m0 + row, kb + c * 8, va[i]);
        }
    };
    load_a(kz0);
    for (int n0 = 0; n0 < N; n0 += BN, ++ntile) {
        for (int kb = kz0; kb < kz1; kb += kTgBK, ++fill) {
            const int stage = fill & 1, use = fill >> 1;
            uint8_t* sA_hi = smem + stage * stage_bytes;
            uint8_t* sA_lo = sA_hi + a_bytes;
            uint8_t* sB_hi = sA_lo + a_bytes;
            uint8_t* sB_lo = sB_hi + b_bytes;
            // ---- issue the B loads of this k-block (first 2 groups) ...
            float vb[2][8];
#pragma unroll
            for (int i = 0; i < 2; ++i) {
                const int g = tid + i * kTgThreads;
                if (g < BN * 8) {
                    const int row = BOp::kContigK ? (g >> 3) : (g % BN);
                    const int c = BOp::kContigK ? (g & 7) : (g / BN);
                    b_op.load8(n0 + row, kb + c * 8, vb[i]);
                }
            }
            if (use > 0) ptx::mbar_wait(&empty[stage], (uint32_t)(use - 1) & 1u);   // MMAs that read this stage retired
            // ---- ... convert + store the prefetched A, then fetch the next k-block's A behind it
#pragma unroll
            for (int i = 0; i < 2; ++i) {
                const int g = tid + i * kTgThreads;
                const int row = AOp::kContigK ? (g >> 3) : (g & (kTgBM - 1));
                const int c = AOp::kContigK ? (g & 7) : (g >> 7);
                tg_store_split8(sA_hi, sA_lo, row, c, va[i]);
            }
            {
                const int kb_next = kb + kTgBK < kz1 ? kb + kTgBK : kz0;      // wraps to the next column tile
                if (kb + kTgBK < kz1 || n0 + BN < N) load_a(kb_next);
            }
#pragma unroll
            for (int i = 0; i < 2; ++i) {
                const int g = tid + i * kTgThreads;
                if (g < BN * 8) {
                    const int row = BOp::kContigK ? (g >> 3) : (g % BN);
                    const int c = BOp::kContigK ? (g & 7) : (g / BN);
                    tg_store_split8(sB_hi, sB_lo, row, c, vb[i]);
                }
            }
            // ---- rest of B in batches of 2 groups per thread
            for (int g0 = 2 * kTgThreads; g0 < BN * 8; g0 += 2 * kTgThreads) {
#pragma unroll
                for (int i = 0; i < 2; ++i) {
                    const int g = g0 + tid + i * kTgThreads;
                    if (g < BN * 8) {
                        const int row = BOp::kContigK ? (g >> 3) : (g % BN);
                        const int c = BOp::kContigK ? (g & 7) : (g / BN);
                        b_op.load8(n0 + row, kb + c * 8, vb[i]);
                    }
                }
#pragma unroll
                for (int i = 0; i < 2; ++i) {
                    const int g = g0 + tid + i * kTgThreads;
                    if (g < BN * 8) {
                        const int row = BOp::kContigK ? (g >> 3) : (g % BN);
                        const int c = BOp::kContigK ? (g & 7) : (g / BN);
                        tg_store_split8(sB_hi, sB_lo, row, c, vb[i]);
                    }
                }
            }
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
            __syncthreads();
            dbg_stamp(2 + fill);
            if (tid == 0) {
                ptx::tc_fence_after();
                const uint32_t a_hi = ptx::smem_u32(sA_hi), a_lo = ptx::smem_u32(sA_lo);
                const uint32_t b_hi = ptx::smem_u32(sB_hi), b_lo = ptx::smem_u32(sB_lo);
#pragma unroll
                for (int term = 0; term < 3; ++term) {
                    const uint32_t a = term == 0 ? a_lo : a_hi, b = term == 1 ? b_lo : b_hi;
#pragma unroll
                    for (int kk = 0; kk < kTgBK / 16; ++kk)
                        ptx::mma_bf16_ss(tmem_base, ptx::umma_desc_k_sw128(a + kk * 32), ptx::umma_desc_k_sw128(b + kk * 32),
                                         idesc, (uint32_t)(kb != kz0 || term != 0 || kk != 0));
                }
                ptx::mma_commit(&empty[stage]);
                if (kb + kTgBK >= kz1) ptx::mma_commit(acc_done);
            }
        }
        // ---- epilogue of this column tile (all MMAs retired -> the stage buffers double as transpose tiles)
        ptx::mbar_wait(acc_done, (uint32_t)ntile & 1u);
        ptx::tc_fence_after();
        dbg_stamp(20 + ntile);
        const uint32_t taddr = tmem_base + ((uint32_t)(quarter * 32) << 16);
        const int ncols = min(BN, N - n0);
        for (int c0 = cgroup * 32; c0 < ncols; c0 += 32 * (kTgWarps / 4)) {
            uint32_t v[32];
            ptx::tmem_ld_32x32(taddr + c0, v);
            ptx::tmem_ld_wait(v);
            if (c0 == 0) dbg_stamp(21);
            if (m_row < M) epi.transform(st, m_row, n0 + c0, v);
            if (Epi::kDirect) continue;
            __syncwarp();
            if (c0 == 0) dbg_stamp(22);
#pragma unroll
            for (int j = 0; j < 32; j += 2)
                *reinterpret_cast<float2*>(&tstage[lane * 34 + j]) = make_float2(__uint_as_float(v[j]), __uint_as_float(v[j + 1]));
            __syncwarp();
            if (c0 == 0) dbg_stamp(23);
            // half-warp per row, two adjacent columns per lane: 16 lanes x 8 B = one 128 B line per row
            const int cn = 2 * (lane & 15), n = n0 + c0 + cn;
            if (n < N) {
#pragma unroll 4
                for (int r2 = 0; r2 < 32; r2 += 2) {
                    const int r = r2 + (lane >> 4);
                    if (m0 + quarter * 32 + r < M) {
                        const float2 q = *reinterpret_cast<const float2*>(&tstage[r * 34 + cn]);
                        epi.store2(rowptr + (quarter * 32 + r) * 3, n, q.x, q.y);
                    }
                }
            }
            if (c0 == 0) dbg_stamp(24);
        }
        ptx::tc_fence_before();
        __syncthreads();                           // TMEM reads + transpose tiles done before the next tile's fill / MMAs
        ptx::tc_fence_after();
    }
    dbg_stamp(28);
    epi.finish(st, m_row, quarter * 32 + lane, cgroup, scratch, m_row < M);
    ptx::tc_fence_before();
    __syncthreads();
    dbg_stamp(29);
    if (warp == 1) {
        ptx::tc_fence_after();
        ptx::tmem_dealloc(tmem_base, 256);
    }
}

template <class AOp, class BOp, class Epi>
inline int launch_tcgemm(int M, int N, int Kd, int BN, int splits, AOp a, BOp b, Epi e, cudaStream_t st,
                         const char* what) {
    auto kern = tcgemm_kernel<AOp, BOp, Epi>;
    const size_t smem = tcgemm_smem_bytes(BN);
    {   // per call: the attribute is per device and setting it is cheap
        cudaError_t err = opt_in_smem(kern, (int)tcgemm_smem_bytes(kTgMaxBN));
        if (err != cudaSuccess) { set_error("%s: cudaFuncSetAttribute: %s", what, cudaGetErrorString(err)); return (int)err; }
    }
    if (splits < 1) splits = 1;
    int k_per_split = ceil_div(ceil_div(Kd, splits), kTgBK) * kTgBK;
    splits = ceil_div(Kd, k_per_split);
    dim3 grid(ceil_div(M, kTgBM), splits);
    launch_k(kern, dim3(grid), dim3(kTgThreads), (size_t)(smem), st, M, N, Kd, BN, k_per_split, a, b, e);
    return launch_status(what);
}

// column-tile width for an N-wide output: a multiple of 16, <= 256, balanced over ceil(N/256) tiles
inline int tcgemm_pick_bn(int N) {
    const int tiles = ceil_div(N, kTgMaxBN);
    return ceil_div(ceil_div(N, tiles), 16) * 16;
}

}  // namespace pph
