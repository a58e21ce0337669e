// "Single-shot" small GEMM on tcgen05 for the add-on layer products (K <= 192 per CTA):
//
//   C[m, n] (+)= sum_{k in this CTA's k range} A(m, k) * B(n, k)        A, B: fp32 functors (contracts of pph_tcgemm.cuh)
//
// pph_tcgemm.cuh walks column tiles and k-blocks inside one CTA with a two-stage fill -> MMA pipeline: at the add-on
// shapes (K = 192 = three k-blocks) that is three global-load round trips, three CTA-wide barriers and 41-82 CTAs --
// latency bound (ncu: tensor pipe < 3 % active, 20-35 us).  Here every CTA owns ONE 128 x BN output tile and its whole
// k range fits in shared memory, so the structure collapses to
//   all global loads of k-block 0 and 1 in flight -> convert / split to bf16 hi + lo -> swizzled shared stores ->
//   one barrier -> 3 passes x KB x 4 tcgen05.mma into one TMEM accumulator -> epilogue
// and the grid is (row tiles) x (column tiles) x (k splits): 82-164 CTAs at the add-on shapes.  With k splits the
// partial tiles are reduced by ALL CTAs after one grid-wide barrier (fixed order: deterministic).
// Precision: the 3-term bf16 split of pph_tcgemm.cuh (A_lo B_hi + A_hi B_lo + A_hi B_hi, fp32 accumulation in TMEM).
#pragma once

#include "pph_common.cuh"
#include "pph_tc_ptx.cuh"
#include "pph_tcgemm.cuh"      // tg_store_split8, constants

namespace pph {

constexpr int kTsThreads = 512;
constexpr int kTsWarps = kTsThreads / 32;
constexpr int kTsBM = 128;
constexpr int kTsBK = 64;
constexpr int kTsMaxKB = 3;         // k-blocks per CTA (K <= 192)
constexpr int kTsMaxBN = 128;

// operand buffers double as the per-warp transpose tiles of the epilogue (16 warps x 32 x 34 floats)
__host__ __device__ inline size_t tcshot_operand_bytes(int BN, int KB) {
    const size_t ops = (size_t)KB * 2 * (kTsBM + BN) * kTsBK * 2, tiles = (size_t)kTsWarps * 32 * 34 * 4;
    return ((ops > tiles ? ops : tiles) + 1023) / 1024 * 1024;
}
inline size_t tcshot_smem_bytes(int BN, int KB) {
    return 1024 + tcshot_operand_bytes(BN, KB) + 128 * 16 * 4 + 128 * 3 * 8 + 256;
}

// Optional operand contract (row-contiguous operands, kContigK == false):
//   static constexpr bool kQuad = true;
//   __device__ void load8x4(int row0, int k0, float (&v)[4][8]) const;     // rows row0..row0+3 (row0 % 4 == 0) x k0..k0+7
// lets a thread fetch its values with 128-bit loads along the rows (4x fewer load instructions and index look-ups
// than eight scalar loads per row) -- the transposed operands of the weight gradient are what this is for.
template <class Op, class = void>
struct op_is_quad { static constexpr bool value = false; };
template <class Op>
struct op_is_quad<Op, decltype((void)Op::kQuad)> { static constexpr bool value = Op::kQuad; };

// A operands that compute their own row list first (FwdSelAOp): prologue(m0, smem words, write_out) by all threads, then
// load8(r, k0, v, m0, smem words).  The words live in the epilogue's scratch area, idle until the accumulator is drained.
template <class Op, class = void>
struct op_selects { static constexpr bool value = false; };
template <class Op>
struct op_selects<Op, decltype((void)Op::kSelect)> { static constexpr bool value = Op::kSelect; };

// Extra epilogue contract on top of pph_tcgemm.cuh's:
//   static constexpr bool kGridReduce;                       // run reduce() on every CTA after a grid-wide barrier
//   __device__ void reduce(int cta, int n_ctas, int tid, int nthreads) const;
template <class AOp, class BOp, class Epi>
__global__ void __launch_bounds__(kTsThreads, 1)
tcshot_kernel(int M, int N, int Kd, int BN, int k_per_split, unsigned int* sync_ctr, AOp a_op, BOp b_op, Epi epi) {
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
    const int kz0 = blockIdx.z * k_per_split, kz1 = min(Kd, kz0 + k_per_split);
    const int KB = (kz1 - kz0 + kTsBK - 1) / kTsBK;                  // 1..kTsMaxKB
    const int KBmax = (k_per_split + kTsBK - 1) / kTsBK;             // layout is sized by the launch, not by this split
    const int a_bytes = kTsBM * kTsBK * 2, b_bytes = BN * kTsBK * 2;
    uint8_t* sA_hi = smem;
    uint8_t* sA_lo = sA_hi + (size_t)KBmax * a_bytes;
    uint8_t* sB_hi = sA_lo + (size_t)KBmax * a_bytes;
    uint8_t* sB_lo = sB_hi + (size_t)KBmax * b_bytes;
    uint8_t* tail = smem + tcshot_operand_bytes(BN, KBmax);
    float* scratch = reinterpret_cast<float*>(tail);                                     // [128][16]
    void** rowptr = reinterpret_cast<void**>(tail + 128 * 16 * 4);                        // [128][3]
    uint64_t* acc_done = reinterpret_cast<uint64_t*>(tail + 128 * 16 * 4 + 128 * 3 * 8);
    uint32_t* tmem_ptr = reinterpret_cast<uint32_t*>(acc_done + 1);

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int m0 = blockIdx.x * kTsBM, n0 = blockIdx.y * BN;
    if (tid == 0) {
        ptx::mbar_init(acc_done, 1);
        ptx::fence_mbar_init();
    }
    if (warp == 1) ptx::tmem_alloc(tmem_ptr, 128);
    if (tid >= 128 && tid < 256) {
        void* p3[3] = {nullptr, nullptr, nullptr};
        if (m0 + tid - 128 < M) epi.row_ptrs(m0 + tid - 128, p3);
        rowptr[(tid - 128) * 3 + 0] = p3[0]; rowptr[(tid - 128) * 3 + 1] = p3[1]; rowptr[(tid - 128) * 3 + 2] = p3[2];
    }

    if constexpr (op_selects<AOp>::value) {
        a_op.prologue(m0, reinterpret_cast<int*>(scratch), blockIdx.y == 0 && blockIdx.z == 0);
        __syncthreads();
    }

    // ---- fill: k-block kb+1's global loads are in flight while k-block kb is converted and stored -------------------
    constexpr bool kAQ = op_is_quad<AOp>::value, kBQ = op_is_quad<BOp>::value;
    const int nbg = BN * 8;                                  // B groups of 8 k per k-block (<= 1024: two per thread)
    // quad items: (4 adjacent rows, one 8-wide k chunk).  A has 32 x 8 = 256 of them, B (BN / 4) x 8 <= 256; when both
    // operands are quad the first half of the CTA serves A and the second half B
    const int a_item = tid, b_item = kAQ ? tid - 256 : tid;
    const int nbq = (BN >> 2) * 8;
    float va[2][4][8], vb_own[2][4][8];                      // [set][group or quad row][k]
    // both operands quad: a thread serves ONE of them, so the two roles share one register array
    float (&vb)[2][4][8] = *((kAQ && kBQ) ? &va : &vb_own);
    auto zero8v = [](float (&v)[8]) {
#pragma unroll
        for (int e = 0; e < 8; ++e) v[e] = 0.f;
    };
    auto load_kb = [&](int kb, int set) {
        const int k0 = kz0 + kb * kTsBK;
        if constexpr (kAQ) {
            if (a_item < 256) {
                const int rq = a_item & 31, c = a_item >> 5;
                if (k0 + c * 8 < kz1) a_op.load8x4(m0 + 4 * rq, k0 + c * 8, va[set]);
                else {
#pragma unroll
                    for (int i = 0; i < 4; ++i) zero8v(va[set][i]);
                }
            }
        } else {
#pragma unroll
            for (int i = 0; i < 2; ++i) {
                const int g = tid + i * kTsThreads;
                const int row = AOp::kContigK ? (g >> 3) : (g & (kTsBM - 1));
                const int c = AOp::kContigK ? (g & 7) : (g >> 7);
                if (k0 + c * 8 < kz1) {
                    if constexpr (op_selects<AOp>::value)
                        a_op.load8(m0 + row, k0 + c * 8, va[set][i], m0, reinterpret_cast<const int*>(scratch));
                    else
                        a_op.load8(m0 + row, k0 + c * 8, va[set][i]);
                } else {
                    zero8v(va[set][i]);
                }
            }
        }
        if constexpr (kBQ) {
            if (b_item >= 0 && b_item < nbq) {
                const int nq = BN >> 2;
                const int rq = b_item % nq, c = b_item / nq;
                if (k0 + c * 8 < kz1) b_op.load8x4(n0 + 4 * rq, k0 + c * 8, vb[set]);
                else {
#pragma unroll
                    for (int i = 0; i < 4; ++i) zero8v(vb[set][i]);
                }
            }
        } else {
#pragma unroll
            for (int i = 0; i < 2; ++i) {
                const int g = tid + i * kTsThreads;
                if (g < nbg) {
                    const int row = BOp::kContigK ? (g >> 3) : (g % BN);
                    const int c = BOp::kContigK ? (g & 7) : (g / BN);
                    if (k0 + c * 8 < kz1) b_op.load8(n0 + row, k0 + c * 8, vb[set][i]);
                    else zero8v(vb[set][i]);
                }
            }
        }
    };
    auto store_kb = [&](int kb, int set) {
        uint8_t* ah = sA_hi + (size_t)kb * a_bytes;
        uint8_t* al = sA_lo + (size_t)kb * a_bytes;
        uint8_t* bh = sB_hi + (size_t)kb * b_bytes;
        uint8_t* bl = sB_lo + (size_t)kb * b_bytes;
        if constexpr (kAQ) {
            if (a_item < 256) {
                const int rq = a_item & 31, c = a_item >> 5;
#pragma unroll
                for (int i = 0; i < 4; ++i) tg_store_split8(ah, al, 4 * rq + i, c, va[set][i]);
            }
        } else {
#pragma unroll
            for (int i = 0; i < 2; ++i) {
                const int g = tid + i * kTsThreads;
                const int row = AOp::kContigK ? (g >> 3) : (g & (kTsBM - 1));
                const int c = AOp::kContigK ? (g & 7) : (g >> 7);
                tg_store_split8(ah, al, row, c, va[set][i]);
            }
        }
        if constexpr (kBQ) {
            if (b_item >= 0 && b_item < nbq) {
                const int nq = BN >> 2;
                const int rq = b_item % nq, c = b_item / nq;
#pragma unroll
                for (int i = 0; i < 4; ++i) tg_store_split8(bh, bl, 4 * rq + i, c, vb[set][i]);
            }
        } else {
#pragma unroll
            for (int i = 0; i < 2; ++i) {
                const int g = tid + i * kTsThreads;
                if (g < nbg) {
                    const int row = BOp::kContigK ? (g >> 3) : (g % BN);
                    const int c = BOp::kContigK ? (g & 7) : (g / BN);
                    tg_store_split8(bh, bl, row, c, vb[set][i]);
                }
            }
        }
    };
    load_kb(0, 0);
#pragma unroll
    for (int kb = 0; kb < kTsMaxKB; ++kb) {
        if (kb < KB) {
            if (kb + 1 < KB) load_kb(kb + 1, (kb + 1) & 1);
            store_kb(kb, kb & 1);
        }
    }
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    ptx::tc_fence_before();
    __syncthreads();
    ptx::tc_fence_after();
    const uint32_t tmem_base = *tmem_ptr;
    if (tid == 0) {
        const uint32_t idesc = ptx::umma_idesc_bf16(kTsBM, BN);
        bool first = true;
        for (int kb = 0; kb < KB; ++kb) {
            const uint32_t a_hi = ptx::smem_u32(sA_hi + (size_t)kb * a_bytes), a_lo = ptx::smem_u32(sA_lo + (size_t)kb * a_bytes);
            const uint32_t b_hi = ptx::smem_u32(sB_hi + (size_t)kb * b_bytes), b_lo = ptx::smem_u32(sB_lo + (size_t)kb * b_bytes);
#pragma unroll
            for (int term = 0; term < 3; ++term) {
                const uint32_t a = term == 0 ? a_lo : a_hi, b = term == 1 ? b_lo : b_hi;
#pragma unroll
                for (int kk = 0; kk < kTsBK / 16; ++kk) {
                    ptx::mma_bf16_ss(tmem_base, ptx::umma_desc_k_sw128(a + kk * 32), ptx::umma_desc_k_sw128(b + kk * 32), idesc,
                                     first ? 0u : 1u);
                    first = false;
                }
            }
        }
        ptx::mma_commit(acc_done);
    }

    // ---- epilogue (as pph_tcgemm.cuh: thread = row for the transform, transposed through shared memory for stores) --
    typename Epi::State st;
    epi.init(st);
    const int quarter = warp & 3, cgroup = warp >> 2;
    const int m_row = m0 + quarter * 32 + lane;
    ptx::mbar_wait(acc_done, 0u);
    ptx::tc_fence_after();
    float* tstage = reinterpret_cast<float*>(smem) + warp * (32 * 34);        // operand buffers are idle now
    const uint32_t taddr = tmem_base + ((uint32_t)(quarter * 32) << 16);
    const int ncols = min(BN, N - n0);
    for (int c0 = cgroup * 32; c0 < ncols; c0 += 32 * (kTsWarps / 4)) {
        uint32_t v[32];
        ptx::tmem_ld_32x32(taddr + c0, v);
        ptx::tmem_ld_wait(v);
        if (m_row < M) epi.transform(st, m_row, n0 + c0, v);
        if (Epi::kDirect) continue;
        __syncwarp();
#pragma unroll
        for (int j = 0; j < 32; j += 2)
            *reinterpret_cast<float2*>(&tstage[lane * 34 + j]) = make_float2(__uint_as_float(v[j]), __uint_as_float(v[j + 1]));
        __syncwarp();
        const int cn = 2 * (lane & 15), n = n0 + c0 + cn;
        if (c0 + cn < ncols) {             // BN need not be a multiple of 32: columns past the tile belong to the next CTA
#pragma unroll 4
            for (int r2 = 0; r2 < 32; r2 += 2) {
                const int r = r2 + (lane >> 4);
                if (m0 + quarter * 32 + r < M) {
                    const float2 q = *reinterpret_cast<const float2*>(&tstage[r * 34 + cn]);
                    epi.store2(rowptr + (quarter * 32 + r) * 3, n, q.x, q.y);
                }
            }
        }
    }
    epi.finish(st, m_row, quarter * 32 + lane, cgroup, scratch, m_row < M);
    ptx::tc_fence_before();
    __syncthreads();
    if (warp == 1) {
        ptx::tc_fence_after();
        ptx::tmem_dealloc(tmem_base, 128);
    }
    if constexpr (Epi::kGridReduce) {
        const unsigned int n_ctas = gridDim.x * gridDim.y * gridDim.z;
        const int cta = blockIdx.x + gridDim.x * (blockIdx.y + gridDim.y * blockIdx.z);
        grid_barrier(sync_ctr, n_ctas);
        epi.reduce(cta, (int)n_ctas, tid, kTsThreads);
        grid_finish(sync_ctr, sync_ctr + 1, n_ctas);
    }
}

template <class AOp, class BOp, class Epi>
inline int launch_tcshot(int M, int N, int Kd, int BN, int k_per_split, unsigned int* sync_ctr, AOp a, BOp b, Epi e,
                         cudaStream_t st, const char* what) {
    auto kern = tcshot_kernel<AOp, BOp, Epi>;
    const int KB = ceil_div(k_per_split, kTsBK);
    if (KB < 1 || KB > kTsMaxKB || BN % 16 != 0 || BN < 16 || BN > kTsMaxBN || k_per_split % kTsBK != 0) {
        set_error("%s: tcshot plan BN=%d k_per_split=%d", what, BN, k_per_split);
        return PPH_EUNSUP;
    }
    const size_t smem = tcshot_smem_bytes(BN, KB);
    cudaError_t err = opt_in_smem(kern, (int)smem);
    if (err != cudaSuccess) { set_error("%s: cudaFuncSetAttribute: %s", what, cudaGetErrorString(err)); return (int)err; }
    dim3 grid(ceil_div(M, kTsBM), ceil_div(N, BN), ceil_div(Kd, k_per_split));
    if (Epi::kGridReduce) {
        int sms = pph_sm_count();
        if (sms <= 0) sms = 148;
        if ((int)(grid.x * grid.y * grid.z) > sms) {       // one CTA per SM (shared memory): all must be co-resident
            set_error("%s: %u CTAs cannot be co-resident on %d SMs", what, grid.x * grid.y * grid.z, sms);
            return PPH_EUNSUP;
        }
    }
    launch_k(kern, grid, dim3(kTsThreads), smem, st, M, N, Kd, BN, k_per_split, sync_ctr, a, b, e);
    return launch_status(what);
}

}  // namespace pph
