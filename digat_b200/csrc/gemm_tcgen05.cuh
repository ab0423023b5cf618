// tcgen05 tensor-core GEMM with fp32-level accuracy (3xTF32 error compensation), TMA-fed, accumulators in TMEM.
//
//   C[M,N] = A[M,K] * W[N,K]^T (+ bias)        A fp32 (split on the fly), W pre-split into two TF32 planes
//   A = A_hi + A_lo  (A_hi = rna_tf32(A), A_lo = rna_tf32(A - A_hi));  W = W_hi + W_lo likewise
//   C = A_hi*W_hi + A_lo*W_hi + A_hi*W_lo      (the dropped A_lo*W_lo term is ~2^-22 relative)
//
// This is the projection GEMM of the DIGAT layer: h | K1 | K2 = X * [W; ffn1; ffn2]^T (reference
// graphEncoders.py:146-148 / 166-168), M = batch*nodes, N = 3D = 1200, K = D = 400.
//
// CTA = 192 threads, one output tile of 128 x BN:
//   warp 0      TMA producer: per k-block (16 fp32 = one 64-byte swizzle row) loads the raw A tile and both W planes
//   warps 2..5  operand transform: split the raw fp32 A tile in smem into A_hi (in place) and A_lo, fence to the
//               async proxy, signal the MMA warp; after the main loop the same warps run the epilogue
//               (tcgen05.ld TMEM -> registers, + bias, 128-bit global stores)
//   warp 1      MMA issuer (one elected lane): 3 x tcgen05.mma.kind::tf32 per 8-wide k-step, commit to the stage's
//               "empty" barrier; owns the TMEM allocation (2*BN fp32 columns).
// Pipeline: full[s] (TMA bytes landed) -> ready[s] (A split done) -> MMA -> empty[s] (tcgen05.commit) -> TMA.
#pragma once
#include "common.cuh"
#include "tma.cuh"
#include "gemm_simt.cuh"   // GroupBias

namespace digat {

constexpr int kTcBK = 16;                       // fp32 elements per k-block = 64 bytes = SWIZZLE_64B span
constexpr int kTcThreads = 192;
constexpr int kTcTransformThreads = 128;
constexpr int kTcPrefetchBlocks = 40;          // M blocks between a CTA and the block whose A rows it prefetches into L2
constexpr int kTcSmallRows = 1024;             // GEMMs of at most this many rows take 32-wide tiles
constexpr int kTcBigRows = 16384;              // GEMMs of more rows take the persistent kernel or the wide tiles

// K-major operand tile, SWIZZLE_64B: rows of 64 bytes, 8-row groups of 512 bytes (SBO), version 1 (sm_100).
__device__ __forceinline__ uint64_t umma_desc_sw64(uint32_t smem_addr) {
    uint64_t d = 0;
    d |= (uint64_t)((smem_addr >> 4) & 0x3FFF);        // start address  [0,14)
    d |= (uint64_t)1 << 16;                             // leading byte offset (unused for swizzled K-major)
    d |= (uint64_t)(512 >> 4) << 32;                    // stride byte offset [32,46)
    d |= (uint64_t)1 << 46;                             // descriptor version
    d |= (uint64_t)4 << 61;                             // SWIZZLE_64B
    return d;
}

// K-major bf16 operand tile of 16 elements per row, SWIZZLE_32B: rows of 32 bytes, 8-row groups of 256 bytes (SBO).
__device__ __forceinline__ uint64_t umma_desc_sw32(uint32_t smem_addr) {
    uint64_t d = 0;
    d |= (uint64_t)((smem_addr >> 4) & 0x3FFF);
    d |= (uint64_t)1 << 16;
    d |= (uint64_t)(256 >> 4) << 32;
    d |= (uint64_t)1 << 46;
    d |= (uint64_t)6 << 61;                             // SWIZZLE_32B
    return d;
}
// kind::f16 with bf16 operands (K = 16 per instruction), fp32 accumulate, both operands K-major.
__host__ __device__ constexpr uint32_t umma_idesc_bf16(int M, int N) {
    return (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}
__device__ __forceinline__ void umma_bf16(uint32_t tmem_d, uint64_t da, uint64_t db, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
        :: "r"(tmem_d), "l"(da), "l"(db), "r"(idesc), "r"(accumulate) : "memory");
}

// kind::tf32, fp32 accumulate, both operands K-major, M=128, N=BN.
__host__ __device__ constexpr uint32_t umma_idesc_tf32(int M, int N) {
    return (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}

__device__ __forceinline__ void umma_tf32(uint32_t tmem_d, uint64_t da, uint64_t db, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}"
        :: "r"(tmem_d), "l"(da), "l"(db), "r"(idesc), "r"(accumulate) : "memory");
}
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];"
                 :: "r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ float tf32_trunc(float x) {      // what the tensor core sees of an fp32 operand
    return __uint_as_float(__float_as_uint(x) & 0xFFFFE000u);
}
__device__ __forceinline__ float to_tf32_rna(float x) {
    uint32_t r;
    asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(x));
    return __uint_as_float(r);
}

// The correction products (A_lo*W_hi + A_hi*W_lo, ~2^-11 of the main term) get their own TMEM accumulator.
// The tensor core adds into the fp32 accumulator with truncation, aligned to the accumulator's exponent; keeping the
// small terms out of the large accumulator removes most of that error (measured: see profiles/ and DESIGN.md).
template <int BN>
struct TcCfg {
    static constexpr int BM = 128;
    static constexpr int A_BYTES = BM * kTcBK * 4;             // one plane of the A tile
    static constexpr int W_BYTES = BN * kTcBK * 4;
    static constexpr int STAGE_BYTES = 2 * A_BYTES + 2 * W_BYTES;
    // BN = 128 is the two-CTAs-per-SM configuration (256 TMEM columns and <= 110 KB of smem each): one CTA's prologue /
    // epilogue overlaps the other's main loop.  The other widths own the SM (up to 512 TMEM columns, ~200 KB).
    static constexpr int SMEM_BUDGET = (BN == 128 ? 108 : 200) * 1024;
    static constexpr int STAGES = SMEM_BUDGET / STAGE_BYTES > 6 ? 6 : SMEM_BUDGET / STAGE_BYTES;
    static constexpr int ACC_COLS = 2 * BN;                    // main + correction accumulators
    static constexpr int TMEM_COLS = (ACC_COLS <= 32) ? 32 : (ACC_COLS <= 64) ? 64 : (ACC_COLS <= 128) ? 128
                                     : (ACC_COLS <= 256) ? 256 : 512;
    static constexpr size_t SMEM = (size_t)STAGES * STAGE_BYTES + 1024 /*alignment slack*/ + 256 /*barriers*/;
    static_assert(ACC_COLS <= 512, "accumulators exceed TMEM");
    static_assert(BN % 16 == 0 && BN <= 256, "invalid UMMA N");
    static_assert(A_BYTES % 1024 == 0 && W_BYTES % 1024 == 0, "operand tiles must keep 1024-byte alignment");
    static_assert(STAGES >= 2, "not enough shared memory for a pipeline");
};

template <int BN>
__global__ void __launch_bounds__(kTcThreads, BN == 128 ? 2 : 1)
gemm_tf32x3_kernel(const __grid_constant__ CUtensorMap map_a, const __grid_constant__ CUtensorMap map_whi,
                   const __grid_constant__ CUtensorMap map_wlo, const float* __restrict__ bias,
                   float* __restrict__ C, int ldc, int M, int N, int K, GroupBias gb) {
    using Cfg = TcCfg<BN>;
    extern __shared__ __align__(1024) uint8_t smem_raw[];   // SWIZZLE_64B operand tiles: keep 1024-byte alignment
    uint8_t* smem = smem_raw;                               // stays a __shared__ pointer (LDS/STS in the transform warps)
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem + (size_t)Cfg::STAGES * Cfg::STAGE_BYTES);
    uint64_t* full = bars;                       // [STAGES] TMA bytes landed
    uint64_t* ready = bars + Cfg::STAGES;        // [STAGES] A split into hi/lo
    uint64_t* empty = bars + 2 * Cfg::STAGES;    // [STAGES] MMAs reading the stage have completed
    uint64_t* accum_full = bars + 3 * Cfg::STAGES;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 3 * Cfg::STAGES + 1);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int n0 = blockIdx.x * BN, m0 = blockIdx.y * Cfg::BM;
    const int nkb = (K + kTcBK - 1) / kTcBK;
    __shared__ float bias_s[BN];
    for (int i = threadIdx.x; i < BN; i += kTcThreads) bias_s[i] = (bias != nullptr && n0 + i < N) ? bias[n0 + i] : 0.f;

    auto a_hi = [&](int s) { return smem + (size_t)s * Cfg::STAGE_BYTES; };
    auto a_lo = [&](int s) { return smem + (size_t)s * Cfg::STAGE_BYTES + Cfg::A_BYTES; };
    auto w_hi = [&](int s) { return smem + (size_t)s * Cfg::STAGE_BYTES + 2 * Cfg::A_BYTES; };
    auto w_lo = [&](int s) { return smem + (size_t)s * Cfg::STAGE_BYTES + 2 * Cfg::A_BYTES + Cfg::W_BYTES; };

    if (warp == 0 && lane == 0) {
        asm volatile("prefetch.tensormap [%0];" :: "l"(reinterpret_cast<uint64_t>(&map_a)) : "memory");
        asm volatile("prefetch.tensormap [%0];" :: "l"(reinterpret_cast<uint64_t>(&map_whi)) : "memory");
        asm volatile("prefetch.tensormap [%0];" :: "l"(reinterpret_cast<uint64_t>(&map_wlo)) : "memory");
        for (int s = 0; s < Cfg::STAGES; ++s) {
            mbar_init(&full[s], 1);
            mbar_init(&ready[s], kTcTransformThreads / 32);      // one arrival per transform warp
            mbar_init(&empty[s], 1);
        }
        mbar_init(accum_full, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 1) {   // TMEM allocation (whole warp), address lands in smem
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;"
                     :: "r"(smem_u32(tmem_slot)), "r"((uint32_t)Cfg::TMEM_COLS) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tmem_base = *tmem_slot;

    if (warp == 0) {
        // ------------------------------------------------------------------ TMA producer
        if (lane == 0) {
            // A is touched first by the CTAs of one M block, all at the same time: every one of them would wait for DRAM.
            // The first N tile of each M block therefore pulls the A rows of a LATER M block (one that starts roughly a
            // wave from now) into L2, so that the loads of the main loop see L2 latency instead of DRAM latency.
            if (blockIdx.x == 0) {
                const int ahead = (int)blockIdx.y + kTcPrefetchBlocks;
                if (ahead < (int)gridDim.y)
                    for (int kb = 0; kb < nkb; ++kb)
                        asm volatile("cp.async.bulk.prefetch.tensor.2d.L2.global [%0, {%1, %2}];"
                                     :: "l"(reinterpret_cast<uint64_t>(&map_a)), "r"(kb * kTcBK), "r"(ahead * Cfg::BM) : "memory");
            }
            for (int kb = 0; kb < nkb; ++kb) {
                const int s = kb % Cfg::STAGES;
                const uint32_t ph = (kb / Cfg::STAGES) & 1;
                mbar_wait(&empty[s], ph ^ 1);
                mbar_arrive_expect_tx(&full[s], Cfg::A_BYTES + 2 * Cfg::W_BYTES);
                tma_load_2d(a_hi(s), &map_a, &full[s], kb * kTcBK, m0);
                tma_load_2d(w_hi(s), &map_whi, &full[s], kb * kTcBK, n0);
                tma_load_2d(w_lo(s), &map_wlo, &full[s], kb * kTcBK, n0);
            }
        }
    } else if (warp == 1) {
        // ------------------------------------------------------------------ MMA issuer
        // The tensor core reads only the upper 19 bits of an fp32 operand (TF32 = truncation), so the RAW A tile is the
        // "hi" operand as it lands from TMA: the main product and the A_hi*W_lo correction are issued as soon as the
        // stage is full, and only the A_lo*W_hi correction waits for the transform warps -- one stage later, so the
        // split of stage s is hidden behind the four independent MMAs of stage s+1.
        if (lane == 0) {
            constexpr uint32_t idesc = umma_idesc_tf32(128, BN);
            auto issue_raw = [&](int kb) {                        // products that need no transformed operand
                const int s = kb % Cfg::STAGES;
                mbar_wait(&full[s], (kb / Cfg::STAGES) & 1);
                asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                const uint64_t d_whi = umma_desc_sw64(smem_u32(w_hi(s))), d_wlo = umma_desc_sw64(smem_u32(w_lo(s)));
                const uint64_t d_ahi = umma_desc_sw64(smem_u32(a_hi(s)));
                const uint32_t d_main = tmem_base, d_corr = tmem_base + (uint32_t)BN;
#pragma unroll
                for (int k = 0; k < kTcBK / 8; ++k) {
                    const uint64_t koff = (uint64_t)((k * 8 * 4) >> 4);   // 32 bytes per k-step, in 16-byte units
                    const uint32_t first = (kb > 0 || k > 0) ? 1u : 0u;
                    umma_tf32(d_main, d_ahi + koff, d_whi + koff, idesc, first);
                    umma_tf32(d_corr, d_ahi + koff, d_wlo + koff, idesc, first);
                }
            };
            auto issue_lo = [&](int kb) {                         // A_lo * W_hi, then release the stage
                const int s = kb % Cfg::STAGES;
                mbar_wait(&ready[s], (kb / Cfg::STAGES) & 1);
                asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                const uint64_t d_whi = umma_desc_sw64(smem_u32(w_hi(s)));
                const uint64_t d_alo = umma_desc_sw64(smem_u32(a_lo(s)));
                const uint32_t d_corr = tmem_base + (uint32_t)BN;
#pragma unroll
                for (int k = 0; k < kTcBK / 8; ++k) {
                    const uint64_t koff = (uint64_t)((k * 8 * 4) >> 4);
                    umma_tf32(d_corr, d_alo + koff, d_whi + koff, idesc, 1u);
                }
                umma_commit(&empty[s]);            // frees the smem stage once every MMA issued so far has retired
            };
            issue_raw(0);
            for (int kb = 0; kb < nkb; ++kb) {
                if (kb + 1 < nkb) issue_raw(kb + 1);
                issue_lo(kb);
            }
            umma_commit(accum_full);               // accumulators complete
        }
    } else {
        // ------------------------------------------------------------------ operand transform, then epilogue
        const int t = threadIdx.x - 64;            // 0..127
        for (int kb = 0; kb < nkb; ++kb) {
            const int s = kb % Cfg::STAGES;
            const uint32_t ph = (kb / Cfg::STAGES) & 1;
            mbar_wait(&full[s], ph);
            float4* hi = reinterpret_cast<float4*>(a_hi(s));
            float4* lo = reinterpret_cast<float4*>(a_lo(s));
#pragma unroll
            for (int i = 0; i < Cfg::A_BYTES / 16 / kTcTransformThreads; ++i) {
                const int idx = t + i * kTcTransformThreads;     // elementwise: the swizzle pattern is irrelevant
                // the raw tile stays untouched (the tensor core truncates it to TF32 itself); lo = rna_tf32(A - trunc(A))
                const float4 v = hi[idx];
                float4 vl;
                vl.x = to_tf32_rna(v.x - tf32_trunc(v.x)); vl.y = to_tf32_rna(v.y - tf32_trunc(v.y));
                vl.z = to_tf32_rna(v.z - tf32_trunc(v.z)); vl.w = to_tf32_rna(v.w - tf32_trunc(v.w));
                lo[idx] = vl;
            }
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // generic-proxy writes -> visible to tcgen05.mma
            __syncwarp();
            if (lane == 0) mbar_arrive(&ready[s]);       // (128 per-thread arrivals serialised on the barrier: ~0.3 us per k-block)
        }
        // epilogue: this warp may touch TMEM lanes [32*(warp%4), +32).  Software-pipelined over 16-column groups: the
        // TMEM loads (and the row-group-bias loads) of group c+1 are in flight while group c is finished and stored.
        mbar_wait(accum_full, 0);
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        const int q = warp & 3;
        const bool has_gb = gb.ptr != nullptr;
        float* stage = reinterpret_cast<float*>(smem) + q * (32 * 20);     // per-warp 32 x (16+4) staging block
        const int m = m0 + q * 32 + lane;
        const bool row_ok = m < M;
        const float* grow = (has_gb && row_ok) ? gb.ptr + (size_t)(m / gb.rows) * gb.ld - gb.col0 + n0 : nullptr;
        const uint32_t tbase = tmem_base + ((uint32_t)(q * 32) << 16);
        uint32_t rm[16], rc[16];
        float4 gq[4];
        auto issue_group = [&](int c) {
            asm volatile(
                "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
                : "=r"(rm[0]), "=r"(rm[1]), "=r"(rm[2]), "=r"(rm[3]), "=r"(rm[4]), "=r"(rm[5]), "=r"(rm[6]), "=r"(rm[7]),
                  "=r"(rm[8]), "=r"(rm[9]), "=r"(rm[10]), "=r"(rm[11]), "=r"(rm[12]), "=r"(rm[13]), "=r"(rm[14]), "=r"(rm[15])
                : "r"(tbase + (uint32_t)c));
            asm volatile(
                "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
                : "=r"(rc[0]), "=r"(rc[1]), "=r"(rc[2]), "=r"(rc[3]), "=r"(rc[4]), "=r"(rc[5]), "=r"(rc[6]), "=r"(rc[7]),
                  "=r"(rc[8]), "=r"(rc[9]), "=r"(rc[10]), "=r"(rc[11]), "=r"(rc[12]), "=r"(rc[13]), "=r"(rc[14]), "=r"(rc[15])
                : "r"(tbase + (uint32_t)(BN + c)));
#pragma unroll
            for (int v4 = 0; v4 < 4; ++v4) {
                const int col = n0 + c + v4 * 4;       // col0 / cols are multiples of 4: a quad is entirely in or out
                gq[v4] = (grow != nullptr && col >= gb.col0 && col < gb.col0 + gb.cols)
                             ? *reinterpret_cast<const float4*>(grow + c + v4 * 4) : make_float4(0.f, 0.f, 0.f, 0.f);
            }
        };
        issue_group(0);
#pragma unroll 1
        for (int c = 0; c < BN; c += 16) {
            asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
            float o[16];
#pragma unroll
            for (int i = 0; i < 16; ++i)        // main + correction accumulators (IEEE add), then the bias
                o[i] = (__uint_as_float(rm[i]) + __uint_as_float(rc[i])) + bias_s[c + i];
#pragma unroll
            for (int v4 = 0; v4 < 4; ++v4) {
                o[v4 * 4 + 0] += gq[v4].x; o[v4 * 4 + 1] += gq[v4].y;
                o[v4 * 4 + 2] += gq[v4].z; o[v4 * 4 + 3] += gq[v4].w;
            }
            if (c + 16 < BN) issue_group(c + 16);                // next group's loads overlap these stores
            // A thread owns one ROW of the tile, so direct stores would scatter 16-byte pieces over 32 rows per
            // instruction (measured: the epilogue was LSU-transaction-bound, 10.5k of 36k cycles per tile).  Stage the
            // 32 x 16 block through shared memory (the pipeline stages are idle now) and write 64-byte row segments:
            // 4 lanes per row, 8 rows per instruction.
            __syncwarp();
#pragma unroll
            for (int v4 = 0; v4 < 4; ++v4)
                *reinterpret_cast<float4*>(stage + lane * 20 + v4 * 4) =
                    make_float4(o[v4 * 4 + 0], o[v4 * 4 + 1], o[v4 * 4 + 2], o[v4 * 4 + 3]);
            __syncwarp();
#pragma unroll
            for (int t4 = 0; t4 < 4; ++t4) {
                const int f = t4 * 32 + lane, row = f >> 2, cq = f & 3;
                const int mr = m0 + q * 32 + row;
                if (mr < M && n0 + c + cq * 4 < N)          // N % 4 == 0; the last N tile may be partial
                    *reinterpret_cast<float4*>(C + (size_t)mr * ldc + n0 + c + cq * 4) =
                        *reinterpret_cast<const float4*>(stage + row * 20 + cq * 4);
            }
        }
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if (warp == 1) {
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;"
                     :: "r"(tmem_base), "r"((uint32_t)Cfg::TMEM_COLS) : "memory");
    }
}

// ------------------------------------------------------------------------------------------------ host side
__global__ void split_tf32_kernel(const float* __restrict__ w, float* __restrict__ hi, float* __restrict__ lo, int64_t n) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) {
        const float x = w[i];
        const float h = to_tf32_rna(x);
        hi[i] = h;
        lo[i] = to_tf32_rna(x - h);
    }
}

template <int BN>
inline int launch_tf32x3_cfg(const float* A, int lda, const float* W_hi, const float* W_lo, int ldw, const float* bias,
                             float* C, int ldc, int M, int N, int K, GroupBias gb, cudaStream_t st) {
    using Cfg = TcCfg<BN>;
    CUtensorMap ma, mh, ml;
    int rc;
    if ((rc = make_tensor_map_2d(&ma, A, M, K, lda, Cfg::BM, kTcBK, CU_TENSOR_MAP_SWIZZLE_64B)) != DIGAT_OK) return rc;
    if ((rc = make_tensor_map_2d(&mh, W_hi, N, K, ldw, BN, kTcBK, CU_TENSOR_MAP_SWIZZLE_64B)) != DIGAT_OK) return rc;
    if ((rc = make_tensor_map_2d(&ml, W_lo, N, K, ldw, BN, kTcBK, CU_TENSOR_MAP_SWIZZLE_64B)) != DIGAT_OK) return rc;
    if (int rc_ = ensure_dynamic_smem(gemm_tf32x3_kernel<BN>, (size_t)(Cfg::SMEM))) return rc_;
    dim3 grid((N + BN - 1) / BN, (M + Cfg::BM - 1) / Cfg::BM);
    gemm_tf32x3_kernel<BN><<<grid, kTcThreads, Cfg::SMEM, st>>>(ma, mh, ml, bias, C, ldc, M, N, K, gb);
    return check_launch("digat_linear_tf32x3");
}

// Row-group bias accepted by both tcgen05 projection GEMMs (digat_linear_tf32x3, digat_linear_bf16).
inline int check_group_bias(const char* who, const GroupBias& gb, int N) {
    DIGAT_REQUIRE(gb.ptr == nullptr || (gb.rows > 0 && gb.col0 >= 0 && gb.cols > 0 && gb.col0 + gb.cols <= N &&
                                        (gb.col0 & 3) == 0 && (gb.cols & 3) == 0 && (gb.ld & 3) == 0 && gb.ld >= gb.cols &&
                                        aligned16(gb.ptr)),
                  "%s: bad row-group bias (col0/cols must be multiples of 4)", who);
    return DIGAT_OK;
}

template <int BN>
int launch_tf32x3_persistent(const float* A, int lda, const float* W_hi, const float* W_lo, int ldw, const float* bias,
                             float* C, int ldc, int M, int N, int K, GroupBias gb, cudaStream_t st);   // gemm_tcgen05_persistent.cuh

inline int launch_linear_tf32x3(const float* A, int lda, const float* W_hi, const float* W_lo, int ldw, const float* bias,
                                float* C, int ldc, int M, int N, int K, GroupBias gb, cudaStream_t st) {
    if (M == 0) return DIGAT_OK;
    DIGAT_REQUIRE(A && W_hi && W_lo && C, "digat_linear_tf32x3: null pointer");
    if (int rc_ = check_group_bias("digat_linear_tf32x3", gb, N)) return rc_;
    DIGAT_REQUIRE(M >= 0 && N > 0 && K > 0, "digat_linear_tf32x3: bad shape M=%d N=%d K=%d", M, N, K);
    DIGAT_REQUIRE((K & 3) == 0 && (lda & 3) == 0 && (ldw & 3) == 0 && (ldc & 3) == 0,
                  "digat_linear_tf32x3: K, lda, ldw, ldc must be multiples of 4");
    DIGAT_REQUIRE(lda >= K && ldw >= K && ldc >= N, "digat_linear_tf32x3: leading dimension too small");
    DIGAT_REQUIRE(aligned16(A) && aligned16(W_hi) && aligned16(W_lo) && aligned16(C) && (!bias || aligned16(bias)),
                  "digat_linear_tf32x3: pointers must be 16-byte aligned");
    DIGAT_REQUIRE(N % 16 == 0, "digat_linear_tf32x3: N=%d must be a multiple of 16", N);
    DIGAT_REQUIRE(gb.kbatches >= 1, "digat_linear_tf32x3: bad split-K batch count");
    const bool scatter = gb.out_rows != nullptr || gb.kbatches > 1;    // row scatter / split-K live in the persistent kernel only
    if (scatter) DIGAT_REQUIRE(N <= 1280, "digat_linear_tf32x3: c_row_index needs N <= 1280 (N=%d)", N);
    const bool big = M > kTcBigRows;
    // Large M: persistent 128 x 240 tiles, or 208-wide ones for widths that 240 does not divide (N = 400: featureAffine)
    // when they waste < 10 % of the MMA columns (400 -> 2 x 208 = 4 %; the 128-wide tiles below compute 512 columns = 28 %).
    if (scatter || (big && N <= 1280 && (N % 240 == 0 || ((N + 207) / 208) * 208 * 10 < N * 11))) {
        if (N % 240 == 0) return launch_tf32x3_persistent<240>(A, lda, W_hi, W_lo, ldw, bias, C, ldc, M, N, K, gb, st);
        return launch_tf32x3_persistent<208>(A, lda, W_hi, W_lo, ldw, bias, C, ldc, M, N, K, gb, st);
    }
    // a few hundred rows (the context projections of a training step, M = batch): three 128-row tiles x N/128 columns
    // would occupy a dozen SMs, each pulling its whole A panel and 2 W planes through one SM's ingest; narrow tiles
    // spread the same MMAs over N/32 times as many SMs (results are bit-identical: the k order per element is unchanged)
    if (M <= kTcSmallRows) return launch_tf32x3_cfg<32>(A, lda, W_hi, W_lo, ldw, bias, C, ldc, M, N, K, gb, st);
    // Large M keeps a wide tile (fewer re-reads of A: measured 185 vs 158 TFLOP/s at 240 against 128).  Small problems
    // (few tiles) and the other widths: 128-wide tiles, two CTAs per SM (measured 1.45x faster at M = 4096); the last N
    // tile may be partial.
    if (big && N % 240 == 0) return launch_tf32x3_cfg<240>(A, lda, W_hi, W_lo, ldw, bias, C, ldc, M, N, K, gb, st);
    if (big && N % 160 == 0) return launch_tf32x3_cfg<160>(A, lda, W_hi, W_lo, ldw, bias, C, ldc, M, N, K, gb, st);
    return launch_tf32x3_cfg<128>(A, lda, W_hi, W_lo, ldw, bias, C, ldc, M, N, K, gb, st);
}

}  // namespace digat
