// Persistent variant of the tcgen05 3xTF32 projection GEMM (gemm_tcgen05.cuh) for large M.
//
// Measured on the one-tile-per-CTA kernel (clock64 instrumentation, M=278528, N=1200, K=400): of ~33k cycles per
// 128x240 tile the MMA main loop takes 18.2k (tensor-bound, 122 cycles per MMA); the rest is CTA launch, barrier init,
// TMEM alloc, pipeline fill and the epilogue, none of which overlaps because the tile's accumulators and ~190 KB of
// stages own the SM.  Here one CTA per SM loops over tiles:
//   * barriers, TMEM and the bias vector are set up once per CTA;
//   * the TMA producer and the transform warps run ahead into the NEXT tile while the epilogue warps (now separate
//     warps) drain the accumulators of the current one -- the pipeline fill hides behind the epilogue;
//   * the MMA warp starts the next tile as soon as the epilogue has released TMEM (tmem_empty barrier).
// Warp roles (448 threads): 0 = TMA producer, 1 = MMA issuer + TMEM owner, 2-5 = operand transform (A_lo),
// 6-13 = epilogue (TMEM lane quarter = warp % 4, two warps per quarter split the columns).  Arithmetic is identical to gemm_tf32x3_kernel<BN>.
#pragma once
#include <cuda_bf16.h>
#include "gemm_tcgen05.cuh"

namespace digat {

constexpr int kTcEpiWarps = 8;                  // two epilogue warps per TMEM lane quarter, each takes half of the columns
constexpr int kTcPersistThreads = (2 + 4 + kTcEpiWarps) * 32;

// kBf16: the BF16 GEMM (gemm_bf16.cuh): a stage holds the raw fp32 A tile, bf16(A) and ONE bf16 plane of W.
template <int BN, bool kBf16 = false>
struct TcPersistCfg {
    static constexpr int A_BYTES = 128 * kTcBK * 4;
    static constexpr int W_BYTES = BN * kTcBK * 4;
    static constexpr int STAGE_BYTES = kBf16 ? A_BYTES + A_BYTES / 2 + W_BYTES / 2 : 2 * A_BYTES + 2 * W_BYTES;
    static constexpr int ACC_BUFS = kBf16 ? 2 : 1;                       // TMEM accumulator buffers (tiles in flight)
    static constexpr int MAX_N = 1280;                                   // bias vector kept in smem for the whole N
    static constexpr int GB_GROUPS = 16;                                 // row groups of one 128-row tile staged in smem
    static constexpr int EXTRA = 512 /*barriers*/ + MAX_N * 4 + kTcEpiWarps * 32 * 20 * 4 /*epilogue staging*/ + GB_GROUPS * BN * 4;
    static constexpr int MAX_STAGES = kBf16 ? 8 : 6;
    static constexpr int STAGES = (226 * 1024 - EXTRA) / STAGE_BYTES > MAX_STAGES ? MAX_STAGES : (226 * 1024 - EXTRA) / STAGE_BYTES;
    static constexpr int TMEM_COLS = 2 * BN <= 256 ? 256 : 512;
    static constexpr size_t SMEM = (size_t)STAGES * STAGE_BYTES + EXTRA;
    static_assert(STAGES >= 3, "not enough shared memory for the pipeline");
    static_assert(A_BYTES % 512 == 0 && W_BYTES % 512 == 0 && STAGE_BYTES % 512 == 0,
                  "operand tiles must start on a swizzle-atom boundary");
    static_assert(!kBf16 || 2 * BN <= 512, "the BF16 GEMM keeps two accumulators in TMEM");
};

// kBf16: C = bf16_rn(A) * W_b^T, one kind::f16 MMA (K = 16) per k-block into ONE accumulator (map_whi = W_b, SWIZZLE_32B;
// map_wlo is unused).  The transform warps write bf16_rn(A) instead of A_lo.  Two accumulator buffers alternate between
// tiles: the MMA warp fills buffer (j+1)&1 while the epilogue drains buffer j&1.  The epilogue is the same code as the
// 3xTF32 scheme's (bias, row-group bias, row scatter, staged row-segment stores).
template <int BN, bool kBf16>
__global__ void __launch_bounds__(kTcPersistThreads, 1)
gemm_tf32x3_persistent_kernel(const __grid_constant__ CUtensorMap map_a, const __grid_constant__ CUtensorMap map_whi,
                              const __grid_constant__ CUtensorMap map_wlo, const float* __restrict__ bias,
                              float* __restrict__ C, int ldc, int M, int N, int K, GroupBias gb) {
    using Cfg = TcPersistCfg<BN, kBf16>;
    extern __shared__ __align__(1024) uint8_t smem_raw[];
    uint8_t* smem = smem_raw;
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem + (size_t)Cfg::STAGES * Cfg::STAGE_BYTES);
    uint64_t* full = bars;                                  // [STAGES] TMA bytes landed
    uint64_t* ready = bars + Cfg::STAGES;                   // [STAGES] A_lo written by the transform warps
    uint64_t* empty = bars + 2 * Cfg::STAGES;               // [STAGES] MMAs reading the stage have retired
    uint64_t* accum_full = bars + 3 * Cfg::STAGES;          // [ACC_BUFS] accumulators of the current tile complete
    uint64_t* tmem_empty = accum_full + Cfg::ACC_BUFS;      // [ACC_BUFS] epilogue has drained the accumulators
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tmem_empty + Cfg::ACC_BUFS);
    float* bias_s = reinterpret_cast<float*>(smem + (size_t)Cfg::STAGES * Cfg::STAGE_BYTES + 512);   // [N]
    float* stage_base = bias_s + Cfg::MAX_N;                // [4 warps][32][20]
    float* gb_s = stage_base + kTcEpiWarps * 32 * 20;       // [GB_GROUPS][BN] row-group bias slice of the current tile

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int nkb_all = (K + kTcBK - 1) / kTcBK;
    const int nkb = (nkb_all + gb.kbatches - 1) / gb.kbatches;          // k-blocks per split-K slice (tail slices read zeros)
    const int n_tiles_n = (N + BN - 1) / BN, n_tiles_m = (M + 127) / 128;
    const int n_tiles_mn = n_tiles_n * n_tiles_m;
    const int n_tiles = n_tiles_mn * gb.kbatches;                        // tile = slice * n_tiles_mn + (m block, n block)
    const int worker = (int)blockIdx.x, n_workers = (int)gridDim.x;
    auto tile_mb = [&](int t_mn) { return t_mn / n_tiles_n; };
    auto tile_nb = [&](int t_mn) { return t_mn % n_tiles_n; };

    auto a_hi = [&](int s) { return smem + (size_t)s * Cfg::STAGE_BYTES; };
    auto a_lo = [&](int s) { return smem + (size_t)s * Cfg::STAGE_BYTES + Cfg::A_BYTES; };
    auto w_hi = [&](int s) { return smem + (size_t)s * Cfg::STAGE_BYTES + (kBf16 ? Cfg::A_BYTES + Cfg::A_BYTES / 2 : 2 * Cfg::A_BYTES); };
    auto w_lo = [&](int s) { return smem + (size_t)s * Cfg::STAGE_BYTES + 2 * Cfg::A_BYTES + Cfg::W_BYTES; };
    // kBf16: a_lo(s) holds bf16(A) [128x16], w_hi(s) the bf16 W tile [BNx16]

    for (int i = threadIdx.x; i < N; i += kTcPersistThreads) bias_s[i] = bias != nullptr ? bias[i] : 0.f;
    if (warp == 0 && lane == 0) {
        asm volatile("prefetch.tensormap [%0];" :: "l"(reinterpret_cast<uint64_t>(&map_a)) : "memory");
        asm volatile("prefetch.tensormap [%0];" :: "l"(reinterpret_cast<uint64_t>(&map_whi)) : "memory");
        asm volatile("prefetch.tensormap [%0];" :: "l"(reinterpret_cast<uint64_t>(&map_wlo)) : "memory");
        for (int s = 0; s < Cfg::STAGES; ++s) {
            mbar_init(&full[s], 1);
            mbar_init(&ready[s], kTcTransformThreads / 32);      // one arrival per transform warp
            mbar_init(&empty[s], 1);
        }
        for (int b = 0; b < Cfg::ACC_BUFS; ++b) {
            mbar_init(&accum_full[b], 1);
            mbar_init(&tmem_empty[b], kTcEpiWarps);
        }
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
            int it = 0;                                                    // k-blocks issued so far (all tiles)
            for (int tile = worker; tile < n_tiles; tile += n_workers) {
                const int slice = tile / n_tiles_mn, t_mn = tile - slice * n_tiles_mn;
                const int mb = tile_mb(t_mn), m0 = mb * 128, n0 = tile_nb(t_mn) * BN;
                const int kb0 = slice * nkb;                               // first k-block of this split-K slice
                if (n0 == 0 && gb.kbatches == 1) {                         // pull a later M block's A rows into L2
                    const int ahead = mb + kTcPrefetchBlocks;
                    if (ahead < n_tiles_m)
                        for (int kb = 0; kb < nkb; ++kb)
                            asm volatile("cp.async.bulk.prefetch.tensor.2d.L2.global [%0, {%1, %2}];"
                                         :: "l"(reinterpret_cast<uint64_t>(&map_a)), "r"(kb * kTcBK), "r"(ahead * 128) : "memory");
                }
                for (int kb = 0; kb < nkb; ++kb, ++it) {
                    const int s = it % Cfg::STAGES;
                    mbar_wait(&empty[s], ((it / Cfg::STAGES) & 1) ^ 1);
                    if (kBf16) {                                               // raw A + the bf16 W tile
                        mbar_arrive_expect_tx(&full[s], Cfg::A_BYTES + Cfg::W_BYTES / 2);
                        tma_load_2d(a_hi(s), &map_a, &full[s], (kb0 + kb) * kTcBK, m0);
                        tma_load_2d(w_hi(s), &map_whi, &full[s], (kb0 + kb) * kTcBK, n0);
                        continue;
                    }
                    mbar_arrive_expect_tx(&full[s], Cfg::A_BYTES + 2 * Cfg::W_BYTES);      // A + both W planes
                    tma_load_2d(a_hi(s), &map_a, &full[s], (kb0 + kb) * kTcBK, m0);        // k past K arrives as zeros
                    tma_load_2d(w_hi(s), &map_whi, &full[s], (kb0 + kb) * kTcBK, n0);
                    tma_load_2d(w_lo(s), &map_wlo, &full[s], (kb0 + kb) * kTcBK, n0);
                }
            }
        }
    } else if (warp == 1) {
        // ------------------------------------------------------------------ MMA issuer (raw A = hi operand, see gemm_tcgen05.cuh)
        if (kBf16 && lane == 0) {
            // one bf16 MMA per k-block, into the accumulator buffer of the tile's parity
            constexpr uint32_t idesc16 = umma_idesc_bf16(128, BN);
            int it = 0, j = 0;
            for (int tile = worker; tile < n_tiles; tile += n_workers, ++j) {
                const int b = j & 1;
                const uint32_t d_acc = tmem_base + (uint32_t)(b * BN);
                if (j >= 2) {                                              // tile j-2's epilogue has drained buffer b
                    mbar_wait(&tmem_empty[b], (uint32_t)((j >> 1) - 1) & 1u);
                    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                }
                for (int kb = 0; kb < nkb; ++kb, ++it) {
                    const int s = it % Cfg::STAGES;
                    mbar_wait(&full[s], (it / Cfg::STAGES) & 1);           // W tile landed
                    mbar_wait(&ready[s], (it / Cfg::STAGES) & 1);          // bf16(A) written
                    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                    umma_bf16(d_acc, umma_desc_sw32(smem_u32(a_lo(s))), umma_desc_sw32(smem_u32(w_hi(s))), idesc16,
                              kb > 0 ? 1u : 0u);
                    umma_commit(&empty[s]);
                }
                umma_commit(&accum_full[b]);
            }
        } else if (lane == 0) {
            constexpr uint32_t idesc = umma_idesc_tf32(128, BN);
            const uint32_t d_main = tmem_base, d_corr = tmem_base + (uint32_t)BN;
            int it = 0, j = 0;
            for (int tile = worker; tile < n_tiles; tile += n_workers, ++j) {
                if (j > 0) {                                               // the previous tile's accumulators are drained
                    mbar_wait(tmem_empty, (uint32_t)(j - 1) & 1u);
                    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                }
                auto issue_raw = [&](int kb, int g) {
                    const int s = g % Cfg::STAGES;
                    mbar_wait(&full[s], (g / Cfg::STAGES) & 1);
                    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                    const uint64_t d_ahi = umma_desc_sw64(smem_u32(a_hi(s)));
                    const uint64_t d_whi = umma_desc_sw64(smem_u32(w_hi(s))), d_wlo = umma_desc_sw64(smem_u32(w_lo(s)));
#pragma unroll
                    for (int k = 0; k < kTcBK / 8; ++k) {
                        const uint64_t koff = (uint64_t)((k * 8 * 4) >> 4);
                        const uint32_t first = (kb > 0 || k > 0) ? 1u : 0u;
                        umma_tf32(d_main, d_ahi + koff, d_whi + koff, idesc, first);
                        umma_tf32(d_corr, d_ahi + koff, d_wlo + koff, idesc, first);
                    }
                };
                auto issue_lo = [&](int g) {
                    const int s = g % Cfg::STAGES;
                    mbar_wait(&ready[s], (g / Cfg::STAGES) & 1);
                    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                    const uint64_t d_alo = umma_desc_sw64(smem_u32(a_lo(s))), d_whi = umma_desc_sw64(smem_u32(w_hi(s)));
#pragma unroll
                    for (int k = 0; k < kTcBK / 8; ++k) {
                        const uint64_t koff = (uint64_t)((k * 8 * 4) >> 4);
                        umma_tf32(d_corr, d_alo + koff, d_whi + koff, idesc, 1u);
                    }
                    umma_commit(&empty[s]);
                };
                issue_raw(0, it);
                for (int kb = 0; kb < nkb; ++kb) {
                    if (kb + 1 < nkb) issue_raw(kb + 1, it + kb + 1);
                    issue_lo(it + kb);
                }
                it += nkb;
                umma_commit(accum_full);
            }
        }
    } else if (warp < 6) {
        // ------------------------------------------------------------------ operand transform: A_lo = rna_tf32(A - trunc_tf32(A))
        const int t = threadIdx.x - 64;                                    // 0..127
        int it = 0;
        for (int tile = worker; tile < n_tiles; tile += n_workers) {
            for (int kb = 0; kb < nkb; ++kb, ++it) {
                const int s = it % Cfg::STAGES;
                mbar_wait(&full[s], (it / Cfg::STAGES) & 1);
                const float4* hi = reinterpret_cast<const float4*>(a_hi(s));
                float4* lo = reinterpret_cast<float4*>(a_lo(s));
#pragma unroll
                for (int i = 0; i < Cfg::A_BYTES / 16 / kTcTransformThreads; ++i) {
                    const int idx = t + i * kTcTransformThreads;
                    const float4 v = hi[idx];
                    if (kBf16) {
                        // source: fp32 tile, SWIZZLE_64B (16-byte chunk c of row r sits at chunk c ^ ((r >> 1) & 3));
                        // destinations: bf16 tiles, SWIZZLE_32B (rows of 32 bytes, chunk cd at cd ^ ((r >> 2) & 1))
                        const int r = idx >> 2, c = (idx & 3) ^ ((r >> 1) & 3);          // logical columns 4c .. 4c+3
                        const uint32_t off = (uint32_t)(r * 32 + (((c >> 1) ^ ((r >> 2) & 1)) << 4) + ((c & 1) << 3));
                        __nv_bfloat162 p0 = __floats2bfloat162_rn(v.x, v.y), p1 = __floats2bfloat162_rn(v.z, v.w);
                        uint2 full_v;
                        full_v.x = *reinterpret_cast<uint32_t*>(&p0); full_v.y = *reinterpret_cast<uint32_t*>(&p1);
                        *reinterpret_cast<uint2*>(a_lo(s) + off) = full_v;                // bf16(A)
                    } else {
                        float4 vl;
                        vl.x = to_tf32_rna(v.x - tf32_trunc(v.x)); vl.y = to_tf32_rna(v.y - tf32_trunc(v.y));
                        vl.z = to_tf32_rna(v.z - tf32_trunc(v.z)); vl.w = to_tf32_rna(v.w - tf32_trunc(v.w));
                        lo[idx] = vl;
                    }
                }
                asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
                __syncwarp();
                if (lane == 0) mbar_arrive(&ready[s]);
            }
        }
    } else {
        // ------------------------------------------------------------------ epilogue warps 6.. (TMEM lane quarter = warp % 4)
        const int q = warp & 3;
        const int ew = warp - 6;                                           // 0..kTcEpiWarps-1
        // column range of this warp: the first warp of a lane quarter takes [0,128), the second [128,BN)
        const int c_begin = (kTcEpiWarps == 8 && ew >= 4) ? (BN > 128 ? 128 : BN) : 0;
        const int c_end = (kTcEpiWarps == 8 && ew < 4) ? (BN > 128 ? 128 : BN) : BN;
        const bool has_gb = gb.ptr != nullptr;
        float* stage = stage_base + ew * (32 * 20);
        const uint32_t tbase0 = tmem_base + ((uint32_t)(q * 32) << 16);
        int j = 0;
        for (int tile = worker; tile < n_tiles; tile += n_workers, ++j) {
            const int slice = tile / n_tiles_mn, t_mn = tile - slice * n_tiles_mn;
            const int mb = tile_mb(t_mn), m0 = mb * 128, n0 = tile_nb(t_mn) * BN;
            float* __restrict__ Cs = C + (size_t)slice * (size_t)gb.c_batch_stride;       // this slice's output slab
            const int m = m0 + q * 32 + lane;
            const int32_t* orow = gb.out_rows;                             // ascending row scatter, or null
            const int mo = orow != nullptr ? orow[min(m, M - 1)] : m;      // row of C (and of the row-group bias)
            // Row-group bias of this tile: its few distinct rows (128 / group_rows + 2 groups) are staged in smem NOW,
            // while the MMA main loop of this tile is still running, so the epilogue proper never waits on L2.
            const int g0 = has_gb ? (orow != nullptr ? orow[m0] : m0) / gb.rows : 0;
            const int g1 = has_gb ? (orow != nullptr ? orow[min(m0 + 127, M - 1)] : min(m0 + 127, M - 1)) / gb.rows : 0;
            const bool gb_tile = has_gb && n0 < gb.col0 + gb.cols && n0 + BN > gb.col0;      // tile overlaps the bias columns
            const bool gb_smem = gb_tile && (g1 - g0 + 1) <= Cfg::GB_GROUPS;
            if (gb_smem) {
                asm volatile("bar.sync 1, %0;" :: "n"(kTcEpiWarps * 32) : "memory");   // previous tile's readers are done with gb_s
                const int te = threadIdx.x - 192;                          // 0.. over the epilogue warps
                for (int idx = te; idx < (g1 - g0 + 1) * (BN / 4); idx += kTcEpiWarps * 32) {
                    const int gi = idx / (BN / 4), cq = idx - gi * (BN / 4);
                    const int col = n0 + cq * 4;
                    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
                    if (col >= gb.col0 && col < gb.col0 + gb.cols)
                        v = *reinterpret_cast<const float4*>(gb.ptr + (size_t)(g0 + gi) * gb.ld + (col - gb.col0));
                    *reinterpret_cast<float4*>(gb_s + gi * BN + cq * 4) = v;
                }
                asm volatile("bar.sync 1, %0;" :: "n"(kTcEpiWarps * 32) : "memory");
            }
            const float* grow = (gb_tile && !gb_smem && m < M) ? gb.ptr + (size_t)(mo / gb.rows) * gb.ld - gb.col0 + n0 : nullptr;
            const float* gsrow = gb_smem ? gb_s + ((orow != nullptr ? mo : min(m, M - 1)) / gb.rows - g0) * BN : nullptr;
            const int b = Cfg::ACC_BUFS == 2 ? (j & 1) : 0;                // accumulator buffer of this tile
            const uint32_t tbase = tbase0 + (uint32_t)(b * BN);
            mbar_wait(&accum_full[b], (uint32_t)(Cfg::ACC_BUFS == 2 ? j >> 1 : j) & 1u);
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
            uint32_t rm[16], rc[16];
            float4 gq[4];
            auto issue_group = [&](int c) {
                asm volatile(
                    "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
                    : "=r"(rm[0]), "=r"(rm[1]), "=r"(rm[2]), "=r"(rm[3]), "=r"(rm[4]), "=r"(rm[5]), "=r"(rm[6]), "=r"(rm[7]),
                      "=r"(rm[8]), "=r"(rm[9]), "=r"(rm[10]), "=r"(rm[11]), "=r"(rm[12]), "=r"(rm[13]), "=r"(rm[14]), "=r"(rm[15])
                    : "r"(tbase + (uint32_t)c));
                if (!kBf16)                                                // correction accumulator
                    asm volatile(
                        "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
                        : "=r"(rc[0]), "=r"(rc[1]), "=r"(rc[2]), "=r"(rc[3]), "=r"(rc[4]), "=r"(rc[5]), "=r"(rc[6]), "=r"(rc[7]),
                          "=r"(rc[8]), "=r"(rc[9]), "=r"(rc[10]), "=r"(rc[11]), "=r"(rc[12]), "=r"(rc[13]), "=r"(rc[14]), "=r"(rc[15])
                        : "r"(tbase + (uint32_t)(BN + c)));
#pragma unroll
                for (int v4 = 0; v4 < 4; ++v4) {
                    const int col = n0 + c + v4 * 4;
                    gq[v4] = (grow != nullptr && col >= gb.col0 && col < gb.col0 + gb.cols)
                                 ? *reinterpret_cast<const float4*>(grow + c + v4 * 4) : make_float4(0.f, 0.f, 0.f, 0.f);
                }
            };
            if (c_begin < c_end) {
                issue_group(c_begin);
            } else if (lane == 0) {
                mbar_arrive(&tmem_empty[b]);                           // nothing to drain for this warp (BN <= 128)
            }
#pragma unroll 1
            for (int c = c_begin; c < c_end; c += 16) {
                asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
                float o[16];
#pragma unroll
                for (int i = 0; i < 16; ++i)
                    o[i] = (kBf16 ? __uint_as_float(rm[i]) : __uint_as_float(rm[i]) + __uint_as_float(rc[i])) +
                           ((n0 + c + i < N && slice == 0) ? bias_s[n0 + c + i] : 0.f);
#pragma unroll
                for (int v4 = 0; v4 < 4; ++v4) {
                    float4 gv = gq[v4];
                    if (gsrow != nullptr) gv = *reinterpret_cast<const float4*>(gsrow + c + v4 * 4);
                    o[v4 * 4 + 0] += gv.x; o[v4 * 4 + 1] += gv.y;
                    o[v4 * 4 + 2] += gv.z; o[v4 * 4 + 3] += gv.w;
                }
                if (c + 16 < c_end) {
                    issue_group(c + 16);
                } else {
                    // every accumulator column of this tile is in registers: hand TMEM back to the MMA warp
                    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
                    __syncwarp();
                    if (lane == 0) mbar_arrive(&tmem_empty[b]);
                }
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
                    const int mc = __shfl_sync(0xffffffffu, mo, row);         // C row of tile row `row` (== mr without scatter)
                    if (mr < M && n0 + c + cq * 4 < N)
                        *reinterpret_cast<float4*>(Cs + (size_t)mc * ldc + n0 + c + cq * 4) =
                            *reinterpret_cast<const float4*>(stage + row * 20 + cq * 4);
                }
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

// One CTA per SM (or per tile, when there are fewer tiles than SMs); each CTA loops over its tiles.
template <int BN, bool kBf16>
int launch_persistent_inst(const CUtensorMap& ma, const CUtensorMap& mh, const CUtensorMap& ml, const float* bias, float* C,
                           int ldc, int M, int N, int K, GroupBias gb, int sm_count, cudaStream_t st) {
    using Cfg = TcPersistCfg<BN, kBf16>;
    auto kernel = gemm_tf32x3_persistent_kernel<BN, kBf16>;
    if (int rc_ = ensure_dynamic_smem(kernel, (size_t)Cfg::SMEM)) return rc_;
    const int units = ((N + BN - 1) / BN) * ((M + 127) / 128) * gb.kbatches;
    const int grid = units < sm_count ? units : sm_count;
    kernel<<<grid, kTcPersistThreads, Cfg::SMEM, st>>>(ma, mh, ml, bias, C, ldc, M, N, K, gb);
    return check_launch(kBf16 ? "digat_linear_bf16" : "digat_linear_tf32x3(persistent)");
}

template <int BN>
int launch_tf32x3_persistent(const float* A, int lda, const float* W_hi, const float* W_lo, int ldw, const float* bias,
                             float* C, int ldc, int M, int N, int K, GroupBias gb, cudaStream_t st) {
    using Cfg = TcPersistCfg<BN>;
    const DeviceInfo* di = device_info();
    if (!di) return fail(DIGAT_E_CUDA, "digat_linear_tf32x3: no CUDA device");
    DIGAT_REQUIRE(N <= Cfg::MAX_N, "digat_linear_tf32x3(persistent): N=%d exceeds %d", N, Cfg::MAX_N);
    CUtensorMap ma, mh, ml;
    int rc;
    if ((rc = make_tensor_map_2d(&ma, A, M, K, lda, 128, kTcBK, CU_TENSOR_MAP_SWIZZLE_64B)) != DIGAT_OK) return rc;
    if ((rc = make_tensor_map_2d(&mh, W_hi, N, K, ldw, BN, kTcBK, CU_TENSOR_MAP_SWIZZLE_64B)) != DIGAT_OK) return rc;
    if ((rc = make_tensor_map_2d(&ml, W_lo, N, K, ldw, BN, kTcBK, CU_TENSOR_MAP_SWIZZLE_64B)) != DIGAT_OK) return rc;
    return launch_persistent_inst<BN, false>(ma, mh, ml, bias, C, ldc, M, N, K, gb, di->sm_count, st);
}

}  // namespace digat
