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
// 6-13 = epilogue (TMEM lane quarter = warp % 4, two warps per quarter split the columns).  Arithmetic is identical to gemm_tf32x3_kernel<BN,1,true>.
// kCl = 2: two CTAs of a cluster work on the SAME N tile of two adjacent M blocks and share the W tile: each CTA loads
// half of its rows and multicasts them into both CTAs' shared memory (cp.async.bulk.tensor ... .multicast::cluster), so
// every SM pulls A + W/2 instead of A + W through L2 per k-block (38 KB -> 23 KB at BN = 240).  The main loop of the
// single-CTA kernel sits at the L2 -> SM bandwidth of the chip (148 SMs x 38 KB per ~800 cycles = 7.0 KB/clk against the
// ~6.3 KB/clk the L2 slices deliver), which is why fewer MMAs per k-block (the BF16-correction scheme) bought almost
// nothing before.  Everything else (MMA, operand transform, epilogue, TMEM) stays per CTA; only the recycling of a stage is
// coupled: its "empty" barrier counts the commits of BOTH CTAs (tcgen05.commit ... .multicast::cluster), because the
// peer's TMA writes into this CTA's stage too.
#pragma once
#include "gemm_tcgen05.cuh"
#include "gemm_tcgen05_pair.cuh"     // cluster_ctarank, cluster_sync_all, mbar_wait_cluster

namespace digat {

__device__ __forceinline__ void tma_load_2d_multicast(void* dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1,
                                                      uint16_t cta_mask) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes.multicast::cluster [%0], [%1, {%3, %4}], [%2], %5;"
        :: "r"(smem_u32(dst)), "l"(reinterpret_cast<uint64_t>(map)), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "h"(cta_mask) : "memory");
}
__device__ __forceinline__ void umma_commit_multicast(uint64_t* bar, uint16_t cta_mask) {   // arrives on `bar` in every CTA of the mask
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
                 :: "r"(smem_u32(bar)), "h"(cta_mask) : "memory");
}

__device__ __forceinline__ void umma_bf16_2cta(uint32_t tmem_d, uint64_t da, uint64_t db, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}"
        :: "r"(tmem_d), "l"(da), "l"(db), "r"(idesc), "r"(accumulate) : "memory");
}

constexpr int kTcEpiWarps = 8;                  // two epilogue warps per TMEM lane quarter, each takes half of the columns
constexpr int kTcPersistThreads = (2 + 4 + kTcEpiWarps) * 32;

// kCl: 1 = independent CTAs; 2 = W multicast across a CTA pair (experiment); 3 = 2-CTA MMA (cta_group::2, M = 256): each
// CTA of the pair loads and holds only HALF of the W tile, the leader CTA issues the MMAs for both.
// kOne: the plain BF16 GEMM (gemm_bf16.cuh): a stage holds the raw fp32 A tile, bf16(A) and ONE bf16 plane of W.
template <int BN, int kCl = 1, bool kOne = false>
struct TcPersistCfg {
    static constexpr int A_BYTES = 128 * kTcBK * 4;
    static constexpr int W_ROWS = kCl == 3 ? BN / 2 : BN;                // W rows resident in this CTA's shared memory
    static constexpr int W_BYTES = W_ROWS * kTcBK * 4;
    static constexpr int STAGE_BYTES = kOne ? A_BYTES + A_BYTES / 2 + W_BYTES / 2 : 2 * A_BYTES + 2 * W_BYTES;
    static constexpr int ACC_BUFS = kOne ? 2 : 1;                        // TMEM accumulator buffers (tiles in flight)
    static constexpr int MAX_N = 1280;                                   // bias vector kept in smem for the whole N
    static constexpr int GB_GROUPS = 16;                                 // row groups of one 128-row tile staged in smem
    static constexpr int EXTRA = 512 /*barriers*/ + MAX_N * 4 + kTcEpiWarps * 32 * 20 * 4 /*epilogue staging*/ + GB_GROUPS * BN * 4;
    static constexpr int MAX_STAGES = kOne ? 8 : 6;
    static constexpr int STAGES = (226 * 1024 - EXTRA) / STAGE_BYTES > MAX_STAGES ? MAX_STAGES : (226 * 1024 - EXTRA) / STAGE_BYTES;
    static constexpr int TMEM_COLS = 2 * BN <= 256 ? 256 : 512;
    static constexpr size_t SMEM = (size_t)STAGES * STAGE_BYTES + EXTRA;
    static_assert(STAGES >= 3, "not enough shared memory for the pipeline");
    static_assert(A_BYTES % 512 == 0 && W_BYTES % 512 == 0 && STAGE_BYTES % 512 == 0,
                  "operand tiles must start on a swizzle-atom boundary");
    static_assert(!kOne || (kCl == 1 && 2 * BN <= 512), "the BF16 GEMM keeps two accumulators of one CTA in TMEM");
};

// kBf16: the TF32+BF16 scheme.  The two correction products are ~2^-11 of the result, so they only need ~9 good bits:
//   C = A_hi*W_hi [kind::tf32, raw A]  +  bf16(A)*bf16(W_lo)  +  bf16(A_lo)*bf16(W_hi)   [kind::f16, K = 16 per MMA]
// (relative error of the corrections 2^-9 * 2^-10..2^-12 = 2^-19..2^-21 of the result, below the accumulator's own
// truncation error).  bf16 MMAs run at twice the TF32 rate: per 16-wide k-block the tensor pipe does 2 TF32 MMAs + 2 BF16
// MMAs = 4 TF32-MMA times instead of 6.  The stage keeps its size: A_lo (tf32) becomes two bf16 tiles of half the size,
// W_lo (tf32) becomes the two bf16 planes of W (map_w2 = bf16(W_hi), map_w3 = bf16(W_lo); SWIZZLE_32B tiles).
//
// kOne: C = bf16_rn(A) * W_b^T, one kind::f16 MMA (K = 16) per k-block into ONE accumulator (map_whi = W_b, SWIZZLE_32B;
// the other maps are unused).  The transform warps write bf16_rn(A) (the A_hi-free half of the kBf16 transform).  Two
// accumulator buffers alternate between tiles: the MMA warp fills buffer (j+1)&1 while the epilogue drains buffer j&1.
// The epilogue is the same code as the fp32 schemes' (bias, row-group bias, row scatter, staged row-segment stores).
template <int BN, bool kBf16, int kCl, bool kOne = false>
__global__ void __launch_bounds__(kTcPersistThreads, 1)
gemm_tf32x3_persistent_kernel(const __grid_constant__ CUtensorMap map_a, const __grid_constant__ CUtensorMap map_whi,
                              const __grid_constant__ CUtensorMap map_wlo, const __grid_constant__ CUtensorMap map_w3,
                              const float* __restrict__ bias,
                              float* __restrict__ C, int ldc, int M, int N, int K, GroupBias gb) {
    using Cfg = TcPersistCfg<BN, kCl, kOne>;
    extern __shared__ __align__(1024) uint8_t smem_raw[];
    uint8_t* smem = smem_raw;
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem + (size_t)Cfg::STAGES * Cfg::STAGE_BYTES);
    uint64_t* full = bars;                                  // [STAGES] TMA bytes landed
    uint64_t* ready = bars + Cfg::STAGES;                   // [STAGES] A_lo written by the transform warps
    uint64_t* empty = bars + 2 * Cfg::STAGES;               // [STAGES] MMAs reading the stage have retired
    uint64_t* accum_full = bars + 3 * Cfg::STAGES;          // [ACC_BUFS] accumulators of the current tile complete
    uint64_t* tmem_empty = accum_full + Cfg::ACC_BUFS;      // [ACC_BUFS] epilogue has drained the accumulators
    uint64_t* peer_full = tmem_empty + Cfg::ACC_BUFS;       // [STAGES] 2-CTA MMA, leader only: the PEER's TMA bytes of the stage landed
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(peer_full + Cfg::STAGES);
    float* bias_s = reinterpret_cast<float*>(smem + (size_t)Cfg::STAGES * Cfg::STAGE_BYTES + 512);   // [N]
    float* stage_base = bias_s + Cfg::MAX_N;                // [4 warps][32][20]
    float* gb_s = stage_base + kTcEpiWarps * 32 * 20;       // [GB_GROUPS][BN] row-group bias slice of the current tile

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int nkb_all = (K + kTcBK - 1) / kTcBK;
    const int nkb = (nkb_all + gb.kbatches - 1) / gb.kbatches;          // k-blocks per split-K slice (tail slices read zeros)
    const int n_tiles_n = (N + BN - 1) / BN, n_tiles_m = (M + 127) / 128;
    // a "worker" is a CTA (kCl = 1) or a cluster of two CTAs that takes a PAIR of adjacent M blocks of one N tile
    const int cl_rank = kCl >= 2 ? (int)cluster_ctarank() : 0;
    const int worker = kCl >= 2 ? (int)(blockIdx.x >> 1) : (int)blockIdx.x;
    const int n_workers = kCl >= 2 ? (int)(gridDim.x >> 1) : (int)gridDim.x;
    const int n_units_m = kCl >= 2 ? (n_tiles_m + 1) / 2 : n_tiles_m;    // M blocks, or pairs of them
    const int n_tiles_mn = n_tiles_n * n_units_m;
    const int n_tiles = n_tiles_mn * gb.kbatches;                        // tile = slice * n_tiles_mn + (m unit, n block)
    // (a cluster whose second M block lies past M computes zeros there and stores nothing)
    auto tile_mb = [&](int t_mn) { const int u = t_mn / n_tiles_n; return kCl >= 2 ? 2 * u + cl_rank : u; };
    auto tile_nb = [&](int t_mn) { return t_mn % n_tiles_n; };

    auto a_hi = [&](int s) { return smem + (size_t)s * Cfg::STAGE_BYTES; };
    auto a_lo = [&](int s) { return smem + (size_t)s * Cfg::STAGE_BYTES + Cfg::A_BYTES; };
    auto w_hi = [&](int s) { return smem + (size_t)s * Cfg::STAGE_BYTES + (kOne ? Cfg::A_BYTES + Cfg::A_BYTES / 2 : 2 * Cfg::A_BYTES); };
    auto w_lo = [&](int s) { return smem + (size_t)s * Cfg::STAGE_BYTES + 2 * Cfg::A_BYTES + Cfg::W_BYTES; };
    // kBf16: a_lo(s) holds bf16(A) [128x16] then bf16(A_lo); w_lo(s) holds bf16(W_hi) [BNx16] then bf16(W_lo)
    // kOne: a_lo(s) holds bf16(A) [128x16], w_hi(s) the bf16 W tile [BNx16]
    auto a_b2 = [&](int s) { return a_lo(s) + Cfg::A_BYTES / 2; };
    auto w_b3 = [&](int s) { return w_lo(s) + Cfg::W_BYTES / 2; };

    for (int i = threadIdx.x; i < N; i += kTcPersistThreads) bias_s[i] = bias != nullptr ? bias[i] : 0.f;
    if (warp == 0 && lane == 0) {
        asm volatile("prefetch.tensormap [%0];" :: "l"(reinterpret_cast<uint64_t>(&map_a)) : "memory");
        asm volatile("prefetch.tensormap [%0];" :: "l"(reinterpret_cast<uint64_t>(&map_whi)) : "memory");
        asm volatile("prefetch.tensormap [%0];" :: "l"(reinterpret_cast<uint64_t>(&map_wlo)) : "memory");
        for (int s = 0; s < Cfg::STAGES; ++s) {
            mbar_init(&full[s], 1);
            // 2-CTA MMA: the leader's "ready" also counts one arrive forwarded from the peer (its 4 transform warps are done)
            mbar_init(&ready[s], kTcTransformThreads / 32 + ((kCl == 3 && cl_rank == 0) ? 1 : 0));
            mbar_init(&empty[s], kCl == 2 ? 2 : 1);             // kCl = 2: the peer's TMA writes this stage too
            mbar_init(&peer_full[s], 1);
        }
        for (int b = 0; b < Cfg::ACC_BUFS; ++b) {
            mbar_init(&accum_full[b], 1);
            mbar_init(&tmem_empty[b], kCl == 3 ? 2 * kTcEpiWarps : kTcEpiWarps);   // 2-CTA MMA: the leader waits for both epilogues
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 1) {
        if (kCl == 3) {            // both CTAs of the pair issue the 2-CTA allocation from the same logical warp
            asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;"
                         :: "r"(smem_u32(tmem_slot)), "r"((uint32_t)Cfg::TMEM_COLS) : "memory");
            asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
        } else {
            asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;"
                         :: "r"(smem_u32(tmem_slot)), "r"((uint32_t)Cfg::TMEM_COLS) : "memory");
            asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
        }
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    if (kCl >= 2) cluster_sync_all();            // both CTAs' barriers exist before any multicast load / remote commit
    else __syncthreads();
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
                    if (kCl >= 2) mbar_wait_cluster(&empty[s], ((it / Cfg::STAGES) & 1) ^ 1);   // (arrivals come from the peer too)
                    else mbar_wait(&empty[s], ((it / Cfg::STAGES) & 1) ^ 1);
                    if (kOne) {                                                // raw A + the bf16 W tile
                        mbar_arrive_expect_tx(&full[s], Cfg::A_BYTES + Cfg::W_BYTES / 2);
                        tma_load_2d(a_hi(s), &map_a, &full[s], (kb0 + kb) * kTcBK, m0);
                        tma_load_2d(w_hi(s), &map_whi, &full[s], (kb0 + kb) * kTcBK, n0);
                        continue;
                    }
                    mbar_arrive_expect_tx(&full[s], Cfg::A_BYTES + 2 * Cfg::W_BYTES);      // own A + the whole W tile (both halves)
                    tma_load_2d(a_hi(s), &map_a, &full[s], (kb0 + kb) * kTcBK, m0);        // k past K arrives as zeros
                    if (kCl == 2) {
                        // this CTA's half of the W rows, delivered to the same offsets of both CTAs (the maps' boxes are BN/2 rows)
                        constexpr int HR = BN / 2;
                        const int nr = n0 + cl_rank * HR;
                        tma_load_2d_multicast(w_hi(s) + cl_rank * HR * kTcBK * 4, &map_whi, &full[s], (kb0 + kb) * kTcBK, nr, 3);
                        tma_load_2d_multicast(w_lo(s) + cl_rank * HR * kTcBK * (kBf16 ? 2 : 4), &map_wlo, &full[s], (kb0 + kb) * kTcBK, nr, 3);
                        if (kBf16) tma_load_2d_multicast(w_b3(s) + cl_rank * HR * kTcBK * 2, &map_w3, &full[s], (kb0 + kb) * kTcBK, nr, 3);
                    } else {
                        const int nr = kCl == 3 ? n0 + cl_rank * (BN / 2) : n0;                // 2-CTA MMA: this CTA's half of the W rows
                        tma_load_2d(w_hi(s), &map_whi, &full[s], (kb0 + kb) * kTcBK, nr);
                        tma_load_2d(w_lo(s), &map_wlo, &full[s], (kb0 + kb) * kTcBK, nr);      // kBf16: bf16(W_hi), half the bytes
                        if (kBf16) tma_load_2d(w_b3(s), &map_w3, &full[s], (kb0 + kb) * kTcBK, nr);   // bf16(W_lo)
                    }
                }
            }
        }
    } else if (warp == 1) {
        // ------------------------------------------------------------------ MMA issuer (raw A = hi operand, see gemm_tcgen05.cuh)
        if (kCl == 3) {
            if (lane == 0 && cl_rank == 0) {
                // 2-CTA MMA, leader: one M = 256 instruction covers both CTAs' 128 rows; A and the two halves of W are read
                // from both CTAs' shared memory, each CTA's accumulator rows land in its own TMEM.  As in the single-CTA kernel
                // the products that need no transformed operand (raw A x W_hi, raw A x W_lo) are issued as soon as BOTH CTAs'
                // TMA bytes of the stage have landed (own `full`, the peer's forwarded as `peer_full`); only the A_lo products
                // wait for both CTAs' transform warps (`ready`: 4 local arrives + 1 forwarded), one stage later.
                constexpr uint32_t idesc2 = umma_idesc_tf32(256, BN);
                constexpr uint32_t idesc2h = umma_idesc_bf16(256, BN);
                const uint32_t d_main = tmem_base, d_corr = tmem_base + (uint32_t)BN;
                int it = 0, j = 0;
                for (int tile = worker; tile < n_tiles; tile += n_workers, ++j) {
                    if (j > 0) {
                        mbar_wait_cluster(tmem_empty, (uint32_t)(j - 1) & 1u);
                        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                    }
                    auto issue_raw = [&](int kb, int g) {
                        const int s = g % Cfg::STAGES;
                        mbar_wait(&full[s], (g / Cfg::STAGES) & 1);
                        mbar_wait_cluster(&peer_full[s], (g / Cfg::STAGES) & 1);
                        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                        const uint64_t d_ahi = umma_desc_sw64(smem_u32(a_hi(s)));
                        const uint64_t d_whi = umma_desc_sw64(smem_u32(w_hi(s))), d_wlo = umma_desc_sw64(smem_u32(w_lo(s)));
#pragma unroll
                        for (int k = 0; k < kTcBK / 8; ++k) {
                            const uint64_t koff = (uint64_t)((k * 8 * 4) >> 4);
                            const uint32_t first = (kb > 0 || k > 0) ? 1u : 0u;
                            umma_tf32_2cta(d_main, d_ahi + koff, d_whi + koff, idesc2, first);
                            if (!kBf16) umma_tf32_2cta(d_corr, d_ahi + koff, d_wlo + koff, idesc2, first);
                        }
                    };
                    auto issue_lo = [&](int g) {
                        const int s = g % Cfg::STAGES;
                        mbar_wait_cluster(&ready[s], (g / Cfg::STAGES) & 1);
                        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                        if (kBf16) {
                            const uint32_t first = (g - it) > 0 ? 1u : 0u;
                            umma_bf16_2cta(d_corr, umma_desc_sw32(smem_u32(a_lo(s))), umma_desc_sw32(smem_u32(w_b3(s))), idesc2h, first);
                            umma_bf16_2cta(d_corr, umma_desc_sw32(smem_u32(a_b2(s))), umma_desc_sw32(smem_u32(w_lo(s))), idesc2h, 1u);
                        } else {
                            const uint64_t d_alo = umma_desc_sw64(smem_u32(a_lo(s))), d_whi = umma_desc_sw64(smem_u32(w_hi(s)));
#pragma unroll
                            for (int k = 0; k < kTcBK / 8; ++k) {
                                const uint64_t koff = (uint64_t)((k * 8 * 4) >> 4);
                                umma_tf32_2cta(d_corr, d_alo + koff, d_whi + koff, idesc2, 1u);
                            }
                        }
                        umma_commit_2cta(&empty[s]);               // frees stage s in both CTAs
                    };
                    issue_raw(0, it);
                    for (int kb = 0; kb < nkb; ++kb) {
                        if (kb + 1 < nkb) issue_raw(kb + 1, it + kb + 1);
                        issue_lo(it + kb);
                    }
                    it += nkb;
                    umma_commit_2cta(accum_full);                  // both CTAs' epilogues
                }
            } else if (cl_rank == 1 && lane < 2) {
                // peer: two otherwise idle threads forward its per-stage events to the leader as ONE remote arrive each --
                // lane 0 "my TMA bytes have landed" (full -> peer_full), lane 1 "my transform warps are done" (ready -> ready)
                int it = 0;
                for (int tile = worker; tile < n_tiles; tile += n_workers)
                    for (int kb = 0; kb < nkb; ++kb, ++it) {
                        const int s = it % Cfg::STAGES;
                        if (lane == 0) {
                            mbar_wait(&full[s], (it / Cfg::STAGES) & 1);
                            mbar_arrive_cluster(&peer_full[s], 0);
                        } else {
                            mbar_wait(&ready[s], (it / Cfg::STAGES) & 1);
                            mbar_arrive_cluster(&ready[s], 0);
                        }
                    }
            }
        } else if (kOne && lane == 0) {
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
#ifdef DIGAT_TC_TIMING
                const long long t0 = clock64();
#endif
                if (j > 0) {                                               // the previous tile's accumulators are drained
                    mbar_wait(tmem_empty, (uint32_t)(j - 1) & 1u);
                    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                }
#ifdef DIGAT_TC_TIMING
                const long long t1 = clock64();
#endif
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
                        if (!kBf16) umma_tf32(d_corr, d_ahi + koff, d_wlo + koff, idesc, first);
                    }
                };
                auto issue_lo = [&](int g) {
                    const int s = g % Cfg::STAGES;
                    mbar_wait(&ready[s], (g / Cfg::STAGES) & 1);
                    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                    if (kBf16) {
                        // one K=16 bf16 MMA per correction product: bf16(A) x bf16(W_lo), bf16(A_lo) x bf16(W_hi)
                        constexpr uint32_t idesc16 = umma_idesc_bf16(128, BN);
                        const uint32_t first = (g - it) > 0 ? 1u : 0u;                  // first k-block of the tile starts d_corr
                        umma_bf16(d_corr, umma_desc_sw32(smem_u32(a_lo(s))), umma_desc_sw32(smem_u32(w_b3(s))), idesc16, first);
                        umma_bf16(d_corr, umma_desc_sw32(smem_u32(a_b2(s))), umma_desc_sw32(smem_u32(w_lo(s))), idesc16, 1u);
                    } else {
                        const uint64_t d_alo = umma_desc_sw64(smem_u32(a_lo(s))), d_whi = umma_desc_sw64(smem_u32(w_hi(s)));
#pragma unroll
                        for (int k = 0; k < kTcBK / 8; ++k) {
                            const uint64_t koff = (uint64_t)((k * 8 * 4) >> 4);
                            umma_tf32(d_corr, d_alo + koff, d_whi + koff, idesc, 1u);
                        }
                    }
                    if (kCl == 2) umma_commit_multicast(&empty[s], 3);    // frees stage s in both CTAs of the cluster
                    else umma_commit(&empty[s]);
                };
                issue_raw(0, it);
                for (int kb = 0; kb < nkb; ++kb) {
                    if (kb + 1 < nkb) issue_raw(kb + 1, it + kb + 1);
                    issue_lo(it + kb);
                }
                it += nkb;
                umma_commit(accum_full);
#ifdef DIGAT_TC_TIMING
                if (blockIdx.x == 7 && j >= 3 && j <= 5)
                    printf("mma  tile j=%d: waited tmem_empty %lld, issue loop %lld (abs %lld)\n", j, t1 - t0, clock64() - t1, t0);
#endif
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
                    if (kBf16 || kOne) {
                        // source: fp32 tile, SWIZZLE_64B (16-byte chunk c of row r sits at chunk c ^ ((r >> 1) & 3));
                        // destinations: bf16 tiles, SWIZZLE_32B (rows of 32 bytes, chunk cd at cd ^ ((r >> 2) & 1))
                        const int r = idx >> 2, c = (idx & 3) ^ ((r >> 1) & 3);          // logical columns 4c .. 4c+3
                        const uint32_t off = (uint32_t)(r * 32 + (((c >> 1) ^ ((r >> 2) & 1)) << 4) + ((c & 1) << 3));
                        __nv_bfloat162 p0 = __floats2bfloat162_rn(v.x, v.y), p1 = __floats2bfloat162_rn(v.z, v.w);
                        uint2 full_v;
                        full_v.x = *reinterpret_cast<uint32_t*>(&p0); full_v.y = *reinterpret_cast<uint32_t*>(&p1);
                        *reinterpret_cast<uint2*>(a_lo(s) + off) = full_v;                // bf16(A)
                        if (kBf16) {
                            __nv_bfloat162 q0 = __floats2bfloat162_rn(v.x - tf32_trunc(v.x), v.y - tf32_trunc(v.y));
                            __nv_bfloat162 q1 = __floats2bfloat162_rn(v.z - tf32_trunc(v.z), v.w - tf32_trunc(v.w));
                            uint2 lo_v;
                            lo_v.x = *reinterpret_cast<uint32_t*>(&q0); lo_v.y = *reinterpret_cast<uint32_t*>(&q1);
                            *reinterpret_cast<uint2*>(a_b2(s) + off) = lo_v;              // bf16(A - trunc_tf32(A))
                        }
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
#ifdef DIGAT_TC_TIMING
            const long long e0 = clock64();
#endif
            const int b = Cfg::ACC_BUFS == 2 ? (j & 1) : 0;                // accumulator buffer of this tile
            const uint32_t tbase = tbase0 + (uint32_t)(b * BN);
            mbar_wait(&accum_full[b], (uint32_t)(Cfg::ACC_BUFS == 2 ? j >> 1 : j) & 1u);
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
#ifdef DIGAT_TC_TIMING
            const long long e1 = clock64();
#endif
            uint32_t rm[16], rc[16];
            float4 gq[4];
            auto issue_group = [&](int c) {
                asm volatile(
                    "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
                    : "=r"(rm[0]), "=r"(rm[1]), "=r"(rm[2]), "=r"(rm[3]), "=r"(rm[4]), "=r"(rm[5]), "=r"(rm[6]), "=r"(rm[7]),
                      "=r"(rm[8]), "=r"(rm[9]), "=r"(rm[10]), "=r"(rm[11]), "=r"(rm[12]), "=r"(rm[13]), "=r"(rm[14]), "=r"(rm[15])
                    : "r"(tbase + (uint32_t)c));
                if (!kOne)                                                 // correction accumulator
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
                if (kCl == 3 && cl_rank == 1) mbar_arrive_cluster(tmem_empty, 0);
                else mbar_arrive(&tmem_empty[b]);                      // nothing to drain for this warp (BN <= 128)
            }
#pragma unroll 1
            for (int c = c_begin; c < c_end; c += 16) {
                asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
                float o[16];
#pragma unroll
                for (int i = 0; i < 16; ++i)
                    o[i] = (kOne ? __uint_as_float(rm[i]) : __uint_as_float(rm[i]) + __uint_as_float(rc[i])) +
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
                    if (lane == 0) {
                        if (kCl == 3 && cl_rank == 1) mbar_arrive_cluster(tmem_empty, 0);   // the leader issues the next tile's MMAs
                        else mbar_arrive(&tmem_empty[b]);
                    }
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
#ifdef DIGAT_TC_TIMING
            if (blockIdx.x == 7 && j >= 3 && j <= 5 && threadIdx.x == 192)
                printf("epi  tile j=%d: waited accum_full %lld, epilogue %lld (abs %lld)\n", j, e1 - e0, clock64() - e1, e0);
#endif
        }
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    if (kCl >= 2) cluster_sync_all();            // the peer may still multicast into / commit onto this CTA's shared memory
    else __syncthreads();
    if (warp == 1) {
        if (kCl == 3)
            asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;"
                         :: "r"(tmem_base), "r"((uint32_t)Cfg::TMEM_COLS) : "memory");
        else
            asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;"
                         :: "r"(tmem_base), "r"((uint32_t)Cfg::TMEM_COLS) : "memory");
    }
}

// Measured (tools/gemm_bench.py, profiles/r2_gemm_variants.txt): multicast is correct (bit-identical) but NOT faster -- 206 vs
// 214 TFLOP/s (3xTF32), 222 vs 220 (BF16 corrections) at M = 136k.  The full W tile still has to LAND in every SM's shared
// memory: the bound is the ~48 B/clk each SM can take in from the fabric (38 KB per ~800-cycle k-block), not the L2 slices.
// Only the 2-CTA MMA (each SM holds half of W) removes those bytes.  Kept as an experiment, off by default.
static int g_tc_cluster = 0;   // 0 = independent CTAs, 1 = W multicast across CTA pairs, 2 = 2-CTA MMA (digat_debug_set_gemm_variant 6 / 7 / 8)

// Launch of one persistent instantiation; kCl = 2 goes through cudaLaunchKernelEx with a (2,1,1) cluster.
template <int BN, bool kBf16, int kCl, bool kOne = false>
int launch_tf32x3_persistent_inst(const CUtensorMap& ma, const CUtensorMap& mh, const CUtensorMap& ml, const CUtensorMap& m3,
                                  const float* bias, float* C, int ldc, int M, int N, int K, GroupBias gb, int units, int sm_count,
                                  cudaStream_t st) {
    using Cfg = TcPersistCfg<BN, kCl, kOne>;
    auto kernel = gemm_tf32x3_persistent_kernel<BN, kBf16, kCl, kOne>;
    if (int rc_ = ensure_dynamic_smem(kernel, (size_t)Cfg::SMEM)) return rc_;
    if (kCl == 1) {
        const int grid = units < sm_count ? units : sm_count;
        kernel<<<grid, kTcPersistThreads, Cfg::SMEM, st>>>(ma, mh, ml, m3, bias, C, ldc, M, N, K, gb);
        return check_launch(kOne ? "digat_linear_bf16" : "digat_linear_tf32x3(persistent)");
    }
    cudaLaunchConfig_t cfg{};
    cfg.blockDim = dim3(kTcPersistThreads);
    cfg.dynamicSmemBytes = Cfg::SMEM;
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = 2;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    static int max_clusters[16] = {0};                                   // co-resident clusters of this instantiation, per device
    int dev = 0;
    DIGAT_CUDA(cudaGetDevice(&dev));
    if (dev >= 0 && dev < 16 && max_clusters[dev] == 0) {
        cfg.gridDim = dim3(2 * (sm_count / 2));
        int n = 0;
        DIGAT_CUDA(cudaOccupancyMaxActiveClusters(&n, kernel, &cfg));
        max_clusters[dev] = n > 0 ? n : -1;
    }
    int clusters = sm_count / 2;
    if (dev >= 0 && dev < 16 && max_clusters[dev] > 0 && max_clusters[dev] < clusters) clusters = max_clusters[dev];
    if (units < clusters) clusters = units;
    cfg.gridDim = dim3(2 * clusters);
    DIGAT_CUDA(cudaLaunchKernelEx(&cfg, kernel, ma, mh, ml, m3, bias, C, ldc, M, N, K, gb));
    return check_launch("digat_linear_tf32x3(persistent, W multicast)");
}

template <int BN>
int launch_tf32x3_persistent(const float* A, int lda, const float* W_hi, const float* W_lo, int ldw, const float* bias,
                             float* C, int ldc, int M, int N, int K, GroupBias gb, cudaStream_t st,
                             const void* W_hb, const void* W_lb) {
    using Cfg = TcPersistCfg<BN>;
    const DeviceInfo* di = device_info();
    if (!di) return fail(DIGAT_E_CUDA, "digat_linear_tf32x3: no CUDA device");
    DIGAT_REQUIRE(N <= Cfg::MAX_N, "digat_linear_tf32x3(persistent): N=%d exceeds %d", N, Cfg::MAX_N);
    const int tiles_n = (N + BN - 1) / BN, tiles_m = (M + 127) / 128;
    // W multicast pays when every SM streams many tiles (the kernel is then bound by L2 -> SM traffic); short problems and
    // split-K weight gradients (few tiles per CTA) keep the independent CTAs
    const bool cluster = g_tc_cluster != 0 && gb.kbatches == 1 && tiles_m >= 2 && (BN / 2) % 8 == 0 &&
                         (long)tiles_n * tiles_m >= 4L * di->sm_count;
    const int wbox = cluster ? BN / 2 : BN;                               // rows of one W box (a cluster CTA loads half a tile)
    CUtensorMap ma, mh, ml;
    int rc;
    if ((rc = make_tensor_map_2d(&ma, A, M, K, lda, 128, kTcBK, CU_TENSOR_MAP_SWIZZLE_64B)) != DIGAT_OK) return rc;
    if ((rc = make_tensor_map_2d(&mh, W_hi, N, K, ldw, wbox, kTcBK, CU_TENSOR_MAP_SWIZZLE_64B)) != DIGAT_OK) return rc;
    const bool bf16c = W_hb != nullptr && W_lb != nullptr;
    CUtensorMap m3 = mh;
    if (bf16c) {
        if ((rc = make_tensor_map_2d_bf16(&ml, W_hb, N, K, ldw, wbox, kTcBK, CU_TENSOR_MAP_SWIZZLE_32B)) != DIGAT_OK) return rc;
        if ((rc = make_tensor_map_2d_bf16(&m3, W_lb, N, K, ldw, wbox, kTcBK, CU_TENSOR_MAP_SWIZZLE_32B)) != DIGAT_OK) return rc;
    } else {
        if ((rc = make_tensor_map_2d(&ml, W_lo, N, K, ldw, wbox, kTcBK, CU_TENSOR_MAP_SWIZZLE_64B)) != DIGAT_OK) return rc;
    }
    const int units = tiles_n * (cluster ? (tiles_m + 1) / 2 : tiles_m) * gb.kbatches;
    if (cluster && g_tc_cluster == 2) {          // 2-CTA MMA
        if (bf16c) return launch_tf32x3_persistent_inst<BN, true, 3>(ma, mh, ml, m3, bias, C, ldc, M, N, K, gb, units, di->sm_count, st);
        return launch_tf32x3_persistent_inst<BN, false, 3>(ma, mh, ml, m3, bias, C, ldc, M, N, K, gb, units, di->sm_count, st);
    }
    if (cluster) {                               // W multicast (experiment)
        if (bf16c) return launch_tf32x3_persistent_inst<BN, true, 2>(ma, mh, ml, m3, bias, C, ldc, M, N, K, gb, units, di->sm_count, st);
        return launch_tf32x3_persistent_inst<BN, false, 2>(ma, mh, ml, m3, bias, C, ldc, M, N, K, gb, units, di->sm_count, st);
    }
    if (bf16c) return launch_tf32x3_persistent_inst<BN, true, 1>(ma, mh, ml, m3, bias, C, ldc, M, N, K, gb, units, di->sm_count, st);
    return launch_tf32x3_persistent_inst<BN, false, 1>(ma, mh, ml, m3, bias, C, ldc, M, N, K, gb, units, di->sm_count, st);
}

}  // namespace digat
