// BF16 projection GEMM for the opt-in inference mode (DIGAT.projection_precision = 'bf16', DESIGN.md section 4.8):
//
//   C[M,N] = bf16_rn(A) * W_b^T (+ bias) (+ row-group bias),   W_b = bf16_rn(W) [N,K], fp32 accumulation in TMEM
//
// It runs the persistent kernel of gemm_tcgen05_persistent.cuh with kBf16 = true, for every M: the raw fp32 A tile lands
// by TMA exactly as for 3xTF32 (16-wide k-blocks, SWIZZLE_64B), the transform warps round it to a bf16 SWIZZLE_32B
// tile, W arrives as one bf16 plane, and each k-block is ONE tcgen05.mma.kind::f16 (K = 16) into one accumulator.  With
// one accumulator per tile two of them fit in TMEM (2 x 240 or 2 x 208 columns), so the epilogue of tile t overlaps the
// main loop of tile t+1.  A k-block brings in 8 KB of A and BN x 32 bytes of W (7.5 KB at BN = 240) against 38 KB for
// 3xTF32.  Every output row depends on its A row and W only (fixed k order, no dependence on M or on the tile), so
// pruned / row-scattered calls and their dense counterparts are bit-identical.
#pragma once
#include "gemm_tcgen05_persistent.cuh"

namespace digat {

template <int BN>
int launch_bf16_persistent(const float* A, int lda, const void* W_b, int ldw, const float* bias, float* C, int ldc,
                           int M, int N, int K, GroupBias gb, cudaStream_t st) {
    const DeviceInfo* di = device_info();
    if (!di) return fail(DIGAT_E_CUDA, "digat_linear_bf16: no CUDA device");
    CUtensorMap ma, mw;
    int rc;
    if ((rc = make_tensor_map_2d(&ma, A, M, K, lda, 128, kTcBK, CU_TENSOR_MAP_SWIZZLE_64B)) != DIGAT_OK) return rc;
    if ((rc = make_tensor_map_2d_bf16(&mw, W_b, N, K, ldw, BN, kTcBK, CU_TENSOR_MAP_SWIZZLE_32B)) != DIGAT_OK) return rc;
    return launch_persistent_inst<BN, true>(ma, mw, mw, bias, C, ldc, M, N, K, gb, di->sm_count, st);
}

inline int launch_linear_bf16(const float* A, int lda, const void* W_b, int ldw, const float* bias, float* C, int ldc,
                              int M, int N, int K, GroupBias gb, cudaStream_t st) {
    if (M == 0) return DIGAT_OK;
    DIGAT_REQUIRE(A && W_b && C, "digat_linear_bf16: null pointer");
    DIGAT_REQUIRE(M > 0 && N > 0 && K > 0 && (K & 7) == 0 && (lda & 3) == 0 && (ldw & 7) == 0 && (ldc & 3) == 0 &&
                  lda >= K && ldw >= K && ldc >= N && N % 16 == 0 && N <= TcPersistCfg<240>::MAX_N,
                  "digat_linear_bf16: needs K, ldw multiples of 8, lda, ldc multiples of 4, N a multiple of 16 and <= 1280 "
                  "(M=%d N=%d K=%d lda=%d ldw=%d ldc=%d)", M, N, K, lda, ldw, ldc);
    DIGAT_REQUIRE(aligned16(A) && aligned16(W_b) && aligned16(C) && (!bias || aligned16(bias)),
                  "digat_linear_bf16: pointers must be 16-byte aligned");
    if (int rc_ = check_group_bias("digat_linear_bf16", gb, N)) return rc_;
    if (N % 240 == 0) return launch_bf16_persistent<240>(A, lda, W_b, ldw, bias, C, ldc, M, N, K, gb, st);
    return launch_bf16_persistent<208>(A, lda, W_b, ldw, bias, C, ldc, M, N, K, gb, st);
}

}  // namespace digat
