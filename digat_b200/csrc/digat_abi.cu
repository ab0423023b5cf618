// libdigat_sm100.so -- the C ABI (include/digat_sm100.h) over the hand-written sm_100a kernels.
// One translation unit: nvcc -gencode arch=compute_100a,code=sm_100a -lineinfo -O3 -shared -Xcompiler -fPIC
#include "common.cuh"
#include "gemm_simt.cuh"
#include "gemm_small.cuh"
#include "gemm_tcgen05.cuh"
#include "gemm_tcgen05_persistent.cuh"
#include "gemm_bf16.cuh"
#include "pair_attention.cuh"
#include "pair_attention_sparse.cuh"
#include "context.cuh"
#include "gather.cuh"
#include "pair_attention_bwd.cuh"
#include "pair_attention_sparse_bwd.cuh"
#include "context_bwd.cuh"
#include "gemm_wgrad.cuh"
#include "builders.cuh"
#include "news_encoder.cuh"
#include "optimizer.cuh"

using namespace digat;

static inline cudaStream_t as_stream(void* s) { return reinterpret_cast<cudaStream_t>(s); }

extern "C" {

int digat_abi_version(void) { return DIGAT_ABI_VERSION; }

const char* digat_last_error(void) { return g_last_error; }

int digat_device_check(int* sm_count) {
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0)
        return fail(DIGAT_E_CUDA, "no CUDA device: %s", e == cudaSuccess ? "device count is 0" : cudaGetErrorString(e));
    const DeviceInfo* di = device_info();
    if (!di) return fail(DIGAT_E_CUDA, "cannot query the current CUDA device");
    if (di->cc_major != 10)
        return fail(DIGAT_E_UNSUPPORTED, "libdigat_sm100 is built for sm_100a only; device is compute capability %d.x",
                    di->cc_major);
    if (sm_count) *sm_count = di->sm_count;
    return DIGAT_OK;
}

int digat_linear_f32(const float* A, int lda, const float* W, int ldw, const float* bias, float* C, int ldc,
                     int M, int N, int K, int relu, const float* group_bias, int group_rows, int group_col0,
                     int group_cols, int group_ld, void* stream) {
    return launch_linear_f32(A, lda, W, ldw, bias, C, ldc, M, N, K, relu,
                             GroupBias{group_bias, group_rows, group_col0, group_cols, group_ld}, as_stream(stream));
}

int digat_gemm_f32_small(const float* L, int ldl, int l_trans, const float* R, int ldr, int r_trans, const float* bias,
                         float* out, int ldo, int I, int J, int C, void* stream) {
    return launch_gemm_f32_small(L, ldl, l_trans, R, ldr, r_trans, bias, out, ldo, I, J, C, as_stream(stream));
}

int digat_split_tf32(const float* W, float* W_hi, float* W_lo, int64_t count, void* stream) {
    DIGAT_REQUIRE(W && W_hi && W_lo, "digat_split_tf32: null pointer");
    if (count <= 0) return DIGAT_OK;
    split_tf32_kernel<<<(unsigned)((count + 255) / 256), 256, 0, as_stream(stream)>>>(W, W_hi, W_lo, count);
    return check_launch("digat_split_tf32");
}

int digat_linear_tf32x3(const float* A, int lda, const float* W_hi, const float* W_lo, int ldw, const float* bias,
                        float* C, int ldc, int M, int N, int K, const float* group_bias, int group_rows,
                        int group_col0, int group_cols, int group_ld, const int32_t* c_row_index, void* stream) {
    return launch_linear_tf32x3(A, lda, W_hi, W_lo, ldw, bias, C, ldc, M, N, K,
                                GroupBias{group_bias, group_rows, group_col0, group_cols, group_ld, c_row_index},
                                as_stream(stream));
}

int digat_linear_tf32x3_splitk(const float* A, int lda, const float* W_hi, const float* W_lo, int ldw, float* C, int ldc,
                               int M, int N, int K, int kbatches, int64_t c_batch_stride, void* stream) {
    DIGAT_REQUIRE(kbatches >= 1 && (kbatches == 1 || c_batch_stride >= (int64_t)M * ldc),
                  "digat_linear_tf32x3_splitk: bad kbatches / c_batch_stride");
    GroupBias gb{nullptr, 1, 0, 0, 0};
    gb.kbatches = kbatches;
    gb.c_batch_stride = c_batch_stride;
    return launch_linear_tf32x3(A, lda, W_hi, W_lo, ldw, nullptr, C, ldc, M, N, K, gb, as_stream(stream));
}

int digat_linear_bf16(const float* A, int lda, const void* W_b, int ldw, const float* bias, float* C, int ldc,
                      int M, int N, int K, const float* group_bias, int group_rows, int group_col0, int group_cols,
                      int group_ld, const int32_t* c_row_index, void* stream) {
    return launch_linear_bf16(A, lda, W_b, ldw, bias, C, ldc, M, N, K,
                              GroupBias{group_bias, group_rows, group_col0, group_cols, group_ld, c_row_index},
                              as_stream(stream));
}

int digat_debug_set_layer_mode(int mode) {
    g_layer_mode = mode;
    return DIGAT_OK;
}

int digat_graph_layer_fwd(const float* P, int ldp, const float* a, const uint8_t* adj, const float* X, float* Y,
                          int B, int n, int D, const uint8_t* drop_keep, float drop_scale, float* score_out,
                          float* alpha_out, uint8_t* relu_mask_out, const int32_t* px_index, int n_src,
                          const int32_t* adj_index, const float* k3, int ldk3, const uint8_t* row_active,
                          float* Yc, const int32_t* row_pos, const uint16_t* csr_rowptr, const uint16_t* csr_meta,
                          const int32_t* csr_index, void* stream) {
    return launch_graph_layer_fwd(P, ldp, a, adj, X, Y, B, n, D, drop_keep, drop_scale, score_out, alpha_out,
                                  relu_mask_out, px_index, n_src, adj_index, k3, ldk3, row_active, Yc, row_pos,
                                  csr_rowptr, csr_meta, csr_index, as_stream(stream));
}

int digat_build_graph_csr(const uint8_t* adj, const int32_t* adj_index, const uint8_t* row_active, uint16_t* rowptr,
                          uint16_t* meta, uint16_t* colptr, uint16_t* cedge, int64_t G, int n, void* stream) {
    return launch_build_graph_csr(adj, adj_index, row_active, rowptr, meta, colptr, cedge, G, n, as_stream(stream));
}

int digat_gat_layer_fwd(const float* Hm, int ldh, const float* s12, const uint8_t* adj, const float* X, float* Y,
                        int B, int n, int D, void* stream) {
    return launch_gat_layer_fwd(Hm, ldh, s12, adj, X, Y, B, n, D, as_stream(stream));
}

int digat_attention_pool_fwd(const float* F, int64_t strideF, int ldf, const float* resid_F, const float* v,
                             int ldv, const uint8_t* mask, const float* add_in, float* out, int ldo, float* first_out,
                             float* alpha_out, int B, int m, int D, void* stream) {
    return launch_attention_pool_fwd(F, strideF, ldf, resid_F, v, ldv, mask, add_in, out, ldo, first_out, alpha_out, B, m, D,
                                     as_stream(stream));
}

int digat_news_gate_fwd(const float* z, const float* lg, const float* ctx_in, float* ctx_out, int B, int D,
                        void* stream) {
    return launch_news_gate_fwd(z, lg, ctx_in, ctx_out, B, D, as_stream(stream));
}

int digat_topic_segment_fwd(const float* Xu, int64_t strideX, const float* v, int ldv, const int64_t* cidx, float* T,
                            float* alpha_out, int32_t* err_flag, const int32_t* src_index, const uint8_t* cmask,
                            float* Tc, const int32_t* seg_pos, int B, int H, int n_seg, int D, void* stream) {
    return launch_topic_segment_fwd(Xu, strideX, v, ldv, cidx, T, alpha_out, err_flag, src_index, cmask, Tc, seg_pos,
                                    B, H, n_seg, D, as_stream(stream));
}

int digat_gather_rows_i32(const float* table, int64_t n_table, const int32_t* idx, float* out, int64_t ldo,
                          int64_t rows, int D, int32_t* err_flag, void* stream) {
    if (rows <= 0) return DIGAT_OK;
    DIGAT_REQUIRE(table && idx && out, "digat_gather_rows_i32: null pointer");
    DIGAT_REQUIRE(D >= 4 && (D & 3) == 0 && (ldo & 3) == 0 && ldo >= D, "digat_gather_rows_i32: D, ldo must be multiples of 4");
    DIGAT_REQUIRE(aligned16(table) && aligned16(out), "digat_gather_rows_i32: pointers must be 16-byte aligned");
    if (rows <= 0) return DIGAT_OK;
    const DeviceInfo* di = device_info();
    if (!di) return fail(DIGAT_E_CUDA, "digat_gather_rows_i32: no CUDA device");
    gather_rows_kernel<<<gather_grid(rows, di->sm_count), kGatherThreads, 0, as_stream(stream)>>>(
        table, n_table, idx, nullptr, 1, out, ldo, rows, D / 4, err_flag);
    return check_launch("digat_gather_rows_i32");
}

int digat_gather_sag_i32(const float* table, int64_t n_table, const int32_t* node_id, int n_nodes,
                         const int32_t* news, float* out, int64_t rows, int D, int32_t* err_flag, void* stream) {
    if (rows <= 0) return DIGAT_OK;
    DIGAT_REQUIRE(table && node_id && news && out, "digat_gather_sag_i32: null pointer");
    DIGAT_REQUIRE(n_nodes >= 1 && D >= 4 && (D & 3) == 0, "digat_gather_sag_i32: bad n_nodes / D");
    DIGAT_REQUIRE(aligned16(table) && aligned16(out), "digat_gather_sag_i32: pointers must be 16-byte aligned");
    if (rows <= 0) return DIGAT_OK;
    const DeviceInfo* di = device_info();
    if (!di) return fail(DIGAT_E_CUDA, "digat_gather_sag_i32: no CUDA device");
    const int64_t total = rows * n_nodes;
    gather_rows_kernel<<<gather_grid(total, di->sm_count), kGatherThreads, 0, as_stream(stream)>>>(
        table, n_table, news, node_id, n_nodes, out, D, total, D / 4, err_flag);
    return check_launch("digat_gather_sag_i32");
}

int digat_build_user_nodes(const float* table, int64_t n_table, const int32_t* hist_idx, const float* hist,
                           const float* topic_emb, float* Xu, int B, int H, int C, int D, int32_t* err_flag,
                           void* stream) {
    if (B <= 0) return DIGAT_OK;
    DIGAT_REQUIRE(topic_emb && Xu && ((table && hist_idx) || hist), "digat_build_user_nodes: null pointer");
    DIGAT_REQUIRE(H >= 1 && C >= 0 && D >= 4 && (D & 3) == 0, "digat_build_user_nodes: bad H / C / D");
    DIGAT_REQUIRE(aligned16(Xu) && aligned16(topic_emb) && (!table || aligned16(table)) && (!hist || aligned16(hist)),
                  "digat_build_user_nodes: pointers must be 16-byte aligned");
    if (B <= 0) return DIGAT_OK;
    const DeviceInfo* di = device_info();
    if (!di) return fail(DIGAT_E_CUDA, "digat_build_user_nodes: no CUDA device");
    const int64_t rows = (int64_t)B * (H + C);
    build_user_nodes_kernel<<<gather_grid(rows, di->sm_count), kGatherThreads, 0, as_stream(stream)>>>(
        table, n_table, hist_idx, hist, topic_emb, Xu, rows, H, C, D / 4, err_flag);
    return check_launch("digat_build_user_nodes");
}

int digat_logits(const float* news_ctx, const float* user_ctx, float* logits, int B, int D, void* stream) {
    if (B <= 0) return DIGAT_OK;
    DIGAT_REQUIRE(news_ctx && user_ctx && logits, "digat_logits: null pointer");
    DIGAT_REQUIRE(D >= 4 && (D & 3) == 0 && aligned16(news_ctx) && aligned16(user_ctx), "digat_logits: bad D / alignment");
    if (B <= 0) return DIGAT_OK;
    const int warps_per_cta = kGatherThreads / 32;
    logits_kernel<<<(B + warps_per_cta - 1) / warps_per_cta, kGatherThreads, 0, as_stream(stream)>>>(
        news_ctx, user_ctx, logits, B, D / 4);
    return check_launch("digat_logits");
}

int digat_add_inplace(const float* x, float* y, int64_t count, void* stream) {
    DIGAT_REQUIRE(x && y && aligned16(x) && aligned16(y), "digat_add_inplace: null or misaligned pointer");
    if (count <= 0) return DIGAT_OK;
    const int64_t threads = (count + 3) / 4;
    add_inplace_kernel<<<(unsigned)((threads + 255) / 256), 256, 0, as_stream(stream)>>>(x, y, count);
    return check_launch("digat_add_inplace");
}

// ------------------------------------------------------------------------------------------------ backward
int digat_graph_layer_bwd(const float* P, int ldp, const float* a, const uint8_t* adj, const float* score,
                          const float* alpha, const uint8_t* drop_keep, float drop_scale, const float* G, float* dP,
                          int lddp, float* da_partial, int B, int n, int D, void* stream) {
    return launch_graph_layer_bwd(P, ldp, a, adj, score, alpha, drop_keep, drop_scale, G, dP, lddp, da_partial, B, n, D,
                                  as_stream(stream));
}

int digat_graph_layer_bwd_csr(const float* P, int ldp, const float* a, const uint16_t* csr_rowptr, const uint16_t* csr_meta,
                              const uint16_t* csc_colptr, const uint16_t* csc_edge, const float* edge_score,
                              const float* edge_alpha, const uint8_t* drop_keep, float drop_scale, const float* G,
                              const uint8_t* relu_mask, float* dP, int lddp, float* da_partial, float* dh_sum, float* du_sum,
                              int B, int n, int D, void* stream) {
    return launch_graph_layer_bwd_csr(P, ldp, a, csr_rowptr, csr_meta, csc_colptr, csc_edge, edge_score, edge_alpha, drop_keep,
                                      drop_scale, G, relu_mask, dP, lddp, da_partial, dh_sum, du_sum, B, n, D, as_stream(stream));
}

int digat_grad_sumsq(const float* g, int64_t n, float* partials, float* step_counter, void* stream) {
    return launch_grad_sumsq(g, n, partials, step_counter, as_stream(stream));
}

int digat_adam_clip_step(float* p, float* g, float* m, float* v, int64_t n, const float* partials, const float* step_counter,
                         float* grad_norm_out, float max_norm, float lr, float beta1, float beta2, float eps,
                         float weight_decay, void* stream) {
    return launch_adam_clip_step(p, g, m, v, n, partials, step_counter, grad_norm_out, max_norm, lr, beta1, beta2, eps,
                                 weight_decay, as_stream(stream));
}

int digat_graph_layer_bwd_csr_parts(void) { return kSbwdParts; }

int digat_gat_layer_train_fwd(const float* Hm, int ldh, const float* s12, const uint8_t* adj, const float* X, float* Y,
                              int B, int n, int D, const uint8_t* drop_keep, float drop_scale, float* edge_score,
                              float* edge_alpha, uint8_t* relu_mask, const uint16_t* csr_rowptr, const uint16_t* csr_meta,
                              void* stream) {
    return launch_gat_layer_train_fwd(Hm, ldh, s12, adj, X, Y, B, n, D, drop_keep, drop_scale, edge_score, edge_alpha, relu_mask,
                                      csr_rowptr, csr_meta, as_stream(stream));
}

int digat_gat_layer_bwd_csr(const float* Hm, int ldh, const uint16_t* csr_rowptr, const uint16_t* csr_meta,
                            const uint16_t* csc_colptr, const uint16_t* csc_edge, const float* edge_score, const float* edge_alpha,
                            const uint8_t* drop_keep, float drop_scale, const float* dY, const uint8_t* relu_mask, float* dH,
                            int lddh, float* ds12, int B, int n, int D, void* stream) {
    if (B > 0 && ds12 == nullptr) return fail(DIGAT_E_INVALID, "digat_gat_layer_bwd_csr: null ds12");
    return launch_graph_layer_bwd_csr(Hm, ldh, nullptr, csr_rowptr, csr_meta, csc_colptr, csc_edge, edge_score, edge_alpha,
                                      drop_keep, drop_scale, dY, relu_mask, dH, lddh, nullptr, nullptr, nullptr, B, n, D,
                                      as_stream(stream), ds12);
}

int digat_graph_layer_csr_training_supported(int n, int D) { return graph_layer_csr_training_supported(n, D); }

int digat_attention_pool_bwd(const float* F, int64_t strideF, int ldf, const float* resid_F, const float* v,
                             const uint8_t* mask, const float* alpha, const float* dout, int ldg, float* dF,
                             float* dresid, float* dv, int B, int m, int D, void* stream) {
    return launch_attention_pool_bwd(F, strideF, ldf, resid_F, v, mask, alpha, dout, ldg, dF, dresid, dv, B, m, D,
                                     as_stream(stream));
}

int digat_news_gate_bwd(const float* z, const float* lg, const float* dout, float* dz, float* dlg, int B, int D, void* stream) {
    return launch_news_gate_bwd(z, lg, dout, dz, dlg, B, D, as_stream(stream));
}

int digat_topic_segment_bwd(const float* Xu, int64_t strideX, const float* v, const int64_t* cidx, const float* alpha,
                            const float* dT, float* dXu, float* dv, int B, int H, int n_seg, int n_u, int D,
                            void* stream) {
    return launch_topic_segment_bwd(Xu, strideX, v, cidx, alpha, dT, dXu, dv, B, H, n_seg, n_u, D, as_stream(stream));
}

int digat_reduce_workspace_floats(int M, int N, int K, int64_t* floats) {
    DIGAT_REQUIRE(floats != nullptr && M >= 0 && N > 0 && K > 0, "digat_reduce_workspace_floats: bad argument");
    *floats = wgrad_workspace_floats(M, N, K);
    return DIGAT_OK;
}

int digat_linear_wgrad(const float* dC, int lddc, const float* A, int lda, float* dW, float* workspace, int M, int N,
                       int K, void* stream) {
    return launch_linear_wgrad(dC, lddc, A, lda, dW, workspace, M, N, K, as_stream(stream));
}

int digat_colsum(const float* in, int ld, float* out, float* workspace, int M, int N, void* stream) {
    return launch_colsum(in, ld, out, workspace, M, N, as_stream(stream));
}

int digat_transpose_f32(const float* in, int ld_in, float* out, float* out_lo, int ld_out, int rows, int cols, void* stream) {
    return launch_transpose(in, ld_in, out, out_lo, ld_out, rows, cols, as_stream(stream));
}

int digat_groupsum(const float* in, int ld, float* out, int groups, int rows, int col0, int cols, void* stream) {
    return launch_groupsum(in, ld, out, groups, rows, col0, cols, as_stream(stream));
}

int digat_build_user_graphs(const int32_t* hist_cat, const int32_t* hist_len, uint8_t* graph, uint8_t* cmask,
                            int64_t* cidx, int64_t N, int H, int C, int32_t* err_flag, void* stream) {
    return launch_build_user_graphs(hist_cat, hist_len, graph, cmask, cidx, N, H, C, err_flag, as_stream(stream));
}

int digat_user_active_rows(const uint8_t* adj, const int32_t* adj_index, const int64_t* cidx, const uint8_t* cmask,
                           uint8_t* active, uint8_t* pooled, int64_t G, int n, int H, int S, void* stream) {
    return launch_user_active_rows(adj, adj_index, cidx, cmask, active, pooled, G, n, H, S, as_stream(stream));
}

int digat_compact_lists(const uint8_t* flags, const int32_t* csum, int n_lists, const int64_t* lo, const int64_t* size,
                        const int32_t* base, int32_t* const* ids, int32_t* const* pos, void* stream) {
    return launch_compact_lists(flags, csum, n_lists, lo, size, base, ids, pos, as_stream(stream));
}

int digat_news_active_rows(const uint8_t* adj, const uint8_t* mask, uint8_t* active, int64_t G, int n, void* stream) {
    return launch_news_active_rows(adj, mask, active, G, n, as_stream(stream));
}

int digat_graph_layer_supports_row_active(int n, int D, int B) { return graph_layer_supports_row_active(n, D, B); }

int digat_sag_bfs(const int64_t* sim_off, const int32_t* sim_idx, const double* sim_cos, int32_t* node_id,
                  uint8_t* graph, uint8_t* mask, int n_news, int top_M, int hop, int n_nodes, double threshold,
                  int32_t* err_flag, void* stream) {
    return launch_sag_bfs(sim_off, sim_idx, sim_cos, node_id, graph, mask, n_news, top_M, hop, n_nodes, threshold,
                          err_flag, as_stream(stream));
}

int digat_msa_attention_bwd(const float* QKV, int ld, const float* H, int ldh, const float* dH, int lddh, float* dQKV, int ldd,
                            int64_t n_titles, int T, int heads, int dk, void* stream) {
    return launch_msa_attention_bwd(QKV, ld, H, ldh, dH, lddh, dQKV, ldd, n_titles, T, heads, dk, as_stream(stream));
}

int digat_additive_pool_bwd(const float* att_pre, int lda, const float* w2, const float* H, int ldh, const uint8_t* mask,
                            const float* dout, int ldo, float* dH, int lddh, float* datt, int ldda, float* dw2_part,
                            int64_t n_titles, int T, int A, int D, void* stream) {
    return launch_additive_pool_bwd(att_pre, lda, w2, H, ldh, mask, dout, ldo, dH, lddh, datt, ldda, dw2_part, n_titles, T, A, D,
                                    as_stream(stream));
}

int digat_scatter_add_rows(float* dtable, int64_t n_table, const int32_t* idx, const float* src, int64_t lds, int64_t rows, int D,
                           void* stream) {
    return launch_scatter_add_rows(dtable, n_table, idx, src, lds, rows, D, as_stream(stream));
}

int digat_rank_impressions(const float* scores, const int64_t* offsets, int32_t* ranks, int64_t n_imp, void* stream) {
    return launch_rank_impressions(scores, offsets, ranks, n_imp, as_stream(stream));
}

int digat_impression_metrics(const int32_t* ranks, const uint8_t* labels, const int64_t* offsets, double* out,
                             uint8_t* valid, int64_t n_imp, void* stream) {
    return launch_impression_metrics(ranks, labels, offsets, out, valid, n_imp, as_stream(stream));
}

int digat_msa_attention_fwd(const float* QKV, int ld, float* H, int ldh, int64_t n_titles, int T, int heads, int dk,
                            void* stream) {
    return launch_msa_attention(QKV, ld, H, ldh, n_titles, T, heads, dk, as_stream(stream));
}

int digat_additive_pool_fwd(const float* att_pre, int lda, const float* w2, const float* H, int ldh, const uint8_t* mask,
                            float* out, int ldo, int64_t n_titles, int T, int A, int D, void* stream) {
    return launch_additive_pool(att_pre, lda, w2, H, ldh, mask, out, ldo, n_titles, T, A, D, as_stream(stream));
}

}  // extern "C"
