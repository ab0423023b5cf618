/*
 * digat_sm100.h -- C ABI of libdigat_sm100.so: hand-written sm_100a kernels for the DIGAT dual-graph
 * interaction encoder (reference: Veason-silverbullet/DIGAT, graphEncoders.py:48-198).
 *
 * The reference has no native code at all (SURVEY.md section 2): every entry point below replaces a group of
 * PyTorch/torch_scatter library calls on the hot path; the reference lines each one replaces are cited.
 *
 * Conventions
 *   - every pointer is a DEVICE pointer into memory owned by the caller (PyTorch allocates inputs, outputs and
 *     workspaces); the library owns nothing but cached TMA descriptors;
 *   - all matrices are row-major fp32, 16-byte aligned, leading dimensions in ELEMENTS and multiples of 4;
 *   - graphs / masks are 1 byte per element (torch.bool), non-zero = edge / valid;
 *   - `stream` is a cudaStream_t passed as void* (0 = legacy default stream); every call is asynchronous;
 *   - return value: 0 on success, <0 on failure (DIGAT_E_*); digat_last_error() gives the message of the
 *     last failure on the calling thread.  Nothing throws or exits across this boundary.
 *   - entry points are re-entrant (process-wide mutable state: cached device properties, a mutex-guarded TMA
 *     descriptor cache, and the digat_debug_set_layer_mode test switch, which nothing on the reference path sets);
 *     there is no CPU fallback: without an sm_100 device every compute call fails.
 */
#ifndef DIGAT_SM100_H
#define DIGAT_SM100_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DIGAT_OK             0
#define DIGAT_E_INVALID     -1   /* bad argument (null pointer, misaligned, unsupported size) */
#define DIGAT_E_CUDA        -2   /* a CUDA runtime/driver call or a launch failed */
#define DIGAT_E_UNSUPPORTED -3   /* device is not sm_100 */

#define DIGAT_ABI_VERSION 7

int         digat_abi_version(void);
const char* digat_last_error(void);
/* Checks that the current device is compute capability 10.x; fills sm_count if non-null. */
int         digat_device_check(int* sm_count);

/* ---------------------------------------------------------------------------------------------------------
 * Dense projections (replace nn.Linear: graphEncoders.py:146-149,166-169,112,126-127,131; layers.py:200)
 * C[M,N] = A[M,K] * W[N,K]^T (+ bias[N]) (optionally relu), W in nn.Linear layout.
 * --------------------------------------------------------------------------------------------------------- */

/* Optional row-group bias of both GEMMs (group_bias may be NULL):
 *   C[m, group_col0 + c] += group_bias[(m / group_rows) * group_ld + c],  c in [0, group_cols)
 * It folds k3 = ffn3(context) + b3 (graphEncoders.py:149/169, one row per graph) into the K1 block of the node
 * projections, so the GEMM emits U = fl(k3 + K1): the first broadcast add of Eq. (8) with the reference's rounding. */

/* Exact-fp32 CUDA-core GEMM (FFMA, fp32 accumulate).  Any M,N; K % 4 == 0. */
int digat_linear_f32(const float* A, int lda, const float* W, int ldw, const float* bias,
                     float* C, int ldc, int M, int N, int K, int relu,
                     const float* group_bias, int group_rows, int group_col0, int group_cols, int group_ld,
                     void* stream);

/* Exact-fp32 CUDA-core product for the few-hundred-row projections of a training step (context queries / keys / gates,
 * k3): out[I,J] = sum_c L(i,c) R(c,j) (+ bias[j]), no operand copies, sums in c order (deterministic).
 *   l_trans = 0: L stored [I][C] (ldl >= C)      l_trans = 1: L stored [C][I] (ldl >= I)
 *   r_trans = 0: R stored [C][J] (ldr >= J)      r_trans = 1: R stored [J][C] (ldr >= C)
 * forward C = A W^T: (L, R) = (A, W) with r_trans;  dgrad dA = dC W: (dC, W);  wgrad dW = dC^T A: (dC, A) with l_trans.
 * J, the leading dimensions and each operand's contiguous dimension must be multiples of 4. */
int digat_gemm_f32_small(const float* L, int ldl, int l_trans, const float* R, int ldr, int r_trans, const float* bias,
                         float* out, int ldo, int I, int J, int C, void* stream);
/* Splits W into the two TF32 planes used by digat_linear_tf32x3: hi = rna_tf32(W), lo = rna_tf32(W - hi). */
int digat_split_tf32(const float* W, float* W_hi, float* W_lo, int64_t count, void* stream);

/* tcgen05 tensor-core GEMM, operands fed by TMA, fp32 accumulators in TMEM, fp32-level accuracy by 3xTF32 error
 * compensation: C = A_hi*W_hi + A_lo*W_hi + A_hi*W_lo (+ bias).  A is plain fp32 and is split into its TF32 planes
 * on the fly inside the kernel; W_hi / W_lo come from digat_split_tf32 (same ldw).
 * Requires K % 4 == 0, N % 16 == 0, lda/ldw/ldc % 4 == 0.  Replaces the three node projections h, K1, K2 of one
 * layer as ONE GEMM against the stacked [3D, D] weight (graphEncoders.py:146-148 / 166-168).
 * c_row_index (may be NULL; ascending int32 [M]): row scatter -- product row m is written to row c_row_index[m] of C
 * and takes the row-group bias of that row.  A then holds only the node rows worth projecting (see
 * digat_user_active_rows) while C keeps the dense [graphs * n] layout digat_graph_layer_fwd streams with TMA; the
 * rows of C that are not listed are left untouched.  Needs N <= 1280. */
int digat_linear_tf32x3(const float* A, int lda, const float* W_hi, const float* W_lo, int ldw,
                        const float* bias, float* C, int ldc, int M, int N, int K,
                        const float* group_bias, int group_rows, int group_col0, int group_cols, int group_ld,
                        const int32_t* c_row_index, void* stream);

/* C = bf16_rn(A) * W_b^T (+bias)(+row-group bias), fp32 accumulation.  W_b = bf16_rn(W) [N,K] (row pitch ldw).
 * Same bias / group-bias / c_row_index semantics and alignment rules as digat_linear_tf32x3; K, ldw % 8 == 0, N <= 1280.
 * One tcgen05 kind::f16 MMA per 16-wide k-block; every M takes the same kernel, and an output row depends on its A row
 * and W only.  The opt-in inference precision of the DIGAT node projections (DIGAT.projection_precision = 'bf16'). */
int digat_linear_bf16(const float* A, int lda, const void* W_b, int ldw, const float* bias, float* C, int ldc,
                      int M, int N, int K, const float* group_bias, int group_rows, int group_col0, int group_cols,
                      int group_ld, const int32_t* c_row_index, void* stream);

/* Split-K form of digat_linear_tf32x3 (no bias): the contraction range [0,K) is cut into kbatches equal slices and slice
 * s writes its partial product to C + s * c_batch_stride (elements); the caller sums the slabs (digat_colsum over a
 * [kbatches, M*ldc] view: exact fp32 adds in slice order).  Used for weight gradients dW = dC^T A, whose contraction
 * runs over all rows of a batch: more tiles than SMs for a skinny output, and few truncating tensor-core accumulate
 * steps per accumulator.  N <= 1280. */
int digat_linear_tf32x3_splitk(const float* A, int lda, const float* W_hi, const float* W_lo, int ldw,
                               float* C, int ldc, int M, int N, int K, int kbatches, int64_t c_batch_stride,
                               void* stream);

/* digat_graph_layer_fwd kernel choice: 0 = auto (edge-driven kernel when a CTA owns one graph and no training extras are
 * requested, dense kernel otherwise), 1 = always dense, 2 = always edge-driven (inference).  For tests / profiling. */
int digat_debug_set_layer_mode(int mode);

/* ---------------------------------------------------------------------------------------------------------
 * Fused Eq. (8) graph-attention layer (replaces graphEncoders.py:150-153 / 170-173).
 *   P    [B*n, ldp]  node projections of this layer: columns [0,D) = h (bias included), [D,2D) = U = k3 + K1
 *                    (k3 = ffn3(context of the other graph) + bias, folded in by the GEMM's row-group bias),
 *                    [2D,3D) = K2
 *   a    [D]         attention vector                                  (news/user_graph_attention_a[i].weight)
 *   adj  [B, n, n]   bool adjacency, row i = query node, column j = neighbour
 *   X    [B, n, D]   layer input (residual)
 *   Y    [B, n, D]   out: relu(softmax_j(mask(leaky_relu(a . relu(U_j + K2_i)))) * h) + X
 * Training extras (each may be NULL): drop_keep [B,n,n] bool keep-mask of the dropout on the attention weights
 * (graphEncoders.py:152/172; the weights are multiplied by keep * drop_scale, drop_scale = 1/(1-p)); outputs saved
 * for digat_graph_layer_bwd: score_out [B,n,n] raw scores s_ij, alpha_out [B,n,n] softmax weights before dropout,
 * relu_mask_out [B,n,D] bool, 1 where the aggregated message (alpha~ h) is positive.
 * The [B,n,n,D] broadcast tensor of the reference is never materialised: P tiles are streamed through shared memory
 * by TMA (2-deep pipeline).  n <= 128, D % 4 == 0, D <= 1024.
 * De-duplicated scoring (each may be NULL): the ~37 candidate pairs of one impression share the user graph, so its
 * layer-0 projection is computed once per behaviour: px_index [B] makes graph b read P and X of graph px_index[b]
 * (tables with n_src graphs; P then holds K1 WITHOUT k3) and k3 [B,ldk3] is added to the staged K1 tile in-kernel
 * (same fp32 add as the GEMM's row-group bias, so results are bit-identical to the expanded path); adj_index [B]
 * makes graph b read adj of graph adj_index[b] (per-behaviour user graphs, no per-pair copy).
 * Node pruning (may be NULL; edge-driven kernel only, see digat_graph_layer_supports_row_active): row_active [B,n]
 * bool, 0 = node whose output nothing can observe (digat_user_active_rows).  Its P row is never read for arithmetic
 * (it may be uninitialised: digat_linear_tf32x3 with c_row_index skips it), none of its edges is evaluated and its
 * output row is left untouched (neither X nor Y of that row is accessed; every later consumer -- the next layer with
 * the same flags, the pooling kernels with their masks -- skips it too).  An inactive node that an active one has an
 * edge to must have a valid P row (it is still a neighbour): that is the last-layer case, where only the rows a
 * context pools are evaluated.  With row_active, Yc [M_act, D] and
 * row_pos [B*n] int32 (both or neither): the output row of active node row r is ALSO written to Yc[row_pos[r]], the
 * compact operand of the next layer's projection (digat_linear_tf32x3 with c_row_index), saving a gather pass.
 * --------------------------------------------------------------------------------------------------------- */
int digat_graph_layer_fwd(const float* P, int ldp, const float* a, const uint8_t* adj, const float* X, float* Y,
                          int B, int n, int D, const uint8_t* drop_keep, float drop_scale, float* score_out,
                          float* alpha_out, uint8_t* relu_mask_out, const int32_t* px_index, int n_src,
                          const int32_t* adj_index, const float* k3, int ldk3, const uint8_t* row_active,
                          float* Yc, const int32_t* row_pos, const uint16_t* csr_rowptr, const uint16_t* csr_meta,
                          const int32_t* csr_index, void* stream);
/* CSR of each graph's adjacency restricted to its evaluated rows, built once per batch for digat_graph_layer_fwd's
 * csr_rowptr / csr_meta / csr_index (each may be NULL there; with them the kernel does not read `adj` and skips its
 * per-layer, per-pair CSR construction; edge-driven kernel with one graph per CTA, i.e. not the multi-graph news launches):
 *   graph g reads adjacency adj[adj_index ? adj_index[g] : g] ([*,n,n] bool) and row_active [G,n] (NULL = every row);
 *   rowptr [G, n+1] uint16: rowptr[i+1] & 0x7fff = end of row i's edge range (pruned rows are empty), bit 15 = row i has no
 *   edge at all (its range lists every node: the reference's uniform softmax);  meta [G, n*n] uint16: neighbour | row << 8.
 * In digat_graph_layer_fwd graph b uses record csr_index[b] (NULL: b): the pairs of one impression share one record.
 * Transpose for the training backward (both NULL, or both given): colptr [G, n+1] uint16 = start of column j's range,
 * cedge [G, n*n] uint16 = the CSR positions of the edges (i, j) ending in node j, rows ascending.
 * Training (score_out / alpha_out / relu_mask_out given) with a CSR: score_out and alpha_out are then PER EDGE, in
 * CSR order ([B, n*n] capacity, entries past rowptr[n] untouched) instead of dense [B,n,n]; they feed
 * digat_graph_layer_bwd_csr. */
int digat_build_graph_csr(const uint8_t* adj, const int32_t* adj_index, const uint8_t* row_active, uint16_t* rowptr,
                          uint16_t* meta, uint16_t* colptr, uint16_t* cedge, int64_t G, int n, void* stream);
/* Vanilla-GAT layer of the reference's ablation encoders (graphEncoders.py:494-503, 511-520, 640-649, 807-816:
 * wo_interaction, news_graph_wo_inter, user_graph_wo_inter), inference:
 *   Y = relu(softmax_j(mask(leaky_relu(a1 . h_j + a2 . h_i))) * h) + X
 *   Hm [B*n, ldh] = h = W x + b;  s12 [B*n, 2]: s12[r][0] = a1 . h_r (neighbour term), s12[r][1] = a2 . h_r (query term),
 *   both from digat_linear_* ; adj [B,n,n]; X, Y [B,n,D].  Same edge-driven kernel as digat_graph_layer_fwd: an edge's score
 *   is one fp32 add, only h is streamed. */
int digat_gat_layer_fwd(const float* Hm, int ldh, const float* s12, const uint8_t* adj, const float* X, float* Y,
                        int B, int n, int D, void* stream);
/* 1 if an inference call of digat_graph_layer_fwd with these sizes takes the kernel that honours row_active, else 0. */
int digat_graph_layer_supports_row_active(int n, int D, int B);
/* Node pruning flags for user graphs: active [G,n] = 0 iff node i's layer output is unobservable: no other node has
 * an edge to it (column i of adj empty off the diagonal) AND no context reads it (i >= H: topic nodes are never
 * pooled, graphEncoders.py:125; or history slot i belongs to a bucket c = cidx[i] with cmask[c] == 0 while some other
 * bucket is unmasked -- with every bucket masked the softmax is uniform and reads them all).
 * A graph with an edge-less row keeps every node.  adj [*,n,n] read through adj_index [G] when given (then cidx
 * [*,H] int64 is read through the same index); cmask [G,S] is per graph.
 * pooled [G,n] (optional): 1 = the user context pools this node's row directly.  After the LAST layer only those rows
 * are consumed, so they can serve as that layer's row_active (the other active nodes are still projected: they are
 * neighbours). */
int digat_user_active_rows(const uint8_t* adj, const int32_t* adj_index, const int64_t* cidx, const uint8_t* cmask,
                           uint8_t* active, uint8_t* pooled, int64_t G, int n, int H, int S, void* stream);
/* Index lists from flags without a host round trip for the data: up to four flag lists laid out back to back in `flags`
 * (uint8) with their inclusive int32 prefix sums in `csum`.  HOST arrays lo/size (flat range of list k), base (number of
 * set flags before list k) and ids/pos (DEVICE output pointers per list; pos[k] may be NULL): ids_k receives the positions
 * of the set flags of list k in ascending order, pos_k[r] the rank of position r (valid where the flag is set).  The
 * caller sizes ids_k from the counts it read back (one event wait per batch, digat_b200/graphEncoders.py). */
int digat_compact_lists(const uint8_t* flags, const int32_t* csum, int n_lists, const int64_t* lo, const int64_t* size,
                        const int32_t* base, int32_t* const* ids, int32_t* const* pos, void* stream);
/* The same for news graphs: a node is kept iff another node has an edge to it, or the news context reads it
 * (graphEncoders.py:109-114): node 0 (the local context), mask[g,i] != 0 (pooled by the candidate attention), or every
 * mask entry of the graph is 0 (uniform softmax).  adj [G,n,n], mask [G,n], active [G,n]. */
int digat_news_active_rows(const uint8_t* adj, const uint8_t* mask, uint8_t* active, int64_t G, int n, void* stream);

/* ---------------------------------------------------------------------------------------------------------
 * Masked single-query attention pooling (replaces layers.py:199-206 after folding W_K into the query:
 * a_k = F_k . v / sqrt(D) with v = W_K^T (W_Q q + b_Q)):
 *   out[b] = sum_k softmax_k(mask(F[b,k] . v[b] / sqrt(D))) F[b,k]
 *   F [B, m, D] with row stride ldf and batch stride strideF (elements); mask [B,m] bool; v [B,D] with row pitch ldv.
 * If resid_F != NULL the pooled features are F' = relu(F) + resid_F (graphEncoders.py:131, featureAffine output
 * in F, topic embeddings in resid_F).  out has leading dimension ldo (so it can land inside a [B,2D] buffer).
 * add_in [B, ldo] optional: out = add_in + pooled (context accumulation, graphEncoders.py:186/197; may alias out).
 * first_out [B, ldo] optional: receives a copy of F[b,0,:] (the "local" context l of graphEncoders.py:110, so
 * that [l | g] lands in one [B,2D] buffer for the gate projection).  alpha_out [B,m] optional.
 * --------------------------------------------------------------------------------------------------------- */
int digat_attention_pool_fwd(const float* F, int64_t strideF, int ldf, const float* resid_F,
                             const float* v, int ldv, const uint8_t* mask, const float* add_in, float* out, int ldo,
                             float* first_out, float* alpha_out, int B, int m, int D, void* stream);

/* News-graph gate (graphEncoders.py:112-113): ctx_out = ctx_in + sigmoid(z) * l + (1 - sigmoid(z)) * g
 *   z [B,D] = news_graph_W([l;g]) (+bias, from digat_linear_*), lg [B, 2D] = [l | g].  ctx_in may be NULL
 *   (first context, graphEncoders.py:180) and may alias ctx_out. */
int digat_news_gate_fwd(const float* z, const float* lg, const float* ctx_in, float* ctx_out,
                        int B, int D, void* stream);

/* Topic-level aggregation of the user history (replaces torch_scatter.scatter_softmax + scatter_sum,
 * graphEncoders.py:128-130; torch_scatter is an un-vendored third-party dependency, see oracle/scatter_shim.py):
 *   a_t   = Xh[b,t] . v[b] / sqrt(D),                 t in [0,H)      (v = user_news_K^T (user_news_Q c_n + b))
 *   alpha = softmax of a_t inside each segment {t : cidx[b,t] = k}
 *   T[b,k] = sum_{t in segment k, ascending t} alpha_t Xh[b,t],  k in [0, n_seg); empty segments are 0.
 *   Xh = first H rows of X_u [B, n_u, D] (batch stride strideX elements); cidx int64 [B,H] in [0,n_seg).
 * alpha_out [B,H] optional.  err_flag: see the gathers below.  src_index [B] optional: row b reads Xu and cidx of
 * row src_index[b] (user graphs shared by the pairs of one impression).
 * cmask [B,n_seg] bool optional (inference): the mask the user-level attention applies to T afterwards
 * (graphEncoders.py:132).  Segments with cmask == 0 get a softmax weight of exactly 0 there, so their history rows are
 * not read and T[b,k] = 0 -- unless every segment of row b is masked (uniform weights: everything is evaluated).
 * (With Tc, the rows T[b,k] of masked segments are left UNWRITTEN instead: the caller then evaluates featureAffine and the
 * user-level pooling on the visible segments only and nothing reads them.)
 * Tc [M_live, D] + seg_pos [B*n_seg] int32 optional (with cmask): the evaluated segments (cmask != 0, or all of a
 * fully masked row) are also written to Tc[seg_pos[b*n_seg + k]], the compact operand of the featureAffine GEMM. */
int digat_topic_segment_fwd(const float* Xu, int64_t strideX, const float* v, int ldv, const int64_t* cidx,
                            float* T, float* alpha_out, int32_t* err_flag, const int32_t* src_index,
                            const uint8_t* cmask, float* Tc, const int32_t* seg_pos,
                            int B, int H, int n_seg, int D, void* stream);

/* ---------------------------------------------------------------------------------------------------------
 * Gathers (replace index_select at util.py:34-36 and util.py:65-67) and small glue.
 * --------------------------------------------------------------------------------------------------------- */
/* Index errors: the reference's index_select / scatter raise on an out-of-range index.  A kernel cannot raise, so
 * every indexed entry point takes `err_flag` (device int32, may be NULL): it is set to 1 when an index is out of
 * range (the offending row then reads row 0 / the last segment); the host wrapper checks it and raises. */
/* out[r, :] = table[idx[r], :] for r in [0,rows); idx int32; D % 4 == 0; out row stride ldo. */
int digat_gather_rows_i32(const float* table, int64_t n_table, const int32_t* idx, float* out, int64_t ldo,
                          int64_t rows, int D, int32_t* err_flag, void* stream);
/* Two-level gather for SAG node embeddings: out[r, s, :] = table[node_id[news[r], s], :]  (util.py:35 + :66
 * without materialising the [N_news, n_n, D] cache). */
int digat_gather_sag_i32(const float* table, int64_t n_table, const int32_t* node_id, int n_nodes,
                         const int32_t* news, float* out, int64_t rows, int D, int32_t* err_flag,
                         void* stream);
/* X_u[b] = [ hist[b] (H rows, gathered from table through hist_idx or copied from `hist` if table==NULL) ;
 *            topic_emb (C rows) ]   (graphEncoders.py:179/191: cat(user_news_embedding, topic_node_embedding)) */
int digat_build_user_nodes(const float* table, int64_t n_table, const int32_t* hist_idx, const float* hist,
                           const float* topic_emb, float* Xu, int B, int H, int C, int D, int32_t* err_flag,
                           void* stream);
/* logits[b] = sum_d news_ctx[b,d] * user_ctx[b,d]   (model.py:76,89) */
int digat_logits(const float* news_ctx, const float* user_ctx, float* logits, int B, int D, void* stream);
/* y = x + y (fp32, count elements) -- context accumulation (graphEncoders.py:185-186,196-197) */
int digat_add_inplace(const float* x, float* y, int64_t count, void* stream);

/* ---------------------------------------------------------------------------------------------------------
 * Backward kernels (training; replace PyTorch autograd of the forward ops above).  The reference's autograd saves
 * the [B,n,n,D] relu output of Eq. (8) per layer and graph; here its mask is recomputed from P.
 * --------------------------------------------------------------------------------------------------------- */

/* Backward of digat_graph_layer_fwd.
 *   in : P, a, adj as in the forward; score, alpha (saved by the forward); drop_keep/drop_scale as in the forward;
 *        G [B,n,D] = dY * relu_mask (the caller applies the saved relu mask; dX of the residual is dY itself)
 *   out: dP [B*n, lddp] = dh | dU | dK2  (dk3 = sum over a graph's rows of dU: digat_groupsum);
 *        da_partial [B, D] per-graph partial of the attention-vector gradient (digat_colsum over B finishes it). */
int digat_graph_layer_bwd(const float* P, int ldp, const float* a, const uint8_t* adj, const float* score,
                          const float* alpha, const uint8_t* drop_keep, float drop_scale, const float* G,
                          float* dP, int lddp, float* da_partial, int B, int n, int D, void* stream);
/* The same backward, edge-driven: only the E edges of each graph are evaluated (a masked pair has alpha = 0 and
 * ds = 0), through the CSR and its transpose of digat_build_graph_csr (no adj_index / row_active: training evaluates
 * every graph and row) and the per-edge edge_score / edge_alpha [B, n*n] the forward wrote when it was given the
 * same CSR.  drop_keep stays the dense [B,n,n] mask.  dP as in digat_graph_layer_bwd (every row is written).
 * da_partial is [B * PARTS, D] here, PARTS = digat_graph_layer_bwd_csr_parts(): row b * PARTS + w holds the partial of
 * consumer warp w of graph b (digat_colsum over all rows finishes da) -- folding the warps inside the kernel would cost a
 * CTA-wide barrier per feature chunk.
 * Optional (NULL = off): relu_mask [B,n,D] -- G is then the raw dY and the forward's saved mask is applied in-kernel;
 * dh_sum, du_sum [B * PARTS, D] -- column sums of the dh and dU blocks of dP in the same per-warp layout: digat_colsum of
 * dh_sum = the gradient of the projection bias, digat_groupsum of du_sum over each graph's PARTS rows = dk3 (the gradient of
 * the row-group bias), so nothing re-reads dP for them.  All sums run in a fixed order (deterministic). */
int digat_graph_layer_bwd_csr(const float* P, int ldp, const float* a, const uint16_t* csr_rowptr, const uint16_t* csr_meta,
                              const uint16_t* csc_colptr, const uint16_t* csc_edge, const float* edge_score,
                              const float* edge_alpha, const uint8_t* drop_keep, float drop_scale, const float* G,
                              const uint8_t* relu_mask, float* dP, int lddp, float* da_partial, float* dh_sum, float* du_sum,
                              int B, int n, int D, void* stream);
int digat_graph_layer_bwd_csr_parts(void);
/* Training pair of the vanilla-GAT layer (digat_gat_layer_fwd: e_ij = leaky_relu(s12[j,0] + s12[i,1]), Y = relu(alpha~ h) + X),
 * edge-driven like the pair above; the CSR and its transpose come from digat_build_graph_csr:
 *   digat_gat_layer_train_fwd  as digat_gat_layer_fwd, plus the attention dropout (drop_keep [B,n,n] or NULL, drop_scale) and
 *                              the outputs the backward needs: edge_score / edge_alpha [B, n*n] in CSR order, relu_mask [B,n,D]
 *   digat_gat_layer_bwd_csr    dY [B,n,D] (raw: the relu mask is applied in-kernel) -> dH [B*n, lddh] (gradient of h through the
 *                              aggregation) and ds12 [B*n, 2] (ds1_j = sum over the edges entering j of ds_e, ds2_i = sum over
 *                              row i of ds_e); the gradient of X through the residual is dY itself.  The caller adds
 *                              ds12 [a1; a2] to dH and forms da1 / da2 (the backward of its s12 = h [a1; a2]^T product). */
int digat_gat_layer_train_fwd(const float* Hm, int ldh, const float* s12, const uint8_t* adj, const float* X, float* Y,
                              int B, int n, int D, const uint8_t* drop_keep, float drop_scale, float* edge_score,
                              float* edge_alpha, uint8_t* relu_mask, const uint16_t* csr_rowptr, const uint16_t* csr_meta,
                              void* stream);
int digat_gat_layer_bwd_csr(const float* Hm, int ldh, const uint16_t* csr_rowptr, const uint16_t* csr_meta,
                            const uint16_t* csc_colptr, const uint16_t* csc_edge, const float* edge_score, const float* edge_alpha,
                            const uint8_t* drop_keep, float drop_scale, const float* dY, const uint8_t* relu_mask, float* dH,
                            int lddh, float* ds12, int B, int n, int D, void* stream);
/* 1 when graphs of n nodes and width D can train through the CSR pair (digat_graph_layer_fwd with a CSR and training
 * outputs + digat_graph_layer_bwd_csr): both working sets fit one SM.  0: use the dense [B,n,n] score / alpha path. */
int digat_graph_layer_csr_training_supported(int n, int D);

/* Optimizer step of reference trainer.py:98-105 (nn.utils.clip_grad_norm_ + optim.Adam.step) over FLAT fp32 buffers of n
 * elements (parameters, gradients, exp_avg, exp_avg_sq laid out in the same order), two launches:
 *   digat_grad_sumsq      partials [1024] = fixed-chunk partial sums of g^2; step_counter[0] += 1 (device-side Adam step
 *                         count, so a CUDA-graph replay advances it; may be NULL)
 *   digat_adam_clip_step  norm = sqrt(sum partials) (-> grad_norm_out[0], may be NULL); g *= min(1, max_norm / (norm + 1e-6))
 *                         when max_norm > 0 (written back); then torch.optim.Adam's update with L2 weight_decay and the
 *                         bias corrections 1 - beta^step_counter[0]. */
int digat_grad_sumsq(const float* g, int64_t n, float* partials, float* step_counter, void* stream);
int digat_adam_clip_step(float* p, float* g, float* m, float* v, int64_t n, const float* partials, const float* step_counter,
                         float* grad_norm_out, float max_norm, float lr, float beta1, float beta2, float eps,
                         float weight_decay, void* stream);

/* Backward of digat_attention_pool_fwd.  alpha [B,m] saved by the forward; dout [B, ldg].
 * out: dF [B,m,D] dense (w.r.t. F; masked by F > 0 when resid_F is given), dresid [B,m,D] (only with resid_F),
 *      dv [B,D]. */
int digat_attention_pool_bwd(const float* F, int64_t strideF, int ldf, const float* resid_F, const float* v,
                             const uint8_t* mask, const float* alpha, const float* dout, int ldg,
                             float* dF, float* dresid, float* dv, int B, int m, int D, void* stream);

/* Backward of digat_news_gate_fwd (out = ctx_in + s l + (1-s) g, s = sigmoid(z); lg = [l | g], [B, 2D]):
 * dz [B,D] = dout (l - g) s (1 - s),  dlg [B,2D] = [dout s | dout (1 - s)];  the gradient of ctx_in is dout itself. */
int digat_news_gate_bwd(const float* z, const float* lg, const float* dout, float* dz, float* dlg, int B, int D, void* stream);
/* Backward of digat_topic_segment_fwd.  alpha [B,H] saved by the forward; dT [B,n_seg,D].
 * out: dXu [B,n_u,D] (rows >= H are written as zeros: topic nodes are not pooled), dv [B,D]. */
int digat_topic_segment_bwd(const float* Xu, int64_t strideX, const float* v, const int64_t* cidx,
                            const float* alpha, const float* dT, float* dXu, float* dv,
                            int B, int H, int n_seg, int n_u, int D, void* stream);

/* Weight gradient of C = A W^T: dW[N,K] = dC[M,N]^T A[M,K] (exact fp32, deterministic split reduction over M).
 * workspace: digat_reduce_workspace_floats(M, N, K) floats. */
int digat_reduce_workspace_floats(int M, int N, int K, int64_t* floats);
int digat_linear_wgrad(const float* dC, int lddc, const float* A, int lda, float* dW, float* workspace,
                       int M, int N, int K, void* stream);
/* out[n] = sum_m in[m, n] (bias gradients); workspace: digat_reduce_workspace_floats(M, N, 1) floats. */
int digat_colsum(const float* in, int ld, float* out, float* workspace, int M, int N, void* stream);
/* out[c, r] = in[r, c] for an fp32 matrix of `rows` x `cols` (ld_in >= cols, ld_out >= rows).  With out_lo != NULL the
 * transposed matrix is written as its TF32 planes: out = rna_tf32(x), out_lo = rna_tf32(x - out) (digat_split_tf32 of the
 * transpose in one pass).  Operand preparation of the split-K weight gradient: dW = dC^T A contracts over the ROWS of dC and
 * A, and digat_linear_tf32x3_splitk wants the contraction index contiguous. */
int digat_transpose_f32(const float* in, int ld_in, float* out, float* out_lo, int ld_out, int rows, int cols, void* stream);
/* out[g, c] = sum_{r < rows} in[(g*rows + r), col0 + c] -- gradient of the GEMMs' row-group bias (dk3). */
int digat_groupsum(const float* in, int ld, float* out, int groups, int rows, int col0, int cols, void* stream);

/* ---------------------------------------------------------------------------------------------------------
 * Integer builders and ranking either side of the encoder (SURVEY.md section 8(f)); every output is bit-exact.
 * --------------------------------------------------------------------------------------------------------- */

/* User-history graphs (reference MIND_corpus.py:143-176, its O(H^2) Python loops per behaviour).
 *   in : hist_cat [N,H] int32 category id of history slot t (ignored for t >= hist_len[n]); hist_len [N] int32
 *   out: graph [N,H+C,H+C] u8 (bool), cmask [N,C+1] u8 (bool), cidx [N,H] int64 (padding bucket C)
 * err_flag (optional): bit 0 set on a category outside [0,C) or a length outside [0,H] (the reference raises). */
int digat_build_user_graphs(const int32_t* hist_cat, const int32_t* hist_len, uint8_t* graph, uint8_t* cmask,
                            int64_t* cidx, int64_t N, int H, int C, int32_t* err_flag, void* stream);
/* Semantic-augmented graphs by BFS over the similar-news lists (reference construct_SAG.py:449-485).
 *   in : CSR lists sim_off [n_news+1] int64, sim_idx [nnz] int32, sim_cos [nnz] f64, ordered as in the reference's
 *        similarity dict (most similar first); top_M, hop, threshold as construct_SAG.py:15-17,468
 *   out: node_id [n_news,n_nodes] int32, graph [n_news,n_nodes,n_nodes] u8, mask [n_news,n_nodes] u8 (mask[:,0]=1)
 * err_flag (optional): bit 0 = neighbour id out of range, bit 1 = more than n_nodes nodes (the reference raises). */
int digat_sag_bfs(const int64_t* sim_off, const int32_t* sim_idx, const double* sim_cos, int32_t* node_id,
                  uint8_t* graph, uint8_t* mask, int n_news, int top_M, int hop, int n_nodes, double threshold,
                  int32_t* err_flag, void* stream);
/* Backward kernels of the news encoders (training from token tensors, reference model.py:54-77 + autograd):
 *   digat_msa_attention_bwd  QKV, H as the forward saw / wrote them; dH [titles*T, lddh] -> dQKV [titles*T, ldd] (= dQ | dK | dV;
 *                            the relu mask H > 0 is applied to dH in-kernel, the T x T attention is recomputed)
 *   digat_additive_pool_bwd  dout [titles, ldo] -> dH (through the weighted sum only: alpha_t dout), datt [titles*T, ldda]
 *                            (gradient of the pre-tanh affine1 rows), dw2_part [titles, A] (digat_colsum over the titles = dw2)
 *   digat_scatter_add_rows   dtable[idx[r], :] += src[r, :] -- the embedding gather's backward (float atomics, as torch's) */
int digat_msa_attention_bwd(const float* QKV, int ld, const float* H, int ldh, const float* dH, int lddh, float* dQKV, int ldd,
                            int64_t n_titles, int T, int heads, int dk, void* stream);
int digat_additive_pool_bwd(const float* att_pre, int lda, const float* w2, const float* H, int ldh, const uint8_t* mask,
                            const float* dout, int ldo, float* dH, int lddh, float* datt, int ldda, float* dw2_part,
                            int64_t n_titles, int T, int A, int D, void* stream);
int digat_scatter_add_rows(float* dtable, int64_t n_table, const int32_t* idx, const float* src, int64_t lds, int64_t rows, int D,
                           void* stream);

/* ranks[p] = 1-based position of pair p inside its impression under a STABLE descending sort of the scores
 * (reference util.py:70-80).  offsets [n_imp+1] int64 delimit the impressions in the ordered pair list. */
int digat_rank_impressions(const float* scores, const int64_t* offsets, int32_t* ranks, int64_t n_imp, void* stream);
/* Per-impression AUC, MRR, nDCG@5, nDCG@10 of y_score = 1/rank (reference evaluate.py:32-89): out [n_imp,4] f64;
 * valid [n_imp] u8: 1 = scored, 0 = empty impression (skipped, evaluate.py:70), 2 = one class only (sklearn raises). */
int digat_impression_metrics(const int32_t* ranks, const uint8_t* labels, const int64_t* offsets, double* out,
                             uint8_t* valid, int64_t n_imp, void* stream);

/* ---------------------------------------------------------------------------------------------------------
 * News (title) encoder, MSA variant (SURVEY.md section 8(f) row 4; reference newsEncoders.py:58-82, layers.py:50-115),
 * inference.  Word embeddings are gathered with digat_gather_rows_i32 and the Q|K|V and affine1 projections are
 * digat_linear_* calls; these two kernels do the rest.
 * --------------------------------------------------------------------------------------------------------- */
/* Multi-head self-attention over the T <= 32 tokens of each title + relu (layers.py:78-97, newsEncoders.py:78):
 *   QKV [n_titles*T, ld]: columns [0,hd) = Q (bias included), [hd,2hd) = K, [2hd,3hd) = V (bias included), hd = heads*dk,
 *   head h owns columns h*dk .. h*dk+dk of each block;  H [n_titles*T, ldh] = relu(softmax(Q_h K_h^T / sqrt(dk)) V_h).
 * No padding mask (the reference applies none here).  dk <= 32. */
int digat_msa_attention_fwd(const float* QKV, int ld, float* H, int ldh, int64_t n_titles, int T, int heads, int dk,
                            void* stream);
/* Additive attention pooling over the tokens of each title (layers.py:107-115):
 *   a_t = tanh(att_pre[t]) . w2  (att_pre [n_titles*T, lda] = H affine1^T + b1, A columns; w2 [A] = affine2.weight),
 *   alpha = softmax_t(mask[t] ? a_t : -1e9),  out[title] = sum_t alpha_t H[title, t, :]  (out [n_titles, ldo], D columns). */
int digat_additive_pool_fwd(const float* att_pre, int lda, const float* w2, const float* H, int ldh, const uint8_t* mask,
                            float* out, int ldo, int64_t n_titles, int T, int A, int D, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* DIGAT_SM100_H */
