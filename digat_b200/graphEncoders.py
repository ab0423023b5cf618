"""Drop-in for reference graphEncoders.py (``--graph_encoder=DIGAT``): same class names, constructor, parameter
names/shapes (so reference checkpoints ``load_state_dict``), and the same public methods -- but every arithmetic
step runs in the hand-written sm_100a kernels of libdigat_sm100.so (include/digat_sm100.h).

Reference interface mirrored here (paths relative to /root/reference):
  GraphEncoder.__init__/initialize                 graphEncoders.py:10-45
  DIGAT.__init__/initialize                        graphEncoders.py:48-101
  DIGAT.compute_news_graph_context(X, mask)        graphEncoders.py:109-114   (also called by util.py:43)
  DIGAT.compute_user_graph_context(...)            graphEncoders.py:123-134
  DIGAT.compute_news/user_graph_embeddings(...)    graphEncoders.py:143-174   (Eq. (8) at :150/:170)
  DIGAT.forward / DIGAT.inference                  graphEncoders.py:177-198

There is no PyTorch fallback: CPU tensors, a missing library or a non-sm_100 device raise RuntimeError.
"""
import ctypes
import math

import torch
import torch.nn as nn

from . import _lib


def _stream():
    return torch.cuda.current_stream().cuda_stream


def _same_device(t, name):
    """Kernels are launched on the CURRENT device's current stream: a tensor on another device would hand the kernel a
    foreign pointer.  (One process per GPU: call torch.cuda.set_device first, as reference config.py:85-89 does.)"""
    if t.device.index != torch.cuda.current_device():
        raise RuntimeError('%s lives on %s but the current CUDA device is cuda:%d -- call torch.cuda.set_device(%d) '
                           '(digat_b200 launches on the current device)' % (name, t.device, torch.cuda.current_device(),
                                                                            t.device.index))


def _ptr(t):
    return 0 if t is None else t.data_ptr()


def _f32c(t, name):
    if not t.is_cuda:
        raise RuntimeError('%s must be a CUDA tensor (digat_b200 has no CPU fallback)' % name)
    if t.dtype != torch.float32:
        raise RuntimeError('%s must be float32, got %s' % (name, t.dtype))
    _same_device(t, name)
    return t if t.is_contiguous() else t.contiguous()


def _boolc(t, name):
    if not t.is_cuda:
        raise RuntimeError('%s must be a CUDA tensor (digat_b200 has no CPU fallback)' % name)
    if t.dtype not in (torch.bool, torch.uint8):
        raise RuntimeError('%s must be bool, got %s' % (name, t.dtype))
    _same_device(t, name)
    return t if t.is_contiguous() else t.contiguous()


# ------------------------------------------------------------------------------------------- thin op wrappers
_PINNED = {}
_ENDS = {}


def _pinned_ints(n):
    """A small pinned int32 buffer from a free list (cudaHostAlloc per call would cost more than the copy it serves;
    several may be in flight: one per staged batch)."""
    free = _PINNED.setdefault(n, [])
    return free.pop() if free else torch.empty(n, dtype=torch.int32).pin_memory()


def _release_pinned(buf):
    _PINNED.setdefault(buf.shape[0], []).append(buf)


def _ends_tensor(sizes, device):
    """Device tensor of the last flat position of each list (cached per size tuple: building it is a host->device copy)."""
    key = (sizes, str(device))
    t = _ENDS.get(key)
    if t is None:
        t = _ENDS[key] = torch.tensor([sum(sizes[:k + 1]) - 1 for k in range(len(sizes))], device=device)
    return t


class PackedWeight:
    """A projection weight in kernel layout: fp32 [N,K] (nn.Linear layout) plus, when the tcgen05 GEMM can take it
    (N % 16 == 0, K % 4 == 0), its two TF32 planes hi = rna_tf32(W), lo = rna_tf32(W - hi) (digat_split_tf32).
    bf16=True adds wb = bf16_rn(W): linear() then runs this weight's products on the BF16 GEMM (digat_linear_bf16)."""
    __slots__ = ('w', 'hi', 'lo', 'wb')

    def __init__(self, w, bf16=False):
        self.w = w.detach().float().contiguous()
        self.hi = self.lo = self.wb = None
        if bf16:
            if self.w.shape[0] % 16 != 0 or self.w.shape[0] > 1280 or self.w.shape[1] % 8 != 0:
                raise RuntimeError('PackedWeight: the BF16 GEMM needs N %% 16 == 0, N <= 1280, K %% 8 == 0 (got %s)'
                                   % (tuple(self.w.shape),))
            self.wb = self.w.to(torch.bfloat16)             # round to nearest even
        if self.w.shape[0] % 16 == 0 and self.w.shape[1] % 4 == 0:
            self.hi, self.lo = torch.empty_like(self.w), torch.empty_like(self.w)
            _lib.call('digat_split_tf32', self.w.data_ptr(), self.hi.data_ptr(), self.lo.data_ptr(), self.w.numel(),
                      _stream())


# rows below which the exact-fp32 CUDA-core GEMM is used (a 128-row tensor-core tile would be mostly padding)
TENSOR_CORE_MIN_ROWS = 256


def linear(A, W, bias=None, relu=False, M=None, K=None, lda=None, out=None, group_bias=None, group_rows=1,
           group_col0=0, c_rows=None):
    """out[M,N] = A[M,K] W[N,K]^T (+bias).  ``A`` may be a strided row view (pass M, K, lda explicitly).
    W: PackedWeight (tcgen05 3xTF32 GEMM when it has TF32 planes and M is large enough) or a plain fp32 tensor
    (exact-fp32 CUDA-core GEMM).  group_bias [M/group_rows, cols]: out[m, group_col0 + c] += group_bias[m // group_rows, c].
    c_rows [M] int32 ascending (tensor-core path only, ``out`` required): product row m lands in out[c_rows[m]] and takes
    the group bias of that row; the other rows of ``out`` are left untouched."""
    w = W.w if isinstance(W, PackedWeight) else W
    bf16 = isinstance(W, PackedWeight) and W.wb is not None
    if bf16 and relu:
        raise RuntimeError('linear: the BF16 GEMM has no relu epilogue')
    N = w.shape[0]
    if K is None:
        K = w.shape[1]
    if M is None:
        M = A.numel() // K
    if lda is None:
        lda = K
    if out is None:
        out = torch.empty((M, N), device=A.device, dtype=torch.float32)
    gcols = 0 if group_bias is None else group_bias.shape[1]
    gld = 0 if group_bias is None else group_bias.stride(0)
    if bf16:                                                            # every M, with or without c_rows
        _lib.call('digat_linear_bf16', A.data_ptr(), lda, W.wb.data_ptr(), W.wb.stride(0), _ptr(bias), out.data_ptr(),
                  out.stride(0), M, N, K, _ptr(group_bias), group_rows, group_col0, gcols, gld, _ptr(c_rows), _stream())
    elif c_rows is not None:
        if not (isinstance(W, PackedWeight) and W.hi is not None) or relu:
            raise RuntimeError('linear: c_rows needs a PackedWeight with TF32 planes and no relu')
        _lib.call('digat_linear_tf32x3', A.data_ptr(), lda, W.hi.data_ptr(), W.lo.data_ptr(), w.stride(0), _ptr(bias),
                  out.data_ptr(), out.stride(0), M, N, K, _ptr(group_bias), group_rows, group_col0, gcols, gld,
                  c_rows.data_ptr(), _stream())
    elif isinstance(W, PackedWeight) and W.hi is not None and M >= TENSOR_CORE_MIN_ROWS and not relu:
        _lib.call('digat_linear_tf32x3', A.data_ptr(), lda, W.hi.data_ptr(), W.lo.data_ptr(), w.stride(0), _ptr(bias),
                  out.data_ptr(), out.stride(0), M, N, K, _ptr(group_bias), group_rows, group_col0, gcols, gld, 0,
                  _stream())
    else:
        _lib.call('digat_linear_f32', A.data_ptr(), lda, w.data_ptr(), w.stride(0), _ptr(bias), out.data_ptr(),
                  out.stride(0), M, N, K, 1 if relu else 0, _ptr(group_bias), group_rows, group_col0, gcols, gld, _stream())
    return out


def build_graph_csr(adj, row_active=None, adj_index=None, G=None, transpose=False):
    """CSR records of G graphs for graph_layer_fwd(csr=...) (digat_build_graph_csr): built once per batch, reused by every
    layer and by every pair that shares the graph.  adj [*,n,n] bool (read through adj_index [G] int32 when given),
    row_active [G,n] uint8 or None.  Returns (rowptr [G,n+1] int16, meta [G,n*n] int16); with transpose=True also
    (colptr [G,n+1], cedge [G,n*n]), the column-major view the training backward walks."""
    n = adj.shape[1]
    if G is None:
        G = adj.shape[0] if adj_index is None else adj_index.shape[0]
    rowptr = torch.empty((G, n + 1), dtype=torch.int16, device=adj.device)
    meta = torch.empty((G, n * n), dtype=torch.int16, device=adj.device)
    colptr = torch.empty((G, n + 1), dtype=torch.int16, device=adj.device) if transpose else None
    cedge = torch.empty((G, n * n), dtype=torch.int16, device=adj.device) if transpose else None
    _lib.call('digat_build_graph_csr', adj.data_ptr(), _ptr(adj_index), _ptr(row_active), rowptr.data_ptr(), meta.data_ptr(),
              _ptr(colptr), _ptr(cedge), G, n, _stream())
    return (rowptr, meta, colptr, cedge) if transpose else (rowptr, meta)


def graph_layer_fwd(P, a, adj, X, drop_keep=None, drop_scale=1.0, score_out=None, alpha_out=None, relu_mask_out=None,
                    px_index=None, adj_index=None, k3=None, B=None, row_active=None, compact_out=None, row_pos=None,
                    csr=None):
    """P [B*n, 3D] = h | U | K2 with U = k3 + K1 (row-group bias of the projection GEMM).
    Indexed mode (px_index, k3): P / X are per-behaviour tables shared by B pairs, k3 [B,D] is added in-kernel.
    csr = (rowptr, meta, index or None) from build_graph_csr: the kernel loads the record instead of rebuilding it."""
    n_src, n, D = X.shape
    if B is None:
        B = n_src
    Y = torch.empty((B, n, D), device=X.device, dtype=torch.float32)
    _lib.call('digat_graph_layer_fwd', P.data_ptr(), P.stride(0), a.data_ptr(), adj.data_ptr(), X.data_ptr(),
              Y.data_ptr(), B, n, D, _ptr(drop_keep), float(drop_scale), _ptr(score_out), _ptr(alpha_out),
              _ptr(relu_mask_out), _ptr(px_index), n_src, _ptr(adj_index), _ptr(k3),
              0 if k3 is None else k3.stride(0), _ptr(row_active), _ptr(compact_out), _ptr(row_pos),
              0 if csr is None else csr[0].data_ptr(), 0 if csr is None else csr[1].data_ptr(),
              0 if csr is None else _ptr(csr[2]), _stream())
    return Y


def attention_pool_fwd(F, v, mask, resid=None, add_in=None, out=None, ldo=None, first_out=None, alpha_out=None):
    B, m, D = F.shape
    if out is None:
        out = torch.empty((B, D), device=F.device, dtype=torch.float32)
        ldo = D
    _lib.call('digat_attention_pool_fwd', F.data_ptr(), m * D, D, _ptr(resid), v.data_ptr(), v.stride(0), mask.data_ptr(),
              _ptr(add_in), out.data_ptr(), ldo, _ptr(first_out), _ptr(alpha_out), B, m, D, _stream())
    return out


class ScaledDotProductAttention(nn.Module):
    """Parameter container with the names of reference layers.py:181-191 (``K.weight``, ``Q.weight``, ``Q.bias``).
    The arithmetic (layers.py:199-206) is done by digat_attention_pool_fwd after folding K into the query."""

    def __init__(self, feature_dim: int, query_dim: int, attention_dim: int):
        super().__init__()
        self.K = nn.Linear(feature_dim, attention_dim, bias=False)
        self.Q = nn.Linear(query_dim, attention_dim, bias=True)
        self.attention_scalar = math.sqrt(float(attention_dim))

    def initialize(self):
        nn.init.xavier_uniform_(self.K.weight)
        nn.init.xavier_uniform_(self.Q.weight)
        nn.init.zeros_(self.Q.bias)


class GraphEncoder(nn.Module):
    def __init__(self, config, news_embedding_dim: int):
        super().__init__()
        self.news_graph_size = config.news_graph_size
        self.user_graph_size = config.max_history_num + config.category_num
        self.max_history_num = config.max_history_num
        self.category_num = config.category_num + 1
        self.news_embedding_dim = news_embedding_dim
        self.graph_depth = config.graph_depth
        self.attention_scalar = math.sqrt(float(self.news_embedding_dim))
        self.dropout_rate = float(config.dropout_rate)
        self.topic_node_embedding = nn.Parameter(torch.zeros([config.category_num, self.news_embedding_dim]))

    def initialize(self):
        nn.init.zeros_(self.topic_node_embedding)

    def forward(self, news_graph_embeddings, news_graph, news_graph_mask, user_news_embedding, user_graph,
                user_category_mask, user_category_indices):
        raise Exception('Function forward must be implemented at sub-class')

    def inference(self, news_graph_embeddings, news_graph, news_graph_mask, user_news_embedding, user_graph,
                  user_category_mask, user_category_indices, news_graph_context):
        raise Exception('Function inference must be implemented at sub-class')


class DIGAT(GraphEncoder):
    def __init__(self, config, news_embedding_dim: int):
        super().__init__(config, news_embedding_dim)
        D, L = self.news_embedding_dim, self.graph_depth
        if D % 4 != 0:
            raise Exception('news_embedding_dim must be a multiple of 4 for the sm_100a kernels')
        self.candidate_attention = ScaledDotProductAttention(D, D, D)
        self.news_graph_W = nn.Linear(D * 2, D, bias=True)
        self.user_news_K = nn.Linear(D, D, bias=False)
        self.user_news_Q = nn.Linear(D, D, bias=True)
        self.featureAffine = nn.Linear(D, D, bias=True)
        self.userAttention = ScaledDotProductAttention(D, D, D)
        for g in ('news', 'user'):
            setattr(self, g + '_graph_attention_W', nn.ModuleList([nn.Linear(D, D, bias=True) for _ in range(L)]))
            setattr(self, g + '_graph_attention_ffn1', nn.ModuleList([nn.Linear(D, D, bias=False) for _ in range(L)]))
            setattr(self, g + '_graph_attention_ffn2', nn.ModuleList([nn.Linear(D, D, bias=False) for _ in range(L)]))
            setattr(self, g + '_graph_attention_ffn3', nn.ModuleList([nn.Linear(D, D, bias=True) for _ in range(L)]))
            setattr(self, g + '_graph_attention_a', nn.ModuleList([nn.Linear(D, 1, bias=False) for _ in range(L)]))
        self._packed = None
        self._packed_key = None

    def invalidate_packed(self):
        """Drops the kernel-layout copy of the weights (DIGAT._weights).  The copy is keyed on (data_ptr, _version) of every
        parameter, which misses updates that do not bump ``_version``: a CUDA-graph replay of the optimizer step
        (training.GraphedTrainStep), ``param.data`` writes, NCCL broadcasts into parameter storage.  ``train()`` / ``eval()``
        call this on every mode switch, GraphedTrainStep after every replay; call it yourself after any other in-place
        update made behind autograd's back."""
        self._packed = None
        self._packed_key = None

    def train(self, mode: bool = True):
        self.invalidate_packed()          # eval after training must never see the packed weights of an earlier eval
        return super().train(mode)

    def initialize(self):
        super().initialize()
        relu_gain = nn.init.calculate_gain('relu')
        leaky_gain = nn.init.calculate_gain('leaky_relu', 0.2)
        for g in ('news', 'user'):
            for i in range(self.graph_depth):
                W = getattr(self, g + '_graph_attention_W')[i]
                nn.init.xavier_uniform_(W.weight)
                nn.init.zeros_(W.bias)
                nn.init.xavier_uniform_(getattr(self, g + '_graph_attention_a')[i].weight, gain=leaky_gain)
                for f in ('ffn1', 'ffn2', 'ffn3'):
                    nn.init.xavier_uniform_(getattr(self, g + '_graph_attention_' + f)[i].weight, gain=relu_gain)
                nn.init.zeros_(getattr(self, g + '_graph_attention_ffn3')[i].bias)
        self.candidate_attention.initialize()
        nn.init.xavier_uniform_(self.news_graph_W.weight)
        nn.init.zeros_(self.news_graph_W.bias)
        nn.init.xavier_uniform_(self.user_news_K.weight)
        nn.init.xavier_uniform_(self.user_news_Q.weight)
        nn.init.zeros_(self.user_news_Q.bias)
        nn.init.xavier_uniform_(self.featureAffine.weight, gain=relu_gain)
        nn.init.zeros_(self.featureAffine.bias)
        self.userAttention.initialize()

    # ---------------------------------------------------------------------------------- packed weights
    def _bf16_projections(self):
        """True when projection_precision selects the BF16 node projections; raises on an unknown value."""
        mode = self.projection_precision
        if mode not in ('fp32', 'bf16'):
            raise ValueError("projection_precision must be 'fp32' or 'bf16', got %r" % (mode,))
        return mode == 'bf16'

    def _weights(self):
        """Kernel-side weight layout, rebuilt only when a parameter changed (optimizer step / load_state_dict) or
        projection_precision did:
        * per layer and graph: [W; ffn1; ffn2] stacked to [3D, D] so h, K1, K2 come out of ONE projection GEMM;
        * attention K matrices transposed, so the folded query v = K^T (Q q + b) is a plain linear;
        * [user_news_Q; userAttention.Q] stacked: both queries of the user context come from one GEMM on c_n;
        * projection_precision = 'bf16': Wcat and featureAffine also carry their bf16 plane (PackedWeight.wb)."""
        bf16 = self._bf16_projections()
        params = list(self.parameters())
        key = tuple((p.data_ptr(), p._version) for p in params) + (bf16,)
        if self._packed is not None and key == self._packed_key:
            return self._packed
        dev = params[0].device
        if dev.type != 'cuda':
            raise RuntimeError('DIGAT parameters must live on a CUDA device (digat_b200 has no CPU fallback)')
        _lib.require_device(dev.index if dev.index is not None else torch.cuda.current_device())
        D = self.news_embedding_dim
        with torch.no_grad():
            w = {}
            for g in ('news', 'user'):
                for i in range(self.graph_depth):
                    W = getattr(self, g + '_graph_attention_W')[i]
                    f1 = getattr(self, g + '_graph_attention_ffn1')[i]
                    f2 = getattr(self, g + '_graph_attention_ffn2')[i]
                    f3 = getattr(self, g + '_graph_attention_ffn3')[i]
                    av = getattr(self, g + '_graph_attention_a')[i]
                    w[g, i, 'Wcat'] = PackedWeight(torch.cat([W.weight, f1.weight, f2.weight], 0).float().contiguous(),
                                                   bf16=bf16)
                    w[g, i, 'bcat'] = torch.cat([W.bias, torch.zeros(2 * D, device=dev)], 0).float().contiguous()
                    w[g, i, 'W3'] = PackedWeight(f3.weight.detach().float().contiguous())
                    w[g, i, 'b3'] = f3.bias.detach().float().contiguous()
                    w[g, i, 'a'] = av.weight.detach().float().reshape(D).contiguous()
            # attention key folded into the query: a_k = F_k . v / sqrt(D), v = K^T (Q q + b) = (K^T Q) q + K^T b.
            # The [D,D] product is formed once in fp64 and rounded to fp32 (one GEMM per context instead of two).
            def fold(K, Q):
                Kd = K.weight.detach().double()
                return (Kd.t() @ Q.weight.detach().double()).float().contiguous(), \
                       (Kd.t() @ Q.bias.detach().double()).float().contiguous()
            cand_M, cand_m = fold(self.candidate_attention.K, self.candidate_attention.Q)
            w['cand_M'], w['cand_m'] = PackedWeight(cand_M), cand_m
            w['gate_W'] = PackedWeight(self.news_graph_W.weight.detach().float().contiguous())
            w['gate_b'] = self.news_graph_W.bias.detach().float().contiguous()
            # everything the user side needs from c_n comes out of ONE GEMM: [v_topic | v_user | k3 of the next user layer]
            un_M, un_m = fold(self.user_news_K, self.user_news_Q)
            ua_M, ua_m = fold(self.userAttention.K, self.userAttention.Q)
            for j in range(self.graph_depth + 1):
                Ws, bs = [un_M, ua_M], [un_m, ua_m]
                if j < self.graph_depth:
                    f3 = self.user_graph_attention_ffn3[j]
                    Ws.append(f3.weight.detach().float())
                    bs.append(f3.bias.detach().float())
                w['uctx_W', j] = PackedWeight(torch.cat(Ws, 0).contiguous())
                w['uctx_b', j] = torch.cat(bs, 0).contiguous()
            w['fa_W'] = PackedWeight(self.featureAffine.weight.detach().float().contiguous(), bf16=bf16)
            w['fa_b'] = self.featureAffine.bias.detach().float().contiguous()
            w['topic'] = self.topic_node_embedding.detach().float().contiguous()
        self._packed, self._packed_key = w, key
        return w

    # ---------------------------------------------------------------------------------- kernels, no autograd
    def _news_ctx(self, w, X, mask, ctx_in=None):
        B, n, D = X.shape
        v = linear(X, w['cand_M'], w['cand_m'], M=B, K=D, lda=n * D)             # K^T (Q l + b), l = X[:,0,:]
        lg = torch.empty((B, 2 * D), device=X.device, dtype=torch.float32)
        attention_pool_fwd(X, v, mask, out=lg[:, D:], ldo=2 * D, first_out=lg)    # lg = [l | g]
        z = linear(lg, w['gate_W'], w['gate_b'])
        out = torch.empty((B, D), device=X.device, dtype=torch.float32)
        _lib.call('digat_news_gate_fwd', z.data_ptr(), lg.data_ptr(), _ptr(ctx_in), out.data_ptr(), B, D, _stream())
        return out

    def _user_ctx(self, w, Xu, cmask, cidx, c_n, j, ctx_in=None, src_index=None, seg_prune=None):
        """j = index of this call (0 = initial context, i+1 = after layer i).  Returns (context, k3 of user layer j or
        None).  src_index [B] int32: Xu / cidx are per-behaviour tables and row b uses entry src_index[b].
        seg_prune = (rows [M_live] int32, pos [B*S] int32) from _segment_flags / compact_flags: featureAffine runs on the topic
        embeddings the user-level attention can see only (the segment kernel writes them compactly)."""
        nu, D = Xu.shape[1], Xu.shape[2]
        B = c_n.shape[0]
        H, S = self.max_history_num, self.category_num
        vv = linear(c_n, w['uctx_W', j], w['uctx_b', j])                          # [B, 2D or 3D]
        v1, v2 = vv[:, :D], vv[:, D:2 * D]
        k3_next = vv[:, 2 * D:] if vv.shape[1] > 2 * D else None
        T = torch.empty((B, S, D), device=Xu.device, dtype=torch.float32)
        Tc = pos = None
        if seg_prune is not None:
            rows, pos = seg_prune
            Tc = torch.empty((B * S, D), device=Xu.device, dtype=torch.float32)[:rows.shape[0]]
        _lib.call('digat_topic_segment_fwd', Xu.data_ptr(), nu * D, v1.data_ptr(), vv.stride(0), cidx.data_ptr(),
                  T.data_ptr(), 0, self._err_flag(Xu.device).data_ptr(), _ptr(src_index),
                  cmask.data_ptr() if self.prune_user_nodes else 0, _ptr(Tc), _ptr(pos), B, H, S, D, _stream())
        if seg_prune is not None:                                                 # featureAffine on the visible topics only
            Fa = torch.empty((B * S, D), device=Xu.device, dtype=torch.float32)
            linear(Tc, w['fa_W'], w['fa_b'], out=Fa, c_rows=rows)                 # (the pooling never reads the other rows)
        else:
            Fa = linear(T, w['fa_W'], w['fa_b'])                                  # featureAffine(T)  [B*S, D]
        return attention_pool_fwd(Fa.view(B, S, D), v2, cmask, resid=T, add_in=ctx_in), k3_next

    def _layer(self, w, g, i, X, adj, ctx_other, k3=None, share=None, adj_index=None, prune=None, A_c=None,
               want_compact=False, csr=None, csr_last=None):
        """k3 [B,D] (possibly a column view): ffn3(context of the other graph) + bias, computed here when None.
        share [B] int32 (layer 0 of the scoring path): X [n_src,n,D] holds one graph per BEHAVIOUR and pair b uses
        graph share[b]; the projection then runs once per behaviour and k3 is added inside the fused kernel.
        prune = (row_active [B,n] uint8, rows [M_act] int32, row_pos [B*n] int32[, pooled]) from _lists: only the listed
        node rows are projected (compact operand A_c, or gathered here when it is None; scattered back into the dense P)
        and evaluated by the layer kernel.  want_compact: the layer kernel also writes the compact operand of the NEXT
        layer.  Returns (Y [B,n,D], Yc [M_act,D] or None)."""
        n, D = X.shape[1], X.shape[2]
        if k3 is None:
            k3 = linear(ctx_other, w[g, i, 'W3'], w[g, i, 'b3'])                  # [B, D]
        act, rows, pos = (None, None, None) if prune is None else prune[:3]
        kernel_act = act
        if prune is not None and len(prune) > 3 and not want_compact and share is None and i + 1 == self.graph_depth:
            kernel_act = prune[3]         # last layer: only the rows a context pools are evaluated (the rest stay neighbours)
            csr = csr_last                # (its CSR record lists those rows only)
        Yc = None
        if prune is not None and want_compact:
            # capacity = every row (M_act changes from batch to batch: a fixed size lets the caching allocator reuse the block)
            Yc = torch.empty((act.numel(), D), device=X.device, dtype=torch.float32)[:rows.shape[0]]
        if share is not None:
            P = linear(X, w[g, i, 'Wcat'], w[g, i, 'bcat'])                       # h | K1 | K2 per behaviour
            return graph_layer_fwd(P, w[g, i, 'a'], adj, X, px_index=share, adj_index=share, k3=k3, B=k3.shape[0],
                                   row_active=act, compact_out=Yc, row_pos=pos if Yc is not None else None, csr=csr), Yc
        if prune is not None:
            M = rows.shape[0]
            if A_c is None:                                                       # first layer: gather the active rows
                A_c = torch.empty((act.numel(), D), device=X.device, dtype=torch.float32)[:M]
                _lib.call('digat_gather_rows_i32', X.data_ptr(), X.shape[0] * n, rows.data_ptr(), A_c.data_ptr(), D, M, D,
                          self._err_flag(X.device).data_ptr(), _stream())
            P = torch.empty((X.shape[0] * n, w[g, i, 'Wcat'].w.shape[0]), device=X.device, dtype=torch.float32)
            linear(A_c, w[g, i, 'Wcat'], w[g, i, 'bcat'], out=P, group_bias=k3, group_rows=n, group_col0=D, c_rows=rows)
            return graph_layer_fwd(P, w[g, i, 'a'], adj, X, adj_index=adj_index, row_active=kernel_act, compact_out=Yc,
                                   row_pos=pos if Yc is not None else None, csr=csr), Yc
        P = linear(X, w[g, i, 'Wcat'], w[g, i, 'bcat'], group_bias=k3, group_rows=n, group_col0=D)   # h | k3+K1 | K2
        return graph_layer_fwd(P, w[g, i, 'a'], adj, X, adj_index=adj_index, csr=csr), None

    prune_user_nodes = True      # inference only; switch off to evaluate every node of every user graph
    # Arithmetic of the node projections at inference (the per-layer h | K1 | K2 GEMM of both graphs and featureAffine):
    # 'fp32' (3xTF32, fp32-level accuracy) or 'bf16' (operands rounded to bf16, fp32 accumulation; DESIGN.md section 4.8).
    # Every other GEMM, and the training path (autograd_ops.encode_with_grad), stays fp32 in either mode.
    projection_precision = 'fp32'
    precompute_user_csr = True   # user-graph CSR records built once per batch (build_graph_csr) instead of in every layer launch

    def _user_csr(self, Au, prune, share, first_rows):
        """CSR records of the user graphs for all layers of one batch: (csr, csr_last) for _layer.  The records follow the
        adjacency's granularity: one per behaviour when the pairs of an impression share it (share + first_rows: the first
        pair of each behaviour supplies its pruning flags -- they depend on the behaviour only), else one per row."""
        if not self.precompute_user_csr or Au.shape[1] > 128 or (share is not None and first_rows is None):
            return None, None
        pick = (lambda f: f.index_select(0, first_rows.long())) if share is not None else (lambda f: f)   # noqa: E731
        act = None if prune is None else pick(prune[0])
        csr = build_graph_csr(Au, act) + (share,)
        csr_last = csr
        if prune is not None and len(prune) > 3 and self.graph_depth > 1:
            csr_last = build_graph_csr(Au, pick(prune[3])) + (share,)
        return csr, csr_last

    # ---- pruning lists.  The flags are computed by kernels (no synchronisation); compact_flags turns any number of flag
    # arrays into index lists with ONE host synchronisation (a single nonzero() over their concatenation).
    def _user_flags(self, Au, Mc, ci, adj_index):
        """Node pruning of the user graph at inference (digat_user_active_rows): nodes that no other node attends to and
        no context pools -- in MIND-shaped data the padded history slots and the categories a user never clicked, about
        half of the 68 nodes -- cannot influence (news_ctx, user_ctx); their rows are neither projected nor evaluated.
        Au / ci may be tables read through adj_index [B] int32.  Returns (active [B,n], pooled [B,n]) uint8 or None when
        unsupported / switched off (small batches stay on the exact-fp32 GEMM, which has no row scatter)."""
        B, n = Mc.shape[0], Au.shape[1]
        if not self.prune_user_nodes or B * n < TENSOR_CORE_MIN_ROWS or \
           not _lib.load().digat_graph_layer_supports_row_active(n, self.news_embedding_dim, B):
            return None
        act = torch.empty((B, n), dtype=torch.uint8, device=Au.device)
        pooled = torch.empty((B, n), dtype=torch.uint8, device=Au.device)
        _lib.call('digat_user_active_rows', Au.data_ptr(), _ptr(adj_index), ci.data_ptr(), Mc.data_ptr(), act.data_ptr(),
                  pooled.data_ptr(), B, n, self.max_history_num, self.category_num, _stream())
        return act, pooled

    def _news_flags(self, An, Mn):
        """The same for the news graph (digat_news_active_rows): the unused BFS slots of a SAG (isolated, masked out of the
        candidate attention) are not projected."""
        B, n = Mn.shape
        if not self.prune_user_nodes or B * n < TENSOR_CORE_MIN_ROWS or \
           not _lib.load().digat_graph_layer_supports_row_active(n, self.news_embedding_dim, B):
            return None
        act = torch.empty((B, n), dtype=torch.uint8, device=An.device)
        _lib.call('digat_news_active_rows', An.data_ptr(), Mn.data_ptr(), act.data_ptr(), B, n, _stream())
        return act

    def _segment_flags(self, Mc):
        """Topic embeddings the user-level attention can see: cmask != 0, or every segment of a fully masked row (uniform
        softmax).  [B,S] bool, or None (small batch / pruning off)."""
        B, S = Mc.shape
        if not self.prune_user_nodes or B * S < TENSOR_CORE_MIN_ROWS:
            return None
        return Mc | ~Mc.any(dim=1, keepdim=True)

    @staticmethod
    def compact_begin(flag_list):
        """First half of the flag compaction: enqueue (no host synchronisation) the prefix sums over the concatenated
        flags and an asynchronous copy of the per-list counts to pinned memory, and record an event behind it.
        Returns a state for compact_finish, or None when every entry is None."""
        live = [f for f in flag_list if f is not None]
        if not live:
            return None
        flat = [f.reshape(-1).to(torch.uint8) for f in live]
        sizes = [f.shape[0] for f in flat]
        allf = torch.cat(flat) if len(flat) > 1 else flat[0]
        csum = torch.cumsum(allf, 0, dtype=torch.int32)
        ends = _ends_tensor(tuple(sizes), allf.device)
        counts_host = _pinned_ints(len(sizes))
        counts_host.copy_(csum.index_select(0, ends), non_blocking=True)
        ev = torch.cuda.Event()
        ev.record()
        return dict(flags=flag_list, sizes=sizes, allf=allf, csum=csum, counts=counts_host, event=ev)

    @staticmethod
    def compact_finish(state, n_lists=None):
        """Second half: wait for the counts (the only host synchronisation: an event recorded right behind the prefix
        sums, so it does not wait for anything enqueued afterwards) and build, with ONE launch (digat_compact_lists),
        [(ids int32 [count], pos int32 [numel]) or None, ...]: ids = flat positions of the nonzero flags, pos[r] = rank
        of position r among them (valid where the flag is set)."""
        if state is None:
            return [None] * (n_lists or 0)
        state['event'].synchronize()
        cum = state['counts'].tolist()
        _release_pinned(state['counts'])
        allf, csum, sizes = state['allf'], state['csum'], state['sizes']
        dev = allf.device
        total_set = cum[-1]
        ids_all = torch.empty(max(total_set, 1), dtype=torch.int32, device=dev)      # the lists, back to back
        pos_all = torch.empty(allf.shape[0], dtype=torch.int32, device=dev)
        out, lo, size, base, ids_p, pos_p = [], [], [], [], [], []
        k, lo_pos, b0 = 0, 0, 0
        for f in state['flags']:
            if f is None:
                out.append(None)
                continue
            count, sz = cum[k] - b0, sizes[k]
            ids, pos = ids_all[b0:b0 + count], pos_all[lo_pos:lo_pos + sz]
            out.append((ids, pos))
            lo.append(lo_pos); size.append(sz); base.append(b0)
            ids_p.append(ids_all.data_ptr() + 4 * b0); pos_p.append(pos.data_ptr())
            b0, lo_pos, k = cum[k], lo_pos + sz, k + 1
        n = len(lo)
        if n > 4:
            raise RuntimeError('compact_finish: at most four lists per call')
        pad = lambda v: v + [0] * (4 - n)
        _lib.call('digat_compact_lists', allf.data_ptr(), csum.data_ptr(), n, (ctypes.c_int64 * 4)(*pad(lo)),
                  (ctypes.c_int64 * 4)(*pad(size)), (ctypes.c_int32 * 4)(*pad(base)), (ctypes.c_void_p * 4)(*pad(ids_p)),
                  (ctypes.c_void_p * 4)(*pad(pos_p)), _stream())
        return out

    @classmethod
    def compact_flags(cls, flag_list):
        """compact_begin + compact_finish back to back (one host synchronisation)."""
        return cls.compact_finish(cls.compact_begin(flag_list), len(flag_list))

    def _lists(self, uf, nf, sf):
        """(user flags (active, pooled) | None, news flags | None, segment flags | None) -> (prune, prune_n, seg_prune)
        as consumed by _layer / _user_ctx; a list that would keep every row is dropped (None)."""
        cu, cn, cs = self.compact_flags([None if uf is None else uf[0], nf, sf])
        prune = prune_n = seg_prune = None
        if cu is not None and cu[0].shape[0] < uf[0].numel():
            prune = (uf[0], cu[0], cu[1], uf[1])        # 4th entry: the rows the user context pools (last layer)
        if cn is not None and cn[0].shape[0] < nf.numel():
            prune_n = (nf, cn[0], cn[1])
        if cs is not None and cs[0].shape[0] < sf.numel():
            seg_prune = cs
        return prune, prune_n, seg_prune

    def _err_flag(self, device):
        f = getattr(self, '_err', None)
        if f is None or f.device != device:
            f = torch.zeros(1, dtype=torch.int32, device=device)
            self._err = f
        return f

    def check_index_errors(self):
        """Raises if a kernel saw an out-of-range category index since the last check (synchronises)."""
        f = getattr(self, '_err', None)
        if f is not None and int(f.item()) != 0:
            f.zero_()
            raise RuntimeError('index out of range in user_category_indices (reference: torch_scatter raises)')

    def _user_nodes(self, w, user_news_embedding):
        B, H, D = user_news_embedding.shape
        C = w['topic'].shape[0]
        Xu = torch.empty((B, H + C, D), device=user_news_embedding.device, dtype=torch.float32)
        _lib.call('digat_build_user_nodes', 0, 0, 0, user_news_embedding.data_ptr(), w['topic'].data_ptr(),
                  Xu.data_ptr(), B, H, C, D, 0, _stream())
        return Xu

    def _check_inputs(self, news_graph_embeddings, news_graph, news_graph_mask, user_news_embedding, user_graph,
                      user_category_mask, user_category_indices):
        Xn = _f32c(news_graph_embeddings, 'news_graph_embeddings')
        Xh = _f32c(user_news_embedding, 'user_news_embedding')
        An = _boolc(news_graph, 'news_graph')
        Au = _boolc(user_graph, 'user_graph')
        Mn = _boolc(news_graph_mask, 'news_graph_mask')
        Mc = _boolc(user_category_mask, 'user_category_mask')
        if user_category_indices.dtype != torch.int64 or not user_category_indices.is_cuda:
            raise RuntimeError('user_category_indices must be a CUDA int64 tensor')
        ci = user_category_indices.contiguous()
        B = Xn.shape[0]
        if Xn.shape[1:] != (self.news_graph_size, self.news_embedding_dim) or \
           Xh.shape != (B, self.max_history_num, self.news_embedding_dim) or \
           An.shape != (B, self.news_graph_size, self.news_graph_size) or \
           Au.shape != (B, self.user_graph_size, self.user_graph_size) or \
           Mn.shape != (B, self.news_graph_size) or Mc.shape != (B, self.category_num) or \
           ci.shape != (B, self.max_history_num):
            raise RuntimeError('DIGAT: inconsistent input shapes')
        return Xn, An, Mn, Xh, Au, Mc, ci

    # ---------------------------------------------------------------------------------- reference API
    def compute_news_graph_context(self, news_graph_embeddings, news_graph_mask):
        w = self._weights()
        with torch.no_grad():
            return self._news_ctx(w, _f32c(news_graph_embeddings, 'news_graph_embeddings'),
                                  _boolc(news_graph_mask, 'news_graph_mask'))

    def compute_user_graph_context(self, user_graph_embeddings, user_category_mask, user_category_indices,
                                   news_graph_context):
        w = self._weights()
        with torch.no_grad():
            return self._user_ctx(w, _f32c(user_graph_embeddings, 'user_graph_embeddings'),
                                  _boolc(user_category_mask, 'user_category_mask'), user_category_indices.contiguous(),
                                  _f32c(news_graph_context, 'news_graph_context'), self.graph_depth)[0]

    def compute_news_graph_embeddings(self, index, news_graph_embeddings, news_graph, user_graph_context):
        w = self._weights()
        with torch.no_grad():
            return self._layer(w, 'news', index, _f32c(news_graph_embeddings, 'news_graph_embeddings'),
                               _boolc(news_graph, 'news_graph'), _f32c(user_graph_context, 'user_graph_context'))[0]

    def compute_user_graph_embeddings(self, index, user_graph_embeddings, user_graph, news_graph_context):
        w = self._weights()
        with torch.no_grad():
            return self._layer(w, 'user', index, _f32c(user_graph_embeddings, 'user_graph_embeddings'),
                               _boolc(user_graph, 'user_graph'), _f32c(news_graph_context, 'news_graph_context'))[0]

    def _encode(self, w, Xn, An, Mn, Xu, Au, Mc, ci, c_n, share=None, lists=None, first_rows=None):
        """The L-layer dual-graph schedule of graphEncoders.py:180-198 on prebuilt node tensors.
        Xu [B, H+C, D] already holds [history ; topic nodes]; c_n None = compute the initial news context.
        share [B] int32 (scoring path): Xu / Au / ci are per-BEHAVIOUR tables and pair b uses entry share[b]; the
        user graph's layer-0 projection and node build then run once per behaviour (results are bit-identical).
        lists = (prune, prune_n, seg_prune) when the caller prepared the pruning lists already (scoring.Scorer does, on a
        side stream); otherwise they are computed here (one nonzero() host synchronisation)."""
        if c_n is None:
            c_n = self._news_ctx(w, Xn, Mn)
        if lists is not None:
            prune, prune_n, seg_prune = lists
        else:
            prune, prune_n, seg_prune = self._lists(self._user_flags(Au, Mc, ci, share), self._news_flags(An, Mn),
                                                    self._segment_flags(Mc))
        c_u, k3u = self._user_ctx(w, Xu, Mc, ci, c_n, 0, src_index=share, seg_prune=seg_prune)
        csr_u, csr_u_last = self._user_csr(Au, prune, share, first_rows)
        if share is not None:
            ci = ci.index_select(0, share.long())      # [B,H] int64: from layer 1 on every pair owns its user nodes
        Ac_n = Ac_u = None                               # compact projection operands written by the previous layer
        for i in range(self.graph_depth):
            more = i + 1 < self.graph_depth
            Xn_new, Ac_n = self._layer(w, 'news', i, Xn, An, c_u, prune=prune_n, A_c=Ac_n, want_compact=more)
            Xu, Ac_u = self._layer(w, 'user', i, Xu, Au, c_n, k3=k3u, share=share if i == 0 else None,
                                   adj_index=share if i > 0 else None, prune=prune, A_c=Ac_u, want_compact=more,
                                   csr=csr_u, csr_last=csr_u_last)
            Xn = Xn_new
            c_n = self._news_ctx(w, Xn, Mn, ctx_in=c_n)
            c_u, k3u = self._user_ctx(w, Xu, Mc, ci, c_n, i + 1, ctx_in=c_u, seg_prune=seg_prune)
        return c_n, c_u

    def inference(self, news_graph_embeddings, news_graph, news_graph_mask, user_news_embedding, user_graph,
                  user_category_mask, user_category_indices, news_graph_context):
        w = self._weights()
        args = self._check_inputs(news_graph_embeddings, news_graph, news_graph_mask, user_news_embedding, user_graph,
                                  user_category_mask, user_category_indices)
        Xn, An, Mn, Xh, Au, Mc, ci = args
        with torch.no_grad():
            return self._encode(w, Xn, An, Mn, self._user_nodes(w, Xh), Au, Mc, ci,
                                _f32c(news_graph_context, 'news_graph_context'))

    def forward(self, news_graph_embeddings, news_graph, news_graph_mask, user_news_embedding, user_graph,
                user_category_mask, user_category_indices):
        args = self._check_inputs(news_graph_embeddings, news_graph, news_graph_mask, user_news_embedding, user_graph,
                                  user_category_mask, user_category_indices)
        if torch.is_grad_enabled() and (any(p.requires_grad for p in self.parameters())
                                        or news_graph_embeddings.requires_grad or user_news_embedding.requires_grad):
            from . import autograd_ops   # training path: autograd.Functions over the backward kernels
            return autograd_ops.encode_with_grad(self, *args)
        Xn, An, Mn, Xh, Au, Mc, ci = args
        w = self._weights()               # (inference branch only: the training path packs its own, differentiable, layout)
        with torch.no_grad():
            return self._encode(w, Xn, An, Mn, self._user_nodes(w, Xh), Au, Mc, ci, None)


# The reference keeps its five ablation encoders in the same module (graphEncoders.py:201-842) and model.py:20-29 looks
# them up here by name (`graphEncoders.wo_SA(...)`): resolve them lazily (PEP 562; ablation_encoders imports this module) so
# that `from digat_b200 import graphEncoders` stays a one-line swap.
_ABLATIONS = ('wo_SA', 'Seq_SA', 'wo_interaction', 'News_graph_wo_inter', 'User_graph_wo_inter')


def __getattr__(name):
    if name in _ABLATIONS:
        from . import ablation_encoders
        return getattr(ablation_encoders, name)
    raise AttributeError('module %r has no attribute %r' % (__name__, name))
