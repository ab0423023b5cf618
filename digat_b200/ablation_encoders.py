"""The five ablation graph encoders of the reference (``--graph_encoder`` = wo_SA | Seq_SA | wo_interaction |
news_graph_wo_inter | user_graph_wo_inter; reference graphEncoders.py:201-842, dispatched by model.py:20-29 and
util.py:39-50) on the same sm_100a kernels as DIGAT.  Same class names, constructor, parameter names / shapes / order
(reference checkpoints load with ``strict=True``) and public methods.

  wo_SA                (:201-295)  no news graph: the candidate's own embedding X_n[:,0] drives L user-graph layers
                                   (Eq. (8) with k3 = ffn3(candidate)), ONE user context at the end
  Seq_SA               (:298-407)  news side = one attention pooling over the SAG node sequence (compute_news_sequence_context),
                                   fixed over the layers; user side as DIGAT
  wo_interaction       (:410-548)  both graphs are vanilla GATs (e_ij = leaky_relu(a1.h_j + a2.h_i)), contexts as DIGAT
  News_graph_wo_inter  (:551-695)  news graph vanilla GAT, user graph the DIGAT layer
  User_graph_wo_inter  (:698-842)  news graph the DIGAT layer, user graph vanilla GAT

A vanilla-GAT layer is a degenerate Eq. (8): ``digat_gat_layer_fwd`` runs the edge-driven layer kernel with the edge score
formed by one add of two per-node dot products, streaming h only.  All five TRAIN through autograd_ops.encode_with_grad
(``forward`` with gradients enabled): ``wo_SA`` / ``Seq_SA`` as their own schedules of the DIGAT layer and contexts, the
vanilla-GAT layers through GATLayerFn (digat_gat_layer_train_fwd / digat_gat_layer_bwd_csr); ``inference`` is a no-grad path.  Node pruning is off here
(every node is projected and evaluated): these are not the benchmarked path."""
import torch
import torch.nn as nn

from . import _lib
from .graphEncoders import (DIGAT, GraphEncoder, PackedWeight, ScaledDotProductAttention, _boolc, _f32c, _stream, linear)


def gat_layer_fwd(h, s12, adj, X):
    """Y = relu(softmax_j(mask(leaky_relu(s12[j,0] + s12[i,1]))) h) + X   (reference graphEncoders.py:498-502)."""
    B, n, D = X.shape
    Y = torch.empty((B, n, D), device=X.device, dtype=torch.float32)
    _lib.call('digat_gat_layer_fwd', h.data_ptr(), h.stride(0), s12.data_ptr(), adj.data_ptr(), X.data_ptr(), Y.data_ptr(),
              B, n, D, _stream())
    return Y


class _AblationEncoder(DIGAT):
    NEWS_CONTEXT = True          # candidate_attention + news_graph_W (compute_news_graph_context)
    NEWS_LAYER = None            # None | 'digat' | 'gat'
    USER_LAYER = 'digat'         # 'digat' | 'gat'
    USER_K3_FROM_CONTEXT = True  # the user layer's k3 input is the running news context (False: a fixed vector, wo_SA)
    prune_user_nodes = False

    def __init__(self, config, news_embedding_dim: int):
        GraphEncoder.__init__(self, config, news_embedding_dim)
        D, L = self.news_embedding_dim, self.graph_depth
        if D % 4 != 0:
            raise Exception('news_embedding_dim must be a multiple of 4 for the sm_100a kernels')
        lin = lambda o, b: nn.ModuleList([nn.Linear(D, o, bias=b) for _ in range(L)])     # noqa: E731
        if self.NEWS_CONTEXT:
            self.candidate_attention = ScaledDotProductAttention(D, D, D)
            self.news_graph_W = nn.Linear(D * 2, D, bias=True)
        self.user_news_K = nn.Linear(D, D, bias=False)
        self.user_news_Q = nn.Linear(D, D, bias=True)
        self.featureAffine = nn.Linear(D, D, bias=True)
        self.userAttention = ScaledDotProductAttention(D, D, D)
        for g, kind in (('news', self.NEWS_LAYER), ('user', self.USER_LAYER)):       # the reference's definition order
            p = g + '_graph_attention_'
            if kind == 'digat':
                setattr(self, p + 'W', lin(D, True))
                setattr(self, p + 'ffn1', lin(D, False))
                setattr(self, p + 'ffn2', lin(D, False))
                setattr(self, p + 'ffn3', lin(D, True))
                setattr(self, p + 'a', lin(1, False))
            elif kind == 'gat':
                setattr(self, p + 'W', lin(D, True))
                setattr(self, p + 'a1', lin(1, False))
                setattr(self, p + 'a2', lin(1, False))
        self._packed = None
        self._packed_key = None

    def initialize(self):
        GraphEncoder.initialize(self)
        relu_gain = nn.init.calculate_gain('relu')
        leaky_gain = nn.init.calculate_gain('leaky_relu', 0.2)
        for g, kind in (('news', self.NEWS_LAYER), ('user', self.USER_LAYER)):
            p = g + '_graph_attention_'
            for i in range(self.graph_depth if kind else 0):
                W = getattr(self, p + 'W')[i]
                nn.init.xavier_uniform_(W.weight)
                nn.init.zeros_(W.bias)
                if kind == 'digat':
                    for f in ('ffn1', 'ffn2', 'ffn3'):
                        nn.init.xavier_uniform_(getattr(self, p + f)[i].weight, gain=relu_gain)
                    nn.init.zeros_(getattr(self, p + 'ffn3')[i].bias)
                    nn.init.xavier_uniform_(getattr(self, p + 'a')[i].weight, gain=leaky_gain)
                else:
                    nn.init.xavier_uniform_(getattr(self, p + 'a1')[i].weight, gain=leaky_gain)
                    nn.init.xavier_uniform_(getattr(self, p + 'a2')[i].weight, gain=leaky_gain)
        if self.NEWS_CONTEXT:
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
    def _weights(self):
        """Kernel-side layout of whatever this variant owns (same conventions as DIGAT._weights)."""
        if self._bf16_projections():
            raise RuntimeError("%s: projection_precision = 'bf16' is implemented for DIGAT only" % type(self).__name__)
        params = list(self.parameters())
        key = tuple((p.data_ptr(), p._version) for p in params)
        if self._packed is not None and key == self._packed_key:
            return self._packed
        dev = params[0].device
        if dev.type != 'cuda':
            raise RuntimeError('%s parameters must live on a CUDA device (digat_b200 has no CPU fallback)' % type(self).__name__)
        _lib.require_device(dev.index if dev.index is not None else torch.cuda.current_device())
        D, L = self.news_embedding_dim, self.graph_depth
        f = lambda t: t.detach().float().contiguous()                                     # noqa: E731
        with torch.no_grad():
            w = {}
            for g, kind in (('news', self.NEWS_LAYER), ('user', self.USER_LAYER)):
                p = g + '_graph_attention_'
                for i in range(L if kind else 0):
                    W = getattr(self, p + 'W')[i]
                    if kind == 'digat':
                        f1, f2, f3 = (getattr(self, p + n)[i] for n in ('ffn1', 'ffn2', 'ffn3'))
                        w[g, i, 'Wcat'] = PackedWeight(torch.cat([W.weight, f1.weight, f2.weight], 0).float().contiguous())
                        w[g, i, 'bcat'] = torch.cat([W.bias, torch.zeros(2 * D, device=dev)], 0).float().contiguous()
                        w[g, i, 'W3'] = PackedWeight(f(f3.weight))
                        w[g, i, 'b3'] = f(f3.bias)
                        w[g, i, 'a'] = f(getattr(self, p + 'a')[i].weight).reshape(D).contiguous()
                    else:
                        w[g, i, 'Wh'] = PackedWeight(f(W.weight))
                        w[g, i, 'bh'] = f(W.bias)
                        w[g, i, 'a12'] = torch.cat([getattr(self, p + 'a1')[i].weight, getattr(self, p + 'a2')[i].weight],
                                                   0).detach().float().contiguous()       # [2, D]: neighbour term, query term

            def fold(K, Q):
                Kd = K.weight.detach().double()
                return (Kd.t() @ Q.weight.detach().double()).float().contiguous(), \
                       (Kd.t() @ Q.bias.detach().double()).float().contiguous()
            if self.NEWS_CONTEXT:
                cand_M, cand_m = fold(self.candidate_attention.K, self.candidate_attention.Q)
                w['cand_M'], w['cand_m'] = PackedWeight(cand_M), cand_m
                w['gate_W'] = PackedWeight(f(self.news_graph_W.weight))
                w['gate_b'] = f(self.news_graph_W.bias)
            un_M, un_m = fold(self.user_news_K, self.user_news_Q)
            ua_M, ua_m = fold(self.userAttention.K, self.userAttention.Q)
            for j in range(L + 1):
                Ws, bs = [un_M, ua_M], [un_m, ua_m]
                if j < L and self.USER_LAYER == 'digat' and self.USER_K3_FROM_CONTEXT:
                    f3 = self.user_graph_attention_ffn3[j]
                    Ws.append(f3.weight.detach().float())
                    bs.append(f3.bias.detach().float())
                w['uctx_W', j] = PackedWeight(torch.cat(Ws, 0).contiguous())
                w['uctx_b', j] = torch.cat(bs, 0).contiguous()
            w['fa_W'] = PackedWeight(f(self.featureAffine.weight))
            w['fa_b'] = f(self.featureAffine.bias)
            w['topic'] = f(self.topic_node_embedding)
        self._packed, self._packed_key = w, key
        return w

    # ---------------------------------------------------------------------------------- layers
    def _gat(self, w, g, i, X, adj):
        """Vanilla-GAT layer (reference :494-503 / :511-520): h = W x + b, a1.h and a2.h per node, fused layer kernel."""
        B, n, D = X.shape
        h = linear(X, w[g, i, 'Wh'], w[g, i, 'bh'])                 # [B*n, D]
        s12 = linear(h, w[g, i, 'a12'])                             # [B*n, 2]  (exact-fp32 CUDA-core GEMM)
        return gat_layer_fwd(h, s12, adj, X)

    def _news_layer(self, w, i, Xn, An, c_u):
        return self._gat(w, 'news', i, Xn, An) if self.NEWS_LAYER == 'gat' else self._layer(w, 'news', i, Xn, An, c_u)[0]

    def _user_layer(self, w, i, Xu, Au, c_n, k3=None):
        return self._gat(w, 'user', i, Xu, Au) if self.USER_LAYER == 'gat' else self._layer(w, 'user', i, Xu, Au, c_n, k3=k3)[0]

    def _run(self, w, Xn, An, Mn, Xu, Au, Mc, ci, c_n):
        """The dual-graph schedule shared by wo_interaction / News_graph_wo_inter / User_graph_wo_inter (= DIGAT's,
        reference :537-548, :685-695, :832-842); c_n None = compute the initial news context (forward)."""
        if c_n is None:
            c_n = self._news_ctx(w, Xn, Mn)
        c_u, k3u = self._user_ctx(w, Xu, Mc, ci, c_n, 0)
        for i in range(self.graph_depth):
            Xn_new = self._news_layer(w, i, Xn, An, c_u)
            Xu = self._user_layer(w, i, Xu, Au, c_n, k3=k3u)
            Xn = Xn_new
            c_n = self._news_ctx(w, Xn, Mn, ctx_in=c_n)
            c_u, k3u = self._user_ctx(w, Xu, Mc, ci, c_n, i + 1, ctx_in=c_u)
        return c_n, c_u

    # ---------------------------------------------------------------------------------- reference API
    def _no_grad_only(self, *tensors):
        if torch.is_grad_enabled() and (any(p.requires_grad for p in self.parameters())
                                        or any(t.requires_grad for t in tensors)):
            raise RuntimeError('%s: this entry point is a no-grad path (run it under torch.no_grad(); training goes through '
                               'forward())' % type(self).__name__)

    def compute_news_graph_embeddings(self, index, news_graph_embeddings, news_graph, user_graph_context=None):
        w = self._weights()
        with torch.no_grad():
            return self._news_layer(w, index, _f32c(news_graph_embeddings, 'news_graph_embeddings'),
                                    _boolc(news_graph, 'news_graph'),
                                    None if user_graph_context is None else _f32c(user_graph_context, 'user_graph_context'))

    def compute_user_graph_embeddings(self, index, user_graph_embeddings, user_graph, news_graph_context=None):
        w = self._weights()
        with torch.no_grad():
            return self._user_layer(w, index, _f32c(user_graph_embeddings, 'user_graph_embeddings'),
                                    _boolc(user_graph, 'user_graph'),
                                    None if news_graph_context is None else _f32c(news_graph_context, 'news_graph_context'))

    def inference(self, news_graph_embeddings, news_graph, news_graph_mask, user_news_embedding, user_graph,
                  user_category_mask, user_category_indices, news_graph_context):
        self._no_grad_only(news_graph_embeddings, user_news_embedding)
        w = self._weights()
        Xn, An, Mn, Xh, Au, Mc, ci = self._check_inputs(news_graph_embeddings, news_graph, news_graph_mask,
                                                        user_news_embedding, user_graph, user_category_mask,
                                                        user_category_indices)
        with torch.no_grad():
            return self._run(w, Xn, An, Mn, self._user_nodes(w, Xh), Au, Mc, ci,
                             _f32c(news_graph_context, 'news_graph_context'))

    TRAIN_SCHEDULE = None        # name of the autograd_ops.encode_with_grad schedule, for the encoders that can train

    def forward(self, news_graph_embeddings, news_graph, news_graph_mask, user_news_embedding, user_graph,
                user_category_mask, user_category_indices):
        wants_grad = torch.is_grad_enabled() and (any(p.requires_grad for p in self.parameters())
                                                  or news_graph_embeddings.requires_grad or user_news_embedding.requires_grad)
        if wants_grad and self.TRAIN_SCHEDULE is not None:
            from . import autograd_ops   # training path: the DIGAT layer / context autograd nodes in this encoder's schedule
            args = self._check_inputs(news_graph_embeddings, news_graph, news_graph_mask, user_news_embedding, user_graph,
                                      user_category_mask, user_category_indices)
            return autograd_ops.encode_with_grad(self, *args, schedule=self.TRAIN_SCHEDULE)
        self._no_grad_only(news_graph_embeddings, user_news_embedding)
        w = self._weights()
        Xn, An, Mn, Xh, Au, Mc, ci = self._check_inputs(news_graph_embeddings, news_graph, news_graph_mask,
                                                        user_news_embedding, user_graph, user_category_mask,
                                                        user_category_indices)
        with torch.no_grad():
            return self._run(w, Xn, An, Mn, self._user_nodes(w, Xh), Au, Mc, ci, None)


class wo_SA(_AblationEncoder):
    """Reference graphEncoders.py:201-295: no semantic-augmented news graph."""
    NEWS_CONTEXT = False
    NEWS_LAYER = None
    USER_LAYER = 'digat'
    USER_K3_FROM_CONTEXT = False
    TRAIN_SCHEDULE = 'wo_SA'

    def compute_news_graph_context(self, news_graph_embeddings, news_graph_mask):
        raise Exception('wo_SA has no news-graph context (reference graphEncoders.py:201-295)')

    def _run(self, w, Xn, An, Mn, Xu, Au, Mc, ci, c_n):
        cand = Xn[:, 0, :].contiguous()                         # single_candidate_news_representation (:281 / :290)
        for i in range(self.graph_depth):
            Xu = self._layer(w, 'user', i, Xu, Au, cand)[0]     # k3 = ffn3_i(candidate) + b
        c_u, _ = self._user_ctx(w, Xu, Mc, ci, cand, self.graph_depth)
        return cand, c_u

    def inference(self, news_graph_embeddings, news_graph, news_graph_mask, user_news_embedding, user_graph,
                  user_category_mask, user_category_indices, news_graph_context=None):
        return self.forward(news_graph_embeddings, news_graph, news_graph_mask, user_news_embedding, user_graph,
                            user_category_mask, user_category_indices)        # the cached context is ignored (:288-295)


class Seq_SA(_AblationEncoder):
    """Reference graphEncoders.py:298-407: the SAG nodes as a sequence, pooled once."""
    NEWS_CONTEXT = True
    NEWS_LAYER = None
    USER_LAYER = 'digat'
    TRAIN_SCHEDULE = 'Seq_SA'

    def compute_news_sequence_context(self, news_graph_embeddings, news_graph_mask):
        """util.py:48 calls this instead of compute_news_graph_context (same arithmetic, reference :342-347)."""
        return DIGAT.compute_news_graph_context(self, news_graph_embeddings, news_graph_mask)

    def _run(self, w, Xn, An, Mn, Xu, Au, Mc, ci, c_n):
        if c_n is None:
            c_n = self._news_ctx(w, Xn, Mn)
        c_u, k3u = self._user_ctx(w, Xu, Mc, ci, c_n, 0)
        for i in range(self.graph_depth):
            Xu = self._layer(w, 'user', i, Xu, Au, c_n, k3=k3u)[0]
            c_u, k3u = self._user_ctx(w, Xu, Mc, ci, c_n, i + 1, ctx_in=c_u)
        return c_n, c_u


class wo_interaction(_AblationEncoder):
    """Reference graphEncoders.py:410-548: both graphs vanilla GAT."""
    NEWS_LAYER = 'gat'
    USER_LAYER = 'gat'
    TRAIN_SCHEDULE = 'digat'     # the dual-graph schedule; the layer kinds come from NEWS_LAYER / USER_LAYER


class News_graph_wo_inter(_AblationEncoder):
    """Reference graphEncoders.py:551-695."""
    NEWS_LAYER = 'gat'
    USER_LAYER = 'digat'
    TRAIN_SCHEDULE = 'digat'


class User_graph_wo_inter(_AblationEncoder):
    """Reference graphEncoders.py:698-842."""
    NEWS_LAYER = 'digat'
    USER_LAYER = 'gat'
    TRAIN_SCHEDULE = 'digat'


ENCODERS = {'DIGAT': DIGAT, 'wo_SA': wo_SA, 'Seq_SA': Seq_SA, 'wo_interaction': wo_interaction,
            'news_graph_wo_inter': News_graph_wo_inter, 'user_graph_wo_inter': User_graph_wo_inter}
