"""Training path of the sm_100a DIGAT encoder: torch.autograd.Functions whose forward AND backward are the kernels of
libdigat_sm100.so, plus ``encode_with_grad`` -- reference DIGAT.forward (graphEncoders.py:177-187) including its
dropout sites.  PyTorch only provides the autograd graph, the dropout random numbers (elementwise masks) and
trivial glue (cat / slicing / the [B,D] gate arithmetic); every contraction, the fused Eq. (8) layer and the
segment / pooling ops run in the hand-written kernels, forward and backward.

Works under DistributedDataParallel (reference trainer.py:19): parameters receive ordinary ``.grad`` tensors, so DDP's
bucketed NCCL all-reduce overlaps with this backward exactly as it does with PyTorch's own.
"""
import torch
import torch.nn.functional as F
from torch.autograd import Function

from . import _lib
from .graphEncoders import PackedWeight, _ptr, _stream, attention_pool_fwd, build_graph_csr, graph_layer_fwd, linear

# Training walks each graph's edges (CSR + transpose built once per step) instead of all n^2 pairs; False = dense kernels.
TRAIN_EDGE_DRIVEN = True


def _workspace(M, N, K, device):
    n = torch.zeros(1, dtype=torch.int64)
    _lib.call('digat_reduce_workspace_floats', M, N, K, n.data_ptr())
    return torch.empty(int(n.item()), device=device, dtype=torch.float32)


def colsum(x2d, bufs=None):
    """bufs = (out, workspace) allocated by colsum_bufs (side-stream launches), else allocated here."""
    M, N = x2d.shape
    out, ws = bufs if bufs is not None else colsum_bufs(M, N, x2d.device)
    if M == 0:
        return out.zero_()
    _lib.call('digat_colsum', x2d.data_ptr(), x2d.stride(0), out.data_ptr(), ws.data_ptr(), M, N, _stream())
    return out


def colsum_bufs(M, N, device):
    return torch.empty(N, device=device, dtype=torch.float32), _workspace(max(M, 1), N, 1, device)


# Kernel-layout copies (TF32 planes of W for the forward, of W^T for dgrad) of the weights of ONE training step.  A weight
# that feeds several GEMMs of a step -- the context projections are applied L+1 times -- is split once per direction
# instead of once per call (ADVICE r1: 1.4 ms of a 10.3 ms step were redundant splits).  encode_with_grad clears the cache
# when a step starts (the optimizer has changed the weights); entries pin their source tensor, so a pointer is never reused
# while its entry is alive.
_STEP_PLANES = {}


def _planes(W, transposed):
    key = (W.data_ptr(), tuple(W.shape), tuple(W.stride()), W._version, transposed)
    hit = _STEP_PLANES.get(key)
    if hit is None:
        hit = _STEP_PLANES[key] = (PackedWeight(W.t().contiguous() if transposed else W.contiguous()), W)
    return hit[0]


WGRAD_TC_MIN_ROWS = 2048     # shorter contractions keep the exact-fp32 CUDA-core wgrad kernel (measured faster up to M ~ 2k: no transposes)
WGRAD_SLICE = 512            # rows per split-K slice: 64 truncating accumulate steps per accumulator (DESIGN.md 4.1)


# Independent kernels of one backward node (dgrad / wgrad / bias sums) are issued on a second stream and joined before the
# node returns: in the captured training step they become parallel graph branches, so the latency-bound small products overlap
# instead of queueing behind each other.  Every buffer a side-stream kernel touches is allocated on the MAIN stream before the
# fork (the caching allocator ties a block to the stream that was current when it was allocated).
PARALLEL_BACKWARD = True
PARALLEL_BRANCHES = True     # encode_with_grad: the small-row chain (contexts, news layer) beside the user layer (second stream)
_SIDE_STREAMS = {}
_BRANCH_STREAMS = {}


class _Fork:
    """with _Fork() as f: <launches on the side stream>  ...  f.join() on the main stream."""

    def __init__(self, enabled=True):
        self.enabled = enabled and PARALLEL_BACKWARD

    def __enter__(self):
        if self.enabled:
            self.cur = torch.cuda.current_stream()
            key = (self.cur.device_index, self.cur.cuda_stream)          # one helper stream per forking stream
            side = _SIDE_STREAMS.get(key)
            if side is None:
                side = _SIDE_STREAMS[key] = torch.cuda.Stream(device=self.cur.device)
            self.side = side
            side.wait_stream(self.cur)
            self.ctx = torch.cuda.stream(side)
            self.ctx.__enter__()
        return self

    def __exit__(self, *exc):
        if self.enabled:
            self.ctx.__exit__(*exc)
        return False

    def join(self):
        if self.enabled:
            self.cur.wait_stream(self.side)


class _WgradPlan:
    """Buffers of wgrad(dC, A), allocated up front so that the launches can run on a side stream."""

    def __init__(self, M, N, K, device, force_simt=False):
        self.M, self.N, self.K = M, N, K
        self.dW = torch.empty((N, K), device=device, dtype=torch.float32)
        self.tensor_path = not (force_simt or M < WGRAD_TC_MIN_ROWS or (M & 3) != 0 or K > 1280 or (K & 15) != 0 or (N & 3) != 0)
        if not self.tensor_path:
            self.ws = _workspace(M, N, K, device)
            return
        self.dCt = torch.empty((N, M), device=device, dtype=torch.float32)
        self.At_hi = torch.empty((K, M), device=device, dtype=torch.float32)
        self.At_lo = torch.empty((K, M), device=device, dtype=torch.float32)
        self.S = (M + WGRAD_SLICE - 1) // WGRAD_SLICE
        self.out = self.dW if self.S == 1 else torch.empty((self.S, N, K), device=device, dtype=torch.float32)
        self.ws = _workspace(self.S, N * K, 1, device) if self.S > 1 else None

    def run(self, dC, A):
        M, N, K = self.M, self.N, self.K
        if not self.tensor_path:
            _lib.call('digat_linear_wgrad', dC.data_ptr(), dC.stride(0), A.data_ptr(), A.stride(0), self.dW.data_ptr(),
                      self.ws.data_ptr(), M, N, K, _stream())
            return self.dW
        _lib.call('digat_transpose_f32', dC.data_ptr(), dC.stride(0), self.dCt.data_ptr(), 0, M, M, N, _stream())
        _lib.call('digat_transpose_f32', A.data_ptr(), A.stride(0), self.At_hi.data_ptr(), self.At_lo.data_ptr(), M, M, K, _stream())
        _lib.call('digat_linear_tf32x3_splitk', self.dCt.data_ptr(), M, self.At_hi.data_ptr(), self.At_lo.data_ptr(), M,
                  self.out.data_ptr(), K, N, K, M, self.S, N * K, _stream())
        if self.S > 1:
            _lib.call('digat_colsum', self.out.data_ptr(), N * K, self.dW.data_ptr(), self.ws.data_ptr(), self.S, N * K, _stream())
        return self.dW


def wgrad(dC, A):
    """dW[N,K] = dC[M,N]^T A[M,K].  Long contractions run on the tensor cores: both operands are transposed so that the
    contraction index is contiguous (digat_transpose_f32; A^T directly as its TF32 planes), digat_linear_tf32x3_splitk writes one
    partial product per slice of WGRAD_SLICE rows and digat_colsum adds the slabs in slice order (deterministic)."""
    return _WgradPlan(A.shape[0], dC.shape[1], A.shape[1], A.device).run(dC, A)


SMALL_GEMM_ROWS = 1024       # products with at most this many rows run on the exact-fp32 CUDA-core kernel (digat_gemm_f32_small)


def _rows16(x):
    """x usable as a strided operand (unit inner stride, 16-byte aligned rows) -- else a contiguous copy."""
    if x.stride(1) == 1 and (x.stride(0) & 3) == 0 and (x.data_ptr() & 15) == 0 and x.stride(0) >= x.shape[1]:
        return x
    return x.contiguous()


def _small_gemm(L, l_trans, R, r_trans, ldr, bias, I, J, C, out=None):
    if out is None:
        out = torch.empty((I, J), device=L.device, dtype=torch.float32)
    _lib.call('digat_gemm_f32_small', L.data_ptr(), L.stride(0), int(l_trans), R.data_ptr(), ldr, int(r_trans), _ptr(bias),
              out.data_ptr(), J, I, J, C, _stream())
    return out


def _weight_layout(W):
    """W [N,K] as stored: (tensor to point at, 'nk' if rows of K are contiguous, 'kn' if W is the transposed view of a
    row-major [K,N] matrix, leading dimension).  The context keys enter as ``K.weight.t()``: no copy is made of them."""
    if W.stride(1) == 1 and (W.stride(0) & 3) == 0 and (W.data_ptr() & 15) == 0:
        return W, 'nk', W.stride(0)
    if W.stride(0) == 1 and (W.stride(1) & 3) == 0 and (W.data_ptr() & 15) == 0:
        return W, 'kn', W.stride(1)
    W = W.contiguous()
    return W, 'nk', W.stride(0)


class LinearFn(Function):
    """out = A W^T (+bias) (+row-group bias).  Few-hundred-row products (the context projections): all three directions on the
    exact-fp32 CUDA-core kernel, operands read in place.  Large ones: dA by the tcgen05 GEMM against W^T, dW by split-K."""

    @staticmethod
    def forward(ctx, A, W, bias, group_bias, group_rows, group_col0):
        M, K = A.shape
        N = W.shape[0]
        # (N < 16: the two attention columns of a vanilla-GAT layer over all node rows -- too thin for a tensor-core tile)
        ctx.small = (M <= SMALL_GEMM_ROWS or N < 16) and group_bias is None and (K & 3) == 0 and (N & 3) == 0
        ctx.has_bias = bias is not None
        ctx.group = None if group_bias is None else (group_rows, group_col0, group_bias.shape[1])
        if ctx.small:
            A = _rows16(A)
            ctx.save_for_backward(A, W)
            Wt, lay, ldw = _weight_layout(W)
            return _small_gemm(A, False, Wt, lay == 'nk', ldw, None if bias is None else bias.contiguous(), M, N, K)
        A = A.contiguous()
        ctx.save_for_backward(A, W)
        return linear(A, _planes(W, False), None if bias is None else bias.contiguous(),
                      group_bias=None if group_bias is None else group_bias.contiguous(), group_rows=group_rows,
                      group_col0=group_col0)

    @staticmethod
    def backward(ctx, dC):
        A, W = ctx.saved_tensors
        M, K = A.shape
        N = W.shape[0]
        dA = dW = db = dg = None
        want_db = ctx.has_bias and ctx.needs_input_grad[2]
        if ctx.small:
            dC = _rows16(dC)
            dev = dC.device
            tall = M > SMALL_GEMM_ROWS                                 # thin-and-tall: the contraction needs row slices
            plan = _WgradPlan(M, N, K, dev, force_simt=True) if (tall and ctx.needs_input_grad[1]) else None
            if ctx.needs_input_grad[1]:
                dW = plan.dW if plan is not None else torch.empty((N, K), device=dev, dtype=torch.float32)
            db_bufs = colsum_bufs(M, N, dev) if want_db else None
            with _Fork(ctx.needs_input_grad[0]) as side:               # weight / bias gradients beside the dgrad product
                if plan is not None:
                    plan.run(dC, A)
                elif dW is not None:
                    _small_gemm(dC, True, A, False, A.stride(0), None, N, K, M, out=dW)
                if want_db:
                    db = colsum(dC, db_bufs)
            if ctx.needs_input_grad[0]:
                Wt, lay, ldw = _weight_layout(W)
                dA = _small_gemm(dC, False, Wt, lay == 'kn', ldw, None, M, K, N)
            side.join()
            return dA, dW, db, None, None, None
        dC = dC.contiguous()
        plan = _WgradPlan(M, N, K, A.device) if ctx.needs_input_grad[1] else None
        db_bufs = colsum_bufs(M, N, A.device) if want_db else None
        with _Fork(ctx.needs_input_grad[0]) as side:
            if plan is not None:
                dW = plan.run(dC, A)
            if want_db:
                db = colsum(dC, db_bufs)
        if ctx.needs_input_grad[0]:
            dA = linear(dC, _planes(W, True))
        side.join()
        if ctx.group is not None and ctx.needs_input_grad[3]:
            rows, col0, cols = ctx.group
            dg = torch.empty((M // rows, cols), device=A.device, dtype=torch.float32)
            _lib.call('digat_groupsum', dC.data_ptr(), dC.stride(0), dg.data_ptr(), M // rows, rows, col0, cols, _stream())
        return dA, dW, db, dg, None, None


def lin(A, W, bias=None, group_bias=None, group_rows=1, group_col0=0):
    return LinearFn.apply(A, W, bias, group_bias, group_rows, group_col0)


class GraphLayerFn(Function):
    """Fused Eq. (8) layer; backward recomputes the [n,n,D] relu mask instead of storing it.  With csr = (rowptr, meta,
    colptr, cedge) from build_graph_csr(transpose=True) both directions are edge-driven (digat_graph_layer_fwd with
    per-edge score / alpha + digat_graph_layer_bwd_csr); without it the dense [B,n,n] kernels run."""

    @staticmethod
    def forward(ctx, P, a, adj, X, drop_keep, drop_scale, csr=None):
        B, n, D = X.shape
        P, a, X = P.contiguous(), a.contiguous(), X.contiguous()
        score = torch.empty((B, n, n), device=X.device, dtype=torch.float32)
        alpha = torch.empty((B, n, n), device=X.device, dtype=torch.float32)
        rmask = torch.empty((B, n, D), device=X.device, dtype=torch.uint8)
        Y = graph_layer_fwd(P, a, adj, X, drop_keep=drop_keep, drop_scale=drop_scale, score_out=score,
                            alpha_out=alpha, relu_mask_out=rmask, csr=None if csr is None else (csr[0], csr[1], None))
        ctx.save_for_backward(P, a, adj, score, alpha, rmask)
        ctx.drop = (drop_keep, float(drop_scale))
        ctx.csr = csr
        return Y

    @staticmethod
    def backward(ctx, dY):
        P, a, adj, score, alpha, rmask = ctx.saved_tensors
        keep, scale = ctx.drop
        B, n, D = rmask.shape
        dY = dY.contiguous()
        G = dY * rmask                                    # dZ = dY * 1[Z > 0]
        dP = torch.empty_like(P)
        parts = _lib.load().digat_graph_layer_bwd_csr_parts() if ctx.csr is not None else 1
        da_part = torch.empty((B * parts, D), device=P.device, dtype=torch.float32)
        if ctx.csr is not None:
            rowptr, meta, colptr, cedge = ctx.csr
            _lib.call('digat_graph_layer_bwd_csr', P.data_ptr(), P.stride(0), a.data_ptr(), rowptr.data_ptr(), meta.data_ptr(),
                      colptr.data_ptr(), cedge.data_ptr(), score.data_ptr(), alpha.data_ptr(), _ptr(keep), scale, G.data_ptr(),
                      0, dP.data_ptr(), dP.stride(0), da_part.data_ptr(), 0, 0, B, n, D, _stream())
        else:
            _lib.call('digat_graph_layer_bwd', P.data_ptr(), P.stride(0), a.data_ptr(), adj.data_ptr(), score.data_ptr(),
                      alpha.data_ptr(), _ptr(keep), scale, G.data_ptr(), dP.data_ptr(), dP.stride(0), da_part.data_ptr(),
                      B, n, D, _stream())
        return dP, colsum(da_part), None, dY, None, None, None


class ProjectedGraphLayerFn(Function):
    """One graph-attention layer as ONE autograd node: the projection P = [h | U | K2] = Xd [W; f1; f2]^T + [b; 0; 0] with
    the row-group bias k3 on U, then the fused Eq. (8) layer with residual Xd.  Fusing the two lets the edge-driven backward
    kernel hand over what the projection's backward would otherwise re-read the [B*n, 3D] gradient for: the bias gradient
    (per-graph column sums of dh) and dk3 (per-graph column sums of dU); the relu mask is applied in that kernel too."""

    @staticmethod
    def forward(ctx, Xd, W, Wb, f1w, f2w, k3, a, adj, drop_keep, drop_scale, csr):
        B, n, D = Xd.shape
        Xd = Xd.contiguous()
        Wcat = torch.cat([W, f1w, f2w], 0)
        bcat = torch.cat([Wb, Wb.new_zeros(2 * D)], 0)
        a = a.contiguous()
        P = linear(Xd.view(B * n, D), _planes(Wcat, False), bcat, group_bias=k3.contiguous(), group_rows=n, group_col0=D)
        score = torch.empty((B, n, n), device=Xd.device, dtype=torch.float32)
        alpha = torch.empty((B, n, n), device=Xd.device, dtype=torch.float32)
        rmask = torch.empty((B, n, D), device=Xd.device, dtype=torch.uint8)
        Y = graph_layer_fwd(P, a, adj, Xd, drop_keep=drop_keep, drop_scale=drop_scale, score_out=score, alpha_out=alpha,
                            relu_mask_out=rmask, csr=None if csr is None else (csr[0], csr[1], None))
        ctx.save_for_backward(Xd, Wcat, P, a, adj, score, alpha, rmask)
        ctx.drop = (drop_keep, float(drop_scale))
        ctx.csr = csr
        return Y

    @staticmethod
    def backward(ctx, dY):
        Xd, Wcat, P, a, adj, score, alpha, rmask = ctx.saved_tensors
        keep, scale = ctx.drop
        B, n, D = Xd.shape
        dev = Xd.device
        dY = dY.contiguous()
        dP = torch.empty_like(P)
        parts = _lib.load().digat_graph_layer_bwd_csr_parts() if ctx.csr is not None else 1
        da_part = torch.empty((B * parts, D), device=dev, dtype=torch.float32)
        if ctx.csr is not None:
            rowptr, meta, colptr, cedge = ctx.csr
            dh_sum = torch.empty((B * parts, D), device=dev, dtype=torch.float32)     # per-warp partials (see the header)
            du_sum = torch.empty((B * parts, D), device=dev, dtype=torch.float32)
            _lib.call('digat_graph_layer_bwd_csr', P.data_ptr(), P.stride(0), a.data_ptr(), rowptr.data_ptr(), meta.data_ptr(),
                      colptr.data_ptr(), cedge.data_ptr(), score.data_ptr(), alpha.data_ptr(), _ptr(keep), scale, dY.data_ptr(),
                      rmask.data_ptr(), dP.data_ptr(), dP.stride(0), da_part.data_ptr(), dh_sum.data_ptr(), du_sum.data_ptr(),
                      B, n, D, _stream())
            dWb = colsum(dh_sum)
            dk3 = torch.empty((B, D), device=dev, dtype=torch.float32)
            _lib.call('digat_groupsum', du_sum.data_ptr(), D, dk3.data_ptr(), B, parts, 0, D, _stream())
        else:
            G = dY * rmask
            _lib.call('digat_graph_layer_bwd', P.data_ptr(), P.stride(0), a.data_ptr(), adj.data_ptr(), score.data_ptr(),
                      alpha.data_ptr(), _ptr(keep), scale, G.data_ptr(), dP.data_ptr(), dP.stride(0), da_part.data_ptr(),
                      B, n, D, _stream())
            dWb = colsum(dP[:, :D])
            dk3 = torch.empty((B, D), device=dev, dtype=torch.float32)
            _lib.call('digat_groupsum', dP.data_ptr(), dP.stride(0), dk3.data_ptr(), B, n, D, D, _stream())
        plan = _WgradPlan(B * n, 3 * D, D, dev)
        da_bufs = colsum_bufs(B * parts, D, dev)
        with _Fork() as side:                                          # weight gradients beside the dgrad product
            dWcat = plan.run(dP, Xd.view(B * n, D))
            da = colsum(da_part, da_bufs)
        dXd = linear(dP, _planes(Wcat, True)).view(B, n, D)
        dXd += dY                                                      # the residual path
        side.join()
        return dXd, dWcat[:D], dWb, dWcat[D:2 * D], dWcat[2 * D:], dk3, da, None, None, None, None


class GATLayerFn(Function):
    """Vanilla-GAT layer of the ablation encoders (reference graphEncoders.py:494-503): Y = relu(softmax(mask(leaky_relu(s1_j +
    s2_i))) h) + X, edge-driven both ways (digat_gat_layer_train_fwd / digat_gat_layer_bwd_csr).  s12 [B*n, >=2]: column 0 =
    a1.h (neighbour term), column 1 = a2.h (query term); wider inputs (zero-padded weights) are read through their first two."""

    @staticmethod
    def forward(ctx, h, s12, adj, X, drop_keep, drop_scale, csr):
        B, n, D = X.shape
        h, X = h.contiguous(), X.contiguous()
        s2 = s12[:, :2].contiguous()
        score = torch.empty((B, n * n), device=X.device, dtype=torch.float32)
        alpha = torch.empty((B, n * n), device=X.device, dtype=torch.float32)
        rmask = torch.empty((B, n, D), device=X.device, dtype=torch.uint8)
        Y = torch.empty((B, n, D), device=X.device, dtype=torch.float32)
        _lib.call('digat_gat_layer_train_fwd', h.data_ptr(), h.stride(0), s2.data_ptr(), adj.data_ptr(), X.data_ptr(), Y.data_ptr(),
                  B, n, D, _ptr(drop_keep), float(drop_scale), score.data_ptr(), alpha.data_ptr(), rmask.data_ptr(),
                  csr[0].data_ptr(), csr[1].data_ptr(), _stream())
        ctx.save_for_backward(h, score, alpha, rmask)
        ctx.extra = (drop_keep, float(drop_scale), csr, s12.shape[1], (B, n, D))
        return Y

    @staticmethod
    def backward(ctx, dY):
        h, score, alpha, rmask = ctx.saved_tensors
        keep, scale, csr, s_cols, (B, n, D) = ctx.extra
        dY = dY.contiguous()
        dh = torch.empty_like(h)
        ds12 = torch.zeros((B * n, s_cols), device=h.device, dtype=torch.float32)
        ds2 = ds12 if s_cols == 2 else torch.empty((B * n, 2), device=h.device, dtype=torch.float32)
        rowptr, meta, colptr, cedge = csr
        _lib.call('digat_gat_layer_bwd_csr', h.data_ptr(), h.stride(0), rowptr.data_ptr(), meta.data_ptr(), colptr.data_ptr(),
                  cedge.data_ptr(), score.data_ptr(), alpha.data_ptr(), _ptr(keep), scale, dY.data_ptr(), rmask.data_ptr(),
                  dh.data_ptr(), dh.stride(0), ds2.data_ptr(), B, n, D, _stream())
        if s_cols != 2:
            ds12[:, :2] = ds2
        return dh, ds12, None, dY, None, None, None


class AttentionPoolFn(Function):
    @staticmethod
    def forward(ctx, Fm, v, mask, resid):
        Fm, v = Fm.contiguous(), v.contiguous()
        resid = None if resid is None else resid.contiguous()
        B, m, D = Fm.shape
        alpha = torch.empty((B, m), device=Fm.device, dtype=torch.float32)
        out = attention_pool_fwd(Fm, v, mask, resid=resid, alpha_out=alpha)
        ctx.save_for_backward(Fm, v, mask, alpha, *(() if resid is None else (resid,)))
        ctx.has_resid = resid is not None
        return out

    @staticmethod
    def backward(ctx, dout):
        Fm, v, mask, alpha = ctx.saved_tensors[:4]
        resid = ctx.saved_tensors[4] if ctx.has_resid else None
        B, m, D = Fm.shape
        dout = dout.contiguous()
        dF = torch.empty_like(Fm)
        dres = torch.empty_like(Fm) if resid is not None else None
        dv = torch.empty_like(v)
        _lib.call('digat_attention_pool_bwd', Fm.data_ptr(), m * D, D, _ptr(resid), v.data_ptr(), mask.data_ptr(),
                  alpha.data_ptr(), dout.data_ptr(), dout.stride(0), dF.data_ptr(), _ptr(dres), dv.data_ptr(), B, m, D,
                  _stream())
        return dF, dv, None, dres


class NewsGateFn(Function):
    """ctx_out = ctx_in + sigmoid(z) * l + (1 - sigmoid(z)) * g with lg = [l | g]  (graphEncoders.py:112-113, 185): one kernel
    each way instead of sigmoid / mul / rsub / mul / add / add and their autograd nodes."""

    @staticmethod
    def forward(ctx, z, lg, ctx_in):
        z, lg = z.contiguous(), lg.contiguous()
        B, D = z.shape
        out = torch.empty((B, D), device=z.device, dtype=torch.float32)
        _lib.call('digat_news_gate_fwd', z.data_ptr(), lg.data_ptr(), 0 if ctx_in is None else ctx_in.contiguous().data_ptr(),
                  out.data_ptr(), B, D, _stream())
        ctx.save_for_backward(z, lg)
        ctx.has_ctx = ctx_in is not None
        return out

    @staticmethod
    def backward(ctx, dout):
        z, lg = ctx.saved_tensors
        B, D = z.shape
        dout = dout.contiguous()
        dz = torch.empty_like(z)
        dlg = torch.empty_like(lg)
        _lib.call('digat_news_gate_bwd', z.data_ptr(), lg.data_ptr(), dout.data_ptr(), dz.data_ptr(), dlg.data_ptr(), B, D,
                  _stream())
        return dz, dlg, dout if ctx.has_ctx else None


class TopicSegmentFn(Function):
    @staticmethod
    def forward(ctx, Xu, v, cidx, H, S, err_flag):
        Xu, v = Xu.contiguous(), v.contiguous()
        B, nu, D = Xu.shape
        T = torch.empty((B, S, D), device=Xu.device, dtype=torch.float32)
        alpha = torch.empty((B, H), device=Xu.device, dtype=torch.float32)
        _lib.call('digat_topic_segment_fwd', Xu.data_ptr(), nu * D, v.data_ptr(), D, cidx.data_ptr(), T.data_ptr(),
                  alpha.data_ptr(), err_flag.data_ptr(), 0, 0, 0, 0, B, H, S, D, _stream())
        ctx.save_for_backward(Xu, v, cidx, alpha)
        ctx.dims = (H, S)
        return T

    @staticmethod
    def backward(ctx, dT):
        Xu, v, cidx, alpha = ctx.saved_tensors
        H, S = ctx.dims
        B, nu, D = Xu.shape
        dT = dT.contiguous()
        dXu = torch.empty_like(Xu)
        dv = torch.empty_like(v)
        _lib.call('digat_topic_segment_bwd', Xu.data_ptr(), nu * D, v.data_ptr(), cidx.data_ptr(), alpha.data_ptr(),
                  dT.data_ptr(), dXu.data_ptr(), dv.data_ptr(), B, H, S, nu, D, _stream())
        return dXu, dv, None, None, None, None


def encode_with_grad(enc, Xn, An, Mn, Xh, Au, Mc, ci, schedule='digat'):
    """Reference DIGAT.forward (graphEncoders.py:177-187) with autograd; dropout active iff enc.training.
    schedule: 'digat' (the dual-graph schedule), or one of the two ablations built from the same pieces --
    'wo_SA' (graphEncoders.py:277-284: the candidate's own embedding drives L user layers, one user context at the end) and
    'Seq_SA' (:388-396: a fixed news-sequence context, user layers and contexts as DIGAT).
    Every GEMM here is fp32 (3xTF32 or exact): enc.projection_precision applies to the no-grad inference paths only."""
    D, L, H, S = enc.news_embedding_dim, enc.graph_depth, enc.max_history_num, enc.category_num
    p = enc.dropout_rate if enc.training else 0.0
    B = Xn.shape[0]
    dev = Xn.device
    _lib.require_device(dev.index if dev.index is not None else torch.cuda.current_device())
    err = enc._err_flag(dev)
    _STEP_PLANES.clear()

    def drop(x, rate):
        return F.dropout(x, rate, True) if rate > 0 else x

    # differentiable packing of the parameters (same layout as DIGAT._weights)
    cand, ua = getattr(enc, 'candidate_attention', None), enc.userAttention          # (wo_SA has no news context)
    cand_Kt = None if cand is None else cand.K.weight.t()
    ua_Kt, un_Kt = ua.K.weight.t(), enc.user_news_K.weight.t()
    uq_W = torch.cat([enc.user_news_Q.weight, ua.Q.weight], 0)
    uq_b = torch.cat([enc.user_news_Q.bias, ua.Q.bias], 0)

    def news_ctx(X, c_prev=None):
        """c_prev + gated news context (graphEncoders.py:104-113, 185)."""
        l = X[:, 0, :]
        q = lin(l, cand.Q.weight, cand.Q.bias)
        v = lin(q, cand_Kt)
        g = AttentionPoolFn.apply(X, v, Mn, None)
        lg = torch.cat([l, g], 1)
        z = drop(lin(lg, enc.news_graph_W.weight, enc.news_graph_W.bias), p / 2)
        return NewsGateFn.apply(z, lg, c_prev)

    def user_ctx(Xu, c_n):
        qq = lin(c_n, uq_W, uq_b)
        v1 = lin(qq[:, :D], un_Kt)
        v2 = lin(qq[:, D:], ua_Kt)
        T = TopicSegmentFn.apply(Xu, v1, ci, H, S, err)
        Fa = lin(T.reshape(B * S, D), enc.featureAffine.weight, enc.featureAffine.bias).view(B, S, D)
        if p > 0:
            return AttentionPoolFn.apply(drop(torch.relu(Fa) + T, p), v2, Mc, None)
        return AttentionPoolFn.apply(Fa, v2, Mc, T)

    def train_csr(adj):
        n = adj.shape[1]
        if not TRAIN_EDGE_DRIVEN or not _lib.load().digat_graph_layer_csr_training_supported(n, D):
            return None
        return build_graph_csr(adj, transpose=True)

    main = torch.cuda.current_stream()
    branch = None
    if PARALLEL_BRANCHES:
        branch = _BRANCH_STREAMS.get(main.device_index)
        if branch is None:
            branch = _BRANCH_STREAMS[main.device_index] = torch.cuda.Stream(device=main.device)
    # CSR + transpose of both graph families, once per step (every layer walks the same edges); on the second stream they are
    # built beside the initial contexts
    if schedule != 'digat':
        branch = None
        csr_of = {'user': train_csr(Au)}
    elif branch is None:
        csr_of = {'news': train_csr(An), 'user': train_csr(Au)}
    else:
        branch.wait_stream(main)
        with torch.cuda.stream(branch):
            csr_of = {'news': train_csr(An), 'user': train_csr(Au)}
        for c in csr_of.values():
            for t in (c or ()):
                t.record_stream(main)

    def layer(g, i, X, adj, ctx_other):
        n = X.shape[1]
        W = getattr(enc, g + '_graph_attention_W')[i]
        f1 = getattr(enc, g + '_graph_attention_ffn1')[i]
        f2 = getattr(enc, g + '_graph_attention_ffn2')[i]
        f3 = getattr(enc, g + '_graph_attention_ffn3')[i]
        av = getattr(enc, g + '_graph_attention_a')[i]
        Xd = drop(X, p / 2)                                        # the residual uses the DROPPED input (:145,153)
        k3 = lin(ctx_other, f3.weight, f3.bias)
        keep = (torch.rand((B, n, n), device=dev) >= p) if p > 0 else None
        return ProjectedGraphLayerFn.apply(Xd, W.weight, W.bias, f1.weight, f2.weight, k3, av.weight.reshape(D), adj, keep,
                                           1.0 / (1.0 - p) if p > 0 else 1.0, csr_of[g])

    def gat_layer(g, i, X, adj, ctx_other=None):
        """Vanilla-GAT layer (reference :494-503 / :511-520): h = W x + b, s1 = a1.h, s2 = a2.h per node, edge-driven layer."""
        n = X.shape[1]
        W = getattr(enc, g + '_graph_attention_W')[i]
        a1 = getattr(enc, g + '_graph_attention_a1')[i]
        a2 = getattr(enc, g + '_graph_attention_a2')[i]
        if csr_of[g] is None:
            raise RuntimeError('vanilla-GAT training needs the edge-driven kernels (graph of %d nodes does not fit)' % n)
        Xd = drop(X, p / 2)
        h = lin(Xd.reshape(B * n, D), W.weight, W.bias)
        a12 = torch.cat([a1.weight, a2.weight, a1.weight.new_zeros((2, D))], 0)       # [4, D]: zero rows keep the GEMM shapes legal
        s12 = lin(h, a12)
        keep = (torch.rand((B, n, n), device=dev) >= p) if p > 0 else None
        return GATLayerFn.apply(h, s12, adj, Xd, keep, 1.0 / (1.0 - p) if p > 0 else 1.0, csr_of[g])

    news_layer = gat_layer if getattr(enc, 'NEWS_LAYER', 'digat') == 'gat' else layer
    user_layer = gat_layer if getattr(enc, 'USER_LAYER', 'digat') == 'gat' else layer

    if schedule != 'digat':                                        # single-graph ablations: sequential on the current stream
        topic = drop(enc.topic_node_embedding.unsqueeze(0).expand(B, -1, -1), p / 2)
        Xu = torch.cat([Xh, topic], 1)
        if schedule == 'wo_SA':
            cand_vec = Xn[:, 0, :]
            for i in range(L):
                Xu = layer('user', i, Xu, Au, cand_vec)
            return cand_vec, user_ctx(Xu, cand_vec)
        if schedule != 'Seq_SA':
            raise ValueError('unknown schedule %r' % (schedule,))
        c_n = news_ctx(Xn)                                          # compute_news_sequence_context: the same gate (:342-347)
        c_u = user_ctx(Xu, c_n)
        for i in range(L):
            Xu = layer('user', i, Xu, Au, c_n)
            c_u = c_u + user_ctx(Xu, c_n)
        return c_n, c_u
    topic = drop(enc.topic_node_embedding.unsqueeze(0).expand(B, -1, -1), p / 2)
    Xu = torch.cat([Xh, topic], 1)
    c_n = news_ctx(Xn)
    c_u = user_ctx(Xu, c_n)
    if branch is not None:
        main.wait_stream(branch)                                   # the CSR records
    if branch is None:
        for i in range(L):
            Xn_new = news_layer('news', i, Xn, An, c_u)
            Xu = user_layer('user', i, Xu, Au, c_n)
            Xn = Xn_new
            c_n = news_ctx(Xn, c_n)
            c_u = c_u + user_ctx(Xu, c_n)
        return c_n, c_u
    # Two streams.  The user layer of iteration i (tens of thousands of rows: the big GEMMs and the layer kernel) needs only
    # X_u and c_n of iteration i; everything else -- the user context of the previous iteration's outputs, the news layer that
    # needs it, the news context -- is a chain of small, latency-bound launches (a few hundred or thousand rows) that runs
    # beside it on a second stream.  Autograd replays each node on its forward stream, so the backward forks the same way, and
    # in the captured step the two become parallel graph branches.  Same arithmetic as the sequential order above.
    for i in range(L):
        branch.wait_stream(main)
        with torch.cuda.stream(branch):
            if i > 0:
                c_u = c_u + user_ctx(Xu, c_n)                      # context of the previous iteration's user graph
            Xn_new = news_layer('news', i, Xn, An, c_u)
            c_n_new = news_ctx(Xn_new, c_n)
        Xu_new = user_layer('user', i, Xu, Au, c_n)
        main.wait_stream(branch)
        for t in (Xn_new, c_n_new, c_u):
            t.record_stream(main)
        Xu_new.record_stream(branch)
        Xn, c_n, Xu = Xn_new, c_n_new, Xu_new
    c_u = c_u + user_ctx(Xu, c_n)
    return c_n, c_u
