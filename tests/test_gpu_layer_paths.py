"""Every launch path of the fused Eq. (8) layer (digat_graph_layer_fwd / digat_graph_layer_bwd / digat_graph_layer_bwd_csr)
against one fp64 reference of the same operation, called through the C entry point at shapes chosen to reach each path:

  1  edge-driven kernel, one graph per CTA            graph_layer_fwd_sparse_kernel<false, false, false>
  2  edge-driven kernel, G > 1 graphs per CTA          graph_layer_fwd_sparse_kernel<false, true, false>
  3  indexed (de-duplicated) scoring                   graph_layer_fwd_sparse_kernel<true, false, false>, dense <true>
  4  node pruning (row_active, Yc / row_pos)           graph_layer_fwd_sparse_kernel<false, false, false>
  5  dense kernel, R graphs per CTA / multi-tile       graph_layer_fwd_kernel<true> / <false>
  6  training outputs (score, alpha, relu mask)        graph_layer_fwd_kernel<*>, graph_layer_fwd_sparse_kernel<false, false, true>
  7  backward, dense multi-tile and CSR                graph_layer_bwd_kernel<false>, graph_layer_bwd_sparse_kernel
  8  numerical edges (exact integer scores of |s| ~ 1e3, all-negative scores, a = 0, X = 0)
  9  memory contract (P with ldp > 3D and NaN pads, tensors inside NaN / sentinel buffers)

test_layer_cases_reach_their_kernels confirms with torch.profiler that a representative case of each path runs the
instantiation listed above, so a geometry change that moves a shape off its path fails instead of silently dropping
coverage."""
import ctypes
import re

import pytest
import torch

pytestmark = pytest.mark.gpu

TOL = 2e-6              # max|got - fp64| / max|fp64| for Y, scores and alpha (fp32 sums of <= 1024 terms)
GRAD_TOL = 5e-6         # dP, da vs fp64 autograd: <= 4e-7 measured on these inputs (B200), the softmax backward amplifies
                        # rounding with the score spread, so this is a margin over the measurement, not a general bound
SENTINEL = 0x7FC0DEAD   # a NaN bit pattern no kernel produces: untouched memory is recognised bit for bit
W = 400                 # the encoder's width; the reduced sets below also run D = 36 and 132 (D % 32, 64, 68 != 0)
NARROW = (36, 132)


# ---------------------------------------------------------------------------------------------------------------- helpers
def _lib():
    from digat_b200 import _lib as lib
    if not torch.cuda.is_available():
        pytest.fail('-m gpu tests need a CUDA device')
    lib.require_device(0)
    return lib


class _layer_mode:
    """digat_debug_set_layer_mode for the duration of a with-block (1 = dense kernel, 2 = edge-driven), reset to auto."""

    def __init__(self, mode):
        self.mode = mode

    def __enter__(self):
        _lib().call('digat_debug_set_layer_mode', self.mode)

    def __exit__(self, *exc):
        _lib().call('digat_debug_set_layer_mode', 0)


def _gen(seed):
    return torch.Generator(device='cuda').manual_seed(seed)


def _inputs(B, n, D, density, seed, special=True):
    """P = h | U | K2 [B*n, 3D], a [D], X [B,n,D], adj [B,n,n] with self-loops.  With `special`, graph 0 has only its
    self-loops, graph 1 is fully dense and graph 2 has an edge-less row (uniform softmax over the graph)."""
    g = _gen(seed)
    P = torch.randn(B * n, 3 * D, device='cuda', generator=g) * 0.5
    a = torch.randn(D, device='cuda', generator=g) * 0.1
    X = torch.randn(B, n, D, device='cuda', generator=g)
    adj = (torch.rand(B, n, n, device='cuda', generator=g) < density) | torch.eye(n, dtype=torch.bool, device='cuda')
    if special:
        if B > 0:
            adj[0] = torch.eye(n, dtype=torch.bool, device='cuda')
        if B > 1:
            adj[1] = True
        if B > 2:
            adj[2, n // 2] = False
    return P, a, X, adj


def _ptr(t):
    return 0 if t is None else t.data_ptr()


def _fwd(P, a, adj, X, Y=None, B=None, keep=None, scale=1.0, score=None, alpha=None, rmask=None, px_index=None,
         adj_index=None, k3=None, row_active=None, Yc=None, row_pos=None, csr=None):
    """digat_graph_layer_fwd with every argument exposed, Y included (the caller may place it inside a larger buffer)."""
    n_src, n, D = X.shape
    B = n_src if B is None else B
    if Y is None:
        Y = torch.empty((B, n, D), device='cuda')
    _lib().call('digat_graph_layer_fwd', P.data_ptr(), P.stride(0), a.data_ptr(), adj.data_ptr(), X.data_ptr(),
                Y.data_ptr(), B, n, D, _ptr(keep), float(scale), _ptr(score), _ptr(alpha), _ptr(rmask), _ptr(px_index),
                n_src, _ptr(adj_index), _ptr(k3), 0 if k3 is None else k3.stride(0), _ptr(row_active), _ptr(Yc),
                _ptr(row_pos), 0 if csr is None else csr[0].data_ptr(), 0 if csr is None else csr[1].data_ptr(),
                0 if csr is None else _ptr(csr[2]), torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    return Y


def _ref(P, a, adj, X, px_index=None, adj_index=None, k3=None, keep=None, scale=1.0):
    """fp64 Eq. (8) layer from the fp32 inputs, on the GPU, chunked over the batch:
        s_ij = sum_d a_d relu(U_jd + K2_id);  e = leaky_relu(s, 0.2);  alpha = softmax_j(adj ? e : -1e9)
        z = (alpha * keep * scale) h;  Y = relu(z) + X
    Graph b reads P / X of graph px_index[b] and adj of graph adj_index[b].  In indexed mode U = fl32(K1 + k3[b]): the
    kernel's rounding of the shared K1 tile, then promoted.  -> s, alpha (before dropout), z, Y; float64."""
    n_src, n, D = X.shape
    B = n_src if px_index is None else px_index.shape[0]
    dev = X.device
    src = torch.arange(B, device=dev) if px_index is None else px_index.long()
    ai = torch.arange(B, device=dev) if adj_index is None else adj_index.long()
    Pv = P[:, :3 * D].reshape(n_src, n, 3 * D)
    a64 = a.double()
    out = {'s': [], 'alpha': [], 'z': [], 'Y': []}
    chunk = max(1, (1 << 24) // (n * n * D))
    for b0 in range(0, B, chunk):
        sl = slice(b0, min(B, b0 + chunk))
        Pg = Pv[src[sl]]
        h, U, K2 = Pg[..., :D].double(), Pg[..., D:2 * D], Pg[..., 2 * D:].double()
        if k3 is not None:
            U = U + k3[sl, :D].unsqueeze(1)                                     # fp32 add, as in the kernel
        U = U.double()
        s = (torch.relu(U.unsqueeze(1) + K2.unsqueeze(2)) * a64).sum(-1)       # [b, i, j]
        e = torch.nn.functional.leaky_relu(s, 0.2).masked_fill(~adj[ai[sl]].bool(), -1e9)
        al = torch.softmax(e, dim=2)
        alt = al if keep is None else al * keep[sl].double() * scale
        z = torch.bmm(alt, h)
        out['s'].append(s)
        out['alpha'].append(al)
        out['z'].append(z)
        out['Y'].append(torch.relu(z) + X[src[sl]].double())
    return {k: torch.cat(v) for k, v in out.items()}


def _rel(got, want):
    """max|got - want| / max|want| (tests/helpers.py:rel_err), on the GPU; NaN / inf in `got` count as infinite error."""
    got = got.double()
    if not bool(torch.isfinite(got).all()):
        return float('inf')
    return float((got - want).abs().max() / want.abs().max().clamp_min(1e-30))


def _check(label, got, want, tol=TOL):
    err = _rel(got, want)
    print('%-60s rel err %.2e' % (label, err))
    assert err < tol, '%s: rel err vs fp64 %.3e (gate %.0e)' % (label, err, tol)
    return err


def _bits(t):
    return t.contiguous().view(torch.int32)


def _sentinel(*shape):
    return torch.full(shape, SENTINEL, dtype=torch.int32, device='cuda').view(torch.float32)


def _f32(x):
    return float(torch.tensor(x, dtype=torch.float32))


# -- geometry of the edge-driven kernel (pair_attention_sparse.cuh: sparse_geometry / sparse_graphs_per_cta).  The path
#    check below confirms the kernel these numbers select, so a drift between this copy and the launcher fails there.
def _sparse_smem(n, D, G):
    NB = G * n
    tile = ((NB * 32 * 4 + 1023) // 1024) * 1024 // 4
    return (4 * 2 * tile * 4 + 2 * 4 * 8 + 2 * D * 4 + NB * n * 4 + (NB + 2) * 4 + 2 * NB * n + ((NB * n + 15) & ~15)
            + 2 * NB + 4 * NB + NB + 8 + 64)


def _sm_count():
    c = ctypes.c_int(0)
    assert _lib().load().digat_device_check(ctypes.addressof(c)) == 0
    return c.value


def _graphs_per_cta(n, D, B):
    max_smem = torch.cuda.get_device_properties(0).shared_memory_per_block_optin
    budget = min(227 * 1024 // 2 - 1024, max_smem)
    slots = _sm_count() * 2
    best, best_cost, G = 1, -1, 1
    while G * n <= 128 and G <= B:
        if G > 1 and _sparse_smem(n, D, G) > budget:
            break
        cost = ((B + G - 1) // G + slots - 1) // slots * (G * n + 24)
        if best_cost < 0 or cost < best_cost:
            best, best_cost = G, cost
        G += 1
    return best


def _multi_batch(n, D, B0):
    """Smallest B >= B0 for which the launcher batches G > 1 graphs per CTA and the last CTA is partial (B % G != 0)."""
    B = B0
    while True:
        G = _graphs_per_cta(n, D, B)
        if G > 1 and B % G != 0:
            return B, G
        B += 1


# ------------------------------------------------------------------------------------------- 1. edge-driven, one graph / CTA
EDGE_N = (1, 2, 3, 5, 8, 17, 31, 32, 33, 63, 64, 65, 68, 69, 100, 120)


def _case_edge(n, D, density, B=6):
    P, a, X, adj = _inputs(B, n, D, density, seed=1000 * n + D + int(100 * density))
    assert _graphs_per_cta(n, D, B) == 1
    Y = _fwd(P, a, adj, X)
    ref = _ref(P, a, adj, X)
    err = _check('edge n=%d D=%d density=%.2f' % (n, D, density), Y, ref['Y'])
    # adjacency through adj_index from a 1-byte-misaligned base: the byte-loop copy instead of the 16-byte loads
    buf = torch.zeros(B * n * n + 32, dtype=torch.bool, device='cuda')
    adj_m = buf[1:1 + B * n * n].view(B, n, n)
    perm = torch.randperm(B, generator=_gen(n), device='cuda').to(torch.int32)
    adj_m.copy_(adj[perm.long().argsort()])                  # adj_m[perm[b]] = adj[b]
    Y2 = _fwd(P, a, adj_m, X, adj_index=perm)
    assert torch.equal(Y2, Y), 'adj_index from a misaligned base changed the result (n=%d)' % n
    return err


@pytest.mark.parametrize('density', [0.05, 0.5])
@pytest.mark.parametrize('n', EDGE_N)
def test_edge_driven_one_graph_per_cta(n, density):
    _case_edge(n, W, density)


@pytest.mark.parametrize('D', NARROW)
@pytest.mark.parametrize('n', [1, 5, 32, 33, 69, 120])
def test_edge_driven_one_graph_per_cta_narrow(n, D):
    _case_edge(n, D, 0.3)


# ------------------------------------------------------------------------------------------- 2. edge-driven, G > 1 per CTA
def _case_multi(n, D, B0):
    B, G = _multi_batch(n, D, B0)
    P, a, X, adj = _inputs(B, n, D, 0.3, seed=2000 + n + D, special=False)
    tail = (B // G) * G
    for b, row in ((G, 0), (G + 1, n // 2), (2 * G - 1, n - 1), (tail, n - 1), (B - 1, 0)):
        adj[b, row] = False                    # edge-less rows at positions 0, 1, G-1 of a CTA and in the tail CTA
    Y = _fwd(P, a, adj, X)
    ref = _ref(P, a, adj, X)
    err = _check('multi n=%d D=%d B=%d G=%d' % (n, D, B, G), Y, ref['Y'])
    Y1 = _fwd(P, a, adj, X, adj_index=torch.arange(B, dtype=torch.int32, device='cuda'))      # forces G = 1
    _check('multi n=%d D=%d vs one graph per CTA' % (n, D), Y, Y1.double())
    return err


@pytest.mark.parametrize('n,B0', [(5, 3000), (10, 3000), (19, 600), (33, 600)])
def test_edge_driven_several_graphs_per_cta(n, B0):
    _case_multi(n, W, B0)


@pytest.mark.parametrize('D', NARROW)
@pytest.mark.parametrize('n,B0', [(5, 2000), (19, 600)])
def test_edge_driven_several_graphs_per_cta_narrow(n, B0, D):
    _case_multi(n, D, B0)


def test_multi_graph_uniform_row_spans_its_own_graph():
    """The smallest case of the rule: two graphs of 5 nodes per CTA, an edge-less row in the second graph of a CTA gets
    1/5 on each node of ITS graph (not 1/10 over the CTA's block-diagonal graph)."""
    n, D = 5, W
    B, G = _multi_batch(n, D, 300)
    P, a, X, adj = _inputs(B, n, D, 0.3, seed=7, special=False)
    adj[1, 2] = False
    Y = _fwd(P, a, adj, X)
    h = P.view(B, n, 3 * D)[1, :, :D].double()
    want = torch.relu(h.mean(0)) + X[1, 2].double()
    _check('multi uniform row', Y[1, 2], want)


# ------------------------------------------------------------------------------------------- 3. indexed (shared user graphs)
def _case_indexed(n, D, dense=False, n_src=7, B=19, n_adj=5):
    g = _gen(3000 + n)
    P = torch.randn(n_src * n, 3 * D, device='cuda', generator=g) * 0.5           # h | K1 | K2 per source graph
    a = torch.randn(D, device='cuda', generator=g) * 0.1
    X = torch.randn(n_src, n, D, device='cuda', generator=g)
    adj = (torch.rand(n_adj, n, n, device='cuda', generator=g) < 0.2) | torch.eye(n, dtype=torch.bool, device='cuda')
    adj[1, n // 2] = False
    px = torch.tensor([4, 4, 0, 6, 2, 2, 2, 5, 1, 3, 6, 0, 4, 1, 5, 3, 2, 6, 0][:B], dtype=torch.int32, device='cuda')
    ai = torch.tensor([1, 3, 0, 2, 4, 1, 1, 0, 3, 2, 4, 4, 0, 1, 2, 3, 1, 0, 2][:B], dtype=torch.int32, device='cuda')
    k3buf = torch.randn(B, D + 12, device='cuda', generator=g) * 0.5                 # ldk3 = D + 12 > D
    k3buf[:, D:] = float('nan')
    k3 = k3buf[:, :D]
    ref = _ref(P, a, adj, X, px_index=px, adj_index=ai, k3=k3)
    if dense:
        with _layer_mode(1):
            Y = _fwd(P, a, adj, X, B=B, px_index=px, adj_index=ai, k3=k3)
        return _check('indexed dense n=%d D=%d' % (n, D), Y, ref['Y'])
    Y = _fwd(P, a, adj, X, B=B, px_index=px, adj_index=ai, k3=k3)
    err = _check('indexed n=%d D=%d' % (n, D), Y, ref['Y'])
    from digat_b200.graphEncoders import build_graph_csr
    uniq, inv = torch.unique(ai, return_inverse=True)
    rowptr, meta = build_graph_csr(adj, adj_index=uniq.to(torch.int32))
    Yp = _fwd(P, a, adj, X, B=B, px_index=px, adj_index=ai, k3=k3, csr=(rowptr, meta, inv.to(torch.int32)))
    assert torch.equal(Yp, Y), 'precomputed CSR (csr_index) differs from the in-kernel CSR'
    return err


@pytest.mark.parametrize('dense', [False, True], ids=['edge', 'dense'])
@pytest.mark.parametrize('n', [10, 33, 68])
def test_indexed_mode(n, dense):
    _case_indexed(n, W, dense)


# ------------------------------------------------------------------------------------------- 4. pruned rows
def _case_pruned(n, D, B, use_csr):
    P, a, X, adj = _inputs(B, n, D, 0.2, seed=4000 + n + B, special=False)
    g = _gen(4001 + n)
    act = torch.rand(B, n, device='cuda', generator=g) < 0.6
    act[0] = True
    act[1] = True                                                    # all-active graphs
    act[2] = False
    act[2, n // 2] = True                                            # a graph with a single active row
    adj &= ~(act.unsqueeze(2) & ~act.unsqueeze(1))                   # contract: no active row has an edge to a pruned node
    Y0 = _fwd(P, a, adj, X)                                          # unpruned call, clean P
    ref = _ref(P, a, adj, X)
    Pn = P.clone().view(B, n, 3 * D)
    Pn[~act] = float('nan')                                          # P rows of pruned nodes: never read
    Pn = Pn.view(B * n, 3 * D)
    M = int(act.sum())
    holes = 9
    perm = torch.randperm(M + holes, generator=g, device='cuda')
    row_pos = torch.empty(B * n, dtype=torch.int64, device='cuda')
    flat = act.view(-1)
    row_pos[flat] = perm[:M]
    row_pos[~flat] = perm[M]                                         # pruned rows point at a hole: it must stay untouched
    row_pos = row_pos.to(torch.int32)
    Y = _sentinel(B, n, D)
    Yc = _sentinel(M + holes, D)
    row_active = act.to(torch.uint8)
    csr = None
    if use_csr:
        from digat_b200.graphEncoders import build_graph_csr
        csr = (*build_graph_csr(adj, row_active=row_active), None)
    _fwd(Pn, a, adj, X, Y=Y, row_active=row_active, Yc=Yc, row_pos=row_pos, csr=csr)
    assert torch.equal(_bits(Y[act]), _bits(Y0[act])), 'active rows differ from the unpruned call'
    assert bool((_bits(Y[~act]) == SENTINEL).all()), 'a pruned row of Y was written'
    assert torch.equal(_bits(Yc[row_pos[flat].long()]), _bits(Y[act])), 'Yc[row_pos[r]] != Y[r]'
    unused = torch.ones(M + holes, dtype=torch.bool, device='cuda')
    unused[row_pos[flat].long()] = False
    assert bool((_bits(Yc[unused]) == SENTINEL).all()), 'a Yc row no active node maps to was written'
    return _check('pruned n=%d B=%d csr=%s' % (n, B, use_csr), Y[act], ref['Y'][act])


@pytest.mark.parametrize('use_csr', [False, True], ids=['in_kernel_csr', 'precomputed_csr'])
@pytest.mark.parametrize('n', [19, 68])
def test_pruned_rows(n, use_csr):
    _case_pruned(n, W, 6, use_csr)


def test_pruned_rows_several_graphs_per_cta():
    n = 19
    B, G = _multi_batch(n, W, 600)
    _case_pruned(n, W, B, False)


# ------------------------------------------------------------------------------------------- 5. dense forward
def _case_dense(n, D, B, auto=False):
    P, a, X, adj = _inputs(B, n, D, 0.3, seed=5000 + n + D)
    if auto:
        Y = _fwd(P, a, adj, X)
    else:
        with _layer_mode(1):
            Y = _fwd(P, a, adj, X)
    return _check('dense n=%d D=%d B=%d%s' % (n, D, B, ' (auto)' if auto else ''), Y, _ref(P, a, adj, X)['Y'])


@pytest.mark.parametrize('n,B,auto', [(10, 23, False), (19, 23, False), (68, 5, False), (69, 5, False),
                                      (121, 3, True), (127, 3, True), (128, 3, True)])
def test_dense_kernel(n, B, auto):
    _case_dense(n, W, B, auto)


@pytest.mark.parametrize('D', NARROW)
@pytest.mark.parametrize('n,B,auto', [(10, 23, False), (19, 23, False), (69, 3, False), (128, 2, True)])
def test_dense_kernel_narrow(n, B, auto, D):
    _case_dense(n, D, B, auto)


# ------------------------------------------------------------------------------------------- 6. training outputs
def _edges(rowptr, meta, B, n):
    """(graph, CSR position, row i, column j) of every edge of the records, in CSR order."""
    E = rowptr[:, n].int() & 0x7FFF
    on = torch.arange(n * n, device='cuda').unsqueeze(0) < E.unsqueeze(1)
    b, e = on.nonzero(as_tuple=True)
    m = meta[b, e].int()
    return b, e, (m >> 8).long(), (m & 255).long()


def _check_relu_mask(label, rmask, z):
    big = z.abs() >= 1e-6 * z.abs().max()
    bad = int((rmask.bool() != (z > 0))[big].sum())
    assert bad == 0, '%s: relu mask wrong at %d entries' % (label, bad)


def _case_train(n, D, p, edge, B=5, inputs=None):
    P, a, X, adj = inputs if inputs is not None else _inputs(B, n, D, 0.3, seed=6000 + n)
    B = X.shape[0]
    keep = (torch.rand(B, n, n, device='cuda', generator=_gen(6001 + n)) >= p) if p > 0 else None
    scale = _f32(1.0 / (1.0 - p))
    ref = _ref(P, a, adj, X, keep=keep, scale=scale)
    rmask = torch.empty(B, n, D, dtype=torch.uint8, device='cuda')
    tag = '%s train n=%d D=%d p=%.1f' % ('edge' if edge else 'dense', n, D, p)
    if edge:
        from digat_b200.graphEncoders import build_graph_csr
        assert _lib().load().digat_graph_layer_csr_training_supported(n, D) == 1
        rowptr, meta, _, _ = build_graph_csr(adj, transpose=True)
        score = torch.full((B, n * n), float('nan'), device='cuda')
        alpha = torch.full((B, n * n), float('nan'), device='cuda')
        Y = _fwd(P, a, adj, X, keep=keep, scale=scale, score=score, alpha=alpha, rmask=rmask, csr=(rowptr, meta, None))
        b, e, i, j = _edges(rowptr, meta, B, n)
        got_s, want_s = score[b, e], ref['s'][b, i, j]
        got_a, want_a = alpha[b, e], ref['alpha'][b, i, j]
    else:
        score = torch.empty(B, n, n, device='cuda')
        alpha = torch.empty(B, n, n, device='cuda')
        Y = _fwd(P, a, adj, X, keep=keep, scale=scale, score=score, alpha=alpha, rmask=rmask)
        got_s, want_s, got_a, want_a = score, ref['s'], alpha, ref['alpha']
    errs = {'Y': _check(tag + ' Y', Y, ref['Y']),
            'score': _check(tag + ' score', got_s, want_s),
            'alpha': _check(tag + ' alpha', got_a, want_a)}
    _check_relu_mask(tag, rmask, ref['z'])
    return errs, (got_s, want_s, got_a, want_a)


@pytest.mark.parametrize('edge', [False, True], ids=['dense', 'edge'])
@pytest.mark.parametrize('p', [0.0, 0.3])
@pytest.mark.parametrize('n', [7, 26, 68, 100])
def test_training_outputs(n, p, edge):
    _case_train(n, W, p, edge)


# ------------------------------------------------------------------------------------------- 7. backward
def _case_bwd(n, D, p, csr, B=3):
    from digat_b200.autograd_ops import GraphLayerFn
    from digat_b200.graphEncoders import build_graph_csr
    P, a, X, adj = _inputs(B, n, D, 0.3, seed=7000 + n + D)
    adj[min(2, B - 1), :, 0] = False                                # a node nobody attends to
    g = _gen(7001 + n)
    keep = (torch.rand(B, n, n, device='cuda', generator=g) >= p) if p > 0 else None
    scale = _f32(1.0 / (1.0 - p))
    dY = torch.randn(B, n, D, device='cuda', generator=g)
    P64, a64, X64 = (t.double().requires_grad_(True) for t in (P, a, X))
    h, U, K2 = P64.view(B, n, 3 * D).split(D, dim=2)
    s = (torch.relu(U.unsqueeze(1) + K2.unsqueeze(2)) * a64).sum(-1)
    al = torch.softmax(torch.nn.functional.leaky_relu(s, 0.2).masked_fill(~adj, -1e9), dim=2)
    if keep is not None:
        al = al * keep.double() * scale
    Y64 = torch.relu(torch.bmm(al, h)) + X64
    Y64.backward(dY.double())
    Pc, ac, Xc = (t.clone().requires_grad_(True) for t in (P, a, X))
    rec = build_graph_csr(adj, transpose=True) if csr else None
    Y = GraphLayerFn.apply(Pc, ac, adj, Xc, keep, scale, rec)
    Y.backward(dY)
    torch.cuda.synchronize()
    tag = '%s bwd n=%d D=%d p=%.1f' % ('csr' if csr else 'dense', n, D, p)
    errs = {'Y': _check(tag + ' Y', Y.detach(), Y64.detach()),
            'dP': _check(tag + ' dP', Pc.grad, P64.grad, GRAD_TOL),
            'da': _check(tag + ' da', ac.grad, a64.grad, GRAD_TOL),
            'dX': _check(tag + ' dX', Xc.grad, X64.grad, 1e-6)}
    return errs


@pytest.mark.parametrize('p', [0.0, 0.3])
@pytest.mark.parametrize('n', [69, 100, 128])
def test_dense_backward_multi_tile(n, p):
    _case_bwd(n, W, p, csr=False)


def _largest_csr_training_n(D):
    lib = _lib().load()
    n = max(k for k in range(1, 129) if lib.digat_graph_layer_csr_training_supported(k, D) == 1)
    assert n < 128, 'every n is CSR-trainable at D=%d: there is no dense fall-back to test' % D
    return n


def test_csr_backward_at_the_largest_supported_graph():
    _case_bwd(_largest_csr_training_n(W), W, 0.3, csr=True)


def test_dense_backward_one_past_the_largest_csr_graph():
    """One node past the CSR limit, digat_graph_layer_csr_training_supported says 0, the CSR backward refuses the call
    (no launch), and the dense pair that training falls back to matches fp64."""
    n = _largest_csr_training_n(W) + 1
    lib = _lib()
    assert lib.load().digat_graph_layer_csr_training_supported(n, W) == 0
    from digat_b200.graphEncoders import build_graph_csr
    B, D = 1, W
    adj = torch.ones(B, n, n, dtype=torch.bool, device='cuda')
    rowptr, meta, colptr, cedge = build_graph_csr(adj, transpose=True)
    f = torch.zeros(B * n, 3 * D, device='cuda')
    with pytest.raises(RuntimeError, match='dense'):
        lib.call('digat_graph_layer_bwd_csr', f.data_ptr(), 3 * D, f.data_ptr(), rowptr.data_ptr(), meta.data_ptr(),
                 colptr.data_ptr(), cedge.data_ptr(), f.data_ptr(), f.data_ptr(), 0, 1.0, f.data_ptr(), 0, f.data_ptr(),
                 3 * D, f.data_ptr(), 0, 0, B, n, D, torch.cuda.current_stream().cuda_stream)
    _case_bwd(n, W, 0.3, csr=False)


@pytest.mark.parametrize('D', NARROW)
@pytest.mark.parametrize('n,csr', [(69, False), (33, True)])
def test_backward_narrow(n, csr, D):
    _case_bwd(n, D, 0.3, csr)


# ------------------------------------------------------------------------------------------- 8. numerical edges
def _integer_inputs(B, n, D, a_value, seed):
    """U, K2 small integers and a = a_value (a multiple of 5): every score is an integer multiple of 5 below 2^24, exact in
    fp32 whatever the summation order, and so is leaky_relu(s) = s * 0.2f.  The kernel's scores then equal the fp64 ones
    bit for bit and only the softmax / aggregation arithmetic is left to compare."""
    g = _gen(seed)
    P = torch.randn(B * n, 3 * D, device='cuda', generator=g)
    P[:, D:] = torch.randint(-2, 3, (B * n, 2 * D), device='cuda', generator=g).float()
    a = torch.full((D,), float(a_value), device='cuda')
    X = torch.randn(B, n, D, device='cuda', generator=g)
    adj = (torch.rand(B, n, n, device='cuda', generator=g) < 0.3) | torch.eye(n, dtype=torch.bool, device='cuda')
    adj[1, n // 2] = False
    return P, a, X, adj


def _case_numeric(kind, n, D=W, B=4):
    if kind == 'zero_x':
        P, a, X, adj = _inputs(B, n, D, 0.3, seed=8000 + n)
        X = torch.zeros_like(X)
    else:
        P, a, X, adj = _integer_inputs(B, n, D, {'large': 5, 'negative': -5, 'zero_a': 0}[kind], seed=8001 + n)
    ref = _ref(P, a, adj, X)
    if kind == 'large':
        assert float(ref['s'].abs().min()) > 500              # |s| ~ 1e3: exp overflows without the max subtraction
    if kind == 'negative':
        assert float(ref['s'].max()) <= 0 and float(ref['s'].min()) < -500
    if kind in ('large', 'negative', 'zero_a'):
        assert torch.equal(ref['s'], ref['s'].float().double())
    Ys = {'edge': _fwd(P, a, adj, X)}
    with _layer_mode(1):
        Ys['dense'] = _fwd(P, a, adj, X)
    for path, Y in Ys.items():
        _check('numeric %s n=%d %s Y' % (kind, n, path), Y, ref['Y'])
        if kind == 'zero_x':                                   # Y = relu(alpha h) + 0 exactly
            clearly_negative = ref['z'] < -1e-6 * ref['z'].abs().max()
            assert bool((Y >= 0).all()) and bool((Y[clearly_negative] == 0).all())
    if n <= 109:
        for edge in (False, True):
            _, (got_s, want_s, got_a, want_a) = _case_train(n, D, 0.0, edge, inputs=(P, a, X, adj))
            if kind in ('large', 'negative', 'zero_a'):
                assert torch.equal(got_s.double(), want_s), 'exact integer scores differ'
            if kind == 'zero_a':                               # uniform weights over each row's edges: fl(1/deg)
                if edge:
                    continue
                deg = adj.sum(2, keepdim=True).float()
                deg = torch.where(deg == 0, float(n), deg)
                want = torch.where(adj | (adj.sum(2, keepdim=True) == 0), 1.0 / deg, 0.0)
                assert torch.equal(got_a, want)


@pytest.mark.parametrize('kind', ['large', 'negative', 'zero_a', 'zero_x'])
@pytest.mark.parametrize('n', [26, 68, 120])
def test_numerical_edges(kind, n):
    _case_numeric(kind, n)


# ------------------------------------------------------------------------------------------- 9. memory contract
def _case_memory(path, n, D, B, pre=5, post=7, pad=64):
    """P = columns [0, 3D) of a [rows, 3D + 64] buffer whose pad columns are NaN; P, X and Y sit in the middle of larger
    NaN (P, X) or sentinel (Y) buffers, with `pre` rows before and `post` rows after them."""
    Pc, a, Xc, adj = _inputs(B, n, D, 0.3, seed=9000 + n + D)
    R = B * n
    Pbuf = torch.full((pre + R + post, 3 * D + pad), float('nan'), device='cuda')
    Pbuf[pre:pre + R, :3 * D] = Pc
    P = Pbuf[pre:pre + R, :3 * D]
    Xbuf = torch.full((pre + R + post, D), float('nan'), device='cuda')
    Xbuf[pre:pre + R] = Xc.view(R, D)
    X = Xbuf[pre:pre + R].view(B, n, D)
    Ybuf = _sentinel(pre + R + post, D)
    Y = Ybuf[pre:pre + R].view(B, n, D)
    assert P.stride(0) == 3 * D + pad
    if path == 'dense':
        with _layer_mode(1):
            _fwd(P, a, adj, X, Y=Y)
    else:
        _fwd(P, a, adj, X, Y=Y)
    assert bool(torch.isfinite(Y).all())
    assert bool((_bits(Ybuf[:pre]) == SENTINEL).all()) and bool((_bits(Ybuf[pre + R:]) == SENTINEL).all()), \
        'rows around Y were written'
    return _check('memory %s n=%d D=%d B=%d' % (path, n, D, B), Y, _ref(P, a, adj, X)['Y'])


@pytest.mark.parametrize('D', [W, 132])
@pytest.mark.parametrize('path,n,B', [('edge', 33, 6), ('edge', 120, 3), ('multi', 10, 0), ('dense', 10, 23),
                                      ('dense', 19, 23), ('dense', 69, 3)])
def test_memory_contract(path, n, B, D):
    if path == 'multi':
        B, _ = _multi_batch(n, D, 600)
    _case_memory(path, n, D, B)


# ------------------------------------------------------------------------------------------- path check
def _kernel_name(name):
    """'...kernel<false, true>(...)' whichever way the profiler spells the template arguments: demangled with '(bool)0',
    or still mangled ('_ZN5digat...kernelILb0ELb1EEEv...')."""
    m = re.match(r'_ZN5digat\d+(\w+?)(I(?:Lb[01]E)+E)?E?v', name)
    if m:
        args = re.findall(r'Lb([01])E', m.group(2) or '')
        return m.group(1) + ('<%s>' % ', '.join('true' if x == '1' else 'false' for x in args) if args else '')
    return name.replace('(bool)0', 'false').replace('(bool)1', 'true')


def _kernels(fn):
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    return {_kernel_name(ev.name) for ev in prof.events()}


PATHS = [
    ('1 edge-driven, G = 1', lambda: _case_edge(33, W, 0.05), ['graph_layer_fwd_sparse_kernel<false, false, false>'], []),
    ('2 edge-driven, G > 1', lambda: _case_multi(10, W, 3000), ['graph_layer_fwd_sparse_kernel<false, true, false>'], []),
    ('3 indexed', lambda: _case_indexed(68, W), ['graph_layer_fwd_sparse_kernel<true, false, false>'], ['graph_layer_fwd_kernel']),
    ('3 indexed, dense', lambda: _case_indexed(68, W, dense=True), ['graph_layer_fwd_kernel<true>'],
     ['graph_layer_fwd_sparse_kernel']),
    ('4 pruned', lambda: _case_pruned(68, W, 6, False), ['graph_layer_fwd_sparse_kernel<false, false, false>'],
     ['graph_layer_fwd_kernel']),
    ('5 dense, R > 1', lambda: _case_dense(10, W, 23), ['graph_layer_fwd_kernel<true>'], ['graph_layer_fwd_sparse_kernel']),
    ('5 dense, multi-tile', lambda: _case_dense(69, W, 5), ['graph_layer_fwd_kernel<false>'], ['graph_layer_fwd_sparse_kernel']),
    ('5 dense, auto fall-back', lambda: _case_dense(121, W, 3, auto=True), ['graph_layer_fwd_kernel<false>'],
     ['graph_layer_fwd_sparse_kernel']),
    ('6 training, dense', lambda: _case_train(26, W, 0.3, False), ['graph_layer_fwd_kernel<true>'],
     ['graph_layer_fwd_sparse_kernel']),
    ('6 training, edge-driven', lambda: _case_train(26, W, 0.3, True), ['graph_layer_fwd_sparse_kernel<false, false, true>'],
     ['graph_layer_fwd_kernel']),
    ('7 backward, dense multi-tile', lambda: _case_bwd(69, W, 0.3, csr=False), ['graph_layer_bwd_kernel<false>'],
     ['graph_layer_bwd_sparse_kernel']),
    ('7 backward, CSR', lambda: _case_bwd(_largest_csr_training_n(W), W, 0.3, csr=True), ['graph_layer_bwd_sparse_kernel'],
     ['graph_layer_bwd_kernel']),
    ('9 memory, dense', lambda: _case_memory('dense', 10, W, 23), ['graph_layer_fwd_kernel<true>'], []),
]


def test_layer_cases_reach_their_kernels():
    for label, fn, want, never in PATHS:
        names = _kernels(fn)
        layer = sorted(k for k in names if 'graph_layer' in k)
        print('%-32s %s' % (label, layer))
        for w in want:
            assert any(w in k for k in names), '%s: %s did not run (ran: %s)' % (label, w, layer)
        for w in never:
            assert not any(w in k for k in names), '%s: %s ran (ran: %s)' % (label, w, layer)
