"""GPU tests of the tcgen05 3xTF32 projection GEMM against fp64 (and against the exact-fp32 CUDA-core GEMM)."""
import numpy as np
import pytest
import torch

from tests.helpers import rel_err

pytestmark = pytest.mark.gpu


def _split(W):
    from digat_b200 import _lib
    hi, lo = torch.empty_like(W), torch.empty_like(W)
    _lib.call('digat_split_tf32', W.data_ptr(), hi.data_ptr(), lo.data_ptr(), W.numel(),
              torch.cuda.current_stream().cuda_stream)
    return hi, lo


def _tf32x3(A, W, bias, lda=None):
    from digat_b200 import _lib
    M, K = A.shape
    N = W.shape[0]
    hi, lo = _split(W)
    C = torch.full((M, N), float('nan'), device=A.device)
    _lib.call('digat_linear_tf32x3', A.data_ptr(), lda or A.stride(0), hi.data_ptr(), lo.data_ptr(), W.stride(0),
              0 if bias is None else bias.data_ptr(), C.data_ptr(), N, M, N, K, 0, 1, 0, 0, 0, 0,
              torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    return C


def test_split_planes_are_exact_tf32():
    g = torch.Generator().manual_seed(0)
    W = (torch.randn(1200, 400, generator=g) * 0.1).cuda()
    hi, lo = _split(W)
    torch.cuda.synchronize()
    assert int((hi.view(torch.int32) & 0x1FFF).abs().max()) == 0 and int((lo.view(torch.int32) & 0x1FFF).abs().max()) == 0
    # hi + lo reproduces W to 2^-22 relative
    assert float(((hi.double() + lo.double() - W.double()).abs() / W.double().abs().clamp_min(1e-30)).max()) < 2 ** -21


@pytest.mark.parametrize('M,N,K', [(128, 240, 16), (128, 80, 400), (256, 1200, 400), (1000, 400, 400),
                                   (4096, 400, 800), (20000, 1200, 400), (69632, 1200, 400), (16385, 800, 400),
                                   (20000, 640, 400), (20000, 1440, 400)])
def test_tf32x3_matches_fp64(M, N, K):
    g = torch.Generator().manual_seed(M + N + K)
    A = torch.randn(M, K, generator=g)
    W = torch.randn(N, K, generator=g) * 0.05
    bias = torch.randn(N, generator=g)
    C = _tf32x3(A.cuda(), W.cuda(), bias.cuda()).cpu()
    assert torch.isfinite(C).all()
    # row-sampled fp64 reference (full fp64 GEMM of the largest case is slow on the host)
    rows = torch.randperm(M, generator=g)[:min(M, 512)]
    rows = torch.cat([rows, torch.tensor([0, M - 1])])
    ref = A[rows].double() @ W.double().t() + bias.double()
    e = rel_err(C[rows].numpy(), ref.numpy())
    ref32 = (A[rows] @ W.t() + bias)
    e32 = rel_err(ref32.numpy(), ref.numpy())
    assert e < 4e-6, "tf32x3 rel err %.3e (torch fp32 on CPU: %.3e)" % (e, e32)


def test_tf32x3_strided_A_and_no_bias():
    g = torch.Generator().manual_seed(4)
    X = torch.randn(300, 10, 400, generator=g).cuda()       # A = X[:, 0, :] with lda = 10*400
    W = (torch.randn(400, 400, generator=g) * 0.05).cuda()
    from digat_b200 import _lib
    hi, lo = _split(W)
    C = torch.empty(300, 400, device='cuda')
    _lib.call('digat_linear_tf32x3', X.data_ptr(), 4000, hi.data_ptr(), lo.data_ptr(), 400, 0, C.data_ptr(), 400,
              300, 400, 400, 0, 1, 0, 0, 0, 0, torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    ref = X[:, 0, :].double().cpu() @ W.double().cpu().t()
    assert rel_err(C.cpu().numpy(), ref.numpy()) < 2e-6


@pytest.mark.parametrize('M,n', [(680, 68), (100, 10), (5440, 68)])
def test_group_bias_folds_k3_into_K1_block(M, n):
    """U = fl(k3 + K1): the row-group bias of both GEMMs (tensor-core path for M >= 256, CUDA-core path below)."""
    from digat_b200.graphEncoders import PackedWeight, linear
    g = torch.Generator().manual_seed(M)
    D = 400
    X = torch.randn(M, D, generator=g).cuda()
    W = (torch.randn(3 * D, D, generator=g) * 0.05).cuda()
    bias = torch.randn(3 * D, generator=g).cuda()
    k3 = torch.randn(M // n, D, generator=g).cuda()
    base = linear(X, PackedWeight(W), bias)
    out = linear(X, PackedWeight(W), bias, group_bias=k3, group_rows=n, group_col0=D)
    torch.cuda.synchronize()
    expect = base.clone()
    expect[:, D:2 * D] = base[:, D:2 * D] + k3.repeat_interleave(n, 0)       # exactly one fp32 add
    assert torch.equal(out, expect)


@pytest.mark.parametrize('M,N,K', [(300, 64, 64), (1000, 256, 256), (20000, 512, 128), (40000, 128, 512), (700, 48, 32)])
def test_tf32x3_widths_that_80_does_not_divide(M, N, K):
    """news_embedding_dim values such as 64 / 128 / 256 / 512 (ADVICE r1): partial last N tiles on every tile variant."""
    g = torch.Generator().manual_seed(M + N + K)
    A = torch.randn(M, K, generator=g)
    W = torch.randn(N, K, generator=g) * 0.05
    bias = torch.randn(N, generator=g)
    C = _tf32x3(A.cuda(), W.cuda(), bias.cuda()).cpu()
    ref = A.double() @ W.double().t() + bias.double()
    assert torch.isfinite(C).all()
    assert rel_err(C.numpy(), ref.numpy()) < 4e-6


@pytest.mark.parametrize('M,D', [(512, 64), (1000, 256), (300, 128)])
def test_linear_backward_other_embedding_dims(M, D):
    """Weight gradients on the split-K tensor-core path for D not a multiple of 80 (used to crash: no TF32 planes)."""
    from digat_b200.autograd_ops import lin
    g = torch.Generator().manual_seed(M + D)
    A = torch.randn(M, D, generator=g)
    W = torch.randn(3 * D, D, generator=g) * 0.05
    bias = torch.randn(3 * D, generator=g)
    dC = torch.randn(M, 3 * D, generator=g)
    A64, W64, b64 = (t.double().requires_grad_(True) for t in (A, W, bias))
    (A64 @ W64.t() + b64).backward(dC.double())
    Ac, Wc, bc = (t.cuda().requires_grad_(True) for t in (A, W, bias))
    lin(Ac, Wc, bc).backward(dC.cuda())
    torch.cuda.synchronize()
    assert rel_err(Ac.grad.cpu().numpy(), A64.grad.numpy()) < 5e-6
    assert rel_err(Wc.grad.cpu().numpy(), W64.grad.numpy()) < 5e-6
    assert rel_err(bc.grad.cpu().numpy(), b64.grad.numpy()) < 2e-6


@pytest.mark.parametrize('M,N,K', [(100000, 1200, 400), (77824, 400, 400), (136000 + 77, 1200, 400), (30000, 480, 96)])
def test_persistent_kernel_row_scatter_is_dense_product_plus_group_bias(M, N, K):
    """The persistent kernel with bias, row-group bias, an odd M-block tail and ascending row scatter: row m of the product
    lands in C[rows[m]] as the dense product D[m] of the same call without scatter or group bias, plus the group bias of
    row rows[m] in one fp32 add on the bias columns, bit for bit; the rows of C that are not listed stay untouched."""
    from digat_b200 import _lib
    g = torch.Generator().manual_seed(M + N)
    A = torch.randn(M, K, generator=g).cuda()
    W = (torch.randn(N, K, generator=g) * 0.05).cuda()
    bias = torch.randn(N, generator=g).cuda()
    gcols = min(400, N)
    gbias = torch.randn((2 * M + 67) // 68, gcols, generator=g).cuda()
    rows = torch.sort(torch.randperm(2 * M, generator=g)[:M]).values.to(torch.int32).cuda()      # ascending scatter targets
    hi, lo = _split(W)
    st = torch.cuda.current_stream().cuda_stream
    C = torch.zeros((2 * M, N), device='cuda')
    _lib.call('digat_linear_tf32x3', A.data_ptr(), K, hi.data_ptr(), lo.data_ptr(), K, bias.data_ptr(), C.data_ptr(), N,
              M, N, K, gbias.data_ptr(), 68, 0, gcols, gcols, rows.data_ptr(), st)
    D = torch.full((M, N), float('nan'), device='cuda')
    _lib.call('digat_linear_tf32x3', A.data_ptr(), K, hi.data_ptr(), lo.data_ptr(), K, bias.data_ptr(), D.data_ptr(), N,
              M, N, K, 0, 1, 0, 0, 0, 0, st)
    torch.cuda.synchronize()
    r = rows.long()
    expect = D.clone()
    expect[:, :gcols] = D[:, :gcols] + gbias[r // 68]
    assert torch.equal(C[r], expect)
    listed = torch.zeros(2 * M, dtype=torch.bool, device='cuda')
    listed[r] = True
    assert int(torch.count_nonzero(C[~listed])) == 0
    sel = torch.randperm(M, generator=g)[:256].cuda()
    ref = A[sel].double() @ W.double().t() + bias.double()
    ref[:, :gcols] += gbias[r[sel] // 68].double()
    assert rel_err(C[r[sel]].cpu().numpy(), ref.cpu().numpy()) < 4e-6


@pytest.mark.parametrize('M,N,K', [(320, 400, 400), (320, 800, 400), (7, 36, 52), (1, 4, 4), (1000, 400, 1200), (33, 400, 68)])
def test_small_exact_fp32_gemm_three_products(M, N, K):
    """digat_gemm_f32_small: forward (A W^T + bias), dgrad (dC W) and wgrad (dC^T A) read their operands in place -- strided
    slices and the transposed view of a key matrix included -- and match fp64 to fp32 rounding of a K-term sum."""
    from digat_b200.autograd_ops import lin
    g = torch.Generator().manual_seed(M + N + K)
    wide = torch.randn(M, K + 8, generator=g)
    A = wide[:, 4:4 + K]                                   # strided rows (lda = K + 8), 16-byte aligned start
    W = torch.randn(N, K, generator=g) * 0.2
    Kw = torch.randn(K, N, generator=g) * 0.2              # a key matrix applied as lin(q, Kw.t())
    bias = torch.randn(N, generator=g)
    dC = torch.randn(M, N, generator=g)
    for weight, use_bias in ((W, True), (Kw.t(), False)):
        A64, W64 = A.double().requires_grad_(True), weight.double().requires_grad_(True)
        b64 = bias.double().requires_grad_(True)
        ref = A64 @ W64.t() + (b64 if use_bias else 0)
        ref.backward(dC.double())
        wide_c = wide.cuda().requires_grad_(True)
        Wc = (W.cuda() if weight is W else Kw.cuda()).requires_grad_(True)
        bc = bias.cuda().requires_grad_(True)
        out = lin(wide_c[:, 4:4 + K], Wc if weight is W else Wc.t(), bc if use_bias else None)
        out.backward(dC.cuda())
        torch.cuda.synchronize()
        tol = 4e-7 * max(K, M, N) ** 0.5 + 2e-7
        assert rel_err(out.detach().cpu().numpy(), ref.detach().numpy()) < tol
        assert rel_err(wide_c.grad[:, 4:4 + K].cpu().numpy(), A64.grad.numpy()) < tol
        wg = Wc.grad if weight is W else Wc.grad.t()
        assert rel_err(wg.cpu().numpy(), W64.grad.numpy()) < tol
        if use_bias:
            assert rel_err(bc.grad.cpu().numpy(), b64.grad.numpy()) < tol
        assert float(wide_c.grad[:, :4].abs().max()) == 0.0


@pytest.mark.parametrize('rows,cols', [(21760, 400), (680, 1200), (33, 7), (1, 5), (4, 4096)])
def test_transpose_and_tf32_planes(rows, cols):
    """digat_transpose_f32: the transposed matrix bit for bit; with out_lo the TF32 planes of the transpose are exactly
    digat_split_tf32 of it (hi + lo reproduces x to 2^-21 relative)."""
    from digat_b200 import _lib
    from digat_b200.graphEncoders import PackedWeight, _stream
    g = torch.Generator().manual_seed(rows + cols)
    wide = torch.randn(rows, cols + 4, generator=g).cuda()
    x = wide[:, :cols]                                       # strided source rows
    t = torch.empty(cols, rows, device='cuda')
    _lib.call('digat_transpose_f32', x.data_ptr(), x.stride(0), t.data_ptr(), 0, rows, rows, cols, _stream())
    hi, lo = torch.empty(cols, rows, device='cuda'), torch.empty(cols, rows, device='cuda')
    _lib.call('digat_transpose_f32', x.data_ptr(), x.stride(0), hi.data_ptr(), lo.data_ptr(), rows, rows, cols, _stream())
    torch.cuda.synchronize()
    want = x.t().contiguous()
    assert torch.equal(t, want)
    if cols % 16 == 0 and rows % 4 == 0:
        ref = PackedWeight(want)
        assert torch.equal(hi, ref.hi) and torch.equal(lo, ref.lo)
    assert float(((hi.double() + lo.double()) - want.double()).abs().max()) <= 2.0 ** -21 * float(want.abs().max())


@pytest.mark.parametrize('M,N,ld', [(320, 400, 400), (320, 400, 1200), (1, 4, 4), (2048, 1200, 1200), (3200, 400, 400), (4097, 400, 400),
                                    (21760, 1200, 1200), (43, 480000, 480000)])
def test_colsum_paths(M, N, ld):
    """digat_colsum: the single-launch kernel (<= 4096 rows), the sliced two-launch path and its one-slice shortcut."""
    from digat_b200.autograd_ops import colsum
    g = torch.Generator().manual_seed(M)
    x = torch.randn(M, ld, generator=g).cuda()[:, :N]
    got = colsum(x)
    torch.cuda.synchronize()
    want = x.double().sum(0)
    assert rel_err(got.cpu().numpy(), want.cpu().numpy()) < 2e-6
    assert torch.equal(got, colsum(x))                       # deterministic
