"""Small-M GEMMs of the training step (context projections, M = batch rows): tcgen05 3xTF32 vs the exact-fp32 CUDA-core
kernels, forward/dgrad (digat_linear_*) and wgrad.  Warm, back-to-back launches, CUDA events."""
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from digat_b200 import _lib, autograd_ops  # noqa: E402
from digat_b200.graphEncoders import PackedWeight, _stream, linear  # noqa: E402


def timeit(fn, reps=40):
    """fn captured reps times into ONE CUDA graph (no host launch cost, as in the graphed training step), replayed 5 times."""
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        for _ in range(3):
            fn()
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g, stream=s):
        for _ in range(reps):
            fn()
    g.replay()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(5):
        g.replay()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / (5 * reps) * 1e3


def main():
    _lib.require_device(0)
    for M, N, K in ((320, 400, 400), (320, 800, 400), (320, 400, 800), (320, 1200, 400), (6080, 400, 400), (4160, 1200, 400),
                    (4160, 400, 1200), (1280, 400, 400)):
        A = torch.randn(M, K, device='cuda')
        W = torch.randn(N, K, device='cuda')
        dC = torch.randn(M, N, device='cuda')
        pw = PackedWeight(W)
        C = torch.empty(M, N, device='cuda')
        t_tc = timeit(lambda: linear(A, pw))
        t_simt = timeit(lambda: _lib.call('digat_linear_f32', A.data_ptr(), K, W.data_ptr(), K, 0, C.data_ptr(), N, M, N, K, 0,
                                          0, 1, 0, 0, 0, _stream()))
        t_split = timeit(lambda: PackedWeight(W))
        out = torch.empty(M, N, device='cuda'); dA = torch.empty(M, K, device='cuda'); dW = torch.empty(N, K, device='cuda')
        sg = lambda L, ldl, lt, R, ldr, rt, o, ldo, I, J, Cc: _lib.call('digat_gemm_f32_small', L.data_ptr(), ldl, lt, R.data_ptr(), ldr, rt, 0, o.data_ptr(), ldo, I, J, Cc, _stream())  # noqa: E731
        t_sf = timeit(lambda: sg(A, K, 0, W, K, 1, out, N, M, N, K))
        t_sd = timeit(lambda: sg(dC, N, 0, W, K, 0, dA, K, M, K, N))
        t_sw = timeit(lambda: sg(dC, N, 1, A, K, 0, dW, K, N, K, M))
        print('small fp32 kernel: fwd %.1f us  dgrad %.1f us  wgrad %.1f us' % (t_sf, t_sd, t_sw))
        old = autograd_ops.WGRAD_TC_MIN_ROWS
        autograd_ops.WGRAD_TC_MIN_ROWS = 256
        t_wg_tc = timeit(lambda: autograd_ops.wgrad(dC, A))
        autograd_ops.WGRAD_TC_MIN_ROWS = 1 << 30
        t_wg_simt = timeit(lambda: autograd_ops.wgrad(dC, A))
        autograd_ops.WGRAD_TC_MIN_ROWS = old
        print('M=%5d N=%4d K=%4d  linear tcgen05 %6.1f us  simt %6.1f us  split(W) %5.1f us | wgrad tensor path %6.1f us  simt path %6.1f us'
              % (M, N, K, t_tc, t_simt, t_split, t_wg_tc, t_wg_simt), flush=True)


if __name__ == '__main__':
    main()
