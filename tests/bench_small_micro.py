"""Micro-benchmark of the latency-bound (tiny batch) GEMM / conv launches of the GA-tuned MNIST
conv net (batch 6). CUDA events; each shape timed with a cold L2 (256 MB write between launches)
and warm (back-to-back launches). Run on a B200:  python tests/bench_small_micro.py
"""
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from veles.znicz_b200.kernels import load_extension  # noqa: E402

ext = load_extension(required=True)
dev = "cuda"
flush = torch.empty(64 << 20, dtype=torch.float32, device=dev)


def timeit(fn, iters=30, cold=True):
    for _ in range(5):
        fn()
    torch.cuda.synchronize()
    tot = 0.0
    for _ in range(iters):
        if cold:
            flush.fill_(1.0)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        tot += e0.elapsed_time(e1)
    return tot / iters * 1000.0


def gemm_case(M, N, K):
    a = torch.randn(M, K, device=dev).bfloat16()
    b = (torch.randn(N, K, device=dev) / K ** 0.5).bfloat16()
    bias = torch.randn(N, device=dev)
    out = torch.empty(M, N, device=dev, dtype=torch.bfloat16)
    fn = lambda: ext.gemm(a, K, False, b, K, True, out, N, False, M, N, K, bias, 3, 1.0, 0.0, 1, 0, 1)
    r = fn()
    print("gemm M=%d N=%d K=%d rc=%s cold %.1f us warm %.1f us" % (
        M, N, K, r, timeit(fn), timeit(fn, cold=False)))


def conv_case(n, h, w, c, f, k):
    oh, ow = h - k + 1, w - k + 1
    g = [n, h, w, c, oh, ow, f, k, k, 1, 1, 0, 0]
    kw = k * k * c
    x = torch.randn(n, h, w, c, device=dev).bfloat16()
    wl = torch.randn(f, kw, device=dev).bfloat16()
    bias = torch.randn(f, device=dev)
    out = torch.empty(n, oh, ow, f, device=dev, dtype=torch.bfloat16)
    fn = lambda: ext.conv_fprop(x, wl, kw, False, bias, out, g, 3, 1)
    r = fn()
    print("conv n=%d %dx%dx%d f=%d k=%d rc=%s cold %.1f us warm %.1f us" % (
        n, h, w, c, f, k, r, timeit(fn), timeit(fn, cold=False)))


gemm_case(6, 791, 1392)
gemm_case(6, 792, 1392)
gemm_case(6, 792, 128)
gemm_case(128, 128, 1392)
gemm_case(128, 128, 64)
conv_case(6, 12, 12, 64, 87, 5)
conv_case(6, 12, 12, 64, 88, 5)
conv_case(6, 12, 12, 64, 64, 5)
conv_case(6, 12, 12, 64, 64, 1)
