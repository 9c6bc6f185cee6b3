"""Micro-benchmark of the tcgen05 conv kernels on the CIFAR shapes (CUDA events, L2 flushed by a
256 MB write between timed launches). Run on a B200:
    python tests/bench_conv_micro.py
"""
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from veles.znicz_b200.kernels import load_extension  # noqa: E402

ext = load_extension(required=True)
dev = "cuda"
# name, N, H, W, C, F, k, pad      (stride 1)
CIFAR = [("conv1", 100, 32, 32, 8, 32, 5, 2), ("conv2", 100, 16, 16, 32, 32, 5, 2),
         ("conv3", 100, 8, 8, 32, 64, 5, 2)]
ALEXNET = [("alex_conv2", 128, 27, 27, 128, 256, 5, 2), ("alex_conv3", 128, 13, 13, 256, 384, 3, 1),
           ("alex_conv4", 128, 13, 13, 384, 384, 3, 1), ("alex_conv5", 128, 13, 13, 384, 256, 3, 1)]
SHAPES = ALEXNET if (len(sys.argv) > 1 and sys.argv[1] == "alexnet") else CIFAR
flush = torch.empty(64 << 20, dtype=torch.float32, device=dev)


def timeit(fn, iters=50):
    for _ in range(5):
        fn()
    torch.cuda.synchronize()
    tot = 0.0
    for _ in range(iters):
        flush.fill_(1.0)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        tot += e0.elapsed_time(e1)
    return tot / iters * 1000.0


for name, n, h, w, c, f, k, pad in SHAPES:
    g = [n, h, w, c, h, w, f, k, k, 1, 1, pad, pad]
    kw = k * k * c
    x = torch.randn(n, h, w, c, device=dev).bfloat16()
    wl = torch.randn(f, kw, device=dev).bfloat16()
    wd = torch.randn(k * k * f, ((c + 7) // 8) * 8, device=dev).bfloat16()
    bias = torch.randn(f, device=dev)
    out = torch.empty(n, h, w, f, device=dev, dtype=torch.bfloat16)
    eo = torch.randn(n, h, w, f, device=dev).bfloat16()
    ei = torch.empty(n, h, w, c, device=dev, dtype=torch.bfloat16)
    splits = int(ext.pick_splits(kw, f, n * h * w, 64))
    parts = torch.empty(splits, f, kw, device=dev)
    t_f = timeit(lambda: ext.conv_fprop(x, wl, kw, False, bias, out, g, 3, 1))
    t_d = timeit(lambda: ext.conv_dgrad(eo, wd, wd.shape[1], False, ei, g, 1.0, 0.0, 1, None, 0)) if c >= 32 else 0
    t_w = timeit(lambda: ext.conv_wgrad(eo, x, parts, splits, g, False, 1, None))
    fl = 2.0 * n * h * w * kw * f / 1e6           # MFLOP; / us = TFLOP/s
    print("%s fprop %.1f us (%.0f TF)  dgrad %.1f us (%.0f TF)  wgrad %.1f us (%.0f TF, splits %d)  "
          "im2col_tma=%s" % (
              name, t_f, fl / t_f, t_d, fl / t_d if t_d else 0, t_w, fl / t_w, splits,
              os.environ.get("ZNICZ_IM2COL_TMA", "1")))
