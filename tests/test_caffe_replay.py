"""Whole-iteration replay of a Caffe CIFAR-10 training step, layer by layer
(the reference's tests/functional/test_caffe_complex.py:83-534 on
``data/cifar_export.tar.xz``; iteration 0 converted by tools/make_caffe_replay.py into
tests/golden/caffe_cifar_iter0/<layer>.<direction>.npz, batch 3): every layer gets Caffe's
bottom blob / weights / top gradient and must reproduce Caffe's top blob / bottom gradient - on
the numpy oracle (CPU tier) and on the sm_100a path in fp32 and bf16 (GPU tier)."""
import os

import numpy
import pytest

from veles.znicz_b200.core.config import root
from veles.znicz_b200.core.memory import Array
from veles.znicz_b200.core.workflow import DummyWorkflow
from veles.znicz_b200.ops import (activation, all2all, conv, gd, gd_conv, gd_pooling,
                                  normalization, pooling)

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "caffe_cifar_iter0")
D = {}
for _f in sorted(os.listdir(GOLDEN)):
    with numpy.load(os.path.join(GOLDEN, _f)) as _z:
        D.update((k, _z[k]) for k in _z.files)

CONVS = {"conv1": 32, "conv2": 32, "conv3": 64}
POOLS = {"pool1": pooling.MaxPooling, "pool2": pooling.AvgPooling, "pool3": pooling.AvgPooling}
GDPOOLS = {"pool1": gd_pooling.GDMaxPooling, "pool2": gd_pooling.GDAvgPooling,
           "pool3": gd_pooling.GDAvgPooling}


def _rel(a, b):
    a = numpy.asarray(a, numpy.float64).reshape(b.shape)
    return float(numpy.abs(a - b).sum() / max(numpy.abs(b).sum(), 1e-30))


def _arr(x, device, compute):
    a = Array(numpy.ascontiguousarray(x, dtype=numpy.float32))
    if device is not None and compute == "bf16":
        import torch
        a.dev_dtype = torch.bfloat16
    return a


def _get(a):
    a.map_read()
    return a.mem


def replay(device, compute):
    """-> {layer/fwd|bwd: relative L1 error vs Caffe}"""
    root.common.engine.compute_type = compute if device is not None else "fp32"
    wf = DummyWorkflow()
    res = {}
    lrn_kw = dict(n=3, alpha=0.00005, beta=0.75, k=1)
    for name, nk in CONVS.items():
        f = conv.Conv(wf, kx=5, ky=5, padding=(2, 2, 2, 2), sliding=(1, 1), n_kernels=nk)
        f.input = _arr(D[name + "/forward/bottom_0"], device, compute)
        f.initialize(device=device)
        f.weights.map_invalidate()
        f.weights.mem[...] = D[name + "/forward/blob_0"].transpose(0, 2, 3, 1).reshape(nk, -1)
        f.weights.unmap()
        f.bias.map_invalidate()
        f.bias.mem[...] = D[name + "/forward/blob_1"].ravel()
        f.bias.unmap()
        if getattr(f, "on_cuda", False):
            f.refresh_shadows()
        f.run()
        res[name + "/fwd"] = _rel(_get(f.output), D[name + "/forward/top_0"])
        g = gd_conv.GradientDescentConv(wf, kx=5, ky=5, padding=(2, 2, 2, 2), sliding=(1, 1),
                                        n_kernels=nk, learning_rate=0.0, weights_decay=0.0,
                                        apply_gradient=False, gradient_moment=0.0)
        g.err_output = _arr(D[name + "/backward/top_err_0"], device, compute)
        g.link_attrs(f, "input", "output", "weights", "bias")
        g.forward_unit = f
        g.initialize(device=device)
        g.run()
        res[name + "/bwd"] = _rel(_get(g.err_input), D[name + "/backward/bottom_err_0"])
    for name, cls in POOLS.items():
        f = cls(wf, kx=3, ky=3, sliding=(2, 2))
        f.input = _arr(D[name + "/forward/bottom_0"], device, compute)
        f.initialize(device=device)
        f.run()
        res[name + "/fwd"] = _rel(_get(f.output), D[name + "/forward/top_0"])
        g = GDPOOLS[name](wf, kx=3, ky=3, sliding=(2, 2))
        g.err_output = _arr(D[name + "/backward/top_err_0"], device, compute)
        links = ["input", "output"] + (["input_offset"] if name == "pool1" else [])
        g.link_attrs(f, *links)
        g.initialize(device=device)
        g.run()
        res[name + "/bwd"] = _rel(_get(g.err_input), D[name + "/backward/bottom_err_0"])
    for name in ("relu1", "relu2", "relu3"):
        f = activation.ForwardStrictRELU(wf)
        f.input = _arr(D[name + "/forward/bottom_0"], device, compute)
        f.initialize(device=device)
        f.run()
        res[name + "/fwd"] = _rel(_get(f.output), D[name + "/forward/top_0"])
        b = activation.BackwardStrictRELU(wf)
        b.input, b.output = f.input, f.output
        b.err_output = _arr(D[name + "/backward/top_err_0"], device, compute)
        b.initialize(device=device)
        b.run()
        res[name + "/bwd"] = _rel(_get(b.err_input), D[name + "/backward/bottom_err_0"])
    for name in ("norm1", "norm2"):
        f = normalization.LRNormalizerForward(wf, **lrn_kw)
        f.input = _arr(D[name + "/forward/bottom_0"], device, compute)
        f.initialize(device=device)
        f.run()
        res[name + "/fwd"] = _rel(_get(f.output), D[name + "/forward/top_0"])
        b = normalization.LRNormalizerBackward(wf, **lrn_kw)
        b.input, b.output = f.input, f.output
        b.err_output = _arr(D[name + "/backward/top_err_0"], device, compute)
        b.initialize(device=device)
        b.run()
        res[name + "/bwd"] = _rel(_get(b.err_input), D[name + "/backward/bottom_err_0"])
    # inner product + softmax: Caffe flattens NCHW, we flatten NHWC -> permute the weight columns
    f = all2all.All2AllSoftmax(wf, output_sample_shape=10)
    f.input = _arr(D["ip1/forward/bottom_0"], device, compute)
    f.initialize(device=device)
    w = D["ip1/forward/blob_0"].reshape(10, 64, 4, 4).transpose(0, 2, 3, 1).reshape(10, 1024)
    f.weights.map_invalidate()
    f.weights.mem[...] = w
    f.weights.unmap()
    f.bias.map_invalidate()
    f.bias.mem[...] = D["ip1/forward/blob_1"].ravel()
    f.bias.unmap()
    if getattr(f, "on_cuda", False):
        f.refresh_shadows()
    f.run()
    res["ip1+softmax/fwd"] = _rel(_get(f.output), D["loss/forward/top_0"].reshape(3, 10))
    g = gd.GDSoftmax(wf, learning_rate=0.0, weights_decay=0.0, apply_gradient=False,
                     gradient_moment=0.0)
    g.err_output = _arr(D["ip1/backward/top_err_0"].reshape(3, 10), device, compute)
    g.link_attrs(f, "input", "output", "weights", "bias")
    g.forward_unit = f
    g.initialize(device=device)
    g.run()
    res["ip1/bwd"] = _rel(_get(g.err_input), D["ip1/backward/bottom_err_0"])
    root.common.engine.compute_type = "fp32"
    return res


def test_caffe_iteration_replay_numpy():
    res = replay(None, "fp32")
    for k, v in res.items():
        assert v < 2e-3, (k, v, res)


@pytest.mark.gpu
@pytest.mark.parametrize("compute,tol", [("fp32", 2e-3), ("bf16", 4e-2)])
def test_caffe_iteration_replay_gpu(compute, tol):
    from veles.znicz_b200.core.backends import get_device
    res = replay(get_device("cuda"), compute)
    for k, v in res.items():
        assert v < tol, (k, v, compute, res)
