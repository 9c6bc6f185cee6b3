"""Cross-framework golden data: Caffe blob dumps shipped with the reference's functional tests
(``tests/functional/data/*.txt``, stored xz-compressed under tests/golden/caffe) vs our numpy
units — the reference's ``tests/functional/test_caffe.py`` strategy (SURVEY §4, "cross-framework
golden data"). The dump format: ``<name>[\\tnum:N\\tchannels:C\\theight:H\\twidth:W]`` followed by
``num:i`` / ``channels:c`` headers and H tab-separated rows per channel plane."""
import lzma
import os

import numpy
import pytest

from veles.znicz_b200.core.config import root
from veles.znicz_b200.core.memory import Array
from veles.znicz_b200.core.workflow import DummyWorkflow
from veles.znicz_b200.ops import conv, gd_conv, gd_pooling, normalization, pooling

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
DATA = os.path.join(GOLDEN, "caffe")


def read_blob(lines, name, shape=None):
    """→ float64 array [num, height, width, channels] (NHWC) of blob ``name``."""
    start = None
    for i, line in enumerate(lines):
        parts = line.rstrip("\n").split("\t")
        if parts[0].strip() == name:
            dims = dict(p.split(":") for p in parts[1:] if ":" in p)
            if len(dims) >= 4:
                shape = (int(dims["num"]), int(dims["height"]), int(dims["width"]),
                         int(dims["channels"]))
            start = i + 1
            break
    assert start is not None and shape is not None, name
    n, h, w, c = shape
    out = numpy.zeros(shape, numpy.float64)
    cur = start
    for pic in range(n):
        assert lines[cur].strip().split(":") == ["num", str(pic)], lines[cur]
        cur += 1
        for ch in range(c):
            assert lines[cur].strip().split(":") == ["channels", str(ch)]
            cur += 1
            for y in range(h):
                out[pic, y, :, ch] = [float(v) for v in lines[cur].split()]
                cur += 1
    return out


def _lines(name):
    with lzma.open(os.path.join(DATA, name + ".xz"), "rt") as f:
        return f.readlines()


def _rel(a, b):
    return float(numpy.abs(a - b).sum() / max(numpy.abs(b).sum(), 1e-30))


@pytest.fixture(autouse=True)
def _double():
    root.common.engine.precision_type = "double"
    yield
    root.common.engine.precision_type = "float"


def _conv_unit(wf, bottom, weights, n_kernels):
    u = conv.Conv(wf, kx=5, ky=5, padding=(2, 2, 2, 2), sliding=(1, 1), n_kernels=n_kernels)
    u.input = Array(bottom.copy())
    u.initialize(device="numpy")
    u.weights.mem[:] = weights.reshape(n_kernels, -1)
    u.bias.mem[:] = 0
    u.run()
    return u


def test_conv_forward_matches_caffe():
    lines = _lines("conv.txt")
    bottom = read_blob(lines, "bottom", (2, 32, 32, 3))
    weights = read_blob(lines, "weights", (2, 5, 5, 3))
    top = read_blob(lines, "top", (2, 32, 32, 2))
    u = _conv_unit(DummyWorkflow(), bottom, weights, 2)
    assert _rel(u.output.mem, top) < 1e-2      # dumps carry 6 decimals of ~1e-4 weights


def test_conv_backward_matches_caffe():
    lines = _lines("conv_grad.txt")
    bottom = read_blob(lines, "bottom", (2, 32, 32, 3))
    weights = read_blob(lines, "weights", (2, 5, 5, 3))
    top = read_blob(lines, "top", (2, 32, 32, 2))
    top_err = read_blob(lines, "top_diff", (2, 32, 32, 2))
    bot_err = read_blob(lines, "bottom_diff", (2, 32, 32, 3))
    wf = DummyWorkflow()
    u = _conv_unit(wf, bottom, weights, 2)
    assert _rel(u.output.mem, top) < 1e-2      # dumps carry 6 decimals of ~1e-4 weights
    g = gd_conv.GradientDescentConv(wf, kx=5, ky=5, padding=(2, 2, 2, 2), sliding=(1, 1),
                                    n_kernels=2, learning_rate=0.0, weights_decay=0.0,
                                    apply_gradient=False, gradient_moment=0.0)
    g.err_output = Array(top_err.copy())
    g.link_attrs(u, "input", "output", "weights", "bias")
    g.initialize(device="numpy")
    g.run()
    assert _rel(g.err_input.mem, bot_err) < 1e-2


@pytest.mark.parametrize("fname", ["pool.txt", "pool_grad.txt"])
def test_max_pooling_matches_caffe(fname):
    lines = [l.replace("\t\n", "\n") for l in _lines(fname)]
    bottom = read_blob(lines, "bottom", (2, 32, 32, 2))
    top = read_blob(lines, "top", (2, 16, 16, 2))
    wf = DummyWorkflow()
    u = pooling.MaxPooling(wf, kx=3, ky=3, sliding=(2, 2))
    u.input = Array(bottom.copy())
    u.initialize(device="numpy")
    u.run()
    assert _rel(u.output.mem, top) < 1e-6
    if fname == "pool_grad.txt":
        top_err = read_blob(lines, "top_diff", (2, 16, 16, 2))
        bot_err = read_blob(lines, "bottom_diff", (2, 32, 32, 2))
        g = gd_pooling.GDMaxPooling(wf, kx=3, ky=3, sliding=(2, 2))
        g.err_output = Array(top_err.copy())
        g.link_attrs(u, "input", "input_offset", "output")
        g.initialize(device="numpy")
        g.run()
        # errors of ~1e-6 printed with 6 decimals + tie-breaking between equal maxima
        assert _rel(g.err_input.mem, bot_err) < 0.03


def test_lrn_matches_caffe():
    lines = _lines("norm_gd.txt")
    bottom = read_blob(lines, "bottom", (2, 16, 16, 2))
    top = read_blob(lines, "top", (2, 16, 16, 2))
    top_err = read_blob(lines, "top_diff", (2, 16, 16, 2))
    bot_err = read_blob(lines, "bottom_diff", (2, 16, 16, 2))
    wf = DummyWorkflow()
    f = normalization.LRNormalizerForward(wf, k=1)
    f.input = Array(bottom.copy())
    f.initialize(device="numpy")
    f.run()
    assert _rel(f.output.mem, top) < 0.02          # the reference allows 2 %
    b = normalization.LRNormalizerBackward(wf, k=1)
    b.input, b.output = f.input, f.output
    b.err_output = Array(top_err.copy())
    b.initialize(device="numpy")
    b.run()
    assert _rel(b.err_input.mem, bot_err) < 0.02


def test_conv3_golden_arrays_forward_and_err_input():
    """The reference ships golden arrays of the CIFAR net's conv3 (5 x 5, pad 2, 32 -> 64 channels,
    3 images) under tests/data/gd_conv_data (SURVEY Appendix C; copied to tests/golden/gd_conv3):
    forward output and err_input of the numpy oracle against them (relative max error; the arrays
    come from a Caffe fp32 run)."""
    from veles.znicz_b200.core.memory import Array
    from veles.znicz_b200.core.workflow import DummyWorkflow
    from veles.znicz_b200.ops import conv, gd_conv
    base = os.path.join(GOLDEN, "gd_conv3")
    x, w, b, y, eo, ei = [numpy.load(os.path.join(base, n + ".npz"))["arr_0"] for n in
                          ("input", "weights", "bias", "output", "err_output", "err_input")]
    wf = DummyWorkflow()
    kw = dict(n_kernels=64, kx=5, ky=5, padding=(2, 2, 2, 2), sliding=(1, 1))
    c = conv.Conv(wf, weights_stddev=0.1, **kw)
    c.input = Array(x.copy())
    c.initialize(device=None)
    c.weights.map_write()
    c.bias.map_write()
    c.weights.mem[...] = w
    c.bias.mem[...] = b
    c.run()
    assert c.output.mem.shape == y.shape
    assert numpy.abs(c.output.mem - y).max() / numpy.abs(y).max() < 1e-2
    g = gd_conv.GradientDescentConv(wf, learning_rate=0, learning_rate_bias=0, **kw)
    g.err_output = Array(eo.copy())
    g.input, g.output, g.weights, g.bias = c.input, c.output, c.weights, c.bias
    g.initialize(device=None)
    g.run()
    assert numpy.abs(g.err_input.mem - ei).max() / numpy.abs(ei).max() < 1e-3


def _read_any(lines, name, shape):
    """Blob reader for the dumps whose header carries no dimensions; ``*_flat`` blobs hold the
    whole NCHW tensor in one row."""
    start = [i for i, l in enumerate(lines) if l.strip().split("\t")[0] == name][0] + 1
    n, h, w, c = shape
    if name.endswith("_flat"):
        vals = [float(v) for v in lines[start + 2].split()]
        return numpy.array(vals).reshape(n, c, h, w).transpose(0, 2, 3, 1)
    out = numpy.zeros(shape)
    cur = start
    for pic in range(n):
        assert lines[cur].strip() == "num:%d" % pic
        cur += 1
        for ch in range(c):
            assert lines[cur].strip() == "channels:%d" % ch
            cur += 1
            for y in range(h):
                out[pic, y, :, ch] = [float(v) for v in lines[cur].split()]
                cur += 1
    return out


def _conv_relu(wf, bottom, weights):
    u = conv.ConvStrictRELU(wf, kx=5, ky=5, padding=(2, 2, 2, 2), sliding=(1, 1), n_kernels=2)
    u.input = Array(bottom.copy())
    u.initialize(device="numpy")
    u.weights.mem[:] = weights.reshape(2, -1)
    u.bias.mem[:] = 0
    u.run()
    return u


def test_conv_relu_forward_matches_caffe():
    """The reference's tests/functional/test_caffe.py (conv + ReLU pair, `conv_relu.txt`)."""
    lines = _lines("conv_relu.txt")
    bottom = _read_any(lines, "conv_bottom", (2, 32, 32, 3))
    weights = _read_any(lines, "conv_weights", (2, 5, 5, 3))
    relu_top = _read_any(lines, "relu_top_flat", (2, 32, 32, 2))
    u = _conv_relu(DummyWorkflow(), bottom, weights)
    assert _rel(u.output.mem, relu_top) < 5e-3        # weights printed with 6 decimals


def test_conv_relu_backward_matches_caffe():
    """`conv_relu_grad.txt`: the fused conv + ReLU GD unit against Caffe's ReLU backward followed
    by its conv backward - err_input and the raw weight gradient."""
    lines = _lines("conv_relu_grad.txt")
    g = {name: _read_any(lines, name, shape) for name, shape in (
        ("relu_bottom", (2, 32, 32, 2)), ("relu_top_diff", (2, 32, 32, 2)),
        ("relu_bottom_diff", (2, 32, 32, 2)), ("conv_weights", (2, 5, 5, 3)),
        ("conv_top_diff", (2, 32, 32, 2)), ("conv_bottom", (2, 32, 32, 3)),
        ("conv_bottom_diff", (2, 32, 32, 3)), ("conv_weight_delta", (2, 5, 5, 3)),
        ("relu_top_flat", (2, 32, 32, 2)))}
    assert _rel(g["relu_top_diff"] * (g["relu_bottom"] > 0), g["relu_bottom_diff"]) < 1e-9
    wf = DummyWorkflow()
    u = _conv_relu(wf, g["conv_bottom"], g["conv_weights"])
    assert _rel(u.output.mem, g["relu_top_flat"]) < 1e-4
    gd = gd_conv.GDStrictRELUConv(wf, kx=5, ky=5, padding=(2, 2, 2, 2), sliding=(1, 1), n_kernels=2,
                                  learning_rate=0.0, weights_decay=0.0, apply_gradient=False,
                                  gradient_moment=0.0)
    gd.err_output = Array(g["relu_top_diff"].copy())
    gd.link_attrs(u, "input", "output", "weights", "bias")
    gd.initialize(device="numpy")
    gd.run()
    assert _rel(gd.err_input.mem, g["conv_bottom_diff"]) < 1e-5
    assert _rel(gd.gradient_weights.mem.reshape(2, 5, 5, 3), g["conv_weight_delta"]) < 1e-3


def test_softmax_and_loss_gradient_match_caffe():
    """`softmax.txt`: softmax of the logits and the SoftmaxWithLoss gradient (p - onehot) / batch."""
    from veles.znicz_b200.ops import all2all
    from veles.znicz_b200.workflow import evaluator
    lines = _lines("softmax.txt")

    def vec(name, width):
        start = [i for i, l in enumerate(lines) if l.strip() == name][0] + 1
        out = numpy.zeros((2, width))
        cur = start
        for pic in range(2):
            assert lines[cur].strip() == "num:%d" % pic
            cur += 1
            for ch in range(width):
                assert lines[cur].strip() == "channels:%d" % ch
                out[pic, ch] = float(lines[cur + 1].split()[0])
                cur += 2
        return out
    labels = vec("labels", 1)[:, 0].astype(numpy.int32)
    logits, top, bottom_diff = vec("sm_bottom", 10), vec("sm_top", 10), vec("sm_bottom_diff", 10)
    wf = DummyWorkflow()
    f = all2all.All2AllSoftmax(wf, output_sample_shape=10, weights_stddev=0.1)
    f.input = Array(logits.copy())
    f.initialize(device="numpy")
    f.weights.mem[:] = numpy.eye(10)
    f.bias.mem[:] = 0
    f.run()
    assert numpy.abs(f.output.mem - top).max() < 2e-6
    ev = evaluator.EvaluatorSoftmax(wf)
    ev.output, ev.max_idx = f.output, f.max_idx
    ev.labels = Array(labels.copy())
    ev.batch_size = 2
    ev.initialize(device="numpy")
    ev.run()
    assert numpy.abs(ev.err_output.mem - bottom_diff).max() < 2e-6
