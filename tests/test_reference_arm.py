"""The reference arm (``bench.py --impl reference``): the unmodified Samsung/veles.znicz units
on the Veles-core / cuda4py stand-in of ``baseline/veles_core``.

CPU tier: the vendored tree is byte-identical to its manifest, its CUDA sources compile with
NVRTC against the stand-in core includes, and the whole cuda_init / cuda_run control flow of the
CIFAR sample executes in dry mode (no GPU touched). GPU tier: the stand-in's GEMM / kernel
launch primitives against numpy, and the reference's own numpy back end against its CUDA back
end on a small net (the stock oracle style of the reference's unit tests)."""
import json
import os
import subprocess
import sys

import pytest

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BASE = os.path.join(REPO, "baseline")

# build() vendors the reference tree into baseline/_ref where the reference is available; the
# stand-in core's own primitives need no reference code
needs_reference = pytest.mark.skipif(
    not os.path.isfile(os.path.join(BASE, "_ref", "veles", "znicz", "MANIFEST.sha256.json")),
    reason="reference tree not vendored")


def _run(code, env=None, timeout=900):
    e = dict(os.environ)
    e.pop("PYTHONPATH", None)
    e.update(env or {})
    r = subprocess.run([sys.executable, "-W", "ignore", "-c", code], capture_output=True,
                       text=True, timeout=timeout, env=e, cwd="/tmp")
    assert r.returncode == 0, r.stderr[-4000:]
    return r.stdout


@needs_reference
def test_vendored_reference_is_unmodified():
    sys.path.insert(0, BASE)
    import install_reference
    install_reference.install()
    assert install_reference.verify("/root/reference") == []


# Hyper-parameters are chosen so that the reference's OWN numpy and GPU update rules coincide:
# no momentum (gd.py:315-327 vs cuda/gradient_descent.store_output.cu differ), and bias == weights
# learning rate / decay (its numpy_update applies learning_rate and weights_decay to the bias as
# well, gd.py:363-365, while the GPU kernel uses learning_rate_bias / weights_decay_bias).
TINY = """
import sys, json, numpy
sys.path.insert(0, %r)
import run_reference as rr
tiny = [
 {"name": "conv1", "type": "conv", "->": {"n_kernels": 8, "kx": 5, "ky": 5, "padding": (2,2,2,2), "sliding": (1,1), "weights_filling": "gaussian", "weights_stddev": 0.01, "bias_filling": "constant", "bias_stddev": 0},
  "<-": {"learning_rate": 0.001, "learning_rate_bias": 0.001, "weights_decay": 0.0005, "weights_decay_bias": 0.0005, "factor_ortho": 0.001, "gradient_moment": 0, "gradient_moment_bias": 0}},
 {"name": "pool1", "type": "max_pooling", "->": {"kx": 3, "ky": 3, "sliding": (2, 2)}},
 {"name": "relu1", "type": "activation_str"},
 {"name": "norm1", "type": "norm", "alpha": 0.00005, "beta": 0.75, "n": 3, "k": 1},
 {"name": "pool2", "type": "avg_pooling", "->": {"kx": 8, "ky": 8, "sliding": (8, 8)}},
 {"name": "fc_softmax4", "type": "softmax", "->": {"output_sample_shape": 10, "weights_filling": "gaussian", "weights_stddev": 0.01, "bias_filling": "constant", "bias_stddev": 0},
  "<-": {"learning_rate": 0.001, "learning_rate_bias": 0.001, "weights_decay": 0.01, "weights_decay_bias": 0.01, "gradient_moment": 0, "gradient_moment_bias": 0}}]
"""


@pytest.fixture(scope="module")
def data_dir(tmp_path_factory):
    return str(tmp_path_factory.mktemp("ref_cifar"))


@needs_reference
def test_reference_cuda_control_flow_dry_run(data_dir):
    """All 12 forward + 12 GD units of the stock CIFAR config: NVRTC build of the reference's
    sources, kernel lookup, argument marshalling, launch geometry — without a GPU."""
    code = ("import sys; sys.path.insert(0, %r)\n"
            "import run_reference as rr, json\n"
            "wf, dev = rr.launch('cuda', data_dir=%r)\n"
            "import cuda4py\n"
            "wf.run(iterations=100); l0 = cuda4py.dry_stats['launches']; g0 = cuda4py.dry_stats['gemms']\n"
            "n = wf.run(iterations=3)\n"
            "print(json.dumps({'n': n, 'cls': wf.loader.minibatch_class,\n"
            "  'launches': cuda4py.dry_stats['launches'] - l0, 'gemms': cuda4py.dry_stats['gemms'] - g0,\n"
            "  'kernels': sorted(cuda4py.dry_stats['kernels'])}))\n") % (BASE, data_dir)
    out = json.loads(_run(code, {"CUDA4PY_DRY": "1"}).strip().splitlines()[-1])
    assert out["n"] == 3 and out["cls"] == 2
    # > 100 tiny launches + ~60 GEMMs per minibatch (SURVEY §3.3): 16-image sub-blocks
    assert out["launches"] >= 3 * 80 and out["gemms"] >= 3 * 50
    for k in ("Unpack1D", "DirectPack", "apply_bias_with_activation", "max_pooling", "avg_pooling",
              "gd_max_pooling", "gd_avg_pooling", "forward", "backward", "forward_strict_relu",
              "backward_strict_relu", "apply_exp", "evaluate_softmax", "weights_update",
              "bias_update", "compute_col_sums"):
        assert k in out["kernels"], k


@needs_reference
def test_bench_reference_arm_dry(tmp_path, data_dir):
    env = dict(os.environ, CUDA4PY_DRY="1", ZNICZ_REF_DATA_DIR=data_dir)
    r = subprocess.run([sys.executable, "-W", "ignore", os.path.join(REPO, "bench.py"), "--impl",
                        "reference", "--steps", "3", "--warmup", "3", "--skip-e2e"],
                       capture_output=True, text=True, timeout=900, env=env, cwd=str(tmp_path))
    assert r.returncode == 0, r.stderr[-3000:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and "unavailable" not in line, line
    assert line["steps"] == 3 and line["config"]["per_gpu_batch"] == 100
    assert line["gpu_launches"] > 300


@pytest.mark.gpu
def test_cuda4py_standin_primitives():
    code = ("import sys; sys.path.insert(0, %r)\n" % os.path.join(BASE, "veles_core") +
            "import numpy, cuda4py as cu, cuda4py.blas as cb\n"
            "ctx = cu.Context(cu.Devices()[0]); blas = cb.CUBLAS(ctx)\n"
            "rs = numpy.random.RandomState(1)\n"
            "for (m, n, k, ta, tb) in [(10, 100, 1024, 1, 0), (1024, 100, 10, 0, 0), (1024, 10, 100, 0, 1), (75, 1600, 32, 0, 0)]:\n"
            "    A = rs.randn(k, m).astype('f') if ta else rs.randn(m, k).astype('f').T.copy()\n"   # column-major storage
            "    opA = A.T if ta else A.T\n"
            "    a_cm = rs.randn(m, k).astype('f'); b_cm = rs.randn(k, n).astype('f')\n"
            "    a_store = numpy.asfortranarray(a_cm.T if ta else a_cm); b_store = numpy.asfortranarray(b_cm.T if tb else b_cm)\n"
            "    da = ctx.mem_alloc(a_store.nbytes); db = ctx.mem_alloc(b_store.nbytes); dc = ctx.mem_alloc(m * n * 4)\n"
            "    da.to_device(numpy.ravel(a_store, order='F')); db.to_device(numpy.ravel(b_store, order='F'))\n"
            "    blas.sgemm(ta, tb, m, n, k, numpy.ones(1, 'f'), da, db, numpy.zeros(1, 'f'), dc)\n"
            "    c = numpy.zeros(m * n, 'f'); dc.to_host(c); c = c.reshape(n, m).T\n"
            "    ref = a_cm @ b_cm\n"
            "    assert numpy.abs(c - ref).max() < 1e-3 * numpy.abs(ref).max(), (m, n, k, ta, tb)\n"
            "mod = cu.Module(ctx, source='extern \"C\" __global__ void axpy(float* y, const float* x, const float a, const int n) { int i = blockIdx.x * blockDim.x + threadIdx.x; if (i < n) y[i] += a * x[i]; }')\n"
            "f = mod.create_function('axpy')\n"
            "x = rs.randn(1000).astype('f'); y = rs.randn(1000).astype('f')\n"
            "dx = ctx.mem_alloc(4000); dy = ctx.mem_alloc(4000); dx.to_device(x); dy.to_device(y)\n"
            "f.set_args(dy, dx, numpy.array([2.5], 'f'), numpy.array([1000], numpy.int64))\n"
            "bs = f.max_potential_block_size()[1]; assert bs % 32 == 0 and bs >= 32\n"
            "f((4, 1, 1), (256, 1, 1))\n"
            "out = numpy.zeros(1000, 'f'); dy.to_host(out)\n"
            "assert numpy.abs(out - (y + 2.5 * x)).max() < 1e-5\n"
            "dy.memset32_async(); dy.to_host(out); assert not out.any()\n"
            "print('ok')\n")
    assert "ok" in _run(code)


@needs_reference
@pytest.mark.gpu
def test_reference_cuda_backend_matches_its_numpy_backend(tmp_path):
    """Same seeds, same data: 2 validation + 4 training minibatches of the reference
    StandardWorkflow (conv / max-pool / strict-relu / LRN / avg-pool / softmax, momentum + L2 +
    ortho) on its numpy back end and on its CUDA back end through the stand-in core - the
    oracle style of the reference's own unit tests (GPU == numpy)."""
    body = (TINY % BASE) + """
rr.setup_path()
from veles.loader import FullBatchLoader
class TinyLoader(FullBatchLoader):
    MAPPING = "tiny_loader"
    def load_data(self):
        rs = numpy.random.RandomState(3)
        self.class_lengths[:] = [0, 20, 40]
        labels = rs.randint(0, 10, 60)
        protos = rs.rand(10, 16, 16, 3)
        self.original_data.reset((protos[labels] + 0.3 * rs.rand(60, 16, 16, 3)).astype(self.dtype))
        self.original_labels = labels.tolist()
wf, dev = rr.launch(sys.argv[1], layers=tiny, minibatch_size=10, loader_name="tiny_loader")
wf.run(iterations=6)
out = {}
for i, f in enumerate(wf.forwards):
    if getattr(f, 'weights', None):
        f.weights.map_read(); f.bias.map_read()
        out['w%d' % i] = f.weights.mem.ravel()[:64].tolist(); out['b%d' % i] = f.bias.mem.ravel()[:8].tolist()
wf.forwards[-1].output.map_read(); out['y'] = wf.forwards[-1].output.mem.ravel()[:50].tolist()
wf.gds[0].gradient_weights.map_read(); out['gw0'] = wf.gds[0].gradient_weights.mem.ravel()[:64].tolist()
wf.evaluator.n_err.map_read(); out['n_err'] = [None if v is None else int(v) for v in wf.decision.epoch_n_err]; out['cls'] = wf.loader.minibatch_class
print(json.dumps(out))
"""
    tiny_pool = body.replace('"kx": 8, "ky": 8, "sliding": (8, 8)', '"kx": 4, "ky": 4, "sliding": (4, 4)')
    script = tmp_path / "tiny_ref.py"
    script.write_text(tiny_pool)
    res = {}
    for be in ("numpy", "cuda"):
        e = dict(os.environ)
        e.pop("PYTHONPATH", None)
        r = subprocess.run([sys.executable, "-W", "ignore", str(script), be], capture_output=True,
                           text=True, timeout=600, env=e, cwd=str(tmp_path))
        assert r.returncode == 0, r.stderr[-4000:]
        res[be] = json.loads(r.stdout.strip().splitlines()[-1])
    import numpy
    assert res["numpy"]["cls"] == 2 and res["cuda"]["cls"] == 2
    for x, y in zip(res["numpy"]["n_err"], res["cuda"]["n_err"]):
        assert (x is None) == (y is None)
        # (an untrained 10-class net on noise: most argmaxes are near-ties that fp32 vs fp64
        # summation order flips - the weights / outputs below are the real comparison)
        assert x is None or abs(x - y) <= 6
    errs = {}
    for k, v in res["numpy"].items():
        # (gradient_weights is not compared: the reference's numpy path stores the *stepped*
        # gradient there, its GPU path the raw one - SURVEY Appendix B)
        if k[0] in "wby":
            a, b = numpy.array(v), numpy.array(res["cuda"][k])
            errs[k] = float(numpy.abs(a - b).max() / max(numpy.abs(a).max(), 1e-4))
    # weights / outputs tight; biases loose: a conv bias gradient is a sum of ~2.5 K error terms of
    # both signs that nearly cancel, so a max-pooling near-tie routed differently (fp32 vs the
    # numpy path) moves it by a visible fraction of its own (tiny) magnitude
    lim = {"b": 0.3, "w": 2e-3, "y": 2e-2}
    bad = {k: e for k, e in errs.items() if e > lim[k[0]]}
    assert not bad, json.dumps(errs)
