"""package_export + the native C++ runtime (mirrors
/root/reference/tests/functional/test_package_export.py:98-136 and the libZnicz gtest suite)."""
import json
import os
import subprocess
import tarfile
import zipfile

import numpy
import pytest

from veles.znicz_b200.core.workflow import DummyLauncher
from veles.znicz_b200.models import mnist, cifar
from veles.znicz_b200.ops.all2all import All2AllTanh, All2AllSoftmax
from veles.znicz_b200 import native


def _train_fc(tmp_path):
    wf = mnist.build(
        layers=mnist.fc_layers(),
        loader_config={"minibatch_size": 20, "n_train": 100, "n_valid": 40,
                       "normalization_type": "linear"},
        decision_config={"max_epochs": 2, "fail_iterations": 10},
        snapshotter_config={"prefix": "exp", "interval": 100, "time_interval": 1e9})
    wf.initialize(device="numpy")
    wf.run()
    return wf


def _python_forward(wf, x):
    f0, f1 = wf.forwards
    h = 1.7159 * numpy.tanh(0.6666 * (x.reshape(len(x), -1).dot(f0.weights.mem.T) + f0.bias.mem))
    s = h.dot(f1.weights.mem.T) + f1.bias.mem
    e = numpy.exp(s - s.max(1, keepdims=True))
    return e / e.sum(1, keepdims=True)


def test_package_export_formats(tmp_path):
    wf = _train_fc(tmp_path)

    def validate(contents, files):
        unit0 = contents["units"][0]
        assert unit0["class"]["uuid"] == All2AllTanh.__id__
        assert contents["units"][1]["class"]["uuid"] == All2AllSoftmax.__id__
        for unit in contents["units"]:
            for attr in ("bias", "weights"):
                assert "%s.npy" % unit["data"][attr][1:] in files
        assert 1 in unit0["links"]
        assert contents["workflow"] == "MnistWorkflow"

    tgz = str(tmp_path / "pkg.tar.gz")
    wf.package_export(tgz, archive_format="tgz")
    with tarfile.open(tgz, "r:gz") as tar:
        validate(json.load(tar.extractfile("contents.json")), tar.getnames())
    z16 = str(tmp_path / "pkg16.zip")
    wf.package_export(z16, archive_format="zip", precision=16)
    with zipfile.ZipFile(z16) as az:
        validate(json.loads(az.read("contents.json").decode()), az.namelist())
        import io
        w = numpy.load(io.BytesIO(az.read([n for n in az.namelist() if "100x784" in n][0])))
        assert w.dtype == numpy.float16


def test_native_engine_matches_python_fc(tmp_path):
    wf = _train_fc(tmp_path)
    pkg = str(tmp_path / "mnist.zip")
    wf.package_export(pkg, precision=32)
    eng = native.NativeEngine(pkg)
    assert eng.num_units == 2
    x = numpy.random.RandomState(1).uniform(-1, 1, (7, 28, 28, 1)).astype(numpy.float32)
    y = eng.run(x.reshape(7, -1))
    # python forward on the same weights
    f0, f1 = wf.forwards
    h = 1.7159 * numpy.tanh(0.6666 * (x.reshape(7, -1).dot(f0.weights.mem.T) + f0.bias.mem))
    s = h.dot(f1.weights.mem.T) + f1.bias.mem
    e = numpy.exp(s - s.max(1, keepdims=True))
    ref = e / e.sum(1, keepdims=True)
    assert numpy.abs(y - ref).max() < 1e-5


def test_native_engine_matches_python_conv(tmp_path):
    wf = cifar.build(
        loader_config={"minibatch_size": 10, "n_train": 20, "n_valid": 10,
                       "normalization_type": "internal_mean"},
        decision_config={"max_epochs": 1, "fail_iterations": 10},
        snapshotter_config={"prefix": "exp", "interval": 100, "time_interval": 1e9})
    wf.initialize(device="numpy")
    wf.run()
    pkg = str(tmp_path / "cifar.zip")
    wf.package_export(pkg)
    eng = native.NativeEngine(pkg)
    assert eng.num_units == 12
    # reuse the workflow's own forward chain as the oracle
    x = wf.loader.minibatch_data.mem.copy()
    for u in wf.forwards:
        u.run()
    ref = wf.forwards[-1].output.mem
    y = eng.run(x)
    assert numpy.abs(y - ref).max() < 1e-4


def test_native_cpp_test_binary(tmp_path):
    wf = _train_fc(tmp_path)
    pkg = str(tmp_path / "mnist.zip")
    wf.package_export(pkg, precision=16)
    from veles.znicz_b200.native import _build_impl
    _build_impl.build(verbose=False)
    # functional check: python forward of a batch vs the C++ executors on the same package
    x = numpy.random.RandomState(5).uniform(-1, 1, (7, 784)).astype(numpy.float32)
    ref = _python_forward(wf, x)
    numpy.save(str(tmp_path / "x.npy"), x)
    numpy.save(str(tmp_path / "ref.npy"), ref.astype(numpy.float32))
    r = subprocess.run([_build_impl.TEST_BIN, pkg, str(tmp_path / "x.npy"),
                        str(tmp_path / "ref.npy")], stdout=subprocess.PIPE,
                       stderr=subprocess.STDOUT, text=True, timeout=120)
    assert r.returncode == 0, r.stdout
    assert "0 failures" in r.stdout and "functional cpu" in r.stdout


# the MNIST workflow package of the reference's libZnicz tests (tests/workflow_files/mnist.zip)
REF_PKG = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "libznicz_mnist.zip")


def test_native_loads_reference_package():
    eng = native.NativeEngine(REF_PKG)
    assert eng.num_units == 2
    y = eng.run(numpy.zeros((2, 784), numpy.float32))
    assert y.shape == (2, 10) and abs(float(y.sum()) - 2.0) < 1e-4


@pytest.mark.gpu
def test_native_cuda_matches_cpu(tmp_path):
    wf = cifar.build(
        loader_config={"minibatch_size": 10, "n_train": 20, "n_valid": 10,
                       "normalization_type": "internal_mean"},
        decision_config={"max_epochs": 1, "fail_iterations": 10},
        snapshotter_config={"prefix": "exp", "interval": 100, "time_interval": 1e9})
    wf.initialize(device="numpy")
    wf.run()
    pkg = str(tmp_path / "cifar.zip")
    wf.package_export(pkg)
    eng = native.NativeEngine(pkg)
    x = numpy.random.RandomState(2).uniform(-1, 1, (6, 32, 32, 3)).astype(numpy.float32)
    assert numpy.abs(eng.run(x, "cuda") - eng.run(x, "cpu")).max() < 1e-4
    # the conv layers (and every FC layer with >= 32 inputs) ran as split-bf16 tcgen05 launches
    assert eng.tensor_core_launches >= 3
    import os
    os.environ["ZNICZ_NATIVE_TC"] = "0"
    try:
        simt = native.NativeEngine(pkg)
        assert numpy.abs(simt.run(x, "cuda") - eng.run(x, "cpu")).max() < 1e-4
        assert simt.tensor_core_launches == 0
    finally:
        del os.environ["ZNICZ_NATIVE_TC"]


def test_cpu_only_cmake_configuration_builds_and_runs(tmp_path):
    """The portable configuration the Android script cross-compiles (-DZNICZ_WITH_CUDA=OFF, OpenMP
    loops; native/android/build_android.sh, reference: libZnicz/android/Android.mk.in) built with
    the host toolchain: library, CLI and the C++ tests, then inference on the reference's own
    packaged MNIST workflow. (No NDK in this image: the cross build itself stays unexecuted.)"""
    import shutil
    import subprocess
    if shutil.which("cmake") is None:
        pytest.skip("cmake not installed")
    src = os.path.join(os.path.dirname(native.__file__))
    build = str(tmp_path / "cpu")
    for cmd in (["cmake", "-S", src, "-B", build, "-DZNICZ_WITH_CUDA=OFF", "-DZNICZ_OPENMP=ON",
                 "-DCMAKE_BUILD_TYPE=Release"],
                ["cmake", "--build", build, "-j", "4"]):
        r = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
        assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    r = subprocess.run(["ctest", "--test-dir", build, "--output-on-failure"], capture_output=True,
                       text=True, timeout=300)
    assert r.returncode == 0, r.stdout[-2000:]
    numpy.zeros((2, 784), numpy.float32).tofile(tmp_path / "x.f32")
    r = subprocess.run([os.path.join(build, "znicz_infer"), REF_PKG, str(tmp_path / "x.f32"),
                        "2", "1", "1", "784"], capture_output=True, text=True, timeout=120)
    assert r.returncode == 0, r.stderr[-1000:]
    assert "output 2x1x1x10" in r.stdout, r.stdout
