#!/usr/bin/env python
"""Flagship benchmark: CIFAR-10 caffe-conv training throughput (images/s, whole job).

Contract (see the round brief): ``python bench.py --gpus N --steps K --warmup W`` (the
driver launches it with torch.distributed.run for N > 1); rank 0 prints ONE JSON line.

* model/config: /root/reference/samples/CIFAR10/cifar_caffe_config.py:52-145 — conv32-5p2 /
  maxpool3s2 / relu / LRN / conv32-5p2 / relu / avgpool3s2 / LRN / conv64-5p2 / relu / avgpool3s2 /
  softmax; minibatch 100 *per GPU* (the reference's per-process minibatch; weak scaling);
  SGD momentum 0.9 + L2 + factor_ortho, arbitrary_step LR policy; bf16 compute, fp32 master.
* ``value``: device-timed (CUDA events, max over ranks) through the public API
  (``CifarWorkflow.run(iterations=K)``): loader → forward → evaluator → decision → GDs with the
  fused (cross-GPU reduce +) update; the synthetic dataset (50000×32×32×3 fp32 = 614 MB > L2) is
  resident in HBM and every minibatch is a random row gather.
* ``e2e``: same loop in streaming mode — every step copies that step's inputs host→device from
  pinned memory and reads the step's result (n_err) device→host; timed by wall clock around
  the loop with synchronisation on both sides.
"""
import argparse
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

BATCH = 100


class ClockSampler(threading.Thread):
    """Samples SM clock + throttle reasons of one GPU while the timed region runs."""

    def __init__(self, index, period=0.02):
        super().__init__(daemon=True)
        self.index = index
        self.period = period
        self.samples = []
        self.reasons = set()
        self._stop_evt = threading.Event()
        self.max_mhz = None
        self.ok = False
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
            self.ok = True
        except Exception:
            self.nv = None

    def run(self):
        if not self.ok:
            return
        nv = self.nv
        names = {
            getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8): "hw_slowdown",
            getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40): "hw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20): "sw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4): "sw_power_cap",
        }
        while not self._stop_evt.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                try:
                    r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, name in names.items():
                    if r & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            time.sleep(self.period)

    def stop(self):
        self._stop_evt.set()
        self.join(timeout=1.0)
        s = sorted(self.samples)
        return {"sm_mhz": s[len(s) // 2] if s else None, "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(s)}


MODELS = {
    # name: (per-GPU batch, description)
    "cifar_caffe": (100, "cifar_caffe (conv32-5/maxpool3s2/relu/LRN/conv32-5/relu/avgpool/LRN/"
                         "conv64-5/relu/avgpool/softmax10)"),
    "mnist_conv": (6, "mnist_conv_config (conv64-5/mp2/conv87-5/mp2/fc791-softplus/softmax10)"),
    "alexnet": (128, "AlexNet 227x227x3 (5 conv, 2-group zero_filter, LRN, 3 FC, dropout)"),
    "lstm": (128, "lstm_seq 128 features x 32 steps -> LSTM 256 -> softmax10"),
}


def build_workflow(streaming, compute, graphs, n_train, model="cifar_caffe"):
    from veles.znicz_b200.core.config import root
    root.common.engine.compute_type = compute
    root.common.disable.snapshotting = True
    batch = _batch_of(model)
    common = dict(
        use_graphs=graphs,
        decision_config={"max_epochs": 1000000000, "fail_iterations": 1000000},
        snapshotter_config={"prefix": "bench", "interval": 1000000, "time_interval": 1e9})
    if model == "cifar_caffe":
        from veles.znicz_b200.models import cifar
        return cifar.build(
            loader_config={"minibatch_size": batch, "n_train": n_train, "n_valid": 0,
                           "n_test": 0, "normalization_type": "internal_mean",
                           "on_device": not streaming, "shuffle_limit": 2000000000}, **common)
    if model == "mnist_conv":
        from veles.znicz_b200.models import mnist
        return mnist.build(
            layers=mnist.conv_layers(), loader_name="synthetic_mnist",
            loader_config={"minibatch_size": batch, "n_train": min(n_train, 60000),
                           "n_valid": 0, "n_test": 0, "normalization_type": "linear",
                           "on_device": not streaming, "shuffle_limit": 2000000000}, **common)
    if model == "lstm":
        from veles.znicz_b200.models import lstm_seq
        return lstm_seq.build(
            # (per-rank dataset size constant under weak scaling, no epoch end inside the window)
            loader_config={"minibatch_size": batch,
                           "n_train": min(n_train, 32768) * max(1, int(os.environ.get("WORLD_SIZE", "1"))),
                           "n_valid": 0,
                           "n_test": 0, "on_device": not streaming,
                           "shuffle_limit": 2000000000}, **common)
    from veles.znicz_b200.models import alexnet
    return alexnet.build(
        loader_name="synthetic_imagenet", layers=alexnet.alexnet_layers(1000),
        # (per-rank dataset size constant under weak scaling and larger than the measured window:
        # an epoch end - metric reduction incl. a 1000 x 1000 confusion matrix, decision - costs
        # ~13 ms and belongs to the epoch, not to the step)
        loader_config={"minibatch_size": batch,
                       "n_train": min(n_train, int(os.environ.get("ZNICZ_BENCH_ALEXNET_SAMPLES", "5120"))) *
                       max(1, int(os.environ.get("WORLD_SIZE", "1"))),
                       "n_valid": 0,
                       "n_test": 0, "n_classes": 1000, "normalization_type": "internal_mean",
                       "on_device": not streaming, "shuffle_limit": 2000000000}, **common)


GRAPH_CAPTURE_STEPS = 6
ALIGN_STEPS = 3          # untimed, after the pre-timing barrier of a multi-rank run


def _batch_of(model):
    # ZNICZ_BENCH_BATCH: diagnostic only (host- vs device-bound check); the reported config
    # carries whatever batch actually ran
    return int(os.environ.get("ZNICZ_BENCH_BATCH", MODELS[model][0]))


DUMP_SAMPLE = 1 << 19    # elements --dump-outputs keeps of a larger array (fixed, seeded sample)


def dump_outputs(wf, out_dir):
    """Writes what the last training step left to the caller: the network output of the last
    minibatch, the evaluator's error count and every layer's weights and bias, as float32
    ``<out_dir>/<name>.npy``. An array of more than DUMP_SAMPLE elements is replaced by the
    same seeded sample of its flattened elements on every run, so no file exceeds 2 MB."""
    import numpy
    arrays = {"output": wf.forwards[-1].output}
    if getattr(wf.evaluator, "n_err", None):
        arrays["n_err"] = wf.evaluator.n_err
    for i, f in enumerate(wf.forwards):
        for attr in ("weights", "bias"):
            if getattr(f, attr, None):
                arrays["layer%02d_%s_%s" % (i, f.name, attr)] = getattr(f, attr)
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        a.map_read()
        v = numpy.asarray(a.mem, dtype=numpy.float32)
        if v.size > DUMP_SAMPLE:
            pick = numpy.random.RandomState(v.size).choice(v.size, DUMP_SAMPLE, replace=False)
            v = v.ravel()[numpy.sort(pick)]
        numpy.save(os.path.join(out_dir, name + ".npy"), v)


def run_arm(args, streaming):
    import torch
    if os.environ.get("ZNICZ_OVERLAP_WGRAD") == "0":        # diagnostic
        from veles.znicz_b200.core.config import root
        root.common.engine.overlap_wgrad = False
    if os.environ.get("ZNICZ_LOADER_EARLY") == "0":         # diagnostic
        from veles.znicz_b200.core.config import root
        root.common.engine.loader_early_pull = False
    if os.environ.get("ZNICZ_LOADER_PULL") == "0":          # diagnostic
        from veles.znicz_b200.core.config import root
        root.common.engine.loader_pull = False
    if os.environ.get("ZNICZ_LOADER_PREFETCH") == "0":      # diagnostic
        from veles.znicz_b200.core.config import root
        root.common.engine.loader_prefetch = False
    import torch.distributed as dist
    from veles.znicz_b200.kernels import api
    world = int(os.environ.get("WORLD_SIZE", "1"))
    wf = build_workflow(streaming, args.dtype, not args.no_graphs, args.n_train, args.model)
    wf.initialize(device="cuda")
    dev = wf.device
    reader = None
    if streaming:
        from veles.znicz_b200.utils.step_reader import StepResultReader
        reader = StepResultReader(wf.evaluator)
        wf.step_hooks_.append(reader)
    # CUDA graphs are captured during the first steps of a workflow (2 eager passes, the forward /
    # backward captures, then the fused train-step capture): run those outside the timed region
    # whatever --warmup says, then the W warm-up steps proper
    wf.run(iterations=GRAPH_CAPTURE_STEPS)
    if args.warmup > 0:
        wf.run(iterations=args.warmup)
    torch.cuda.synchronize()
    if os.environ.get("ZNICZ_BENCH_STATS"):
        wf.real_loader.__dict__["prof_"] = [0.0, 0.0, 0.0, 0]
    # Everything host-side that can skew the ranks against each other happens BEFORE the final
    # barrier: nvmlInit() enumerates all GPUs under a driver lock (tens of ms, serialised over 8
    # processes) and a late rank makes every peer spin inside the step's cross-GPU flag barrier,
    # on the device, inside the timed events (round-1 driver run: 0.28 efficiency at 8 GPUs).
    sampler = ClockSampler(dev.index)
    e0 = torch.cuda.Event(enable_timing=True)
    e1 = torch.cuda.Event(enable_timing=True)
    sampler.start()
    if world > 1:
        torch.cuda.synchronize()
        dist.barrier()
        # untimed aligned steps: the step's own cross-GPU barrier lines the devices up, and the
        # hosts get their launch queues ahead of the devices again after the barrier's drain
        wf.run(iterations=ALIGN_STEPS)
    if streaming:
        torch.cuda.synchronize()      # e2e is wall-clock timed: synchronised on both sides
    launches0 = api.counters["launches"]
    t0 = time.perf_counter()
    e0.record()
    n_steps = wf.run(iterations=args.steps)
    e1.record()
    t_enq = time.perf_counter()       # host finished enqueueing (the device may still be busy)
    torch.cuda.synchronize()
    t1 = time.perf_counter()
    if n_steps != args.steps:
        raise RuntimeError("the timed region ran %d steps instead of %d" % (n_steps, args.steps))
    if args.dump_outputs and not streaming and int(os.environ.get("RANK", "0")) == 0:
        dump_outputs(wf, args.dump_outputs)
    if world > 1:
        dist.barrier()
    clocks = sampler.stop()
    ms_dev = e0.elapsed_time(e1)
    ms_wall = (t1 - t0) * 1e3
    t = torch.tensor([ms_dev, ms_wall], dtype=torch.float64, device=dev.torch_device)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_dev, ms_wall = float(t[0]), float(t[1])
    res = {
        "ms_dev": ms_dev, "ms_wall": ms_wall, "clocks": clocks,
        "launches": api.counters["launches"] - launches0,
        "h2d": getattr(wf.real_loader, "h2d_bytes_per_step", 0),
        "d2h": reader.bytes_per_step if reader else 0,
        "n_err": int(reader.last[0]) if reader and reader.last is not None else None,
        "dp_algo": getattr(getattr(wf, "fused_step_", None), "algo_name", None),
        "dp_gradients": getattr(getattr(wf, "dp_", None), "gradient_mode", None),
    }
    if os.environ.get("ZNICZ_BENCH_STATS") and int(os.environ.get("RANK", "0")) == 0:
        sys.stderr.write("host enqueue %.4f ms/step, device %.4f ms/step, drain after enqueue "
                         "%.3f ms\n" % ((t_enq - t0) * 1e3 / args.steps, ms_dev / args.steps,
                                        (t1 - t_enq) * 1e3))
        pr = wf.real_loader.__dict__.get("prof_")
        if pr and pr[3]:
            sys.stderr.write("loader per step: slot wait %.1f us, host assembly %.1f us, "
                             "H2D enqueue %.1f us\n" % tuple(1e6 * v / pr[3] for v in pr[:3]))
        pk = wf.real_loader.__dict__.get("_packed_")
        if pk:
            sys.stderr.write("loader prefetch hits: %d\n" % pk.get("hits", 0))
        rows = sorted(((u.total_run_time, u._run_calls, u.name) for u in wf.units), reverse=True)
        for t_, c_, n_ in rows[:25]:
            sys.stderr.write("  %-28s calls %6d  host %9.3f ms  (%.1f us/call)\n" % (
                n_, c_, t_ * 1e3, 1e6 * t_ / max(c_, 1)))
        try:
            sys.stderr.write("conv launches (python-side, incl. capture): pair %d, im2col-TMA %d\n" % (
                dev.ext.conv_pair_launches(), dev.ext.im2col_tma_launches()))
        except Exception:
            pass
        for sg in getattr(wf, "segments_", []):
            sys.stderr.write("  segment %s: replays %d eager %d\n" % (
                sg.name, sg.replays, sg.eager_runs))
    del wf
    return res


def _reference_timed(args, rank, world, streaming):
    """K training minibatches of the unmodified reference sample on its stock cuda_run path
    (see baseline/run_reference.py). Device-timed with driver-API events on the (legacy
    default) stream every reference kernel and cuBLAS call uses; wall clock for e2e."""
    sys.path.insert(0, os.path.join(ROOT, "baseline"))
    import run_reference as rr
    wf, dev = rr.launch("cuda", force_numpy_loader=streaming, pinned=streaming)
    import cuda4py
    read_back = {"n": 0}
    if streaming:
        def hook(_wf):
            wf.evaluator.n_err.map_read()        # the step's result, device -> host
            read_back["n"] = int(wf.evaluator.n_err.mem[0])
        wf.step_hooks_.append(hook)
    # the reference serves VALID (10000 samples = 100 forward-only minibatches) before TRAIN:
    # walk through them untimed, then W warm-up training steps
    valid_steps = wf.loader.class_lengths[1] // wf.loader.max_minibatch_size
    wf.run(iterations=valid_steps)
    assert wf.loader.minibatch_class == 1 and bool(wf.loader.last_minibatch)
    wf.run(iterations=args.warmup)
    assert wf.loader.minibatch_class == 2
    dev.sync()
    sampler = ClockSampler(dev.index)
    sampler.start()
    if world > 1:
        import torch.distributed as dist
        dist.barrier()
    e0, e1 = cuda4py.Event(), cuda4py.Event()
    l0, g0 = cuda4py.dry_stats["launches"], cuda4py.dry_stats["gemms"]
    h0, d0 = dev.h2d_bytes, dev.d2h_bytes
    t0 = time.perf_counter()
    e0.record()
    n = wf.run(iterations=args.steps)
    e1.record()
    dev.sync()
    t1 = time.perf_counter()
    assert n == args.steps and wf.loader.minibatch_class == 2, "timed region left TRAIN"
    ms_dev = e0.elapsed_ms(e1)
    clocks = sampler.stop()
    res = {"ms_dev": ms_dev, "ms_wall": (t1 - t0) * 1e3, "clocks": clocks,
           "launches": cuda4py.dry_stats["launches"] - l0, "gemms": cuda4py.dry_stats["gemms"] - g0,
           "h2d": (dev.h2d_bytes - h0) / args.steps, "d2h": (dev.d2h_bytes - d0) / args.steps,
           "n_err": read_back["n"], "batch": wf.loader.max_minibatch_size}
    if world > 1:
        import torch
        import torch.distributed as dist
        t = torch.tensor([res["ms_dev"], res["ms_wall"]], dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        res["ms_dev"], res["ms_wall"] = float(t[0]), float(t[1])
        dist.barrier()
    del wf
    return res


def run_reference_arm(args, rank, world):
    """``--impl reference``: the UNMODIFIED reference (baseline/_ref) on its own stock GPU path;
    the product package is never imported in this process."""
    try:
        if not os.environ.get("CUDA4PY_DRY"):
            # fail fast (and before any rendezvous) on a box without a GPU
            from cuda.bindings import driver as _drv
            err, = _drv.cuInit(0)
            n_dev = _drv.cuDeviceGetCount()[1] if int(err) == 0 else 0
            if int(err) != 0 or n_dev < 1:
                raise RuntimeError("no CUDA device visible (cuInit: %s)" % getattr(err, "name", err))
        if world > 1:
            os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
            import torch.distributed as dist
            dist.init_process_group(backend="gloo", rank=rank, world_size=world)
        main_res = _reference_timed(args, rank, world, streaming=False)
        e2e_res = None if args.skip_e2e else _reference_timed(args, rank, world, streaming=True)
    except Exception as exc:        # never a fake number: say why the arm could not run
        if rank == 0:
            import traceback
            sys.stderr.write(traceback.format_exc())
            print(json.dumps({"impl": "reference",
                              "unavailable": "%s: %s" % (type(exc).__name__, str(exc)[:300])}))
        return 0
    if rank != 0:
        return 0
    n = max(world, 1)
    batch = main_res["batch"]
    images = args.steps * batch * n
    out = {
        "impl": "reference",
        "metric": "CIFAR-10 caffe-conv training images/sec (whole job, device-timed, max over ranks)",
        "value": round(images / (main_res["ms_dev"] / 1e3), 1), "unit": "images/s", "n_gpus": n,
        "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": round(main_res["ms_dev"] / args.steps, 5),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "fp32", "data": "synthetic",
        "config": {"model": MODELS["cifar_caffe"][1], "global_batch": batch * n,
                   "per_gpu_batch": batch, "image": "32x32x3",
                   "parallelism": "dp1" if n == 1 else
                   "%d independent replicas, no parameter exchange (upper bound of the "
                   "reference's asynchronous master/slave scheme, whose ZeroMQ/Twisted "
                   "transport lives in the absent Veles core)" % n,
                   "code": "unmodified Samsung/veles.znicz (baseline/_ref, sha256 manifest): "
                           "samples/CIFAR10/cifar.py + cifar_caffe_config.py, stock cuda_run "
                           "path (NVRTC build of its cuda/*.cu + cuBLAS SGEMM, precision_type "
                           "float)",
                   "core": "baseline/veles_core: stand-in for the absent Veles core / cuda4py / "
                           "zope.interface (unit graph, Array map/unmap, NVRTC, driver-API "
                           "launches); none of veles.znicz_b200 is imported",
                   "untimed": "100 validation minibatches + W warm-up training steps",
                   "l2": "614 MB fp32 dataset resident in HBM, random rows gathered each step"},
        "clocks": {k: main_res["clocks"][k] for k in ("sm_mhz", "sm_max_mhz", "reasons")},
        "gpu_launches": main_res["launches"] + main_res["gemms"],
        "kernel_launches": main_res["launches"], "cublas_gemms": main_res["gemms"],
    }
    if e2e_res is not None:
        out["e2e"] = {
            "value": round(images / (e2e_res["ms_wall"] / 1e3), 1), "unit": "images/s",
            "h2d_bytes_per_step": int(e2e_res["h2d"]), "d2h_bytes_per_step": int(e2e_res["d2h"]),
            "ms_per_step": round(e2e_res["ms_wall"] / args.steps, 5),
            "timing": "wall clock around workflow.run(), device synchronised on both sides; "
                      "loader force_numpy=True: every minibatch is assembled on the host in "
                      "page-locked memory and uploaded, n_err read back every step",
            "last_n_err": e2e_res["n_err"]}
    print(json.dumps(out))
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=2000)
    ap.add_argument("--warmup", type=int, default=50)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference", "baseline"])
    ap.add_argument("--dtype", default="bf16", choices=["bf16", "fp32"])
    ap.add_argument("--no-graphs", action="store_true")
    ap.add_argument("--n-train", type=int, default=50000)
    ap.add_argument("--skip-e2e", action="store_true")
    ap.add_argument("--strong-global-batch", type=int, default=0,
                    help="strong scaling: fix the GLOBAL batch (per-GPU batch = this / N) instead "
                         "of the per-GPU batch of the config")
    ap.add_argument("--model", default="cifar_caffe", choices=sorted(MODELS),
                    help="cifar_caffe is the north-star config; the others are extra data points")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps write what the last one computed (network output, "
                         "error count, every layer's weights and bias) as DIR/<name>.npy; the "
                         "inputs are seeded, so runs with the same arguments can be compared")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        return run_reference_arm(args, rank, world)
    if args.impl == "baseline":
        # reference-equivalent decomposition inside this repo: fp32, exact SIMT GEMM/conv
        # kernels, one python-driven launch per reference kernel (no CUDA graphs, per-tensor
        # update launches, stand-alone activation units)
        args.dtype = "fp32"
        args.no_graphs = True
        from veles.znicz_b200.core.config import root as _root
        _root.common.engine.fused_step = False
        _root.common.engine.fuse_activations = False
    if args.warmup < 3:
        args.warmup = 3
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
    if args.strong_global_batch:
        if args.strong_global_batch % max(world, 1):
            raise SystemExit("--strong-global-batch must be divisible by the number of GPUs")
        os.environ["ZNICZ_BENCH_BATCH"] = str(args.strong_global_batch // max(world, 1))
    main_res = run_arm(args, streaming=False)
    e2e_res = None if args.skip_e2e else run_arm(args, streaming=True)
    if rank != 0:
        return 0
    n = max(world, 1)
    batch = _batch_of(args.model)
    images = args.steps * batch * n
    value = images / (main_res["ms_dev"] / 1e3)
    unit_name = "sequences" if args.model == "lstm" else "images"
    out = {
        "metric": {"cifar_caffe": "CIFAR-10 caffe-conv", "mnist_conv": "MNIST conv",
                   "alexnet": "AlexNet", "lstm": "LSTM sequence"}[args.model] +
                  " training %s/sec (whole job, device-timed, max over ranks)" % unit_name,
        "value": round(value, 1), "unit": unit_name + "/s", "n_gpus": n, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": round(main_res["ms_dev"] / args.steps, 5),
        "higher_is_better": True, "scaling": "strong" if args.strong_global_batch else "weak",
        "vs_baseline": None,
        "dtype": args.dtype, "data": "synthetic",
        "impl": "znicz_b200" if args.impl == "b200" else "baseline(in-repo, reference-equivalent)",
        "config": {"model": MODELS[args.model][1],
                   "global_batch": batch * n, "per_gpu_batch": batch,
                   "seq_len": 32 if args.model == "lstm" else None,
                   "image": {"cifar_caffe": "32x32x3", "mnist_conv": "28x28x1",
                             "alexnet": "227x227x3", "lstm": None}[args.model],
                   "parallelism": "dp%d" % n,
                   "dp_collective": ("fused peer-memory reduce+update kernel (no NCCL on the "
                                     "step path), algo=%s" % main_res.get("dp_algo")
                                     if os.environ.get("ZNICZ_DP_MODE", "fused") ==
                                     "fused" else "NCCL all-reduce baseline") if n > 1 else None,
                   "dp_gradients": main_res.get("dp_gradients") if n > 1 else None,
                   "optimizer": ("SGD momentum 0.9 + L2 5e-4 + factor_ortho 1e-3, "
                                 "arbitrary_step LR") if args.model == "cifar_caffe" else
                                "SGD momentum + L2 as in the model's layer config",
                   "cuda_graphs": not args.no_graphs,
                   "untimed_graph_capture_steps": GRAPH_CAPTURE_STEPS,
                   "untimed_align_steps_after_barrier": ALIGN_STEPS if n > 1 else 0,
                   "l2": "inputs larger than L2: the whole fp32 dataset (614 MB for 50000x32x32x3 "
                         "in the CIFAR config) is resident in HBM, random minibatch rows gathered "
                         "each step"},
        "clocks": {k: main_res["clocks"][k] for k in ("sm_mhz", "sm_max_mhz", "reasons")},
        "gpu_launches": main_res["launches"],
    }
    if e2e_res is not None:
        out["e2e"] = {
            "value": round(images / (e2e_res["ms_wall"] / 1e3), 1), "unit": unit_name + "/s",
            "h2d_bytes_per_step": int(e2e_res["h2d"]), "d2h_bytes_per_step": int(e2e_res["d2h"]),
            "ms_per_step": round(e2e_res["ms_wall"] / args.steps, 5),
            "timing": "wall clock around the public-API loop, cuda synchronize on both sides",
            "last_n_err": e2e_res["n_err"]}
    print(json.dumps(out))
    return 0


if __name__ == "__main__":
    sys.exit(main())
