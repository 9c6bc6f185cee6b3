"""Synchronous data parallelism: replicated weights, fused reduce+update.

Replaces the reference's asynchronous master/slave parameter exchange
(/root/reference/nn_units.py:644-694, SURVEY §2.6): every rank runs the same unit
graph on its shard of the minibatch; after a GD unit produced its local gradient the
*fused update kernel* reads the gradient tiles of all ranks straight out of their
HBM over NVLink (peer pointers from a symmetric-memory rendezvous), sums them in
rank order — so all replicas compute bit-identical updates — applies the SGD step
and writes the new weights locally. No NCCL call is on that path; NCCL (or gloo on
CPU) is used for bootstrap, metric reduction at epoch ends and as the *baseline*
implementation (``mode="nccl"``) the fused path is measured against.
"""
from __future__ import annotations

import os

import numpy

from ..core.config import root


class RankFailure(RuntimeError):
    """A peer rank died or stalled (raised by ``DataParallel.check_ranks``)."""


class DataParallel(object):
    def __init__(self, device, rank, world_size, mode=None):
        self.device = device
        self.rank = rank
        self.world_size = world_size
        self.mode = mode or os.environ.get("ZNICZ_DP_MODE", "fused")
        self.symm = None
        self._step = 0
        # Gradient semantics: "mean" (default) divides the cross-rank gradient sum by the world
        # size, so N ranks at per-GPU batch b take exactly the step of ONE process at batch N*b
        # with the same hyper-parameters (every evaluator already divides by its local batch);
        # "sum" keeps the plain sum (step N times larger - the reference's asynchronous
        # master applied every slave's gradient in full, /root/reference/nn_units.py:679-691).
        from ..core.config import root
        self.gradient_mode = os.environ.get(
            "ZNICZ_DP_GRADIENTS", root.common.engine.get("dp_gradients", "mean"))
        if self.gradient_mode not in ("mean", "sum"):
            raise ValueError("dp_gradients must be 'mean' or 'sum'")
        self.gradient_scale = 1.0 / world_size if self.gradient_mode == "mean" else 1.0

    @classmethod
    def from_env(cls, device):
        ws = int(os.environ.get("WORLD_SIZE", "1"))
        if ws <= 1:
            return None
        import torch.distributed as dist
        rank = int(os.environ.get("RANK", "0"))
        if not dist.is_initialized():
            backend = "nccl" if device is not None and device.is_cuda else "gloo"
            kw = {}
            if backend == "nccl":
                kw["device_id"] = device.torch_device
            # failure detection: a collective (or the monitored barrier of check_ranks) that a
            # dead rank never joins raises after this many seconds instead of hanging the job
            import datetime
            kw["timeout"] = datetime.timedelta(seconds=float(os.environ.get(
                "ZNICZ_DP_TIMEOUT_S", root.common.engine.get("dp_timeout_s", 600))))
            attempt = int(os.environ.get("TORCHELASTIC_RESTART_COUNT", "0"))
            if attempt > 0:
                # torchrun gives a restarted group the rendezvous store of the failed attempt,
                # which still holds the dead ranks' process-group keys (gloo peer addresses):
                # a peer reading one connects to a closed port. Keep each attempt's keys apart.
                store, _, _ = next(dist.rendezvous("env://", rank, ws, timeout=kw["timeout"]))
                kw["store"] = dist.PrefixStore("attempt%d/" % attempt, store)
            dist.init_process_group(backend=backend, rank=rank, world_size=ws, **kw)
        return cls(device, rank, ws)

    def check_ranks(self, timeout_s=None):
        """Epoch-end health check: every rank must arrive within ``timeout_s``; a missing rank
        raises ``RankFailure`` naming it (gloo) or the backend's timeout error (nccl). Together
        with rank-0 snapshots, ``--snapshot latest`` and ``torchrun --max-restarts`` this is the
        recovery path: the group is restarted and resumes from the last snapshot - on fewer
        ranks if need be (the loader re-shards). The reference's master re-queued the jobs of a
        dropped slave (``drop_slave``, /root/reference/nn_rollback.py:94-95); with synchronous
        replicas there is nothing to re-queue, the epoch is simply repeated."""
        import datetime
        import torch.distributed as dist
        t = datetime.timedelta(seconds=float(timeout_s if timeout_s is not None else os.environ.get(
            "ZNICZ_DP_TIMEOUT_S", root.common.engine.get("dp_timeout_s", 600))))
        try:
            if dist.get_backend() == "gloo":
                dist.monitored_barrier(timeout=t, wait_all_ranks=True)
            else:
                dist.barrier()
        except RuntimeError as e:
            raise RankFailure("rank %d: a peer did not reach the epoch-end barrier: %s" % (
                self.rank, str(e).splitlines()[0] if str(e) else type(e).__name__)) from e

    # -- wiring ---------------------------------------------------------------------------
    def attach(self, workflow):
        """Give every GD unit / decision of ``workflow`` this context, shard the loader
        and broadcast rank 0's initial weights so replicas start identical."""
        from ..ops.nn_units import GradientDescentBase, Forward
        loader = workflow.real_loader
        loader.shard(self.rank, self.world_size)
        for u in workflow.units:
            if isinstance(u, GradientDescentBase):
                u.dp_ = self
            if "dp_" in u.__dict__ and u is not workflow:
                u.dp_ = self
        self.broadcast_parameters(
            [u for u in workflow.forwards if isinstance(u, Forward)])
        if self.device is not None and self.device.is_cuda:
            self.device.ext.set_dp_gradient_scale(self.gradient_scale)
        if self.device is not None and self.device.is_cuda and self.mode == "fused":
            from .symmetric import SymmetricGradients
            gds = [g for g in workflow.gds if g is not None and g.weights]
            self.symm = SymmetricGradients(self, gds)
            # the epoch-end metric exchange buffers exist before the first epoch ends (a
            # symmetric allocation + rendezvous costs tens of milliseconds)
            ev = getattr(workflow, "evaluator", None)
            cm = getattr(ev, "confusion_matrix", None)
            self._metric_state(64 + (int(cm.size) if cm is not None and cm else 0))

    def broadcast_parameters(self, forwards):
        import torch
        import torch.distributed as dist
        for f in forwards:
            for arr in (f.weights, f.bias):
                if not arr:
                    continue
                if arr.devmem is not None:
                    t = arr.dev
                    dist.broadcast(t, src=0)
                    arr.dev_written()
                else:
                    t = torch.from_numpy(arr.mem)
                    dist.broadcast(t, src=0)
            if getattr(f, "on_cuda", False):
                f.refresh_shadows()

    # -- reductions on the slow path (epoch ends) ----------------------------------------------
    # -- epoch-end metrics through the symmetric-memory mechanism (no library collective) ---------
    def _metric_state(self, n):
        import torch
        import torch.distributed as dist
        st = self.__dict__.get("_mstate_")
        if st is None or st["cap"] < n:
            cap = max(int(n), 4096)
            t, h = self.symm._alloc(2 * cap, torch.float64)
            t.zero_()
            flags, epoch_ptr = self.symm.sync_state(("metrics", cap))
            st = {"cap": cap, "t": t, "h": h, "ptrs": [int(p) for p in h.buffer_ptrs],
                  "flags": flags, "epoch_ptr": epoch_ptr, "calls": 0,
                  "out": torch.zeros(cap, dtype=torch.float64, device=self.device.torch_device)}
            torch.cuda.synchronize()
            dist.barrier()
            self.__dict__["_mstate_"] = st
        return st

    def _reduce_symm(self, sums, maxs):
        """Element-wise SUM of the ``sums`` arrays and MAX of the ``maxs`` arrays over all ranks by
        ``metric_reduce_k`` (csrc/update.cu): every rank publishes its packed doubles in a
        symmetric slot and reduces all peers' slots in fixed rank order."""
        import torch
        flat = [numpy.asarray(a, dtype=numpy.float64).ravel() for a in sums + maxs]
        n_sum = sum(a.size for a in flat[:len(sums)])
        n = sum(a.size for a in flat)
        st = self._metric_state(n)
        st["calls"] += 1
        slot = st["calls"] & 1
        packed = torch.from_numpy(numpy.concatenate(flat) if flat else numpy.zeros(0))
        st["t"][slot * n:slot * n + n].copy_(packed)
        self.device.ext.metric_reduce(st["ptrs"], st["flags"], st["epoch_ptr"], self.rank, st["out"],
                                      n_sum, n - n_sum, slot)
        res = st["out"][:n].cpu().numpy()
        out, off = [], 0
        for a in flat:
            out.append(res[off:off + a.size])
            off += a.size
        return out[:len(sums)], out[len(sums):]

    def reduce_metrics(self, n_err=None, confusion=None, max_err=None, mse_metrics=None):
        import torch
        import torch.distributed as dist
        if self.symm is not None and os.environ.get("ZNICZ_METRICS_NCCL", "0") != "1":
            def host(arr):
                arr.map_read()
                return arr.mem
            sums = [a for a in (n_err, confusion) if a is not None and a]
            maxs = [a for a in (max_err,) if a is not None and a]
            s_in = [host(a) for a in sums]
            m_in = [host(a) for a in maxs]
            mse = mse_metrics is not None and bool(mse_metrics)
            if mse:
                m = host(mse_metrics)
                s_in.append(numpy.array([float(m[0])]))
                m_in.append(numpy.array([float(m[1]), -float(m[2])]))
            s_out, m_out = self._reduce_symm(s_in, m_in)
            for arr, res in zip(sums + maxs, s_out[:len(sums)] + m_out[:len(maxs)]):
                arr.map_invalidate()
                arr.mem[...] = res.reshape(arr.mem.shape).astype(arr.mem.dtype)
                arr.unmap()
            if mse:
                mse_metrics.map_invalidate()
                mse_metrics.mem[0] = s_out[-1][0]
                mse_metrics.mem[1] = m_out[-1][0]
                mse_metrics.mem[2] = -m_out[-1][1]
                mse_metrics.unmap()
            return

        def _reduce(arr, op):
            if arr is None or not arr:
                return
            arr.map_read()
            t = torch.from_numpy(numpy.ascontiguousarray(arr.mem))
            if self.device is not None and self.device.is_cuda:
                t = t.to(self.device.torch_device)
            dist.all_reduce(t, op=op)
            arr.map_invalidate()
            arr.mem[...] = t.cpu().numpy()
            arr.unmap()
        _reduce(n_err, dist.ReduceOp.SUM)
        _reduce(confusion, dist.ReduceOp.SUM)
        _reduce(max_err, dist.ReduceOp.MAX)
        if mse_metrics is not None and mse_metrics:
            mse_metrics.map_read()
            m = mse_metrics.mem
            vals = torch.tensor([float(m[0]), float(m[1]), -float(m[2])],
                                dtype=torch.float64)
            if self.device is not None and self.device.is_cuda:
                vals = vals.to(self.device.torch_device)
            s = vals[:1].clone()
            dist.all_reduce(s, op=dist.ReduceOp.SUM)
            mx = vals[1:].clone()
            dist.all_reduce(mx, op=dist.ReduceOp.MAX)
            mse_metrics.map_invalidate()
            m[0] = float(s[0])
            m[1] = float(mx[0])
            m[2] = -float(mx[1])
            mse_metrics.unmap()

    def all_reduce_scalar(self, value, op="sum"):
        import torch
        import torch.distributed as dist
        if self.symm is not None and op in ("sum", "max", "min") and \
                os.environ.get("ZNICZ_METRICS_NCCL", "0") != "1":
            v = numpy.array([float(value)])
            if op == "sum":
                return float(self._reduce_symm([v], [])[0][0][0])
            sign = -1.0 if op == "min" else 1.0
            return sign * float(self._reduce_symm([], [sign * v])[1][0][0])
        t = torch.tensor([float(value)], dtype=torch.float64)
        if self.device is not None and self.device.is_cuda:
            t = t.to(self.device.torch_device)
        dist.all_reduce(t, op={"sum": dist.ReduceOp.SUM, "min": dist.ReduceOp.MIN,
                               "max": dist.ReduceOp.MAX}[op])
        return float(t[0])

    def barrier(self):
        import torch.distributed as dist
        dist.barrier()

    # -- numpy / gloo gradient path (CPU multi-process tests) ------------------------------------
    def all_reduce_numpy(self, arr):
        import torch
        import torch.distributed as dist
        t = torch.from_numpy(arr)
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        if self.gradient_scale != 1.0:
            arr *= arr.dtype.type(self.gradient_scale)
        return arr
