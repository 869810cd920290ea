"""A whole training step of a converted model as ONE CUDA graph (EXTENSION; the reference has no counterpart).

The reference's layers are host-scheduled: step counters, schedules and EMA indices are Python values
(qsparse/quantize.py:340-348, sparse.py:82-113), i.e. frozen into the launch arguments of a captured graph.  In
*graph mode* the steady-state routes of this package index their running means by DEVICE counters instead — the
prune callback's own ``t`` Parameter, a per-quantizer int64 counter — which the kernels read and advance
themselves (``step_counter_dev`` of the C-ABI), so a replay computes exactly what the next eager step would.

    step = GraphedTrainStep(model, train_step, warmup=3)     # model already in its steady state
    for x, y in data:
        static_x.copy_(x); static_y.copy_(y)
        step.replay()
    step.sync_host()                                          # host counters catch up with the device

Capturable routes: every stock quantizer (Decimal / Scaler / Adaptive / Percentile; per tensor, per channel, the
row-resident weight kernel, the fused weight chain), the stock magnitude prune callback with a channel mask or a
full-size mask (the one-pass step K9, per layer or batched by ``WeightSetPruner``) or a frozen mask, and fused
prune -> quantize activation sites
(``convert(..., fuse=True)``; Decimal / Scaler, and Adaptive whose lines index keeps a constant offset to the prune
callback's counter, up to 1 024 channels), past their timeouts and schedules, with the default mask refresh (every step, never
stopping).  Every other stateful route (gradient / l0 importance, sparser refresh intervals on full-size masks,
group-wise scale sharing before its clustering step, ...) raises ``NotCapturable`` while graph mode
is on rather than silently freezing a step index."""
from __future__ import annotations

import contextlib
from typing import Callable, List

import torch
import torch.nn as nn

_ACTIVE = False


class NotCapturable(RuntimeError):
    pass


def active() -> bool:
    return _ACTIVE


@contextlib.contextmanager
def graph_mode():
    global _ACTIVE
    prev, _ACTIVE = _ACTIVE, True
    try:
        yield
    finally:
        _ACTIVE = prev


def require_eager(what: str):
    """Called by every route that passes a HOST step index to a kernel."""
    if _ACTIVE:
        raise NotCapturable(f"{what} indexes its running mean by a host-side step counter and cannot be part of a "
                            "captured training step (GraphedTrainStep supports per-tensor Decimal / Scaler layers and "
                            "fused prune -> quantize activation sites in their steady state)")


NO_REFRESH_INTERVAL = 1 << 30   # graph-mode kernels take the refresh INTERVAL: this one never comes round


def host_index(quantizer) -> int:
    """how many estimation calls the quantizer has made (``t``; AdaptiveQuantizer keeps a device Parameter like the
    reference and the host count beside it)"""
    t = quantizer.t
    return int(getattr(quantizer, "_t_host", 0)) if isinstance(t, torch.Tensor) else int(t)


def quantizer_counter(quantizer, device) -> torch.Tensor:
    """the int64 device twin of the quantizer's call count (created and set OUTSIDE capture by GraphedTrainStep);
    kernels index their running mean by it, the caller (or the step kernel itself) advances it"""
    c = getattr(quantizer, "_t_dev", None)
    if c is None or c.device != device:
        if torch.cuda.is_current_stream_capturing():
            raise NotCapturable("a quantizer met its first graph-mode step during capture: run warm-up steps first")
        c = torch.full((1,), host_index(quantizer), dtype=torch.int64, device=device)
        quantizer._t_dev = c
    return c


def callback_counter(callback, device) -> torch.Tensor:
    """the prune callback's own ``t`` Parameter as the device step counter.  Like the reference's, it is created on
    the host and only follows ``model.cuda()``; a callback of a module that was never moved keeps it there (its eager
    steps never need it on the device) — move it now, outside capture."""
    t = callback.t
    if t.device != device:
        if torch.cuda.is_current_stream_capturing():
            raise NotCapturable("a prune callback's step counter is not on the device: run warm-up steps first")
        t.data = t.data.to(device)
        callback._t_mirror._id = None          # re-read once (the Parameter's storage changed)
    if t.dtype != torch.int64:
        raise NotCapturable("the prune callback's step counter is not int64")
    return t.data


def _stateful(model: nn.Module):
    from .quantize import BaseQuantizer, QuantizeLayer
    from .sparse import MagnitudePruningCallback, PruneLayer
    seen, qcbs, qlayers, players, pcbs = set(), [], [], [], []
    for m in model.modules():
        if id(m) in seen:
            continue
        seen.add(id(m))
        if isinstance(m, QuantizeLayer):
            qlayers.append(m)
        elif isinstance(m, PruneLayer):
            players.append(m)
        elif isinstance(m, MagnitudePruningCallback):
            pcbs.append(m)
        elif isinstance(m, BaseQuantizer):
            qcbs.append(m)
    return qcbs, qlayers, players, pcbs


class GraphedTrainStep:
    """Captures ``step_fn()`` (forward + backward + optimizer step on static input tensors) into a CUDA graph.

    ``warmup`` graph-mode steps run eagerly first (on a side stream, as CUDA graph capture requires): they allocate
    every workspace and put the device counters in charge.  They are REAL training steps.  The capture pass itself
    executes nothing on the device; the host-side counters it advanced are rolled back.  (As for any whole-step
    capture in PyTorch: drop references to outputs of earlier eager steps that still carry an autograd graph — a live
    graph pins the leaves' gradient accumulators to the stream they first ran on and invalidates the capture.)
    ``replay()`` runs one
    step; ``sync_host()`` brings the host-side counters (``callback.t``, the counter mirrors) up to date — call it
    before going back to eager steps, ``state_dict()`` needs nothing (the device state is always current)."""

    def __init__(self, model: nn.Module, step_fn: Callable[[], object], warmup: int = 3):
        if not torch.cuda.is_available():
            raise RuntimeError("qsparse_b200 is CUDA-only")
        self.model, self.step_fn = model, step_fn
        self.qcbs, self.qlayers, self.players, self.pcbs = _stateful(model)
        self.fused_sites = [m for m in model.modules() if "fused_steps" in type(m).__dict__ or "fused_steps" in vars(m)]
        from .fused import PruneQuantize
        self.pq_modules = [m for m in model.modules() if isinstance(m, PruneQuantize)]
        for m in self.pq_modules:
            if hasattr(m, "magnitude"):
                m._t_dev = torch.full((1,), int(m.t_prune), dtype=torch.int64, device=m.magnitude.device)
        self._check_steady_state()
        self.replays = 0
        for cb in self.qcbs:                                     # device twins of the host-only EMA indices
            if hasattr(cb, "t"):
                dev = next((p.device for p in model.parameters() if p.is_cuda), torch.device("cuda"))
                cb._t_dev = torch.full((1,), host_index(cb), dtype=torch.int64, device=dev)
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with graph_mode(), torch.cuda.stream(side):
            for _ in range(max(int(warmup), 1)):
                step_fn()
        torch.cuda.current_stream().wait_stream(side)
        self._check_steady_state(after_warmup=True)
        before = self._host_state()
        self.graph = torch.cuda.CUDAGraph()
        with graph_mode(), torch.cuda.graph(self.graph):
            self.result = step_fn()
        after = self._host_state()
        self._per_step = [a - b for a, b in zip(after, before)]  # host increments of ONE step
        self._restore_host_state(before)

    # ---- host-side state that a captured step would have advanced -------------------------------------------
    def _check_steady_state(self, after_warmup: bool = False):
        """every layer the step uses is past its timeout / schedule (run again after the warm-up steps: a layer
        that met its first input there is initialised by now and fails the test)"""
        for q in self.qlayers:
            if not q.initted or q.timeout <= 0:
                continue
            if q._t_mirror.get(q._n_updates) <= q.timeout:
                raise NotCapturable(f"QuantizeLayer {q.name!r} has not passed its timeout yet")
        for cb in self.qcbs:
            # group-wise scale sharing starts at call `group_timeout` (a host-side test, quantize.py:353): a graph
            # captured before that would never start it
            if getattr(cb, "group_num", -1) > 0 and hasattr(cb, "t") and host_index(cb) <= cb.group_timeout:
                raise NotCapturable("a group-wise quantizer has not reached its group_timeout yet")
        for p in self.players:
            if not p.initted:
                raise NotCapturable(f"PruneLayer {p.name!r} has not seen an input yet")
            if p._n_mirror.get(p._n_updates) <= max(p.schedules, default=p.start):
                raise NotCapturable(f"PruneLayer {p.name!r} is still on its sparsity schedule")

    def _host_state(self) -> List[int]:
        vals = [host_index(cb) for cb in self.qcbs if hasattr(cb, "t")]
        vals += [int(q._t_mirror.get(q._n_updates)) for q in self.qlayers if q.initted]
        vals += [int(p._n_mirror.get(p._n_updates)) for p in self.players]
        vals += [int(cb._t()) for cb in self.pcbs]
        vals += [int(m.fused_steps) for m in self.fused_sites]
        for m in self.pq_modules:
            vals += [int(m.t_prune), int(m.t_quant)]
        return vals

    def _restore_host_state(self, vals: List[int]):
        it = iter(vals)
        for cb in self.qcbs:
            if hasattr(cb, "t"):
                v = next(it)
                if isinstance(cb.t, torch.Tensor):
                    cb._t_host = v          # the device Parameter was (or will be) advanced by the graph itself
                else:
                    cb.t = v
        for q in self.qlayers:
            if q.initted:
                q._t_mirror.wrote(q._n_updates, next(it))
        for p in self.players:
            p._n_mirror.wrote(p._n_updates, next(it))
        for cb in self.pcbs:
            cb._t_mirror.wrote(cb.t, next(it))
        for m in self.fused_sites:
            m.fused_steps = next(it)
        for m in self.pq_modules:
            m.t_prune, m.t_quant = next(it), next(it)
            if getattr(m, "_p2p", None) is not None:
                m._p2p.stamp = m.t_prune      # eager steps stamp their peer packets t_prune + 1, like the kernel

    # ---- use ---------------------------------------------------------------------------------------------------
    def replay(self):
        self.graph.replay()
        self.replays += 1
        return self.result

    def sync_host(self):
        """host counters += what the replays since the last call advanced on the device (no device read)"""
        if self.replays:
            cur = self._host_state()
            self._restore_host_state([c + self.replays * d for c, d in zip(cur, self._per_step)])
            self.replays = 0
