"""Fused structured prune -> quantize (K7): the training step of
``Sequential(PruneLayer(dimensions={channel}), QuantizeLayer(channelwise=-1,
callback=DecimalQuantizer()))`` (the adjacency ``convert()`` creates,
ref qsparse/convert.py:214-217) in three launches and 20 B/elem:

    forward   reduce_prune_quant_step(x) 4 B/elem   per-channel sum|x| and max|x| in one read; the
                                                    kernel's last-arriving CTA finalizes, exchanges the
                                                    statistics row with the peer GPUs (NVLink packets)
                                                    and derives magnitude EMA, k-th threshold, mask,
                                                    abs-max of kept channels, scale EMA, decimal
              fq_pow2_fwd(x, mask)       8 B/elem   y = Q(x * mask); pruned channels are not read
    backward  ste_bwd(g, mask)           8 B/elem   gx = clamp(g) * mask

against the reference's ~60 B/elem forward (SURVEY §3.1-3.2).  No host synchronisation:
step counters are host integers, every derived scalar stays on the device.  With a
process group the statistics row is exchanged over peer memory inside that kernel
(parallel.P2PExchange; NCCL all-gather + a parameter kernel when peer mapping is
unavailable) and combined in rank order, so every rank derives identical parameters.

The fusion pass (``FusedPruneQuantSequential``) also takes an ``AdaptiveQuantizer`` site (per-tensor lines, or
per-channel lines on the prune axis), on one GPU, in the same three launches and bytes:

    forward   reduce_prune_line_step(x)  4 B/elem   sum|x| and min / max x; the last CTA derives magnitude EMA,
                                                    threshold, mask, the (min, max) of x * mask and the lines EMA
              fq_line_fwd(x, mask)       8 B/elem   y = Q_lines(x * mask), float zero point
    backward  mask_apply(g, mask)        8 B/elem   gx = g * mask (identity STE: grad_output is not written)

(bf16 / fp16 x: 2 B/elem less for each read of x and the write of gx, 14 B/elem in all.)
"""
from __future__ import annotations

from typing import Optional

import torch
import torch.nn as nn

from . import _native as N
from . import graphs
from . import ops
from .parallel import StatExchange, make_exchange
from .quantize import _grad_buffer, _physical_layout
from .util import kth_rank


def _walked(t, axis):
    """(t, (outer, C, inner) of its memory around ``axis``; axis < 0: per tensor): a contiguous or 4-D channels_last
    tensor as it is (the result keeps its memory format), anything else as a contiguous copy"""
    return _physical_layout(t, axis, axis >= 0)


def _grad_walked(grad_output, axis):
    """grad_output as the backward kernels read it: fp32, and, unless it is contiguous or 4-D channels_last, a
    contiguous copy; with its (outer, C, inner) around ``axis``"""
    return _walked(_grad_buffer(grad_output), axis)


class _PruneQuantizeFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, layer):
        ctx.layer = layer
        xs, layout = _walked(N.as_native(x.detach()), layer.channel_index)
        ctx.x_dtype = xs.dtype
        return layer._forward_impl(xs, layout)

    @staticmethod
    def backward(ctx, grad_output):
        return ctx.layer.backward_kernel(grad_output, ctx.x_dtype), None


class PruneQuantize(nn.Module):
    """State mirrors the two reference layers: ``magnitude`` / ``mask`` (callback.magnitude,
    PruneLayer.mask, shape [C]) and ``scale`` (QuantizeLayer.weight, shape [1, 1])."""

    def __init__(self, sparsity: float = 0.5, bits: int = 8, channel_index: int = 1, running_average: bool = True,
                 mask_refresh_interval: int = 1, group=None, mutate_grad_output: bool = False,
                 exchange_timeout_ms: int = 30000, check_every: int = 16):
        super().__init__()
        self.sparsity = sparsity
        self.bits = bits
        self.channel_index = channel_index
        self.running_average = running_average
        self.mask_refresh_interval = max(int(mask_refresh_interval), 1)
        self.group = group
        self.mutate_grad_output = mutate_grad_output  # also clamp grad_output in place (quantize.py:72)
        self.exchange_timeout_ms = exchange_timeout_ms
        self.check_every = max(int(check_every), 1)   # steps between polls of the exchange's error flag
        self.t_prune = 0   # MagnitudePruningCallback.t
        self.t_quant = 0   # DecimalQuantizer.t
        self._exchange: Optional[StatExchange] = None

    def _step_counter(self, device):
        """device twin of ``t_prune`` for graph mode (created outside capture by ``GraphedTrainStep``)"""
        c = getattr(self, "_t_dev", None)
        if c is None or c.device != device:
            if torch.cuda.is_current_stream_capturing():
                raise graphs.NotCapturable("PruneQuantize met its first graph-mode step during capture")
            c = torch.full((1,), int(self.t_prune), dtype=torch.int64, device=device)
            self._t_dev = c
        return c

    def _allocate(self, x, channels):
        dev = x.device
        self.magnitude = nn.Parameter(torch.zeros(channels, device=dev), requires_grad=False)
        self.mask = nn.Parameter(torch.ones(channels, dtype=torch.bool, device=dev), requires_grad=False)
        self.scale = nn.Parameter(torch.zeros(1, 1, device=dev), requires_grad=False)
        self.decimal = torch.zeros(1, device=dev)
        import torch.distributed as dist
        from .parallel import assert_equal_shards
        multi = dist.is_available() and dist.is_initialized() and dist.get_world_size(self.group) > 1
        if multi:
            assert_equal_shards(x.numel() // channels, self.group)
        self._p2p = make_exchange(channels, dev, self.group, timeout_ms=self.exchange_timeout_ms) \
            if channels <= ops.PARTIALS_ROUTE_MAX_CHANNELS else None
        # NCCL all-gather path only when peer memory is unavailable (or takes more channels than it exchanges)
        self._exchange = StatExchange(channels, dev, self.group) if multi and self._p2p is None else True

    def _forward_impl(self, xs, layout):
        """xs: x as ``_walked`` returns it (bf16 / fp16 read natively, y is fp32 in xs's memory format)"""
        outer, ch, inner = layout
        if self._exchange is None:
            self._allocate(xs, ch)
        if self.training:
            t = self.t_prune
            refresh = (t % self.mask_refresh_interval == 0) and (t > 0 or not self.running_average)
            mode = 1 if self.running_average else 2
            k = kth_rank(self.sparsity, ch)
            if refresh and k >= ch and not graphs.active():   # the reference indexes sorted()[k] on a refresh step
                raise IndexError(f"index {k} is out of bounds for dimension 0 with size {ch}")
            if isinstance(self._exchange, StatExchange):
                # NCCL fallback: finalize into the row, all-gather, combine rows in the kernel
                graphs.require_eager("PruneQuantize over the NCCL all-gather fallback")
                ex = self._exchange
                ops.reduce_stats(xs, layout, abssum=True, absmax=True,
                                 out={"abssum": ex.row.abssum, "absmax": ex.row.absmax})
                rows, n_rows, stride = ex.gather()
                abssum0, absmax0 = ex.views(rows)
                ops.prune_quant_params(self.magnitude.data, self.mask.data, self.scale.data, self.decimal,
                                       {"abssum": abssum0, "absmax": absmax0}, float(outer * inner * n_rows), t,
                                       mode, refresh, k, self.bits, self.t_quant, True, n_rows=n_rows,
                                       row_stride_bytes=stride)
            else:
                world = self._p2p.world if self._p2p is not None else 1
                grp = self._p2p.handle if self._p2p is not None else None
                stamp = self._p2p.next_stamp() if self._p2p is not None else 1
                count = float(outer * inner * world)
                if graphs.active():
                    # graph mode: the step index (and the exchange stamp) come from a device counter that the
                    # kernel reads and advances itself
                    ops.structured_prune_quant_step(xs, layout, self.magnitude.data, self.mask.data, self.scale.data,
                                                    self.decimal, count, 0, mode, self.mask_refresh_interval, k,
                                                    self.bits, self.t_quant - t, True, group=grp,
                                                    step_counter=self._step_counter(xs.device))
                else:
                    ops.structured_prune_quant_step(xs, layout, self.magnitude.data, self.mask.data, self.scale.data,
                                                    self.decimal, count, t, mode, refresh, k, self.bits,
                                                    self.t_quant, True, group=grp, step_stamp=stamp)
                if self._p2p is not None and t % self.check_every == 0 and not graphs.active():
                    self._p2p.check()     # raises when an earlier step timed out waiting for a peer
            self.t_prune += 1
            self.t_quant += 1
        return ops.fq_pow2_fwd(xs, self.decimal, layout, mask=self.mask.data)

    def backward_kernel(self, g, x_dtype=torch.float32):
        """gx in ``x_dtype`` (the input's dtype: bf16 / fp16 are written directly, rounded like autograd's cast) and
        in g's memory format"""
        g, layout = _grad_walked(g, self.channel_index)
        _, gx = ops.ste_bwd(g, self.decimal, True, self.bits, 0, layout, mask=self.mask.data,
                            clamp_in_place=self.mutate_grad_output, want_gx=True, gx_dtype=x_dtype)
        return gx

    def forward(self, x):
        N.require_cuda(x, "x")
        return _PruneQuantizeFn.apply(x, self)


# ----------------------------------------------------------------------------- fusion pass (SURVEY §8 f-1)
def _site_layout(x, d):
    """(outer, C, inner) of x's memory around the prune axis ``d`` when the fused step walks x without a copy:
    contiguous with ``1 <= d < x.dim()`` (the last axis gives [rows, C, 1]), or 4-D channels_last with ``d == 1``
    ([N*H*W, C, 1]); None for every other layout"""
    if not 1 <= d < x.dim():
        return None
    if x.is_contiguous() or (d == 1 and x.dim() == 4 and x.is_contiguous(memory_format=torch.channels_last)):
        return _physical_layout(x, d, True)[1]
    return None


class _FusedLayersFn(torch.autograd.Function):
    """forward value and backward of ``QuantizeLayer(PruneLayer(x))`` in its steady state, on the two
    layers' own state tensors: y = Q(x * mask), gx = clamp(g) * mask (grad_output clamped in place, like
    DecimalQuantization.backward does, ref quantize.py:65-77, sparse.py backward of x * mask).  xs is walked in
    ``layout`` (its memory around the prune axis ``axis``), so y keeps x's memory format; the backward walks
    grad_output in its own memory, so gx keeps g's."""

    @staticmethod
    def forward(ctx, x, xs, layout, axis, mask, param, bits, notch, is_decimal):
        # param: the step's decimal (DecimalQuantizer) or the layer's scale itself (ScalerQuantizer)
        ctx.axis, ctx.mask, ctx.param, ctx.bits, ctx.notch = axis, mask, param, bits, notch
        ctx.is_decimal = is_decimal
        ctx.x_dtype = xs.dtype     # bf16 / fp16 activations: gx is written in their dtype
        if is_decimal:
            return ops.fq_pow2_fwd(xs, param, layout, mask=mask).view(x.shape)
        return ops.fq_scaler_fwd(xs, param, layout, mask=mask).view(x.shape)

    @staticmethod
    def backward(ctx, grad_output):
        g, layout = _grad_walked(grad_output, ctx.axis)
        _, gx = ops.ste_bwd(g, ctx.param, ctx.is_decimal, ctx.bits, ctx.notch, layout, mask=ctx.mask,
                            clamp_in_place=True, want_gx=True, gx_dtype=ctx.x_dtype)
        return (gx,) + (None,) * 8


class _FusedLineLayersFn(torch.autograd.Function):
    """the same for an AdaptiveQuantizer: y = Q_lines(x * mask) with the float zero point of a training step,
    gx = g * mask.  The line quantizer's backward is the identity (ref quantize.py:134-185, SURVEY Q9), so
    grad_output is read, never written."""

    @staticmethod
    def forward(ctx, x, xs, layout, axis, mask, lines, bits):
        ctx.axis, ctx.mask, ctx.x_dtype = axis, mask, xs.dtype
        return ops.fq_line_fwd(xs, lines, bits, True, layout, mask=mask).view(x.shape)

    @staticmethod
    def backward(ctx, grad_output):
        g, layout = _grad_walked(grad_output, ctx.axis)
        return (ops.mask_apply(g, ctx.mask, layout, out_dtype=ctx.x_dtype),) + (None,) * 6


class FusedPruneQuantSequential(nn.Sequential):
    """``Sequential(Sequential(act, PruneLayer), QuantizeLayer)`` (what two ``convert()`` calls build around
    an activation, ref qsparse/convert.py:214-217) or ``Sequential(PruneLayer, QuantizeLayer)``, with the
    SAME children — module tree and ``state_dict`` keys are untouched — whose forward sends every
    steady-state training step through the fused kernels (reduce -> one parameter kernel -> quantize with
    the mask folded in: 20 B/elem with the backward, instead of ~60 + 16).

    A step is fused only when it is provably the plain case: both layers initialised, training, structured
    prune along one axis ``d`` (``dimensions={d}``) by the stock ``MagnitudePruningCallback`` (no gradient / l0 /
    hook variants), pruning started and the sparsity not changing at this step, past the quantizer's timeout,
    with a per-tensor stock ``DecimalQuantizer`` or ``ScalerQuantizer`` (``quantize()``'s default callback) or a
    stock ``AdaptiveQuantizer`` (per tensor, or per channel on the prune axis) after its first estimate, on an
    input the kernels walk without a copy (``_site_layout``): contiguous with ``d >= 1`` (``[N, C, H, W]`` on
    axis 1, ``[tokens, hidden]`` or ``[B, T, H]`` on the last axis) or a 4-D ``channels_last`` tensor with
    ``d == 1``.  Every other step (warm-up, ramp steps, eval, other callbacks, other layouts) runs the two layers
    one after the other, exactly as before.  Counters and parameters advance identically either way, so the two
    routes can alternate freely."""

    fused_steps = 0  # how many forwards took the fused route (per instance once incremented)

    def _layers(self):
        first, q = self[0], self[1]
        if isinstance(first, nn.Sequential):
            return first[0], first[1], q
        return None, first, q

    def _fusable(self, p, q, x):
        from .quantize import AdaptiveQuantizer, DecimalQuantizer, QuantizeLayer, ScalerQuantizer
        from .sparse import MagnitudePruningCallback, PruneLayer

        if not (isinstance(p, PruneLayer) and isinstance(q, QuantizeLayer) and self.training and p.training
                and q.training):
            return False
        if not (isinstance(x, torch.Tensor) and x.is_cuda and x.dim() >= 2 and len(p.dimensions) == 1):
            return False
        d = next(iter(p.dimensions))
        if _site_layout(x, d) is None:
            return False
        cb, qcb = p.callback, q.callback
        if type(cb) is not MagnitudePruningCallback or type(qcb) not in (DecimalQuantizer, ScalerQuantizer,
                                                                         AdaptiveQuantizer):
            return False
        if cb.use_gradient or cb.l0 or cb.forward_hook is not None or not cb.training or not qcb.training:
            return False
        if not p.initted or not q.initted or p.mask.numel() == 1:
            return False
        if p.mask.numel() != x.shape[d] or p.mask.numel() > ops.PARTIALS_ROUTE_MAX_CHANNELS:
            return False
        n = p._n_mirror.get(p._n_updates)
        if n < p.start or n in p.schedules:
            return False
        if not cb.initted or cb._t() >= cb.stop_mask_refresh or cb.mask_refresh_interval <= 0:
            return False
        if cb.running_average and not hasattr(cb, "magnitude"):
            return False
        if q.timeout <= 0 or q._t_mirror.get(q._n_updates) < q.timeout or qcb.group_num > 0:
            return False
        if p._s_mirror.get(p._cur_sparsity) < 0:
            return False
        if type(qcb) is AdaptiveQuantizer:
            # lines per tensor or per channel of the prune axis; not before the first optimize(), which may
            # re-create `t` (like _fused_weight_step)
            rows = 1 if q.channelwise < 0 else p.mask.numel()
            if q.channelwise >= 0 and q.channelwise != d:
                return False
            if tuple(q.weight.shape) != (rows, 2) or not q.weight.is_contiguous():
                return False
            return isinstance(qcb.t, torch.Tensor) or qcb.t != 0
        if q.channelwise >= 0 or qcb.backward_passthrough or qcb.use_uint:
            return False
        if qcb.use_float_scaler != (type(qcb) is ScalerQuantizer):
            return False
        return tuple(q.weight.shape) == (1, 1)

    def _fused_step(self, p, q, x):
        from .quantize import AdaptiveQuantizer
        cb, qcb = p.callback, q.callback
        axis = next(iter(p.dimensions))
        layout = _site_layout(x, axis)
        outer, ch, inner = layout
        xs = N.as_native(x.detach())   # bf16 / fp16 read natively, in x's memory format
        sparsity = p._s_mirror.get(p._cur_sparsity)
        t = cb._t()
        refresh = (t % cb.mask_refresh_interval == 0 and t <= cb.stop_mask_refresh) and \
            (t > 0 or not cb.running_average)
        k = kth_rank(sparsity, ch)
        if refresh and k >= ch:    # the un-fused route only indexes sorted()[k] on a refresh step
            raise IndexError(f"index {k} is out of bounds for dimension 0 with size {ch}")
        if not refresh:
            k = min(k, ch - 1)
        line = type(qcb) is AdaptiveQuantizer
        is_decimal = not line and not qcb.use_float_scaler
        # DecimalQuantizer: this step's decimal (a fresh tensor: the backward must see THIS step's value);
        # ScalerQuantizer: the quantize kernels read the layer's scale itself, like the reference's saved tensor
        decimal = torch.empty(1, dtype=torch.float32, device=x.device) if is_decimal else None
        with torch.no_grad():
            if cb.running_average:
                magnitude, mode = cb.magnitude.data.view(-1), 1
            else:
                magnitude, mode = torch.empty(ch, dtype=torch.float32, device=x.device), 2
            # AdaptiveQuantizer: this call's 1-based index; also advances its device `t` when it has one
            t_line = qcb._next_t() if line else 0
            if graphs.active():
                # graph mode: the step index is the prune callback's own `t` Parameter, read and advanced by the
                # kernel; the quantizer's EMA index keeps its constant distance to it
                if cb.stop_mask_refresh != float("inf"):
                    raise graphs.NotCapturable("a fused site with a stopping mask refresh")
                counter = graphs.callback_counter(cb, x.device)
                if line:
                    ops.structured_prune_line_step(xs, layout, magnitude, p.mask.data.view(-1), q.weight.data,
                                                   float(outer * inner), 0, mode, cb.mask_refresh_interval,
                                                   kth_rank(sparsity, ch), t_line - t, step_counter=counter)
                else:
                    ops.structured_prune_quant_step(xs, layout, magnitude, p.mask.data.view(-1),
                                                    q.weight.data.view(-1), decimal, float(outer * inner), 0, mode,
                                                    cb.mask_refresh_interval, kth_rank(sparsity, ch), q.bits,
                                                    qcb.t - t, True, step_counter=counter)
            else:
                if line:
                    ops.structured_prune_line_step(xs, layout, magnitude, p.mask.data.view(-1), q.weight.data,
                                                   float(outer * inner), t, mode, refresh, k, t_line)
                else:
                    ops.structured_prune_quant_step(xs, layout, magnitude, p.mask.data.view(-1),
                                                    q.weight.data.view(-1), decimal, float(outer * inner), t, mode,
                                                    refresh, k, q.bits, qcb.t, True)
                cb.t.data.add_(1)
            # the counters of the two layers and their callbacks, as their own forwards advance them
            cb._t_mirror.wrote(cb.t, t + 1)
            n = p._n_mirror.get(p._n_updates)
            p._n_updates.data.add_(1)
            p._n_mirror.wrote(p._n_updates, n + 1)
            if not line:
                qcb.t += 1
            q._quantized = True
            tq = q._t_mirror.get(q._n_updates)
            q._n_updates.data.add_(1)
            q._t_mirror.wrote(q._n_updates, tq + 1)
        self.fused_steps += 1
        if line:
            return _FusedLineLayersFn.apply(x, xs, layout, axis, p.mask.data.view(-1), q.weight.data, q.bits)
        return _FusedLayersFn.apply(x, xs, layout, axis, p.mask.data.view(-1),
                                    decimal if is_decimal else q.weight.data.view(-1), q.bits,
                                    1 if qcb.flip_axis else 0, is_decimal)

    def forward(self, x):
        pre, p, q = self._layers()
        if pre is not None:
            x = pre(x)
        if self._fusable(p, q, x):
            return self._fused_step(p, q, x)
        return q(p(x))


# ----------------------------------------------------------------------------- weight chain quantize(prune(layer))
class _FusedWeightFn(torch.autograd.Function):
    """``quantize_layer(prune_layer(w))`` of a weight whose prune mask is frozen (ref qsparse/imitation.py:61-71,
    sparse.py:116, quantize.py:501-508): estimate the row parameters on ``w * mask``, EMA, fake-quantize — one
    launch, 9 B/elem (K8 with an element mask) instead of mask-apply (9) + estimate/quantize (8).  Backward:
    ``clamp(g) * mask`` (Decimal / Scaler, one launch) or ``g * mask`` (Adaptive: identity STE)."""

    @staticmethod
    def forward(ctx, w, ws, mask, q, t_line):
        from .quantize import AdaptiveQuantizer
        qcb = q.callback
        ctx.mask, ctx.rows, ctx.bits = mask, ws.shape[0], q.bits
        counter = graphs.quantizer_counter(qcb, ws.device) if graphs.active() else None
        if type(qcb) is AdaptiveQuantizer:
            if counter is not None:          # graph mode: this call's number is *counter + 1
                y, _ = ops.row_quant_fused_(ws, q.weight.data, ops.ROW_LINE, q.bits, 1, qcb.training, mask=mask,
                                            t_dev=counter)
                counter.add_(1)
            else:
                y, _ = ops.row_quant_fused_(ws, q.weight.data, ops.ROW_LINE, q.bits, t_line, qcb.training, mask=mask)
            ctx.kind = "line"
        else:
            is_decimal = not qcb.use_float_scaler
            kind = ops.ROW_DECIMAL if is_decimal else ops.ROW_SCALER
            if counter is not None:
                y, dec = ops.row_quant_fused_(ws, q.weight.data, kind, q.bits, 0, mask=mask, t_dev=counter)
                counter.add_(1)
            else:
                y, dec = ops.row_quant_fused_(ws, q.weight.data, kind, q.bits, qcb.t, mask=mask)
            qcb.t += 1
            ctx.kind = "ste"
            ctx.is_decimal = is_decimal
            ctx.param = dec if is_decimal else q.weight.data.view(-1)
            ctx.notch = 1 if qcb.flip_axis else 0
            ctx.passthrough = qcb.backward_passthrough
        return y.view(w.shape)

    @staticmethod
    def backward(ctx, grad_output):
        g = N.as_f32_contiguous(grad_output)
        n = g.numel()
        if ctx.kind == "line" or ctx.passthrough:
            return (ops.mask_apply(g, ctx.mask, (1, 1, n)),) + (None,) * 4
        _, gx = ops.ste_bwd(g, ctx.param, ctx.is_decimal, ctx.bits, ctx.notch, (1, ctx.rows, n // ctx.rows),
                            mask=ctx.mask, clamp_in_place=True, want_gx=True)
        return (gx,) + (None,) * 4


def _fused_weight_step(p, q, raw):
    """The fused weight access, or None when this step is not provably the plain frozen-mask case."""
    from .quantize import AdaptiveQuantizer, DecimalQuantizer, QuantizeLayer, ScalerQuantizer
    from .sparse import MagnitudePruningCallback, PruneLayer

    if not (isinstance(p, PruneLayer) and isinstance(q, QuantizeLayer) and p.training and q.training):
        return None
    if not (isinstance(raw, torch.Tensor) and raw.is_cuda and raw.dim() >= 2 and raw.dtype == torch.float32
            and raw.is_contiguous()):
        return None
    cb, qcb = p.callback, q.callback
    if type(cb) is not MagnitudePruningCallback or type(qcb) not in (DecimalQuantizer, ScalerQuantizer,
                                                                     AdaptiveQuantizer):
        return None
    if not p.initted or not q.initted or tuple(p.mask.shape) != tuple(raw.shape):
        return None                                            # unstructured (full-size) masks only
    if cb.use_gradient or cb.forward_hook is not None or not cb.training or not qcb.training or not cb.initted:
        return None
    n = p._n_mirror.get(p._n_updates)
    if n < p.start or n in p.schedules or cb._t() <= cb.stop_mask_refresh:
        return None                                            # the callback still updates magnitude / mask
    if q.channelwise != 0 or q.batch_dimension == 0 or q.timeout <= 0 or qcb.group_num > 0:
        return None
    tq = q._t_mirror.get(q._n_updates)
    if tq < q.timeout:
        return None
    if tuple(q.weight.shape) != (raw.shape[0], qcb.weight_size) or not q.weight.is_contiguous():
        return None
    if type(qcb) is AdaptiveQuantizer and isinstance(qcb.t, torch.Tensor) is False and qcb.t == 0:
        return None                                            # its first optimize() re-creates `t`: unfused
    ws = raw.detach()
    if not ops.row_quant_supported(ws, raw.shape[0]) or p.mask.data_ptr() % 8:
        return None
    with torch.no_grad():
        # the counters of the two layers and their callbacks, as their own forwards advance them
        t = cb._t()
        cb.t.data.add_(1)
        cb._t_mirror.wrote(cb.t, t + 1)
        p._n_updates.data.add_(1)
        p._n_mirror.wrote(p._n_updates, n + 1)
        if graphs.active():
            graphs.quantizer_counter(qcb, raw.device)          # (its device twin exists before the count moves)
        t_line = qcb._next_t() if type(qcb) is AdaptiveQuantizer else 0
        q._quantized = True
        q._n_updates.data.add_(1)
        q._t_mirror.wrote(q._n_updates, tq + 1)
    return _FusedWeightFn.apply(raw, ws, p.mask.data, q, t_line)


def _imitation_chain(mod) -> list:
    """operator names of an ``imitate()`` chain, outermost first (['quantize', 'prune'] = quantize(prune(layer)))"""
    return [c.__dict__["_qsb_imitates"] for c in type(mod).__mro__ if "_qsb_imitates" in c.__dict__]


def _fuse_weight_chain(mod: nn.Module) -> bool:
    if _imitation_chain(mod)[:2] != ["quantize", "prune"] or getattr(type(mod), "_qsb_fused_chain", False):
        return False
    cls = type(mod)

    class FusedChain(cls):
        _qsb_fused_chain = True
        fused_weight_steps = 0

        @property
        def weight(self):
            out = _fused_weight_step(self.prune, self.quantize, self._parameters["weight"])
            if out is not None:
                self.fused_weight_steps += 1
                return out
            return cls.weight.__get__(self)

    FusedChain.__name__ = cls.__name__
    FusedChain.__qualname__ = cls.__qualname__
    mod.__class__ = FusedChain
    return True


def fuse_prune_quantize(model: nn.Module) -> nn.Module:
    """Fusion pass over a converted model (in place): every ``Sequential(Sequential(m, PruneLayer),
    QuantizeLayer)`` / ``Sequential(PruneLayer, QuantizeLayer)`` becomes a ``FusedPruneQuantSequential``
    and every ``quantize(prune(layer))`` weight chain gets a fused ``weight`` property (same children, same
    ``state_dict``).  Returns the model."""
    from .quantize import QuantizeLayer
    from .sparse import PruneLayer

    def is_site(m):
        if type(m) is not nn.Sequential or len(m) != 2 or not isinstance(m[1], QuantizeLayer):
            return False
        first = m[0]
        if isinstance(first, PruneLayer):
            return True
        return type(first) is nn.Sequential and len(first) == 2 and isinstance(first[1], PruneLayer)

    for mod in list(model.modules()):
        if is_site(mod):
            mod.__class__ = FusedPruneQuantSequential
        elif hasattr(mod, "prune") and hasattr(mod, "quantize"):
            _fuse_weight_chain(mod)          # quantize(prune(layer)): frozen-mask steps through K8 with the mask
    return model
