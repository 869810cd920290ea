"""Fake-quantization operators on sm_100a kernels, behind qsparse's own API.

Mirrors ``qsparse/quantize.py`` of mlzxy/qsparse v2.0.1 (same class / function names,
argument order, state and error behaviour), with every tensor op replaced by one
launch of the hand-written kernels in ``csrc/`` through the C-ABI:

=====================  =====================================  ==================
reference              here                                    kernel
=====================  =====================================  ==================
DecimalQuantization    ``DecimalQuantization`` (autograd)      qsb_fq_pow2_fwd / qsb_ste_bwd
ScalerQuantization     ``ScalerQuantization``                  qsb_fq_scaler_fwd / qsb_ste_bwd
LineQuantization       ``LineQuantization``                    qsb_fq_line_fwd (identity bwd)
DecimalQuantizer       ``optimize``: abs-max + EMA             qsb_reduce_stats, qsb_scale_ema
AdaptiveQuantizer      ``optimize``: min/max + EMA             qsb_reduce_stats, qsb_lines_ema
=====================  =====================================  ==================

No CPU path: CPU tensors raise.  bf16 and fp16 activations are read natively by the
kernels, which compute in fp32: outputs are fp32 (the reference's output is always fp32,
SURVEY Q6) and equal bit for bit what the input converted to fp32 gives; input gradients
come back in the input's dtype.  Other dtypes are converted to fp32 first.
"""
from __future__ import annotations

import math
from typing import List, Tuple, Union

import torch
import torch.nn as nn

from . import _native as N
from . import graphs
from . import ops
from .common import TensorOrFloat, TensorOrInt
from .imitation import imitate
from .util import HostMirror, get_option, logging


# Route `channelwise=0` weight layers through the one-launch row kernel (K8).  False keeps the
# reduce -> EMA -> quantize sequence (same results; used by the tests to compare the two).
FUSE_ROW_QUANTIZE = True


# --------------------------------------------------------------------------- helpers
def _physical_layout(x: torch.Tensor, channel_index: int, channelwise: bool):
    """(tensor whose memory the kernel walks, (outer, C, inner)).

    Contiguous tensors are used as they are.  channels_last 4-D tensors are walked
    in their physical NHWC order, so the output keeps the input's memory format like
    the reference's elementwise ops do.  Anything else is made contiguous."""
    if not channelwise:
        if x.is_contiguous() or (x.dim() == 4 and x.is_contiguous(memory_format=torch.channels_last)):
            return x, (1, 1, x.numel())
        x = x.contiguous()
        return x, (1, 1, x.numel())
    ci = channel_index % x.dim() if channel_index < 0 else channel_index
    if x.is_contiguous():
        return x, N.channel_layout(x.shape, ci)
    if x.dim() == 4 and x.is_contiguous(memory_format=torch.channels_last):
        n, c, h, w = (int(s) for s in x.shape)
        phys = {0: (1, n, h * w * c), 1: (n * h * w, c, 1), 2: (n, h, w * c), 3: (n * h, w, c)}[ci]
        return x, phys
    x = x.contiguous()
    return x, N.channel_layout(x.shape, ci)


def _is_channelwise(param) -> bool:
    return isinstance(param, torch.Tensor) and param.numel() > 1


def _broadcast_result(y: torch.Tensor, x_shape, param) -> torch.Tensor:
    """A one-element tensor parameter of higher rank than x broadcasts the result
    shape in the reference (`input * toi` with toi of shape [1, 1])."""
    if isinstance(param, torch.Tensor) and param.numel() == 1 and param.dim() > len(x_shape):
        return y.reshape(torch.broadcast_shapes(tuple(x_shape), tuple(param.shape)))
    return y


def _grad_buffer(grad_output: torch.Tensor) -> torch.Tensor:
    """The STE clamp runs in place on grad_output (quantize.py:72).  A gradient that
    is not a dense fp32 buffer (e.g. the stride-0 expand of `.sum().backward()`, on
    which the reference's in-place clamp raises) gets a dense copy instead."""
    g = grad_output
    if g.dtype != torch.float32:
        g = g.float()
    if not g.is_contiguous() and not (g.dim() == 4 and g.is_contiguous(memory_format=torch.channels_last)):
        g = g.contiguous()
    return g


def _ste_prepare(ctx, input, bits, param, channel_index, backward_passthrough, flip_axis, is_decimal, what):
    """shared forward bookkeeping of the two symmetric quantizers"""
    N.require_cuda(input, "input")
    if isinstance(param, torch.Tensor) and not param.is_cuda and param.numel() > 1:
        raise RuntimeError(f"{what} is a multi-element CPU tensor; qsparse_b200 is CUDA-only")
    channelwise = _is_channelwise(param)
    if channelwise:
        assert len(param) == input.shape[channel_index], \
            "channel of input and decimal must be equal in channel-wise quantization"
    x, layout = _physical_layout(N.as_native(input.detach()), channel_index, channelwise)
    ctx.x_dtype, ctx.x_shape = x.dtype, tuple(input.shape)
    ctx.backward_passthrough = backward_passthrough
    ctx.notch = 1 if flip_axis else 0
    ctx.bits = bits
    ctx.is_decimal = is_decimal
    ctx.channelwise = channelwise
    ctx.channel_index = channel_index
    ctx.param_is_tensor = isinstance(param, torch.Tensor) and param.is_cuda
    if ctx.param_is_tensor:
        p = param.detach()
        p = p if (p.dtype == torch.float32 and p.is_contiguous()) else p.float().contiguous()
        ctx.save_for_backward(p)
        ctx.param_host = None
        param = p
    else:
        ctx.param_host = float(param)
        param = ctx.param_host
    return x, layout, param

def _ste_backward(ctx, grad_output):
    if ctx.backward_passthrough:
        return grad_output
    g = _grad_buffer(grad_output)
    param = ctx.saved_tensors[0] if ctx.param_is_tensor else ctx.param_host
    _, layout = _physical_layout(g, ctx.channel_index, ctx.channelwise)
    x_dtype = getattr(ctx, "x_dtype", torch.float32)
    if x_dtype != torch.float32 and tuple(g.shape) == ctx.x_shape:
        # a 16-bit input: clamp grad_output in place and write its input gradient in the input's dtype, one pass
        _, gx = ops.ste_bwd(g, param, ctx.is_decimal, ctx.bits, ctx.notch, layout, clamp_in_place=True,
                            want_gx=True, gx_dtype=x_dtype)
        return gx
    ops.ste_bwd(g, param, ctx.is_decimal, ctx.bits, ctx.notch, layout, clamp_in_place=True)
    return g


class DecimalQuantization(torch.autograd.Function):
    """Straight-through estimator with a power-of-two scale (ref qsparse/quantize.py:24-77).

    forward  ``y = float(int32_rz(x * 2^d)) * 2^-d`` — the reference's forward clamp acts
    on a temporary and is dropped (SURVEY Q1), so ``bits`` / ``use_uint`` / ``flip_axis``
    only matter in the backward.
    backward ``clamp(g, (-L+notch)*2^-d, (L-1+notch)*2^-d)`` in place on ``grad_output``,
    NaN -> 0 (SURVEY Q2)."""

    @staticmethod
    def forward(ctx, input: torch.Tensor, bits: int = 8, decimal: TensorOrInt = 5, channel_index: int = 1,
                use_uint: bool = False, backward_passthrough: bool = False, flip_axis: bool = False):
        x, layout, dec = _ste_prepare(ctx, input, bits, decimal, channel_index, backward_passthrough,
                                            flip_axis, True, "decimal")
        y = ops.fq_pow2_fwd(x, dec, layout)
        return _broadcast_result(y, input.shape, decimal)

    @staticmethod
    def backward(ctx, grad_output):
        return (_ste_backward(ctx, grad_output),) + (None,) * 6


class ScalerQuantization(torch.autograd.Function):
    """Straight-through estimator with a float scale (ref qsparse/quantize.py:80-131).

    forward  ``y = float(int32_rz(rint(x / s))) * s`` with an IEEE division."""

    @staticmethod
    def forward(ctx, input: torch.Tensor, bits: int = 8, scaler: TensorOrFloat = 0.1, channel_index: int = 1,
                use_uint: bool = False, backward_passthrough: bool = False, flip_axis: bool = False):
        x, layout, s = _ste_prepare(ctx, input, bits, scaler, channel_index, backward_passthrough,
                                          flip_axis, False, "scaler")
        y = ops.fq_scaler_fwd(x, s, layout)
        return _broadcast_result(y, input.shape, scaler)

    @staticmethod
    def backward(ctx, grad_output):
        return (_ste_backward(ctx, grad_output),) + (None,) * 6


class LineQuantization(torch.autograd.Function):
    """Asymmetric quantization between per-channel (lo, hi) lines with an identity
    backward — no STE saturation (ref qsparse/quantize.py:134-185, SURVEY Q9)."""

    @staticmethod
    def forward(ctx, x: torch.Tensor, bits: int = 8, lines=(-0.1, 0.9), channel_index=-1, inplace=False,
                float_zero_point=True):
        N.require_cuda(x, "x")
        if not isinstance(lines, torch.Tensor):
            lines = torch.tensor(lines).view(-1, 2)
        if channel_index >= 0:
            assert x.shape[channel_index] == lines.shape[0]
        assert lines.shape[1] == 2
        channelwise = channel_index >= 0 and lines.shape[0] > 1
        xs, layout = _physical_layout(N.as_native(x.detach()), channel_index, channelwise)
        if lines.is_cuda:
            l = lines.detach().reshape(-1, 2)
        else:
            if lines.shape[0] != 1:
                lines = lines.to(x.device)  # the reference moves a CPU `lines` list to x.device (:152)
            l = lines.detach().reshape(-1, 2)
        return ops.fq_line_fwd(xs, l, bits, bool(float_zero_point), layout)

    @staticmethod
    def backward(ctx, grad_output):
        return (grad_output,) + (None,) * 6


def _block_rows(x: torch.Tensor, rows: str):
    """(tensor whose memory the kernel walks, R, L) of the ``[R, L]`` view of a block-scaled quantizer.

    ``rows="last"``: L is the innermost physical axis — the last axis of a contiguous tensor, C of a 4-D
    ``channels_last`` one (walked in its NHWC order, so the output keeps x's memory format).  ``rows="leading"``:
    the contiguous tensor as ``[x.shape[0], numel / x.shape[0]]``.  Anything else is made contiguous first."""
    x = N.as_native(x)
    if rows == "last" and not x.is_contiguous() and x.dim() == 4 and x.is_contiguous(memory_format=torch.channels_last):
        L = int(x.shape[1])
    else:
        x = x.contiguous()
        if rows == "last":
            L = int(x.shape[-1]) if x.dim() else 1
        else:
            R = int(x.shape[0]) if x.dim() else 1
            L = x.numel() // R if R else 0
    return x, (x.numel() // L if L else 0), L


class BlockScaledQuantization(torch.autograd.Function):
    """Block-scaled FP8 / FP4 fake quantization (``BlockScaledQuantizer``) with an identity backward."""

    @staticmethod
    def forward(ctx, input: torch.Tensor, fmt: str = "nvfp4", rows: str = "last", tensor_amax=None):
        N.require_cuda(input, "input")
        xs, R, L = _block_rows(input.detach(), rows)
        return ops.fq_block_fwd(xs, fmt, R, L, tensor_amax)

    @staticmethod
    def backward(ctx, grad_output):
        return grad_output, None, None, None


class _RowFusedSte(torch.autograd.Function):
    """K8 for the symmetric quantizers on a `channelwise=0` tensor: per-row abs-max -> scale EMA (into
    ``weight``, in place) -> [decimal] -> fake-quantize in ONE launch (``qsb_row_quant_fused``); the backward
    is the ordinary STE kernel with the row's decimal / scale.  Same results as
    ``DecimalQuantizer.optimize`` + ``DecimalQuantization`` / ``ScalerQuantization`` (ref quantize.py:327-349,
    :24-131)."""

    @staticmethod
    def forward(ctx, input, quantizer, bits, weight, xs):
        is_decimal = not quantizer.use_float_scaler
        kind = ops.ROW_DECIMAL if is_decimal else ops.ROW_SCALER
        if graphs.active():
            counter = graphs.quantizer_counter(quantizer, xs.device)
            y, dec = ops.row_quant_fused_(xs, weight.data, kind, bits, 0, t_dev=counter)
            counter.add_(1)
        else:
            y, dec = ops.row_quant_fused_(xs, weight.data, kind, bits, quantizer.t)
        quantizer.t += 1
        ctx.backward_passthrough = quantizer.backward_passthrough
        ctx.notch = 1 if quantizer.flip_axis else 0
        ctx.bits = bits
        ctx.is_decimal = is_decimal
        ctx.channelwise = True
        ctx.channel_index = 0
        ctx.param_is_tensor = True
        ctx.param_host = None
        ctx.save_for_backward(dec if is_decimal else weight.data.view(-1))
        return y.view(input.shape)

    @staticmethod
    def backward(ctx, grad_output):
        return (_ste_backward(ctx, grad_output),) + (None,) * 4


_dummies = {}


def _dummy_state(dev):
    """(magnitude, mask) placeholders of the parameter step for layers that only quantize (never written)"""
    d = _dummies.get(dev)
    if d is None:
        d = (torch.zeros(1, device=dev), torch.ones(1, dtype=torch.bool, device=dev))
        _dummies[dev] = d
    return d


class _TensorFusedSte(torch.autograd.Function):
    """Per-tensor Decimal / Scaler layer step in two launches instead of five: the abs-max reduction,
    whose last-arriving CTA finalizes it and updates scale EMA (into ``weight``) and decimal ->
    fake-quantize; the backward is the ordinary STE kernel.  Same results as ``optimize`` + ``forward``
    (ref quantize.py:327-349, :24-131)."""

    @staticmethod
    def forward(ctx, input, quantizer, bits, weight, xs):
        is_decimal = not quantizer.use_float_scaler
        n = xs.numel()
        layout = (1, 1, n)
        dev = xs.device
        decimal = torch.empty(1, dtype=torch.float32, device=dev) if is_decimal else None
        # ONE launch: abs-max reduction whose last-arriving CTA finalizes and updates scale / decimal
        mag0, mask1 = _dummy_state(dev)
        if graphs.active():
            # graph mode: the EMA index is the quantizer's device counter (read and advanced by the kernel)
            ops.reduce_prune_quant_step(xs, layout, mag0, mask1, weight.data.view(-1), decimal if is_decimal else None,
                                        float(n), 0, 0, graphs.NO_REFRESH_INTERVAL, 0, bits, 0, True,
                                        step_counter=graphs.quantizer_counter(quantizer, dev))
        else:
            ops.reduce_prune_quant_step(xs, layout, mag0, mask1, weight.data.view(-1), decimal if is_decimal else None,
                                        float(n), 0, 0, False, 0, bits, quantizer.t, True)
        quantizer.t += 1
        if is_decimal:
            y = ops.fq_pow2_fwd(xs, decimal, layout)
        else:
            y = ops.fq_scaler_fwd(xs, weight.data.view(-1), layout)
        ctx.x_dtype, ctx.x_shape = xs.dtype, tuple(input.shape)
        ctx.backward_passthrough = quantizer.backward_passthrough
        ctx.notch = 1 if quantizer.flip_axis else 0
        ctx.bits = bits
        ctx.is_decimal = is_decimal
        ctx.channelwise = False
        ctx.channel_index = -1
        ctx.param_is_tensor = True
        ctx.param_host = None
        ctx.save_for_backward(decimal if is_decimal else weight.data.view(-1))
        # a [1, 1] parameter broadcasts a lower-rank input's result, like the unfused functions
        return _broadcast_result(y.view(input.shape), input.shape, weight)

    @staticmethod
    def backward(ctx, grad_output):
        return (_ste_backward(ctx, grad_output),) + (None,) * 4


class _RowFusedLine(torch.autograd.Function):
    """K8 for the asymmetric quantizer: per-row min / max -> lines EMA (in place) -> line fake-quantize in
    ONE launch; identity backward (ref quantize.py:393-430, :134-185)."""

    @staticmethod
    def forward(ctx, input, bits, weight, xs, t, float_zero_point, counter=None):
        if counter is not None:      # graph mode: this call's number is *counter + 1
            y, _ = ops.row_quant_fused_(xs, weight.data, ops.ROW_LINE, bits, 1, float_zero_point, t_dev=counter)
            counter.add_(1)
        else:
            y, _ = ops.row_quant_fused_(xs, weight.data, ops.ROW_LINE, bits, t, float_zero_point)
        return y.view(input.shape)

    @staticmethod
    def backward(ctx, grad_output):
        return (grad_output,) + (None,) * 6


def _row_fusable(quantizer, exact_type, x, weight, channel_index):
    """The fused row kernel replaces optimize() + forward() only for the stock callbacks (a subclass may
    override either), on a CUDA tensor quantized along its leading axis, without channel grouping."""
    if type(quantizer) is not exact_type or channel_index != 0 or quantizer.group_num > 0:
        return None
    if not (isinstance(x, torch.Tensor) and x.is_cuda and x.dim() >= 2 and isinstance(weight, nn.Parameter)):
        return None
    if tuple(weight.shape) != (x.shape[0], quantizer.weight_size) or not weight.is_contiguous():
        return None
    xs = N.as_f32_contiguous(x.detach())
    return xs if ops.row_quant_supported(xs, x.shape[0]) else None


def quantize_with_decimal(input: torch.Tensor, bits: int = 8, decimal: TensorOrInt = 5, channel_index: int = -1,
                          use_uint: bool = False, backward_passthrough: bool = False,
                          flip_axis: bool = False) -> torch.Tensor:
    """Power-of-two uniform fake-quantization (ref qsparse/quantize.py:188-210)."""
    return DecimalQuantization.apply(input, bits, decimal, channel_index, use_uint, backward_passthrough, flip_axis)


def quantize_with_scaler(input: torch.Tensor, bits: int = 8, scaler: TensorOrFloat = 0.1, channel_index: int = -1,
                         use_uint: bool = False, backward_passthrough: bool = False,
                         flip_axis: bool = False) -> torch.Tensor:
    """Scaling-factor uniform fake-quantization (ref qsparse/quantize.py:212-234)."""
    return ScalerQuantization.apply(input, bits, scaler, channel_index, use_uint, backward_passthrough, flip_axis)


def quantize_with_line(x: torch.Tensor, bits: int = 8,
                       lines: Union[Tuple[float, float], List[Tuple[float, float]]] = (-0.1, 0.9),
                       channel_index: int = -1, inplace: bool = False, float_zero_point: bool = True) -> torch.Tensor:
    """Asymmetric uniform fake-quantization (ref qsparse/quantize.py:236-255)."""
    return LineQuantization.apply(x, bits, lines, channel_index, inplace, float_zero_point)


# --------------------------------------------------------------------------- callbacks
class BaseQuantizer(nn.Module):
    """Plug-in protocol of ``quantize`` (ref qsparse/quantize.py:258-272): ``optimize``
    returns the updated ``[C or 1, weight_size]`` parameter, ``forward`` the quantized tensor."""

    weight_size = 1

    def optimize(self, tensor, bits, weight=None, batched=False, channel_index=-1) -> torch.Tensor:
        raise NotImplementedError

    def forward(self, tensor, bits, weight=None, batched=False, channel_index=-1) -> torch.Tensor:
        raise NotImplementedError

    def get_weight_shape(self, x, channelwise):
        return (1 if channelwise < 0 else x.shape[channelwise], self.weight_size)


class DecimalQuantizer(BaseQuantizer):
    """abs-max scale estimation with a running mean, scale restricted to powers of two
    (ref qsparse/quantize.py:275-367)."""

    weight_size = 1

    def __init__(self, use_uint: bool = False, backward_passthrough: bool = False, flip_axis: bool = False,
                 group_num=-1, group_timeout=512):
        super().__init__()
        self.use_uint = use_uint
        self.backward_passthrough = backward_passthrough
        self.flip_axis = flip_axis
        self.use_float_scaler = False
        self.function = DecimalQuantization.apply
        self.t = 0  # Python int, like the reference: not part of state_dict (SURVEY Q16)
        self.group_timeout = group_timeout
        self.groups = None
        self.group_num = group_num

    def quantize(self, tensor, bits, scaler, channel_index=-1, **kwargs):
        # scale -> decimal on the device: round(log2(nan_to_num(1/s)))  (quantize.py:316)
        weight = scaler if self.use_float_scaler else ops.scale_to_decimal(scaler)
        return self.function(tensor, bits, weight, channel_index, self.use_uint, self.backward_passthrough,
                             self.flip_axis)

    def optimize(self, x, bits, weight=None, batched=False, channel_index=-1, **kwargs):
        """new = max|x| / 2^(bits-1) per tensor / channel; running mean over calls
        (ref qsparse/quantize.py:327-349).  One reduction pass + one tiny EMA kernel."""
        N.require_cuda(x, "x")
        wshape = self.get_weight_shape(x, channel_index)
        if batched and channel_index >= 0 and x.shape[0] != 1:
            # the reference reshapes the C per-channel maxima to (-1, batch) and fails
            # for every batch size but 1 (quantize.py:341-343, SURVEY Q10)
            raise RuntimeError(
                f"shape '{list(wshape)}' is invalid for input of size "
                f"{max(int(x.shape[channel_index]) // int(x.shape[0]), 1)}: channel-wise Decimal/Scaler "
                "estimation on batched activations only works for batch size 1 in qsparse 2.0.1")
        with torch.no_grad():
            xs = N.as_native_contiguous(x.detach())
            layout = N.channel_layout(xs.shape, channel_index)
            absmax = ops.reduce_stats(xs, layout, absmax=True)["absmax"]
            if weight is None:
                weight = torch.zeros(wshape, dtype=torch.float32, device=x.device)
            target = weight.data if isinstance(weight, nn.Parameter) else weight
            assert tuple(target.shape) == tuple(wshape) and target.is_contiguous()
            if graphs.active():
                counter = graphs.quantizer_counter(self, x.device)
                ops.scale_ema_(target, absmax, bits, 0, t_dev=counter)
                counter.add_(1)
            else:
                ops.scale_ema_(target, absmax, bits, self.t)
        self.t += 1
        return weight

    def optimize_and_forward(self, x, bits, weight, channel_index=-1, **kwargs):
        """optimize() followed by forward() as one kernel when the tensor allows it (K8); None otherwise."""
        exact = ScalerQuantizer if self.use_float_scaler else DecimalQuantizer
        if channel_index < 0:
            # per tensor: partials -> one parameter kernel -> quantize
            if type(self) is not exact or self.group_num > 0 or not isinstance(weight, nn.Parameter):
                return None
            if not (isinstance(x, torch.Tensor) and x.is_cuda and x.numel() >= 1 and x.is_contiguous()):
                return None
            if tuple(weight.shape) != (1, 1):
                return None
            return _TensorFusedSte.apply(x, self, bits, weight, N.as_native_contiguous(x.detach()))
        xs = _row_fusable(self, exact, x, weight, channel_index)
        if xs is None:
            return None
        return _RowFusedSte.apply(x, self, bits, weight, xs)

    def _group(self, scaler):
        if self.groups is None:
            graphs.require_eager("the one-shot group-wise clustering step (host-side sklearn)")
            from sklearn.cluster import AgglomerativeClustering  # one-shot, host side (quantize.py:355-359)

            logging.danger(f"clustering {len(scaler)} channels into {self.group_num} groups")
            clustering = AgglomerativeClustering(n_clusters=self.group_num)
            clustering.fit(scaler.detach().cpu().numpy())
            self.groups = nn.Parameter(torch.from_numpy(clustering.labels_).to(scaler.device), requires_grad=False)
        # per-group mean of the [C, weight_size] parameter rows (quantize.py:361-366) in ONE launch on the
        # device: the reference's loop does `group_num` boolean-index + mean + scatter steps, each with a host
        # sync.  The mean is the correctly rounded one (<= 1 ulp from torch's fp32 mean).
        return ops.group_mean(scaler, self.groups, self.group_num).view(scaler.shape)

    def forward(self, tensor, bits, scaler, channel_index=-1, **kwargs):
        if self.t >= self.group_timeout and self.group_num > 0 and scaler.numel() > self.group_num:
            scaler = self._group(scaler)
        return self.quantize(tensor, bits, scaler, channel_index, **kwargs)


class PercentileQuantizer(DecimalQuantizer):
    """EXTENSION (not in qsparse 2.0.1; BASELINE.json's north_star asks for "abs-max and percentile statistics"):
    the scale statistic is the ``percentile``-th percentile of ``|x|`` instead of its maximum,

        new = sorted(|x|)[k] / 2^(bits-1),   k = clamp(ceil(percentile / 100 * n) - 1, 0, n - 1)

    per tensor (``channel_index=-1``) or per leading-axis channel (``channel_index=0``), with the same running
    mean as ``DecimalQuantizer`` (ref qsparse/quantize.py:344-348).  The k-th value comes from the exact
    one-pass select of the prune path (``qsb_kth_value(take_abs)``, 4 B/elem, no sort, no host sync).
    ``use_float_scaler=True`` quantizes with the scale itself (like ``ScalerQuantizer``), otherwise with the
    nearest power of two (like ``DecimalQuantizer``).  ``percentile=100`` reproduces the abs-max estimators bit
    for bit.  The forward does not saturate outliers (the reference's fake-quant functions never clamp in the
    forward, SURVEY Q1); the integer export does."""

    def __init__(self, percentile: float = 99.9, use_float_scaler: bool = False, **kwargs):
        super().__init__(**kwargs)
        if not 0.0 < percentile <= 100.0:
            raise ValueError("percentile must be in (0, 100]")
        self.percentile = float(percentile)
        self.use_float_scaler = bool(use_float_scaler)
        self.function = ScalerQuantization.apply if use_float_scaler else DecimalQuantization.apply

    @staticmethod
    def rank(percentile: float, n: int) -> int:
        return min(max(int(math.ceil(percentile / 100.0 * n)) - 1, 0), n - 1)

    def optimize(self, x, bits, weight=None, batched=False, channel_index=-1, **kwargs):
        N.require_cuda(x, "x")
        if channel_index not in (-1, 0) or (batched and channel_index == 0):
            raise NotImplementedError("PercentileQuantizer estimates per tensor or per leading-axis channel")
        wshape = self.get_weight_shape(x, channel_index)
        with torch.no_grad():
            xs = N.as_f32_contiguous(x.detach())
            if channel_index < 0:
                stat = ops.kth_value(xs.reshape(-1), self.rank(self.percentile, xs.numel()), take_abs=True)
            else:
                rows = xs.reshape(xs.shape[0], -1)
                k = self.rank(self.percentile, rows.shape[1])
                stat = torch.cat([ops.kth_value_batched(list(rows[i:i + 32]), [k] * len(rows[i:i + 32]),
                                                        take_abs=True) for i in range(0, rows.shape[0], 32)])
            if weight is None:
                weight = torch.zeros(wshape, dtype=torch.float32, device=x.device)
            target = weight.data if isinstance(weight, nn.Parameter) else weight
            assert tuple(target.shape) == tuple(wshape) and target.is_contiguous()
            if graphs.active():
                counter = graphs.quantizer_counter(self, x.device)
                ops.scale_ema_(target, stat.contiguous(), bits, 0, t_dev=counter)
                counter.add_(1)
            else:
                ops.scale_ema_(target, stat.contiguous(), bits, self.t)
        self.t += 1
        return weight

    def optimize_and_forward(self, *args, **kwargs):
        return None          # the fused abs-max routes do not apply


class BlockScaledQuantizer(BaseQuantizer):
    """EXTENSION (not in qsparse 2.0.1): quantization-aware training for the block-scaled FP8 / FP4 formats whose
    operands B200 tensor cores take natively,

        ``"mxfp8"``  blocks of 32, E4M3 elements, E8M0 power-of-two block scale   (OCP Microscaling v1.0)
        ``"mxfp4"``  blocks of 32, E2M1 elements, E8M0 power-of-two block scale   (OCP Microscaling v1.0)
        ``"nvfp4"``  blocks of 16, E2M1 elements, E4M3 block scale times the tensor scale ``w / 2688``

    Blocks are runs of consecutive elements of the rows of x viewed as ``[R, L]``: ``rows="last"`` splits the
    innermost physical axis (the reduction axis of a Linear weight and of ``[tokens, hidden]`` activations; C of a
    ``channels_last`` tensor), ``rows="leading"`` the contiguous tensor as ``[x.shape[0], -1]`` (the reduction axis of
    a conv weight).  The numerics are DESIGN §2 "Block-scaled formats"; the layer's ``bits`` is not used.

    The block scales are derived from each input, so the layer's ``weight`` ``[1, 1]`` only holds nvfp4's ``w``: the
    running mean of the tensor's abs-max, the ``DecimalQuantizer`` EMA at one bit.  The mx formats keep it at 0 and
    ``optimize`` only counts calls.  Output is fp32; the backward is the identity (straight-through).  Per tensor
    only (``channelwise=-1``).  ``export_block_scaled`` writes the packed codes and scales."""

    weight_size = 1

    def __init__(self, fmt: str = "nvfp4", rows: str = "last"):
        super().__init__()
        if fmt not in ops.BLOCK_FORMATS:
            raise ValueError(f"fmt must be one of {sorted(ops.BLOCK_FORMATS)}, got {fmt!r}")
        if rows not in ("last", "leading"):
            raise ValueError(f'rows must be "last" or "leading", got {rows!r}')
        self.fmt, self.rows = fmt, rows
        self.t = 0  # Python int like DecimalQuantizer's: not part of state_dict

    @staticmethod
    def check_channelwise(channelwise: int):
        if channelwise != -1:
            raise ValueError("BlockScaledQuantizer scales blocks inside each row: it needs channelwise=-1, "
                             f"got {channelwise}")

    def optimize(self, x, bits, weight=None, batched=False, channel_index=-1, **kwargs):
        self.check_channelwise(channel_index)
        N.require_cuda(x, "x")
        if self.fmt == "nvfp4":
            with torch.no_grad():
                xs, layout = _physical_layout(N.as_native(x.detach()), -1, False)
                absmax = ops.reduce_stats(xs, layout, absmax=True)["absmax"]
                if weight is None:
                    weight = torch.zeros((1, 1), dtype=torch.float32, device=x.device)
                target = weight.data if isinstance(weight, nn.Parameter) else weight
                assert tuple(target.shape) == (1, 1) and target.is_contiguous()
                if graphs.active():
                    counter = graphs.quantizer_counter(self, x.device)
                    ops.scale_ema_(target, absmax, 1, 0, t_dev=counter)
                    counter.add_(1)
                else:
                    ops.scale_ema_(target, absmax, 1, self.t)
        self.t += 1
        return weight

    def forward(self, x, bits, weight=None, channel_index=-1, **kwargs):
        self.check_channelwise(channel_index)
        return BlockScaledQuantization.apply(x, self.fmt, self.rows, weight if self.fmt == "nvfp4" else None)

    def optimize_and_forward(self, *args, **kwargs):
        return None          # no fused route: optimize() then forward()


class ScalerQuantizer(DecimalQuantizer):
    """Same estimator without the power-of-two restriction (ref qsparse/quantize.py:370-378)."""

    weight_size = 1

    def __init__(self, *args, **kwargs):
        super().__init__(*args, **kwargs)
        self.use_float_scaler = True
        self.function = ScalerQuantization.apply


class AdaptiveQuantizer(DecimalQuantizer):
    """Asymmetric quantizer: running mean of per-channel (min, max) lines
    (ref qsparse/quantize.py:381-430)."""

    weight_size = 2

    def __init__(self, *args, **kwargs):
        super().__init__(*args, **kwargs)
        self.function = LineQuantization.apply

    def quantize(self, tensor, bits, lines, channel_index=-1, **kwargs):
        # float zero-point while training, integer zero-point in eval (quantize.py:390-391)
        return self.function(tensor, bits, lines, channel_index, kwargs.get("inplace", False), self.training)

    def _next_t(self) -> int:
        """advance the call counter the way optimize() does for an existing weight (quantize.py:426-427)"""
        if isinstance(self.t, torch.Tensor):
            self.t += 1
            self._t_host = getattr(self, "_t_host", 0) + 1
            return self._t_host
        self.t += 1
        return self.t

    def optimize_and_forward(self, x, bits, weight, channel_index=-1, **kwargs):
        xs = _row_fusable(self, AdaptiveQuantizer, x, weight, channel_index)
        if xs is None:
            return None
        counter = graphs.quantizer_counter(self, xs.device) if graphs.active() else None
        with torch.no_grad():
            t = self._next_t()
        return _RowFusedLine.apply(x, bits, weight, xs, t, self.training, counter)

    def optimize(self, x, bits, weight=None, channel_index=-1, batched=False, **kwargs):
        N.require_cuda(x, "x")
        if batched and channel_index == 0:
            # the reference transposes axes 1 and 0 and then calls .view() on the non-contiguous result, which
            # raises for every input (quantize.py:399-402): same error type and message here
            raise RuntimeError("view size is not compatible with input tensor's size and stride (at least one "
                               "dimension spans across two contiguous subspaces). Use .reshape(...) instead.")
        with torch.no_grad():
            xs = N.as_native_contiguous(x.detach())
            # per-(sample, channel) min/max followed by min-of-mins / max-of-maxes over the
            # batch (quantize.py:396-418) == one per-channel reduction with outer = batch
            layout = N.channel_layout(xs.shape, channel_index)
            st = ops.reduce_stats(xs, layout, minmax=True)
            nch = layout[1]
            if weight is None:
                # the reference re-creates `t` as a device Parameter on this path (:423-425)
                self.t = nn.Parameter(torch.zeros(1, device=x.device), requires_grad=False)
                self.t += 1
                self._t_host = 1
                return torch.stack([st["min"], st["max"]], dim=1).view(nch, 2)
            assert (nch, 2) == tuple(weight.shape)
            counter = graphs.quantizer_counter(self, x.device) if graphs.active() else None
            t = self._next_t()
            target = weight.data if isinstance(weight, nn.Parameter) else weight
            if counter is not None:
                ops.lines_ema_(target, st["min"], st["max"], 1, t_dev=counter)
                counter.add_(1)
            else:
                ops.lines_ema_(target, st["min"], st["max"], t)
        return weight


# --------------------------------------------------------------------------- layer
class QuantizeLayer(nn.Module):
    """Fake-quantize the input tensor on a schedule (ref qsparse/quantize.py:434-518).

    State (``state_dict`` keys, dtypes and shapes as in the reference): ``weight``
    ``[C or 1, weight_size]`` fp32 and ``_n_updates`` ``[1]`` int32, both created on the
    first forward.  The step counter is mirrored on the host, so a forward enqueues
    kernels and never waits for the device."""

    def __str__(self):
        return (f"QuantizeLayer(bits={self.bits}, timeout={self.timeout}, "
                f"callback={self.callback.__class__.__name__}, channelwise={self.channelwise})")

    def __repr__(self):
        return str(self)

    def __init__(self, bits: int = 8, channelwise: int = 1, timeout: int = 1000, callback: BaseQuantizer = None,
                 batch_dimension: int = 0, name: str = ""):
        super().__init__()
        if isinstance(callback, BlockScaledQuantizer):
            callback.check_channelwise(channelwise)
        if get_option("log_on_created"):
            logging.info(f"[Quantize{name if name == '' else f' @ {name}'}] bits={bits} "
                         f"channelwise={channelwise} timeout={timeout}")
        self.name = name
        self.channelwise = channelwise
        self.timeout = timeout
        self.bits = bits
        self.callback = callback
        self.batch_dimension = batch_dimension  # 0: activation, -1: weight / bias
        self._quantized = False
        self._t_mirror = HostMirror()

    @property
    def initted(self) -> bool:
        return hasattr(self, "_n_updates")

    def _allocate(self, x):
        N.require_cuda(x, "x")
        rows = 1 if self.channelwise < 0 else x.shape[self.channelwise]
        self.weight = nn.Parameter(torch.zeros(rows, self.callback.weight_size, device=x.device),
                                   requires_grad=False)
        self._n_updates = nn.Parameter(torch.zeros(1, dtype=torch.int, device=x.device), requires_grad=False)
        self._t_mirror.wrote(self._n_updates, 0)

    def forward(self, x):
        if not self.initted:
            self._allocate(x)
        t = self._t_mirror.get(self._n_updates)
        if self.timeout <= 0:
            return x
        out = x
        if t >= self.timeout:
            if self.training:
                if t == self.timeout:
                    logging.warn(f"quantizing {self.name} with {self.bits} bits")
                fused = None
                if FUSE_ROW_QUANTIZE and ((self.channelwise == 0 and self.batch_dimension != 0)
                                          or self.channelwise < 0):
                    # weights quantized along their leading axis: estimate + quantize in one launch (K8);
                    # per-tensor layers: partials -> one parameter kernel -> quantize
                    fuse = getattr(self.callback, "optimize_and_forward", None)
                    fused = fuse(x, self.bits, self.weight, channel_index=self.channelwise) \
                        if fuse is not None else None
                if fused is None:
                    new_weight = self.callback.optimize(x, self.bits, self.weight,
                                                        batched=self.batch_dimension == 0,
                                                        channel_index=self.channelwise)
                    if new_weight is not None and new_weight is not self.weight:
                        self.weight.data[:] = new_weight
                self._quantized = True
                if fused is not None:
                    out = fused
            if self._quantized and out is x:
                out = self.callback(x, self.bits, self.weight, channel_index=self.channelwise,
                                    inplace=self.batch_dimension == 0)
        if self.training:
            self._n_updates.data.add_(1)      # in place: no Module.__setattr__ round trip
            self._t_mirror.wrote(self._n_updates, t + 1)
        return out


def export_integer(layer: "QuantizeLayer", x: torch.Tensor, pack4: bool = False):
    """Integer deployment form of what ``layer`` computes for ``x`` (SURVEY §8 f-3): the int8 / uint8 codes plus
    the parameters that turn them back into the fake-quantized values,

        DecimalQuantizer   q int8,  value = q * 2^-decimal          (decimal per tensor or per channel)
        ScalerQuantizer    q int8,  value = q * scale
        AdaptiveQuantizer  q uint8, value = q * step + lo,  step = (hi - lo) / 2^bits   (float zero-point form)

    one kernel, 5 B/elem (``qsb_quant_export_int8``).  Values outside the ``bits``-bit range saturate (the
    fake-quantizers themselves do not clamp in the forward, SURVEY Q1).  ``pack4`` (layers of <= 4 bits): ``q`` is
    a flat uint8 tensor with two codes per byte, element 2i in the low nibble (4.5 B/elem,
    ``qsb_quant_export_int4``); ``unpack_int4`` turns it back into the int8 form.  Returns a dict."""
    assert isinstance(layer, QuantizeLayer) and layer.initted and layer.bits <= 8
    assert not pack4 or layer.bits <= 4, "pack4 needs a layer of at most 4 bits"
    cb, ci = layer.callback, layer.channelwise
    xs = N.as_f32_contiguous(x.detach())
    layout = N.channel_layout(xs.shape, ci)
    w = layer.weight.data
    if isinstance(cb, AdaptiveQuantizer):
        lines = w.reshape(-1, 2)
        q = ops.quant_export_int8(xs, ops.EXPORT_LINE, lines, layer.bits, layout, pack4)
        return dict(q=q, kind="line", bits=layer.bits, lines=lines.clone(), channel_index=ci, packed=pack4,
                    shape=tuple(xs.shape))
    if cb.use_float_scaler:
        q = ops.quant_export_int8(xs, ops.EXPORT_SCALER, w.reshape(-1), layer.bits, layout, pack4)
        return dict(q=q, kind="scaler", bits=layer.bits, scale=w.reshape(-1).clone(), channel_index=ci, packed=pack4,
                    shape=tuple(xs.shape))
    dec = ops.scale_to_decimal(w).reshape(-1)
    q = ops.quant_export_int8(xs, ops.EXPORT_DECIMAL, dec, layer.bits, layout, pack4)
    return dict(q=q, kind="decimal", bits=layer.bits, decimal=dec, channel_index=ci, packed=pack4,
                shape=tuple(xs.shape))


def unpack_int4(exported: dict) -> torch.Tensor:
    """The int8 / uint8 code tensor of a ``pack4`` export (plain torch ops; a reader-side helper, not a hot path)."""
    q, shape = exported["q"], exported["shape"]
    n = 1
    for s_ in shape:
        n *= int(s_)
    nib = torch.stack([q & 0xF, q >> 4], dim=1).reshape(-1)[:n]
    if exported["kind"] == "line":
        return nib.reshape(shape)
    return ((nib.to(torch.int16) ^ 8) - 8).to(torch.int8).reshape(shape)   # sign-extend the 4-bit code


def export_block_scaled(layer: "QuantizeLayer", x: torch.Tensor) -> dict:
    """Packed deployment form of what a ``BlockScaledQuantizer`` layer computes for ``x``, in one pass
    (``qsb_block_export_dt``):

        codes         uint8 ``[R, L]`` E4M3 (mxfp8) or ``[R, ceil(L / 2)]`` E2M1 pairs, element 2i in the low nibble
        scales        uint8 ``[R, ceil(L / B)]``: E8M0 (mx formats, 0xFF for a NaN block) or E4M3 (nvfp4)
        tensor_scale  nvfp4's fp32 ``[1]`` ``w / 2688`` (None for the mx formats)

    plus ``fmt``, ``shape`` (x's), ``rows``, ``L`` and ``channels_last`` (the ``[R, L]`` view walks x in NHWC
    order).  ``dequantize_block_scaled`` turns it back into the layer's forward output bit for bit."""
    assert isinstance(layer, QuantizeLayer) and layer.initted and isinstance(layer.callback, BlockScaledQuantizer)
    cb = layer.callback
    N.require_cuda(x, "x")
    xs, R, L = _block_rows(x.detach(), cb.rows)
    w = layer.weight.data if cb.fmt == "nvfp4" else None
    codes, scales = ops.block_export(xs, cb.fmt, R, L, w)
    tensor_scale = None
    if w is not None:
        # a tensor divisor: torch turns division by a Python scalar into a multiplication by its reciprocal
        w1 = w.reshape(1).float()
        tensor_scale = torch.div(w1, torch.full_like(w1, 2688.0))
    return dict(codes=codes, scales=scales, tensor_scale=tensor_scale, fmt=cb.fmt, shape=tuple(x.shape),
                rows=cb.rows, L=L, channels_last=not xs.is_contiguous())


_E2M1_VALUES = (0.0, 0.5, 1.0, 1.5, 2.0, 3.0, 4.0, 6.0, -0.0, -0.5, -1.0, -1.5, -2.0, -3.0, -4.0, -6.0)


def dequantize_block_scaled(exported: dict) -> torch.Tensor:
    """The fp32 values of an ``export_block_scaled`` result, in x's shape (plain torch ops; a reader-side helper,
    not a hot path): element code times its block's scale, ``2^(e - 127)`` or ``RN(s_b * tensor_scale)``."""
    fmt, codes, scales, L = exported["fmt"], exported["codes"], exported["scales"], exported["L"]
    B = ops.BLOCK_FORMATS[fmt][1]
    R = codes.shape[0]
    if fmt == "mxfp8":
        v = codes.view(torch.float8_e4m3fn).float()
    else:
        lut = torch.tensor(_E2M1_VALUES, dtype=torch.float32, device=codes.device)
        v = lut[torch.stack([codes & 0xF, codes >> 4], dim=-1).reshape(R, -1)[:, :L].long()]
    if fmt == "nvfp4":
        s = scales.view(torch.float8_e4m3fn).float() * exported["tensor_scale"]
    else:
        e = scales.to(torch.int32)
        bits = torch.where(e == 0, torch.full_like(e, 0x00400000), e << 23)   # E8M0 0 is the subnormal 2^-127
        s = torch.where(e == 255, torch.full_like(e, 0x7FC00000), bits).view(torch.float32)
    y = v * s.repeat_interleave(B, dim=1)[:, :L]
    shape = exported["shape"]
    if exported["channels_last"]:
        n, c, h, w = shape
        return y.reshape(n, h, w, c).permute(0, 3, 1, 2)
    return y.reshape(shape)


def quantize(inp: nn.Module = None, bits: int = 8, channelwise: int = 1, timeout: int = 1000,
             callback: BaseQuantizer = None, bias_bits: int = -1, name: str = "") -> nn.Module:
    """Create a ``QuantizeLayer`` (no input module) or wrap the weight / bias of ``inp``
    with one (ref qsparse/quantize.py:521-585)."""
    callback = callback or ScalerQuantizer()
    kwargs = dict(bits=bits, channelwise=channelwise, timeout=timeout, callback=callback, bias_bits=bias_bits,
                  name=name)

    def make(batch_dimension=0, is_bias=False):
        if is_bias and bias_bits == -1:
            return lambda a: a
        if is_bias:
            layer_bits, layer_channelwise = bias_bits, (0 if channelwise >= 0 else -1)
        else:
            layer_bits, layer_channelwise = bits, channelwise
        # weight and bias layers share one callback instance, as in the reference (SURVEY Q12)
        return QuantizeLayer(bits=layer_bits, channelwise=layer_channelwise, timeout=int(timeout),
                             callback=callback, name=name, batch_dimension=batch_dimension)

    if inp is None:
        layer = make()
        setattr(layer, "_kwargs", kwargs)
        return layer
    if isinstance(inp, nn.Module):
        return imitate(inp, "quantize", make(-1), make(-1, is_bias=True))
    raise ValueError(f"{inp} is not a valid argument for quantize")
