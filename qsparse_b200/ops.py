"""Functional (non-autograd) wrappers of the C-ABI launchers.

Every function takes CUDA tensors, enqueues one or two kernels on torch's
current stream and returns without synchronising.  Argument conventions follow
``include/qsparse_b200.h``; ``layout`` is ``(outer, channels, inner)``.
"""
from __future__ import annotations

from ctypes import c_double, c_float, c_int, c_int64
from typing import Optional, Sequence, Tuple

import torch

from . import _native as N
from . import graphs

Layout = Tuple[int, int, int]


def _mask_kind(mask: Optional[torch.Tensor], numel: int, layout: Layout) -> int:
    if mask is None:
        return N.MASK_NONE
    if mask.dtype not in (torch.bool, torch.uint8):
        raise TypeError("mask must be a bool/uint8 tensor")
    N.require_cuda(mask, "mask")
    if not mask.is_contiguous():
        raise ValueError("mask must be contiguous")
    m = mask.numel()
    if m == layout[1] and (m != numel or layout[0] * layout[2] == 1):
        return N.MASK_CHANNEL
    if m == numel:
        return N.MASK_ELEMENT
    raise ValueError(f"mask with {m} elements fits neither channels={layout[1]} nor numel={numel}")


def _dev_param(p, what: str):
    """(device tensor or None, n, host scalar)."""
    if isinstance(p, torch.Tensor):
        if p.is_cuda:
            q = p.detach()
            if q.dtype != torch.float32 or not q.is_contiguous():
                q = q.float().contiguous()
            return q, q.numel(), 0.0
        if p.numel() == 1:
            return None, 1, float(p)
        raise RuntimeError(f"{what} is a multi-element CPU tensor; qsparse_b200 is CUDA-only")
    return None, 1, float(p)


def mask_layout(x_shape: Sequence[int], mask_shape: Sequence[int]) -> Tuple[str, Layout]:
    """How a broadcastable prune mask maps onto x: ('element', (1,1,n)) for a
    full-size mask, ('channel', (outer, C, inner)) when the kept axes form one
    contiguous run (e.g. [1,C,1,1], [1,C,H,W], [Cout,1,1,1])."""
    x_shape, mask_shape = list(x_shape), list(mask_shape)
    if len(x_shape) != len(mask_shape):
        raise RuntimeError(
            f"The size of tensor a ({len(x_shape)} dims) must match the size of tensor b "
            f"({len(mask_shape)} dims): prune mask and input ranks differ")
    n = 1
    for i, (sx, sm) in enumerate(zip(x_shape, mask_shape)):
        if sm != 1 and sm != sx:
            raise RuntimeError(
                f"The size of tensor a ({sx}) must match the size of tensor b ({sm}) at non-singleton dimension {i}")
        n *= sx
    kept = [i for i, (sx, sm) in enumerate(zip(x_shape, mask_shape)) if sm != 1]
    if not kept:
        return "channel", (1, 1, n)
    lo, hi = kept[0], kept[-1] + 1
    for i in range(lo, hi):
        if mask_shape[i] == 1 and x_shape[i] != 1:
            raise NotImplementedError(
                f"prune mask shape {tuple(mask_shape)} keeps non-adjacent axes of {tuple(x_shape)}; "
                "only one contiguous run of kept axes is supported")
    outer = 1
    for s in x_shape[:lo]:
        outer *= s
    ch = 1
    for s in x_shape[lo:hi]:
        ch *= s
    inner = 1
    for s in x_shape[hi:]:
        inner *= s
    if outer == 1 and inner == 1:
        return "element", (1, 1, n)
    return "channel", (outer, ch, inner)


def mask_perm(x_shape: Sequence[int], mask_shape: Sequence[int]):
    """None when ``mask_layout`` can address the mask directly; otherwise the axis permutation that moves the
    broadcast axes sandwiched between kept ones (``dimensions={1, 3}`` on NCHW -> mask [1,C,1,W]) in front of the
    first kept axis, so that the kept axes form one run ([N,H,C,W] with mask [1,1,C,W]).  The reference takes any
    dimension set through broadcasting (ref qsparse/sparse.py:66, util.py:93-101); here such a mask costs one
    transposing copy each way around the same kernels."""
    x_shape, mask_shape = list(x_shape), list(mask_shape)
    if len(x_shape) != len(mask_shape):
        return None
    kept = [i for i, (sx, sm) in enumerate(zip(x_shape, mask_shape)) if sm != 1]
    if not kept:
        return None
    lo, hi = kept[0], kept[-1] + 1
    between = [i for i in range(lo, hi) if mask_shape[i] == 1 and x_shape[i] != 1]
    if not between:
        return None
    inside = [i for i in range(lo, hi) if i not in between]
    return list(range(lo)) + between + inside + list(range(hi, len(x_shape)))


def invert_perm(perm):
    inv = [0] * len(perm)
    for i, p in enumerate(perm):
        inv[p] = i
    return inv


# ----------------------------------------------------------------------------- K1
def _f32_like(x):
    """the fp32 output of a fake-quantizer (also for a 16-bit x, SURVEY Q6), in x's memory format"""
    return torch.empty_like(x, dtype=torch.float32)


def fq_pow2_fwd(x, decimal, layout: Layout, mask=None, out=None):
    """x: fp32, bf16 or fp16 (read natively); the result is fp32."""
    N.require_cuda(x, "input")
    lib = N.load_library()
    y = _f32_like(x) if out is None else out
    dev, n, host = _dev_param(decimal, "decimal")
    mk = _mask_kind(mask, x.numel(), layout)
    N.check(lib.qsb_fq_pow2_fwd_dt(N.ptr(x), c_int(N.dtype_code(x)), N.ptr(y), N.ptr(dev), c_int64(n), c_double(host),
                                   N.ptr(mask), c_int(mk), c_int64(layout[0]), c_int64(layout[1]), c_int64(layout[2]),
                                   N.stream_ptr(x.device)), "qsb_fq_pow2_fwd_dt")
    return y


def fq_scaler_fwd(x, scaler, layout: Layout, mask=None, out=None):
    N.require_cuda(x, "input")
    lib = N.load_library()
    y = _f32_like(x) if out is None else out
    dev, n, host = _dev_param(scaler, "scaler")
    mk = _mask_kind(mask, x.numel(), layout)
    N.check(lib.qsb_fq_scaler_fwd_dt(N.ptr(x), c_int(N.dtype_code(x)), N.ptr(y), N.ptr(dev), c_int64(n),
                                     c_float(host), N.ptr(mask), c_int(mk), c_int64(layout[0]), c_int64(layout[1]),
                                     c_int64(layout[2]), N.stream_ptr(x.device)), "qsb_fq_scaler_fwd_dt")
    return y


def fq_line_fwd(x, lines, bits: int, float_zero_point: bool, layout: Layout, mask=None, out=None):
    """lines: CUDA float tensor [n, 2] (n == 1 or channels) or a (lo, hi) pair."""
    N.require_cuda(x, "input")
    lib = N.load_library()
    y = _f32_like(x) if out is None else out
    if isinstance(lines, torch.Tensor) and lines.is_cuda:
        dev = lines.detach()
        if dev.dtype != torch.float32 or not dev.is_contiguous():
            dev = dev.float().contiguous()
        n, lo, hi = dev.numel() // 2, 0.0, 0.0
    else:
        flat = torch.as_tensor(lines, dtype=torch.float32).reshape(-1)
        if flat.numel() != 2:
            raise RuntimeError("multi-row `lines` must be a CUDA tensor; qsparse_b200 is CUDA-only")
        dev, n, lo, hi = None, 1, float(flat[0]), float(flat[1])
    mk = _mask_kind(mask, x.numel(), layout)
    N.check(lib.qsb_fq_line_fwd_dt(N.ptr(x), c_int(N.dtype_code(x)), N.ptr(y), N.ptr(dev), c_int64(n), c_float(lo),
                                   c_float(hi), c_int(bits), c_int(1 if float_zero_point else 0), N.ptr(mask),
                                   c_int(mk), c_int64(layout[0]), c_int64(layout[1]), c_int64(layout[2]),
                                   N.stream_ptr(x.device)), "qsb_fq_line_fwd_dt")
    return y


# ----------------------------------------------------------------------------- K2
def ste_bwd(g, scale, is_decimal: bool, bits: int, notch: int, layout: Layout, mask=None, clamp_in_place=True,
            want_gx=False, gx_dtype=torch.float32):
    """Returns (g_clamped or None, gx or None).  clamp_in_place reproduces the
    reference's in-place `grad_output.clamp_` (quantize.py:72).  gx_dtype: bf16 / fp16 writes the input
    gradient of a 16-bit x directly in its dtype (rounded like autograd's cast of the fp32 value)."""
    N.require_cuda(g, "grad_output")
    lib = N.load_library()
    dev, n, host = _dev_param(scale, "scale")
    mk = _mask_kind(mask, g.numel(), layout)
    gc = g if clamp_in_place else None
    gx = torch.empty_like(g, dtype=gx_dtype) if (want_gx or not clamp_in_place) else None
    N.check(lib.qsb_ste_bwd_dt(N.ptr(g), N.ptr(gc), N.ptr(gx), c_int(N.NATIVE_DTYPES[gx_dtype]), N.ptr(dev),
                               c_int64(n), c_double(host), c_int(1 if is_decimal else 0), c_int(bits), c_int(notch),
                               N.ptr(mask), c_int(mk), c_int64(layout[0]), c_int64(layout[1]), c_int64(layout[2]),
                               N.stream_ptr(g.device)), "qsb_ste_bwd_dt")
    return gc, gx


EXPORT_DECIMAL, EXPORT_SCALER, EXPORT_LINE = 0, 1, 2


def quant_export_int8(x, kind: int, param, bits: int, layout: Layout, pack4: bool = False):
    """integer codes of a fake-quantizer: int8 (decimal / scaler) or uint8 (line) tensor of x's shape.
    ``param``: decimal / scale (float or tensor [1] / [C]) or lines ((lo, hi) or tensor [1|C, 2]).
    ``pack4`` (bits <= 4): a flat uint8 tensor of (n + 1) // 2 bytes, element 2i in the low nibble of byte i."""
    lib = N.load_library()
    N.require_cuda(x, "input")
    xs = N.as_f32_contiguous(x.detach())
    if pack4:
        q = torch.empty((xs.numel() + 1) // 2, dtype=torch.uint8, device=x.device)
    else:
        q = torch.empty(xs.shape, dtype=torch.uint8 if kind == EXPORT_LINE else torch.int8, device=x.device)
    dev, n, h1, h2 = None, 1, 0.0, 0.0
    if isinstance(param, torch.Tensor):
        N.require_cuda(param, "param")
        dev = param.detach().float().contiguous()
        n = dev.numel() // (2 if kind == EXPORT_LINE else 1)
    elif kind == EXPORT_LINE:
        h1, h2 = float(param[0]), float(param[1])
    else:
        h1 = float(param)
    fn, what = (lib.qsb_quant_export_int4, "qsb_quant_export_int4") if pack4 else \
        (lib.qsb_quant_export_int8, "qsb_quant_export_int8")
    N.check(fn(N.ptr(xs), N.ptr(q), c_int(kind), N.ptr(dev), c_int64(n), c_double(h1), c_double(h2), c_int(bits),
               c_int64(layout[0]), c_int64(layout[1]), c_int64(layout[2]), N.stream_ptr(x.device)), what)
    return q


# block-scaled FP8 / FP4 formats: name -> (C-ABI code, elements per block)
BLOCK_FORMATS = {"mxfp8": (0, 32), "mxfp4": (1, 32), "nvfp4": (2, 16)}


def _block_args(x, fmt: str, rows: int, L: int, tensor_amax):
    N.require_cuda(x, "input")
    if fmt not in BLOCK_FORMATS:
        raise ValueError(f"fmt must be one of {sorted(BLOCK_FORMATS)}, got {fmt!r}")
    if rows * L != x.numel():
        raise ValueError(f"[rows, L] = [{rows}, {L}] does not cover the {x.numel()} elements of x")
    if fmt == "nvfp4":
        if tensor_amax is None:
            raise ValueError("nvfp4 needs the tensor abs-max `tensor_amax` (a one-element CUDA tensor)")
        N.require_cuda(tensor_amax, "tensor_amax")
        tensor_amax = tensor_amax.detach().reshape(-1)[:1].float().contiguous()
    else:
        tensor_amax = None
    return BLOCK_FORMATS[fmt][0], tensor_amax


def fq_block_fwd(x, fmt: str, rows: int, L: int, tensor_amax=None):
    """Block-scaled fake quantization of x walked as [rows, L] in its memory order (``qsb_fq_block_fwd_dt``).
    x: fp32, bf16 or fp16, read natively; the result is fp32 in x's memory format.  ``tensor_amax``: nvfp4's w."""
    lib = N.load_library()
    code, w = _block_args(x, fmt, rows, L, tensor_amax)
    y = _f32_like(x)
    N.check(lib.qsb_fq_block_fwd_dt(N.ptr(x), c_int(N.dtype_code(x)), N.ptr(y), c_int64(rows), c_int64(L), c_int(code),
                                    N.ptr(w), N.stream_ptr(x.device)), "qsb_fq_block_fwd_dt")
    return y


def block_export(x, fmt: str, rows: int, L: int, tensor_amax=None):
    """(codes, scales) of the same quantizer in one pass (``qsb_block_export_dt``): uint8 codes [rows, L] (E4M3) or
    [rows, ceil(L / 2)] (two E2M1 codes per byte, element 2i in the low nibble), uint8 scales [rows, ceil(L / B)]."""
    lib = N.load_library()
    code, w = _block_args(x, fmt, rows, L, tensor_amax)
    B = BLOCK_FORMATS[fmt][1]
    codes = torch.empty((rows, L if fmt == "mxfp8" else (L + 1) // 2), dtype=torch.uint8, device=x.device)
    scales = torch.empty((rows, (L + B - 1) // B), dtype=torch.uint8, device=x.device)
    N.check(lib.qsb_block_export_dt(N.ptr(x), c_int(N.dtype_code(x)), N.ptr(codes), N.ptr(scales), c_int64(rows),
                                    c_int64(L), c_int(code), N.ptr(w), N.stream_ptr(x.device)), "qsb_block_export_dt")
    return codes, scales


# ----------------------------------------------------------------------------- K6
def mask_apply(x, mask, layout: Layout, out=None, out_dtype=None):
    """``x * mask``; x and the result may differ in dtype when one of them is fp32 and the other bf16 / fp16
    (``out_dtype``, default x's dtype)."""
    N.require_cuda(x, "input")
    lib = N.load_library()
    y = torch.empty_like(x, dtype=out_dtype or x.dtype) if out is None else out
    mk = _mask_kind(mask, x.numel(), layout)
    N.check(lib.qsb_mask_apply_dt(N.ptr(x), c_int(N.dtype_code(x)), N.ptr(y), c_int(N.dtype_code(y)), N.ptr(mask),
                                  c_int(mk), c_int64(layout[0]), c_int64(layout[1]), c_int64(layout[2]),
                                  N.stream_ptr(x.device)), "qsb_mask_apply_dt")
    return y


# ----------------------------------------------------------------------------- K3
def reduce_stats(x, layout: Layout, absmax=False, minmax=False, abssum=False, nnz=False, out=None):
    """One read of x -> dict of per-channel statistics (device tensors).  ``out`` may
    supply pre-allocated result tensors (e.g. views into a statistics row that is
    all-gathered afterwards)."""
    N.require_cuda(x, "input")
    lib = N.load_library()
    outer, ch, inner = layout
    what = (N.STAT_ABSMAX if absmax else 0) | (N.STAT_MINMAX if minmax else 0) | \
           (N.STAT_ABSSUM if (abssum or nnz) else 0) | (N.STAT_NNZ if nnz else 0)
    dev = x.device
    res = dict(out) if out else {}
    if absmax and "absmax" not in res:
        res["absmax"] = torch.empty(ch, dtype=torch.float32, device=dev)
    if (minmax or nnz) and "min" not in res:
        res["min"] = torch.empty(ch, dtype=torch.float32, device=dev)
    if minmax and "max" not in res:
        res["max"] = torch.empty(ch, dtype=torch.float32, device=dev)
    if (abssum or nnz) and "abssum" not in res:
        res["abssum"] = torch.empty(ch, dtype=torch.float64, device=dev)
    if nnz:
        res["nnz"] = torch.empty(ch, dtype=torch.float64, device=dev)
        res["tensor_min"] = torch.empty(1, dtype=torch.float32, device=dev)
    nbytes = lib.qsb_reduce_workspace_bytes(c_int64(outer), c_int64(ch), c_int64(inner))
    ws = N.workspace(dev, nbytes)
    N.check(lib.qsb_reduce_stats_dt(N.ptr(x), c_int(N.dtype_code(x)), c_int(what), c_int64(outer), c_int64(ch),
                                    c_int64(inner), N.ptr(res.get("absmax")), N.ptr(res.get("min")),
                                    N.ptr(res.get("max")), N.ptr(res.get("abssum")), N.ptr(res.get("nnz")),
                                    N.ptr(res.get("tensor_min")), N.ptr(ws), c_int64(ws.numel()), N.stream_ptr(dev)),
            "qsb_reduce_stats_dt")
    return res


# ----------------------------------------------------------------------------- K4
def scale_ema_(weight, absmax, bits: int, t: int, t_dev=None):
    """``t_dev`` (an int64 device counter): the index is ``*t_dev + t``, read by the kernel (CUDA graphs)."""
    lib = N.load_library()
    N.require_cuda(weight, "weight")
    if t_dev is not None:
        N.require_cuda(t_dev, "t_dev")
        N.check(lib.qsb_scale_ema_at(N.ptr(weight), N.ptr(absmax), c_int64(weight.numel()), c_int(bits), N.ptr(t_dev),
                                     c_int64(t), N.stream_ptr(weight.device)), "qsb_scale_ema_at")
        return weight
    N.check(lib.qsb_scale_ema(N.ptr(weight), N.ptr(absmax), c_int64(weight.numel()), c_int(bits), c_int64(t),
                              N.stream_ptr(weight.device)), "qsb_scale_ema")
    return weight


def scale_to_decimal(scale):
    lib = N.load_library()
    N.require_cuda(scale, "scale")
    s = scale.detach()
    if s.dtype != torch.float32 or not s.is_contiguous():
        s = s.float().contiguous()
    d = torch.empty_like(s)
    N.check(lib.qsb_scale_to_decimal(N.ptr(s), N.ptr(d), c_int64(s.numel()), N.stream_ptr(s.device)),
            "qsb_scale_to_decimal")
    return d


def group_mean(values, labels, groups: int):
    """every row of ``values`` [C, weight_size] replaced by the mean of its group's rows (``labels`` int64 [C]);
    one launch, result in a new tensor"""
    lib = N.load_library()
    N.require_cuda(values, "values")
    v = values.detach()
    if v.dtype != torch.float32 or not v.is_contiguous():
        v = v.float().contiguous()
    lab = labels.detach().to(device=v.device, dtype=torch.int64).contiguous()
    out = torch.empty_like(v)
    c = v.shape[0] if v.dim() > 0 else 1
    N.check(lib.qsb_group_mean(N.ptr(v), N.ptr(lab), N.ptr(out), c_int64(c), c_int64(max(v.numel() // max(c, 1), 1)),
                               c_int64(int(groups)), N.stream_ptr(v.device)), "qsb_group_mean")
    return out


def lines_ema_(lines, mn, mx, t: int, t_dev=None):
    lib = N.load_library()
    N.require_cuda(lines, "lines")
    if t_dev is not None:
        N.require_cuda(t_dev, "t_dev")
        N.check(lib.qsb_lines_ema_at(N.ptr(lines), N.ptr(mn), N.ptr(mx), c_int64(lines.numel() // 2), N.ptr(t_dev),
                                     c_int64(t), N.stream_ptr(lines.device)), "qsb_lines_ema_at")
        return lines
    N.check(lib.qsb_lines_ema(N.ptr(lines), N.ptr(mn), N.ptr(mx), c_int64(lines.numel() // 2), c_int64(t),
                              N.stream_ptr(lines.device)), "qsb_lines_ema")
    return lines


ROW_DECIMAL, ROW_SCALER, ROW_LINE = 0, 1, 2


def row_quant_supported(x, rows: int) -> bool:
    """Can ``qsb_row_quant_fused`` take this [rows, inner] fp32 contiguous tensor?"""
    n = x.numel()
    if rows <= 0 or n == 0 or n % rows:
        return False
    inner = n // rows
    return inner % 8 == 0 and inner <= 16384 and x.data_ptr() % 32 == 0


def row_quant_fused_(x, param, kind: int, bits: int, t: int, float_zero_point=True, mask=None, t_dev=None):
    """K8: per-row estimate (abs-max or min/max) -> EMA into ``param`` (in place) -> fake-quantize, one launch.
    x: [rows, ...] fp32 contiguous; param: [rows, 1] (scale) or [rows, 2] (lines).
    ``mask``: optional element prune mask of x's shape: estimate and quantize ``x * mask`` (the weight chain
    ``quantize(prune(layer))`` with a frozen mask).  Returns (y, decimal or None)."""
    lib = N.load_library()
    N.require_cuda(x, "x")
    N.require_cuda(param, "weight")
    rows = param.shape[0]
    inner = x.numel() // rows
    y = torch.empty_like(x)
    dec = torch.empty(rows, dtype=torch.float32, device=x.device) if kind == ROW_DECIMAL else None
    if mask is not None:
        N.require_cuda(mask, "mask")
        if mask.numel() != x.numel() or mask.dtype not in (torch.bool, torch.uint8) or not mask.is_contiguous():
            raise ValueError("mask must be a contiguous bool / uint8 tensor with x's number of elements")
    if t_dev is not None:       # CUDA graphs: the EMA index is *t_dev + t, read by the kernel
        N.require_cuda(t_dev, "t_dev")
        N.check(lib.qsb_row_quant_fused_at(N.ptr(x), N.ptr(y), N.ptr(param), N.ptr(dec), N.ptr(mask), c_int(kind),
                                           c_int(bits), c_int(1 if float_zero_point else 0), c_int64(rows),
                                           c_int64(inner), N.ptr(t_dev), c_int64(t), N.stream_ptr(x.device)),
                "qsb_row_quant_fused_at")
        return y, dec
    if mask is not None:
        N.check(lib.qsb_row_quant_fused_masked(N.ptr(x), N.ptr(y), N.ptr(param), N.ptr(dec), N.ptr(mask), c_int(kind),
                                               c_int(bits), c_int(1 if float_zero_point else 0), c_int64(rows),
                                               c_int64(inner), c_int64(t), N.stream_ptr(x.device)),
                "qsb_row_quant_fused_masked")
        return y, dec
    N.check(lib.qsb_row_quant_fused(N.ptr(x), N.ptr(y), N.ptr(param), N.ptr(dec), c_int(kind), c_int(bits),
                                    c_int(1 if float_zero_point else 0), c_int64(rows), c_int64(inner), c_int64(t),
                                    N.stream_ptr(x.device)), "qsb_row_quant_fused")
    return y, dec


def magnitude_ema_reduced_(magnitude, stats: dict, count: float, t: int, use_l0=False):
    lib = N.load_library()
    N.require_cuda(magnitude, "magnitude")
    N.check(lib.qsb_magnitude_ema_reduced(N.ptr(magnitude), N.ptr(stats["abssum"]), N.ptr(stats.get("nnz")),
                                          N.ptr(stats.get("tensor_min")), c_int(1 if use_l0 else 0),
                                          c_int64(magnitude.numel()), c_double(count), c_int64(t),
                                          N.stream_ptr(magnitude.device)), "qsb_magnitude_ema_reduced")
    return magnitude


def magnitude_ema_full_(magnitude, x, t: int, tensor_min=None, use_l0=False):
    lib = N.load_library()
    N.require_cuda(magnitude, "magnitude")
    N.check(lib.qsb_magnitude_ema_full(N.ptr(magnitude), N.ptr(x), N.ptr(tensor_min), c_int(1 if use_l0 else 0),
                                       c_int64(magnitude.numel()), c_int64(t), N.stream_ptr(magnitude.device)),
            "qsb_magnitude_ema_full")
    return magnitude


# ----------------------------------------------------------------------------- K5 / K6
def new_select_hints(count: int, device) -> torch.Tensor:
    """zeroed pivot-hint state for ``count`` tensors (see ``kth_value(hint=...)``)"""
    return torch.zeros(count, 8, dtype=torch.int32, device=device)


def kth_value(v, k: int, take_abs=False, hint=None):
    """device scalar holding sorted(v)[k] (ascending, NaNs last).

    ``hint``: optional persistent state from ``new_select_hints(1, device)`` for a loop that asks for the same
    order statistic of a slowly drifting tensor every step: from the third call on the pivots come from the
    previous answer instead of a fresh sample (exact either way)."""
    if hint is not None:
        return kth_value_batched([v], [k], take_abs, hints=hint)
    lib = N.load_library()
    N.require_cuda(v, "importance")
    n = v.numel()
    thr = torch.empty(1, dtype=torch.float32, device=v.device)
    nbytes = lib.qsb_kth_workspace_bytes(c_int64(n))
    ws = N.workspace(v.device, nbytes)
    N.check(lib.qsb_kth_value(N.ptr(v), c_int64(n), c_int64(k), c_int(1 if take_abs else 0), N.ptr(thr), N.ptr(ws),
                              c_int64(ws.numel()), N.stream_ptr(v.device)), "qsb_kth_value")
    return thr


def _ptr_array(tensors):
    import ctypes
    return (ctypes.c_void_p * len(tensors))(*[t.data_ptr() for t in tensors])


def _multi_ok(*lists) -> bool:
    """the multi-tensor kernels need fp32 contiguous, 32-byte aligned tensors"""
    for ts in lists:
        for t in ts:
            if t.dtype not in (torch.float32, torch.bool, torch.uint8) or not t.is_contiguous() \
                    or t.data_ptr() % 32:
                return False
    return True


def magnitude_ema_full_multi_(magnitudes, xs, t: int):
    """``magnitude_ema_full_`` for every (magnitude, x) pair in ONE launch (falls back to one launch per
    tensor when a tensor is not 32-byte aligned)."""
    if not _multi_ok(magnitudes, xs):
        for m, x in zip(magnitudes, xs):
            magnitude_ema_full_(m, N.as_f32_contiguous(x.detach()), t)
        return magnitudes
    lib = N.load_library()
    count = len(magnitudes)
    ns = (c_int64 * count)(*[m.numel() for m in magnitudes])
    N.check(lib.qsb_magnitude_ema_full_multi(_ptr_array(magnitudes), _ptr_array(xs), ns, c_int(count), c_int64(t),
                                             N.stream_ptr(magnitudes[0].device)), "qsb_magnitude_ema_full_multi")
    return magnitudes


def mask_build_apply_multi(importances, thr, xs, masks, outs, take_abs=False):
    """``mask_build_apply`` for every layer in ONE launch; ``thr`` is the float32 [L] threshold tensor."""
    if not _multi_ok(importances, xs, outs, masks) or not thr.is_contiguous():
        for i, (imp, x, m, o) in enumerate(zip(importances, xs, masks, outs)):
            mask_build_apply(imp, thr[i:i + 1], x, m, take_abs, out=o)
        return outs
    lib = N.load_library()
    count = len(importances)
    ns = (c_int64 * count)(*[x.numel() for x in xs])
    N.check(lib.qsb_mask_build_apply_multi(_ptr_array(importances), c_int(1 if take_abs else 0), N.ptr(thr),
                                           _ptr_array(xs), _ptr_array(outs), _ptr_array(masks), ns, c_int(count),
                                           N.stream_ptr(xs[0].device)), "qsb_mask_build_apply_multi")
    return outs


def prune_step_supported(magnitudes, xs, masks, outs) -> bool:
    """can ``prune_unstructured_step_batched_`` take these tensors? (fp32 / bool, contiguous, 32-byte aligned)"""
    return _multi_ok(magnitudes, xs, outs, masks) and all(x.dtype == torch.float32 for x in xs)


def prune_unstructured_step_batched_(magnitudes, xs, masks, outs, ks, t: int, hints=None, t_dev=None):
    """K9: the whole unstructured running-average prune step of a set of tensors — magnitude EMA (in place),
    exact k-th value threshold, mask, ``out = x * mask`` — in ONE streaming pass plus a few small launches
    (17 B/elem instead of 29).  Returns the thresholds (float32 [L]).  Same results as
    ``magnitude_ema_full_`` + ``kth_value`` + ``mask_build_apply`` per tensor."""
    lib = N.load_library()
    count = len(magnitudes)
    dev = magnitudes[0].device
    ns = (c_int64 * count)(*[m.numel() for m in magnitudes])
    kk = (c_int64 * count)(*[int(k) for k in ks])
    thr = torch.empty(count, dtype=torch.float32, device=dev)
    nbytes = lib.qsb_prune_step_workspace_bytes(ns, c_int(count))
    ws = N.workspace(dev, nbytes)
    if hints is not None:
        assert hints.dtype == torch.int32 and hints.numel() >= 8 * count and hints.is_contiguous()
    if t_dev is not None:           # CUDA graphs: the EMA index is *t_dev + t, read by the kernels
        N.require_cuda(t_dev, "t_dev")
        N.check(lib.qsb_prune_unstructured_step_batched_at(
            _ptr_array(magnitudes), _ptr_array(xs), _ptr_array(outs), _ptr_array(masks), ns, kk, c_int(count),
            N.ptr(t_dev), c_int64(t), N.ptr(thr), N.ptr(hints), N.ptr(ws), c_int64(ws.numel()), N.stream_ptr(dev)),
            "qsb_prune_unstructured_step_batched_at")
        return thr
    if hints is not None:
        N.check(lib.qsb_prune_unstructured_step_batched_hinted(
            _ptr_array(magnitudes), _ptr_array(xs), _ptr_array(outs), _ptr_array(masks), ns, kk, c_int(count),
            c_int64(t), N.ptr(thr), N.ptr(hints), N.ptr(ws), c_int64(ws.numel()), N.stream_ptr(dev)),
            "qsb_prune_unstructured_step_batched_hinted")
        return thr
    N.check(lib.qsb_prune_unstructured_step_batched(_ptr_array(magnitudes), _ptr_array(xs), _ptr_array(outs),
                                                    _ptr_array(masks), ns, kk, c_int(count), c_int64(t), N.ptr(thr),
                                                    N.ptr(ws), c_int64(ws.numel()), N.stream_ptr(dev)),
            "qsb_prune_unstructured_step_batched")
    return thr


def kth_value_batched(vs, ks, take_abs=False, hints=None):
    """thresholds ``sorted(vs[i])[ks[i]]`` of several tensors (the layers of a weight set) in ONE launch
    sequence: float32 device tensor [len(vs)].  Same kernels as ``kth_value``; blockIdx.y is the tensor."""
    import ctypes
    lib = N.load_library()
    count = len(vs)
    dev = vs[0].device
    flat = []
    for v in vs:
        N.require_cuda(v, "importance")
        flat.append(N.as_f32_contiguous(v.detach()).reshape(-1))
    ptrs = (ctypes.c_void_p * count)(*[t.data_ptr() for t in flat])
    ns = (c_int64 * count)(*[t.numel() for t in flat])
    kk = (c_int64 * count)(*[int(k) for k in ks])
    thr = torch.empty(count, dtype=torch.float32, device=dev)
    nbytes = lib.qsb_kth_batched_workspace_bytes(ns, c_int(count))
    ws = N.workspace(dev, nbytes)
    if hints is not None:
        assert hints.dtype == torch.int32 and hints.numel() >= 8 * count and hints.is_contiguous()
        N.check(lib.qsb_kth_value_batched_hinted(ptrs, ns, kk, c_int(count), c_int(1 if take_abs else 0), N.ptr(thr),
                                                 N.ptr(hints), N.ptr(ws), c_int64(ws.numel()), N.stream_ptr(dev)),
                "qsb_kth_value_batched_hinted")
        return thr
    N.check(lib.qsb_kth_value_batched(ptrs, ns, kk, c_int(count), c_int(1 if take_abs else 0), N.ptr(thr), N.ptr(ws),
                                      c_int64(ws.numel()), N.stream_ptr(dev)), "qsb_kth_value_batched")
    return thr


def mask_from_threshold(importance, thr, mask_out, take_abs=False):
    lib = N.load_library()
    N.check(lib.qsb_mask_from_threshold(N.ptr(importance), c_int(1 if take_abs else 0), N.ptr(thr), N.ptr(mask_out),
                                        c_int64(importance.numel()), N.stream_ptr(importance.device)),
            "qsb_mask_from_threshold")
    return mask_out


def mask_build_apply(importance, thr, x, mask_out, take_abs=False, out=None):
    lib = N.load_library()
    y = torch.empty_like(x) if out is None else out
    N.check(lib.qsb_mask_build_apply(N.ptr(importance), c_int(1 if take_abs else 0), N.ptr(thr), N.ptr(x), N.ptr(y),
                                     N.ptr(mask_out), c_int64(x.numel()), N.stream_ptr(x.device)),
            "qsb_mask_build_apply")
    return y


FUSED_STEP_MAX_CHANNELS = 1024      # the reduction's last CTA runs the step (kStepFusedMaxChannels)
STEP_KERNEL_MAX_CHANNELS = 4096     # the one-CTA step kernel's shared memory (kStepMaxChannels, step_epilogue.cuh)
STEP_MAX_ROWS = 4096                # statistics rows the parameter step combines (qsb_prune_quant_params)
# A route choice, not a kernel limit: up to here the step kernel finalizes the reduction's partials itself (and
# runs the peer exchange); above it the statistics are finalized first.  Moving it changes which launch sequence
# runs for 2049-4096 channels, which has not been measured.
PARTIALS_ROUTE_MAX_CHANNELS = 2048


def prune_quant_params(magnitude, mask, scale, decimal_out, stats: dict, count: float, t_prune: int,
                       update_magnitude: int, refresh_mask: bool, k: int, bits: int, t_quant: int,
                       update_scale: bool, n_rows: int = 1, row_stride_bytes: int = 0):
    """stats["abssum"] / stats["absmax"] point at row 0; further rows (ranks / chunks) follow
    every row_stride_bytes and are combined inside the kernel in row order.  Above
    STEP_KERNEL_MAX_CHANNELS channels the same step runs as a sequence of launches."""
    if mask.numel() > STEP_KERNEL_MAX_CHANNELS:
        return _prune_quant_params_composed(magnitude, mask, scale, decimal_out, stats, count, t_prune,
                                            update_magnitude, refresh_mask, k, bits, t_quant, update_scale,
                                            n_rows, row_stride_bytes)
    lib = N.load_library()
    N.check(lib.qsb_prune_quant_params(N.ptr(magnitude), N.ptr(mask), N.ptr(scale), N.ptr(decimal_out),
                                       N.ptr(stats.get("abssum")), N.ptr(stats.get("absmax")),
                                       c_int64(n_rows), c_int64(row_stride_bytes),
                                       c_int64(mask.numel()), c_double(count), c_int64(t_prune),
                                       c_int(update_magnitude), c_int(1 if refresh_mask else 0), c_int64(k),
                                       c_int(bits), c_int64(t_quant), c_int(1 if update_scale else 0),
                                       N.stream_ptr(mask.device)), "qsb_prune_quant_params")


def _prune_quant_params_composed(magnitude, mask, scale, decimal_out, stats, count, t_prune, update_magnitude,
                                 refresh_mask, k, bits, t_quant, update_scale, n_rows, row_stride_bytes):
    """``prune_quant_params`` for more channels than its one-CTA kernel holds in shared memory: the same
    arithmetic in the same order, as magnitude EMA -> exact k-th value -> mask -> abs-max of the kept channels
    -> scale EMA -> decimal launches."""
    ch = mask.numel()
    # the kernel's row count limit too, so that both routes take the same arguments
    bad = (update_magnitude not in (0, 1, 2) or not 1 <= n_rows <= STEP_MAX_ROWS or (update_magnitude and not count > 0)
           or (refresh_mask and not 0 <= k < ch))
    if bad:
        N.check(-1, "qsb_prune_quant_params")     # QSB_E_BADARG, as the kernel's entry point returns it
    abssum, absmax = stats.get("abssum"), stats.get("absmax")
    if n_rows > 1:
        # rows of other ranks: combined in row order like the kernel (fp64 sums, NaN-propagating maxima)
        def row(t, r):
            off = r * row_stride_bytes
            assert off % t.element_size() == 0
            return torch.as_strided(t, (ch,), (1,), t.storage_offset() + off // t.element_size())
        abssum = abssum.clone() if abssum is not None else None
        absmax = absmax.clone() if absmax is not None else None
        for r in range(1, n_rows):
            if abssum is not None:
                abssum += row(stats["abssum"], r)
            if absmax is not None:
                torch.maximum(absmax, row(stats["absmax"], r), out=absmax)
    if update_magnitude == 2:
        # this step's mean |x| itself: the EMA at t = 0 of a zeroed vector is (0 * 0 + m) / 1 = m
        importance = torch.zeros(ch, dtype=torch.float32, device=mask.device)
        magnitude_ema_reduced_(importance, {"abssum": abssum}, count, 0)
    else:
        importance = magnitude
        if update_magnitude == 1:
            magnitude_ema_reduced_(magnitude, {"abssum": abssum}, count, t_prune)
    if refresh_mask:
        mask_from_threshold(importance, kth_value(importance, k), mask)
    if update_scale:
        # abs-max of x * mask: a pruned channel counts |x * 0|, i.e. 0, or NaN where it holds an inf / NaN
        kept = mask_apply(absmax, mask, (1, ch, 1))
        scale_ema_(scale.view(-1), reduce_stats(kept, (1, 1, ch), absmax=True)["absmax"], bits, t_quant)
    if decimal_out is not None:
        decimal_out.view(-1).copy_(scale_to_decimal(scale.view(-1)))


def reduce_partials(x, layout: Layout):
    """Stage 1 of the sum|x| / max|x| reduction only; the partials stay in the returned
    workspace for prune_quant_step_params (which finalizes them in its own kernel)."""
    N.require_cuda(x, "input")
    lib = N.load_library()
    outer, ch, inner = layout
    nbytes = lib.qsb_reduce_workspace_bytes(c_int64(outer), c_int64(ch), c_int64(inner))
    ws = N.workspace(x.device, nbytes)
    N.check(lib.qsb_reduce_partials_dt(N.ptr(x), c_int(N.dtype_code(x)), c_int64(outer), c_int64(ch), c_int64(inner),
                                       N.ptr(ws), c_int64(ws.numel()), N.stream_ptr(x.device)),
            "qsb_reduce_partials_dt")
    return ws


def prune_quant_step_params(magnitude, mask, scale, decimal_out, workspace, layout: Layout, count: float,
                            t_prune: int, update_magnitude: int, refresh_mask: bool, k: int, bits: int,
                            t_quant: int, update_scale: bool, group=None, step_stamp: int = 1,
                            abssum_out=None, absmax_out=None, step_counter=None):
    """finalize + (peer-memory exchange) + parameter update in ONE kernel.  `group` is a
    parallel.P2PExchange handle (ctypes pointer) or None for a single GPU."""
    lib = N.load_library()
    outer, ch, inner = layout
    N.check(lib.qsb_prune_quant_step_params(
        N.ptr(magnitude), N.ptr(mask), N.ptr(scale), N.ptr(decimal_out), N.ptr(workspace),
        c_int64(workspace.numel()), c_int64(outer), c_int64(ch), c_int64(inner), group, c_int64(step_stamp),
        c_double(count), c_int64(t_prune), c_int(update_magnitude), c_int(int(refresh_mask)), c_int64(k),
        c_int(bits), c_int64(t_quant), c_int(1 if update_scale else 0), N.ptr(abssum_out), N.ptr(absmax_out),
        N.ptr(step_counter), N.stream_ptr(mask.device)), "qsb_prune_quant_step_params")


_arrival_counters = {}


def arrival_counter(device: torch.device) -> torch.Tensor:
    """the zero-initialised uint32 the fused step's last-arriving CTA is elected with: one per
    (device, stream); the kernel leaves it zero"""
    key = N.stream_key(device)
    c = _arrival_counters.get(key)
    if c is None:
        c = torch.zeros(64, dtype=torch.int32, device=device)   # a 256-byte line of its own
        _arrival_counters[key] = c
    return c


def reduce_prune_quant_step(x, layout: Layout, magnitude, mask, scale, decimal_out, count: float, t_prune: int,
                            update_magnitude: int, refresh_mask, k: int, bits: int, t_quant: int,
                            update_scale: bool, group=None, step_stamp: int = 1, abssum_out=None, absmax_out=None,
                            stats_local: bool = False, step_counter=None, arrival=None, timing=None):
    """ONE launch: sum|x| / max|x| reduction of x whose last-arriving CTA finalizes, exchanges with the
    peer GPUs (``group`` = parallel.P2PExchange handle) and updates magnitude / mask / scale / decimal.
    ``arrival``: a caller-owned zeroed int32 tensor (default: one per device and stream, created on first
    use — pass your own when capturing a CUDA graph so that no fill is captured)."""
    N.require_cuda(x, "input")
    if step_counter is not None:
        N.require_cuda(step_counter, "step_counter")
    lib = N.load_library()
    outer, ch, inner = layout
    nbytes = lib.qsb_reduce_workspace_bytes(c_int64(outer), c_int64(ch), c_int64(inner))
    ws = N.workspace(x.device, nbytes)
    N.check(lib.qsb_reduce_prune_quant_step_dt(
        N.ptr(x), c_int(N.dtype_code(x)), c_int64(outer), c_int64(ch), c_int64(inner), N.ptr(ws), c_int64(ws.numel()),
        N.ptr(arrival if arrival is not None else arrival_counter(x.device)), N.ptr(magnitude), N.ptr(mask), N.ptr(scale), N.ptr(decimal_out), group,
        c_int64(step_stamp), c_double(count), c_int64(t_prune), c_int(update_magnitude), c_int(int(refresh_mask)),
        c_int64(k), c_int(bits), c_int64(t_quant), c_int(1 if update_scale else 0), N.ptr(abssum_out),
        N.ptr(absmax_out), c_int(1 if stats_local else 0), N.ptr(step_counter), N.ptr(timing),
        N.stream_ptr(x.device)), "qsb_reduce_prune_quant_step_dt")


def _step_route(channels: int, step_counter=None) -> str:
    """The route of the structured prune -> quantize step by channel count (pow2 and line form alike):

      <= FUSED_STEP_MAX_CHANNELS      "one"       stage 1 whose last-arriving CTA runs the step (one launch)
      <= PARTIALS_ROUTE_MAX_CHANNELS  "partials"  stage 1 + the one-CTA step kernel on its partials
      otherwise                       "stats"     finalized statistics + the step on rows (pow2 form only)

    A device ``step_counter`` (CUDA graphs) is taken by the one-launch route only: with more channels this raises
    ``graphs.NotCapturable``."""
    if channels <= FUSED_STEP_MAX_CHANNELS:
        return "one"
    if step_counter is not None:
        raise graphs.NotCapturable(f"the structured prune -> quantize step with more than {FUSED_STEP_MAX_CHANNELS} "
                                   "channels")
    return "partials" if channels <= PARTIALS_ROUTE_MAX_CHANNELS else "stats"


def structured_prune_quant_step(x, layout: Layout, magnitude, mask, scale, decimal_out, count: float, t_prune: int,
                                update_magnitude: int, refresh_mask, k: int, bits: int, t_quant: int,
                                update_scale: bool, group=None, step_stamp: int = 1, step_counter=None):
    """The structured prune -> pow2 quantize parameter step on x, by channel count (``_step_route``):

      one       reduce_prune_quant_step
      partials  reduce_partials + prune_quant_step_params
      stats     reduce_stats + prune_quant_params (single GPU only)

    Arguments as in ``reduce_prune_quant_step``."""
    route = _step_route(layout[1], step_counter)
    if route == "one":
        reduce_prune_quant_step(x, layout, magnitude, mask, scale, decimal_out, count, t_prune, update_magnitude,
                                refresh_mask, k, bits, t_quant, update_scale, group=group, step_stamp=step_stamp,
                                step_counter=step_counter)
    elif route == "partials":
        ws = reduce_partials(x, layout)
        prune_quant_step_params(magnitude, mask, scale, decimal_out, ws, layout, count, t_prune, update_magnitude,
                                refresh_mask, k, bits, t_quant, update_scale, group=group, step_stamp=step_stamp)
    elif group is not None:
        raise ValueError(f"the peer exchange takes at most {PARTIALS_ROUTE_MAX_CHANNELS} channels")
    else:
        stats = reduce_stats(x, layout, absmax=True, abssum=True)
        prune_quant_params(magnitude, mask, scale, decimal_out, stats, count, t_prune, update_magnitude,
                           refresh_mask, k, bits, t_quant, update_scale)


# ----------------------------------------------------------------------------- the line form (AdaptiveQuantizer)
def reduce_prune_line_step(x, layout: Layout, magnitude, mask, lines, count: float, t_prune: int,
                           update_magnitude: int, refresh_mask, k: int, t_line: int, abssum_out=None, min_out=None,
                           max_out=None, step_counter=None, arrival=None):
    """ONE launch: sum|x| / min / max reduction of x whose last-arriving CTA updates magnitude / mask and the
    ``lines`` [n, 2] (n == 1 or channels) of an AdaptiveQuantizer from the (min, max) of x * mask, at its call index
    ``t_line`` (1-based; an offset to ``*step_counter`` when that is given).  Up to FUSED_STEP_MAX_CHANNELS."""
    N.require_cuda(x, "input")
    if step_counter is not None:
        N.require_cuda(step_counter, "step_counter")
    lib = N.load_library()
    outer, ch, inner = layout
    ws = N.workspace(x.device, lib.qsb_reduce_workspace_bytes(c_int64(outer), c_int64(ch), c_int64(inner)))
    N.check(lib.qsb_reduce_prune_line_step_dt(
        N.ptr(x), c_int(N.dtype_code(x)), c_int64(outer), c_int64(ch), c_int64(inner), N.ptr(ws), c_int64(ws.numel()),
        N.ptr(arrival if arrival is not None else arrival_counter(x.device)), N.ptr(magnitude), N.ptr(mask),
        N.ptr(lines), c_int64(lines.numel() // 2), None, c_double(count), c_int64(t_prune), c_int(update_magnitude),
        c_int(int(refresh_mask)), c_int64(k), c_int64(t_line), N.ptr(abssum_out), N.ptr(min_out), N.ptr(max_out),
        N.ptr(step_counter), N.stream_ptr(x.device)), "qsb_reduce_prune_line_step_dt")


def reduce_line_partials(x, layout: Layout):
    """Stage 1 of the sum|x| / min / max reduction only; the partials stay in the returned workspace for
    ``prune_line_step_params``."""
    N.require_cuda(x, "input")
    lib = N.load_library()
    outer, ch, inner = layout
    ws = N.workspace(x.device, lib.qsb_reduce_workspace_bytes(c_int64(outer), c_int64(ch), c_int64(inner)))
    N.check(lib.qsb_reduce_line_partials_dt(N.ptr(x), c_int(N.dtype_code(x)), c_int64(outer), c_int64(ch),
                                            c_int64(inner), N.ptr(ws), c_int64(ws.numel()), N.stream_ptr(x.device)),
            "qsb_reduce_line_partials_dt")
    return ws


def prune_line_step_params(magnitude, mask, lines, workspace, layout: Layout, count: float, t_prune: int,
                           update_magnitude: int, refresh_mask, k: int, t_line: int, abssum_out=None, min_out=None,
                           max_out=None, step_counter=None):
    """the line step as one one-CTA kernel on the partials of ``reduce_line_partials`` (up to 2048 channels)"""
    lib = N.load_library()
    outer, ch, inner = layout
    N.check(lib.qsb_prune_line_step_params(
        N.ptr(magnitude), N.ptr(mask), N.ptr(lines), c_int64(lines.numel() // 2), N.ptr(workspace),
        c_int64(workspace.numel()), c_int64(outer), c_int64(ch), c_int64(inner), None, c_double(count),
        c_int64(t_prune), c_int(update_magnitude), c_int(int(refresh_mask)), c_int64(k), c_int64(t_line),
        N.ptr(abssum_out), N.ptr(min_out), N.ptr(max_out), N.ptr(step_counter), N.stream_ptr(mask.device)),
        "qsb_prune_line_step_params")


def structured_prune_line_step(x, layout: Layout, magnitude, mask, lines, count: float, t_prune: int,
                               update_magnitude: int, refresh_mask, k: int, t_line: int, step_counter=None):
    """The structured prune -> AdaptiveQuantizer parameter step on x, on the route ``_step_route`` picks:

      one       reduce_prune_line_step
      partials  reduce_line_partials + prune_line_step_params

    Above PARTIALS_ROUTE_MAX_CHANNELS channels there is no line route: ``ValueError``."""
    route = _step_route(layout[1], step_counter)
    if route == "one":
        reduce_prune_line_step(x, layout, magnitude, mask, lines, count, t_prune, update_magnitude, refresh_mask, k,
                               t_line, step_counter=step_counter)
    elif route == "partials":
        ws = reduce_line_partials(x, layout)
        prune_line_step_params(magnitude, mask, lines, ws, layout, count, t_prune, update_magnitude, refresh_mask, k,
                               t_line)
    else:
        raise ValueError(f"the structured prune -> line quantize step takes at most {PARTIALS_ROUTE_MAX_CHANNELS} "
                         "channels")


def prune_quant_rows_step_params(magnitude, mask, scale, decimal_out, stats: dict, count: float, t_prune: int,
                                 update_magnitude: int, refresh_mask: bool, k: int, bits: int, t_quant: int,
                                 update_scale: bool, n_rows: int = 1, row_stride_bytes: int = 0, group=None,
                                 step_stamp: int = 1):
    """``prune_quant_params`` (finalized statistics rows, combined in row order) plus the peer-memory
    exchange of the training step."""
    lib = N.load_library()
    N.check(lib.qsb_prune_quant_rows_step_params(
        N.ptr(magnitude), N.ptr(mask), N.ptr(scale), N.ptr(decimal_out), N.ptr(stats["abssum"]),
        N.ptr(stats["absmax"]), c_int64(n_rows), c_int64(row_stride_bytes), c_int64(mask.numel()), group,
        c_int64(step_stamp), c_double(count), c_int64(t_prune), c_int(update_magnitude),
        c_int(1 if refresh_mask else 0), c_int64(k), c_int(bits), c_int64(t_quant),
        c_int(1 if update_scale else 0), N.stream_ptr(mask.device)), "qsb_prune_quant_rows_step_params")


def set_tuning(key: int, value: int):
    N.check(N.load_library().qsb_set_tuning(c_int(key), c_int(value)), "qsb_set_tuning")
