"""ctypes binding of ``libqsparse_b200.so`` (the C-ABI in ``include/qsparse_b200.h``).

There is deliberately no fallback: if the library is missing, or a tensor is not
a CUDA tensor, the call raises.  torch is used only for device memory and the
current stream.
"""
from __future__ import annotations

import ctypes
import os
from ctypes import c_double, c_float, c_int, c_int64, c_void_p
from pathlib import Path
from typing import Optional, Tuple

import torch

_PKG = Path(__file__).resolve().parent
LIB_PATH = Path(os.environ.get("QSPARSE_B200_LIB", _PKG / "lib" / "libqsparse_b200.so"))

MASK_NONE, MASK_CHANNEL, MASK_ELEMENT = 0, 1, 2
DTYPE_F32, DTYPE_BF16, DTYPE_F16 = 0, 1, 2
# element types the activation kernels read and write natively (QSB_DTYPE_*)
NATIVE_DTYPES = {torch.float32: DTYPE_F32, torch.bfloat16: DTYPE_BF16, torch.float16: DTYPE_F16}
STAT_ABSMAX, STAT_MINMAX, STAT_ABSSUM, STAT_NNZ = 1, 2, 4, 8

# name -> (restype, argtypes); mirrors include/qsparse_b200.h one to one
_P = c_void_p
_SIGNATURES = {
    "qsb_abi_version": (c_int, []),
    "qsb_error_string": (ctypes.c_char_p, [c_int]),
    "qsb_debug_kernel_times": (c_int, [_P, _P]),
    "qsb_device_info": (c_int, [ctypes.POINTER(c_int), ctypes.POINTER(c_int64)]),
    "qsb_fq_pow2_fwd": (c_int, [_P, _P, _P, c_int64, c_double, _P, c_int, c_int64, c_int64, c_int64, _P]),
    "qsb_fq_scaler_fwd": (c_int, [_P, _P, _P, c_int64, c_float, _P, c_int, c_int64, c_int64, c_int64, _P]),
    "qsb_fq_line_fwd": (c_int, [_P, _P, _P, c_int64, c_float, c_float, c_int, c_int, _P, c_int,
                                c_int64, c_int64, c_int64, _P]),
    "qsb_quant_export_int8": (c_int, [_P, _P, c_int, _P, c_int64, c_double, c_double, c_int, c_int64, c_int64,
                                      c_int64, _P]),
    "qsb_quant_export_int4": (c_int, [_P, _P, c_int, _P, c_int64, c_double, c_double, c_int, c_int64, c_int64,
                                      c_int64, _P]),
    "qsb_ste_bwd": (c_int, [_P, _P, _P, _P, c_int64, c_double, c_int, c_int, c_int, _P, c_int,
                            c_int64, c_int64, c_int64, _P]),
    "qsb_mask_apply": (c_int, [_P, _P, _P, c_int, c_int64, c_int64, c_int64, _P]),
    "qsb_fq_pow2_fwd_dt": (c_int, [_P, c_int, _P, _P, c_int64, c_double, _P, c_int, c_int64, c_int64, c_int64, _P]),
    "qsb_fq_scaler_fwd_dt": (c_int, [_P, c_int, _P, _P, c_int64, c_float, _P, c_int, c_int64, c_int64, c_int64, _P]),
    "qsb_fq_line_fwd_dt": (c_int, [_P, c_int, _P, _P, c_int64, c_float, c_float, c_int, c_int, _P, c_int,
                                   c_int64, c_int64, c_int64, _P]),
    "qsb_ste_bwd_dt": (c_int, [_P, _P, _P, c_int, _P, c_int64, c_double, c_int, c_int, c_int, _P, c_int,
                               c_int64, c_int64, c_int64, _P]),
    "qsb_mask_apply_dt": (c_int, [_P, c_int, _P, c_int, _P, c_int, c_int64, c_int64, c_int64, _P]),
    "qsb_reduce_stats_dt": (c_int, [_P, c_int, c_int, c_int64, c_int64, c_int64, _P, _P, _P, _P, _P, _P, _P, c_int64,
                                    _P]),
    "qsb_reduce_partials_dt": (c_int, [_P, c_int, c_int64, c_int64, c_int64, _P, c_int64, _P]),
    "qsb_reduce_prune_quant_step_dt": (c_int, [_P, c_int, c_int64, c_int64, c_int64, _P, c_int64, _P, _P, _P, _P, _P,
                                               _P, c_int64, c_double, c_int64, c_int, c_int, c_int64, c_int, c_int64,
                                               c_int, _P, _P, c_int, _P, _P, _P]),
    "qsb_reduce_prune_line_step_dt": (c_int, [_P, c_int, c_int64, c_int64, c_int64, _P, c_int64, _P, _P, _P, _P,
                                              c_int64, _P, c_double, c_int64, c_int, c_int, c_int64, c_int64, _P, _P,
                                              _P, _P, _P]),
    "qsb_reduce_line_partials_dt": (c_int, [_P, c_int, c_int64, c_int64, c_int64, _P, c_int64, _P]),
    "qsb_prune_line_step_params": (c_int, [_P, _P, _P, c_int64, _P, c_int64, c_int64, c_int64, c_int64, _P, c_double,
                                           c_int64, c_int, c_int, c_int64, c_int64, _P, _P, _P, _P, _P]),
    "qsb_reduce_workspace_bytes": (c_int64, [c_int64, c_int64, c_int64]),
    "qsb_reduce_stats": (c_int, [_P, c_int, c_int64, c_int64, c_int64, _P, _P, _P, _P, _P, _P, _P, c_int64, _P]),
    "qsb_reduce_stats_fused": (c_int, [_P, c_int, c_int64, c_int64, c_int64, _P, _P, _P, _P, _P, _P, _P, c_int64, _P,
                                       _P]),
    "qsb_scale_ema": (c_int, [_P, _P, c_int64, c_int, c_int64, _P]),
    "qsb_scale_to_decimal": (c_int, [_P, _P, c_int64, _P]),
    "qsb_lines_ema": (c_int, [_P, _P, _P, c_int64, c_int64, _P]),
    "qsb_scale_ema_at": (c_int, [_P, _P, c_int64, c_int, _P, c_int64, _P]),
    "qsb_lines_ema_at": (c_int, [_P, _P, _P, c_int64, _P, c_int64, _P]),
    "qsb_row_quant_fused": (c_int, [_P, _P, _P, _P, c_int, c_int, c_int, c_int64, c_int64, c_int64, _P]),
    "qsb_row_quant_fused_masked": (c_int, [_P, _P, _P, _P, _P, c_int, c_int, c_int, c_int64, c_int64, c_int64, _P]),
    "qsb_row_quant_fused_at": (c_int, [_P, _P, _P, _P, _P, c_int, c_int, c_int, c_int64, c_int64, _P, c_int64, _P]),
    "qsb_magnitude_ema_reduced": (c_int, [_P, _P, _P, _P, c_int, c_int64, c_double, c_int64, _P]),
    "qsb_magnitude_ema_full": (c_int, [_P, _P, _P, c_int, c_int64, c_int64, _P]),
    "qsb_magnitude_ema_full_multi": (c_int, [ctypes.POINTER(c_void_p), ctypes.POINTER(c_void_p),
                                             ctypes.POINTER(c_int64), c_int, c_int64, _P]),
    "qsb_mask_build_apply_multi": (c_int, [ctypes.POINTER(c_void_p), c_int, _P, ctypes.POINTER(c_void_p),
                                           ctypes.POINTER(c_void_p), ctypes.POINTER(c_void_p),
                                           ctypes.POINTER(c_int64), c_int, _P]),
    "qsb_prune_step_workspace_bytes": (c_int64, [ctypes.POINTER(c_int64), c_int]),
    "qsb_prune_unstructured_step_batched": (c_int, [ctypes.POINTER(c_void_p), ctypes.POINTER(c_void_p),
                                                    ctypes.POINTER(c_void_p), ctypes.POINTER(c_void_p),
                                                    ctypes.POINTER(c_int64), ctypes.POINTER(c_int64), c_int, c_int64,
                                                    _P, _P, c_int64, _P]),
    "qsb_kth_workspace_bytes": (c_int64, [c_int64]),
    "qsb_kth_value": (c_int, [_P, c_int64, c_int64, c_int, _P, _P, c_int64, _P]),
    "qsb_kth_batched_workspace_bytes": (c_int64, [ctypes.POINTER(c_int64), c_int]),
    "qsb_kth_value_batched": (c_int, [ctypes.POINTER(c_void_p), ctypes.POINTER(c_int64), ctypes.POINTER(c_int64), c_int,
                                      c_int, _P, _P, c_int64, _P]),
    "qsb_kth_value_batched_hinted": (c_int, [ctypes.POINTER(c_void_p), ctypes.POINTER(c_int64),
                                             ctypes.POINTER(c_int64), c_int, c_int, _P, _P, _P, c_int64, _P]),
    "qsb_prune_unstructured_step_batched_hinted": (c_int, [ctypes.POINTER(c_void_p), ctypes.POINTER(c_void_p),
                                                           ctypes.POINTER(c_void_p), ctypes.POINTER(c_void_p),
                                                           ctypes.POINTER(c_int64), ctypes.POINTER(c_int64), c_int,
                                                           c_int64, _P, _P, _P, c_int64, _P]),
    "qsb_prune_unstructured_step_batched_at": (c_int, [ctypes.POINTER(c_void_p), ctypes.POINTER(c_void_p),
                                                       ctypes.POINTER(c_void_p), ctypes.POINTER(c_void_p),
                                                       ctypes.POINTER(c_int64), ctypes.POINTER(c_int64), c_int,
                                                       _P, c_int64, _P, _P, _P, c_int64, _P]),
    "qsb_kth_dist_begin": (c_int, [_P, c_int64, _P]),
    "qsb_kth_dist_pass": (c_int, [_P, c_int64, c_int64, c_int, c_int, _P, c_int64, ctypes.POINTER(c_void_p),
                                  ctypes.POINTER(c_int64), _P]),
    "qsb_kth_dist_final": (c_int, [c_int64, _P, _P, _P]),
    "qsb_mask_from_threshold": (c_int, [_P, c_int, _P, _P, c_int64, _P]),
    "qsb_mask_build_apply": (c_int, [_P, c_int, _P, _P, _P, _P, c_int64, _P]),
    "qsb_group_mean": (c_int, [_P, _P, _P, c_int64, c_int64, c_int64, _P]),
    "qsb_prune_quant_params": (c_int, [_P, _P, _P, _P, _P, _P, c_int64, c_int64, c_int64, c_double, c_int64, c_int,
                                       c_int, c_int64, c_int, c_int64, c_int, _P]),
    "qsb_reduce_partials": (c_int, [_P, c_int64, c_int64, c_int64, _P, c_int64, _P]),
    "qsb_p2p_group_bytes": (c_int64, [c_int, c_int64]),
    "qsb_p2p_alloc": (c_int, [c_int64, ctypes.POINTER(c_void_p), ctypes.c_char_p]),
    "qsb_p2p_open": (c_int, [ctypes.c_char_p, ctypes.POINTER(c_void_p)]),
    "qsb_p2p_close": (c_int, [_P]),
    "qsb_p2p_free": (c_int, [_P]),
    "qsb_p2p_group_create": (c_int, [ctypes.POINTER(c_void_p), c_int, c_int, c_int64, ctypes.POINTER(c_void_p)]),
    "qsb_p2p_group_error": (c_int, [_P, ctypes.POINTER(c_int)]),
    "qsb_p2p_group_error_async": (c_int, [_P, _P, _P]),
    "qsb_p2p_group_set_timeout_ms": (c_int, [_P, c_int64]),
    "qsb_p2p_group_destroy": (c_int, [_P]),
    "qsb_prune_quant_rows_step_params": (c_int, [_P, _P, _P, _P, _P, _P, c_int64, c_int64, c_int64, _P, c_int64,
                                                 c_double, c_int64, c_int, c_int, c_int64, c_int, c_int64, c_int,
                                                 _P]),
    "qsb_reduce_prune_quant_step": (c_int, [_P, c_int64, c_int64, c_int64, _P, c_int64, _P, _P, _P, _P, _P, _P,
                                            c_int64, c_double, c_int64, c_int, c_int, c_int64, c_int, c_int64,
                                            c_int, _P, _P, c_int, _P, _P, _P]),
    "qsb_prune_quant_step_params": (c_int, [_P, _P, _P, _P, _P, c_int64, c_int64, c_int64, c_int64, _P, c_int64,
                                            c_double, c_int64, c_int, c_int, c_int64, c_int, c_int64, c_int, _P, _P,
                                            _P, _P]),
    "qsb_host_ctx_create": (c_int, [ctypes.POINTER(c_void_p), c_int64, c_int64, c_int]),
    "qsb_host_ctx_destroy": (c_int, [_P]),
    "qsb_host_prune_quant_step": (c_int, [_P, _P, _P, _P, _P, _P, _P, _P, _P, c_int64, c_int64, c_int64, c_int64,
                                          c_int64, c_int, c_int64, _P, c_int64, _P]),
    "qsb_host_prune_quant_step_submit": (c_int, [_P, c_int, _P, _P, _P, _P, _P, _P, _P, _P, c_int64, c_int64, c_int64,
                                                 c_int64, c_int64, c_int, c_int64, _P, c_int64, _P]),
    "qsb_host_ctx_wait": (c_int, [_P, c_int]),
    "qsb_set_tuning": (c_int, [c_int, c_int]),
    "qsb_selftest_fastdiv": (c_int, [c_int64, c_int64, ctypes.c_uint64, _P, _P]),
}

_lib = None


class NativeLibraryError(ImportError):
    pass


def load_library() -> ctypes.CDLL:
    """dlopen the C-ABI library once; raise loudly when it is not built."""
    global _lib
    if _lib is not None:
        return _lib
    if not LIB_PATH.exists():
        raise NativeLibraryError(
            f"{LIB_PATH} not found: the CUDA library is not built. Run "
            "`python -m qsparse_b200.build` (needs nvcc; cross-compiles without a GPU). "
            "qsparse_b200 has no CPU or PyTorch fallback."
        )
    lib = ctypes.CDLL(str(LIB_PATH))
    for name, (res, args) in _SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError if the symbol is missing
        fn.restype = res
        fn.argtypes = args
    if lib.qsb_abi_version() != 3:
        raise NativeLibraryError("libqsparse_b200.so ABI version mismatch; rebuild it")
    _lib = lib
    return lib


def exported_symbols():
    return sorted(_SIGNATURES)


def check(rc: int, what: str) -> None:
    if rc != 0:
        msg = load_library().qsb_error_string(rc).decode()
        raise RuntimeError(f"{what} failed: {msg} (code {rc})")


# --------------------------------------------------------------------------
# tensor plumbing
# --------------------------------------------------------------------------
def require_cuda(t: torch.Tensor, name: str = "tensor") -> None:
    if not isinstance(t, torch.Tensor):
        raise TypeError(f"{name} must be a torch.Tensor, got {type(t)}")
    if not t.is_cuda:
        raise RuntimeError(
            f"qsparse_b200 is CUDA-only (no CPU fallback): {name} is on {t.device}. "
            "Move it to a B200 (`.cuda()`)."
        )


def ptr(t: Optional[torch.Tensor]):
    """device address as a plain int (None -> NULL): ctypes converts it through the declared argtypes,
    without building a c_void_p object per argument"""
    return None if t is None else t.data_ptr()


_raw_stream = getattr(torch._C, "_cuda_getCurrentRawStream", None)


def stream_key(device: torch.device) -> Tuple[int, int]:
    """(device index, raw cudaStream_t of torch's current stream) — one C call, not the
    ``torch.cuda.current_stream()`` object round trip (8 us each; a small layer makes a dozen)."""
    idx = device.index
    if idx is None:
        idx = torch.cuda.current_device()
    if _raw_stream is not None:
        return idx, _raw_stream(idx)
    return idx, torch.cuda.current_stream(device).cuda_stream


def stream_ptr(device: torch.device):
    return stream_key(device)[1] or None


_workspaces = {}


def workspace(device: torch.device, nbytes: int) -> torch.Tensor:
    """Per (device, stream) scratch buffer, grown on demand, never shrunk."""
    key = stream_key(device)
    ws = _workspaces.get(key)
    if ws is None or ws.numel() < nbytes:
        ws = torch.empty(max(int(nbytes), 1 << 20), dtype=torch.uint8, device=device)
        _workspaces[key] = ws
    return ws


def as_f32_contiguous(t: torch.Tensor) -> torch.Tensor:
    """The kernels compute in fp32 on contiguous memory (SURVEY Q6: the
    reference's output is fp32 for every input dtype)."""
    if t.dtype != torch.float32:
        t = t.float()
    if not t.is_contiguous():
        t = t.contiguous()
    return t


def dtype_code(t: torch.Tensor) -> int:
    return NATIVE_DTYPES[t.dtype]


def as_native(t: torch.Tensor) -> torch.Tensor:
    """fp32, bf16 and fp16 tensors as they are (the activation kernels read 16-bit values natively and
    compute in fp32, so the results equal those of ``t.float()`` bit for bit); any other dtype as fp32."""
    return t if t.dtype in NATIVE_DTYPES else t.float()


def as_native_contiguous(t: torch.Tensor) -> torch.Tensor:
    t = as_native(t)
    return t if t.is_contiguous() else t.contiguous()


def channel_layout(shape, channel_index: int) -> Tuple[int, int, int]:
    """[outer, channels, inner] factorisation of a contiguous tensor around one
    channel axis; channel_index < 0 means per-tensor."""
    n = 1
    for s in shape:
        n *= int(s)
    if channel_index is None or channel_index < 0:
        return 1, 1, n
    ci = int(channel_index)
    outer = 1
    for s in shape[:ci]:
        outer *= int(s)
    inner = 1
    for s in shape[ci + 1:]:
        inner *= int(s)
    return outer, int(shape[ci]), inner
