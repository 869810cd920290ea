"""Numpy restatement of the block-scaled FP8 / FP4 formats (DESIGN §2 "Block-scaled formats"): MXFP8, MXFP4 and
NVFP4 fake quantization and their packed codes / scales.

Nothing here uses a float8 / float4 library: the E2M1 and E4M3 value grids are enumerated from their bit patterns,
and rounding is "nearest, ties to the even code, saturate to +-max" on that grid, computed in float64 (every grid
point and every fp32 quotient is exact there).  Divisions are fp32 IEEE divisions (numpy float32), exponents come
from the bits of the abs-max."""
from __future__ import annotations

import numpy as np

BLOCK = {"mxfp8": 32, "mxfp4": 32, "nvfp4": 16}


def _grid(mbits: int, ebits: int, bias: int, codes: int) -> np.ndarray:
    """values of the non-negative codes 0 .. codes-1 of a sign/exponent/mantissa format (no inf; subnormals)"""
    out = []
    for c in range(codes):
        e, m = c >> mbits, c & ((1 << mbits) - 1)
        if e == 0:
            out.append(m / (1 << mbits) * 2.0 ** (1 - bias))
        else:
            out.append((1 + m / (1 << mbits)) * 2.0 ** (e - bias))
    return np.array(out, dtype=np.float64)


E2M1 = _grid(1, 2, 1, 8)        # 0, .5, 1, 1.5, 2, 3, 4, 6
E4M3 = _grid(3, 4, 7, 127)      # code 0x7F is NaN; the largest finite value is 448


def round_code(v, grid: np.ndarray) -> np.ndarray:
    """code (index into ``grid``) of |v| rounded to nearest, ties to the even code, saturating at the largest
    value; v must be finite"""
    a = np.minimum(np.abs(np.asarray(v, dtype=np.float64)), grid[-1])
    hi = np.clip(np.searchsorted(grid, a, side="left"), 0, len(grid) - 1)   # first grid point >= a
    lo = np.maximum(hi - 1, 0)
    dlo, dhi = a - grid[lo], grid[hi] - a
    pick_hi = (dhi < dlo) | ((dhi == dlo) & (hi % 2 == 0))
    return np.where(pick_hi, hi, lo)


def cvt(v, grid: np.ndarray) -> np.ndarray:
    """cvt.rn.satfinite onto the grid, keeping the sign (also of a zero); float64 result"""
    v = np.asarray(v, dtype=np.float64)
    return np.copysign(grid[round_code(v, grid)], v)


def exponent(a: np.ndarray) -> np.ndarray:
    """floor(log2 a) of finite fp32 a > 0 from its bits (subnormals included); -150 for a == 0"""
    b = np.asarray(a, dtype=np.float32).view(np.uint32).astype(np.int64) & 0x7FFFFFFF
    e = (b >> 23) - 127
    sub = b < 0x00800000
    msb = np.floor(np.log2(np.maximum(b, 1))).astype(np.int64)  # exact for integers < 2^23
    return np.where(b == 0, -150, np.where(sub, msb - 149, e))


def _blocks(x2d: np.ndarray, B: int):
    """[R, nb, B] view of x2d (fp32), the short last block padded with zeros, and the valid-element mask"""
    R, L = x2d.shape
    nb = -(-L // B)
    pad = np.zeros((R, nb * B), dtype=np.float32)
    pad[:, :L] = x2d
    valid = np.zeros(nb * B, dtype=bool)
    valid[:L] = True
    return pad.reshape(R, nb, B), L


def _quantize(x2d: np.ndarray, fmt: str, w=None):
    """(y [R, L] fp32, element codes [R, L] uint8 (E4M3 byte or E2M1 nibble), scale bytes [R, nb] uint8)"""
    x2d = np.asarray(x2d, dtype=np.float32)
    B = BLOCK[fmt]
    xb, L = _blocks(x2d, B)
    R, nb, _ = xb.shape
    with np.errstate(all="ignore"):
        amax = np.max(np.abs(xb), axis=2)                          # NaN when the block holds one
        bad = ~np.isfinite(amax)
        grid = E4M3 if fmt == "mxfp8" else E2M1
        if fmt == "nvfp4":
            s_t = np.float32(w) / np.float32(2688.0)
            t2 = (amax / np.float32(6.0)) / s_t
            t2_nan = np.isnan(t2)
            mag = round_code(np.where(t2_nan, 0, t2), E4M3)             # +-inf saturates to 448
            s_b = np.where(t2_nan, np.nan, np.copysign(E4M3[mag], t2)).astype(np.float32)
            sb_code = np.where(t2_nan, 0x7F, mag | np.where(np.signbit(t2), 0x80, 0))
            d = (s_b * s_t).astype(np.float32)
            st_zero, st_nan = s_t == 0, np.isnan(s_t)
            nan_blk = bad | st_nan | (~st_zero & np.isnan(d))
            zero_blk = ~nan_blk & (st_zero | (d == 0))
            scale = d
            scale_byte = np.where(bad | st_nan, 0x7F, np.where(st_zero, 0, sb_code)).astype(np.uint8)
            q = (xb / np.where(zero_blk | nan_blk, np.float32(1), d)[..., None]).astype(np.float32)
        else:
            emax = 8 if fmt == "mxfp8" else 2
            k = np.clip(exponent(np.where(bad, 0, amax)) - emax, -127, 127)
            scale = np.ldexp(np.float32(1), k).astype(np.float32)
            q = (xb / scale[..., None]).astype(np.float32)
            nan_blk, zero_blk = bad, np.zeros_like(bad)
            scale_byte = np.where(bad, 0xFF, k + 127).astype(np.uint8)
        q = np.where((nan_blk | zero_blk)[..., None], 0, q)
        codes = round_code(q, grid) | np.where(np.signbit(q), 0x80 if fmt == "mxfp8" else 0x8, 0)
        y = (cvt(q, grid).astype(np.float32) * scale[..., None]).astype(np.float32)
        y = np.where(zero_blk[..., None], np.float32(0), y)
        y = np.where(nan_blk[..., None], np.float32(np.nan), y)
        codes = np.where((nan_blk | zero_blk)[..., None], 0, codes)
    y = y.reshape(R, nb * B)[:, :L]
    codes = codes.reshape(R, nb * B)[:, :L].astype(np.uint8)
    return y, codes, scale_byte


def fake_quant(x2d, fmt: str, w=None) -> np.ndarray:
    """the fp32 fake-quantized [R, L] rows; ``w``: nvfp4's tensor abs-max (fp32 scalar)"""
    return _quantize(x2d, fmt, w)[0]


def export(x2d, fmt: str, w=None):
    """(codes, scales) bytes as the packed export writes them"""
    _, c, s = _quantize(x2d, fmt, w)
    if fmt != "mxfp8":
        R, L = c.shape
        if L % 2:
            c = np.concatenate([c, np.zeros((R, 1), np.uint8)], axis=1)
        c = (c[:, 0::2] | (c[:, 1::2] << 4)).astype(np.uint8)
    return c, s


def rows_view(x: np.ndarray, rows: str = "last", channels_last: bool = False) -> np.ndarray:
    """the [R, L] view of x (a logical-shape array) that the quantizer walks"""
    x = np.asarray(x, dtype=np.float32)
    if rows == "leading":
        return x.reshape(x.shape[0], -1)
    if channels_last:
        x = x.transpose(0, 2, 3, 1)
    return x.reshape(-1, x.shape[-1])
