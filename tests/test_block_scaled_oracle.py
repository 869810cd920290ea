"""Block-scaled FP8 / FP4 formats without a GPU: known answers of the numpy restatement (oracle/block_scaled.py),
its E4M3 rounding against torch's float8_e4m3fn cast, the C-ABI argument checks and the host-side argument
checks of BlockScaledQuantizer."""
import ctypes

import numpy as np
import pytest
import torch

from oracle import block_scaled as bs


def f32(*v):
    return np.array(v, dtype=np.float32)


def test_e2m1_grid_and_e4m3_range():
    assert bs.E2M1.tolist() == [0, 0.5, 1, 1.5, 2, 3, 4, 6]
    assert bs.E4M3[-1] == 448 and bs.E4M3[1] == 2.0 ** -9 and len(bs.E4M3) == 127
    assert np.all(np.diff(bs.E4M3) > 0)


def test_e2m1_ties_to_even_and_saturation():
    # midpoints go to the even code: 0.25 -> 0, 0.75 -> 1, 1.25 -> 1, 1.75 -> 2, 2.5 -> 2, 3.5 -> 4, 5 -> 4
    mids = f32(0.25, 0.75, 1.25, 1.75, 2.5, 3.5, 5.0)
    assert bs.cvt(mids, bs.E2M1).tolist() == [0, 1, 1, 2, 2, 4, 4]
    assert bs.cvt(-mids, bs.E2M1).tolist() == [-0.0, -1, -1, -2, -2, -4, -4]
    assert np.signbit(bs.cvt(f32(-0.1), bs.E2M1))[0]                      # a negative value rounds to -0
    assert bs.cvt(f32(6.5, 7.9, 1e30), bs.E2M1).tolist() == [6, 6, 6]       # satfinite


def test_mxfp4_block_scale_and_saturation():
    # a = 4 -> e(a) = 2, X = 1: the elements round on the grid itself
    x = np.zeros((1, 32), np.float32)
    x[0, :8] = f32(4, 0.25, 0.75, 2.5, 5.0, -3.5, 1.1, -0.2)
    assert bs.fake_quant(x, "mxfp4")[0, :8].tolist() == [4, 0, 1, 2, 4, -4, 1, -0.0]
    # a in (6, 8) * X saturates to 6 * X: a = 7.5 -> X = 1
    x[0, 0] = 7.5
    assert bs.fake_quant(x, "mxfp4")[0, 0] == 6
    x[0, 0] = -7.99
    assert bs.fake_quant(x, "mxfp4")[0, 0] == -6
    c, s = bs.export(x, "mxfp4")
    assert s.tolist() == [[127]] and c.shape == (1, 16) and (c[0, 0] & 0xF) == 0xF   # -6 is nibble 0b1111


def test_power_of_two_amax_and_its_predecessor():
    for fmt, emax in (("mxfp8", 8), ("mxfp4", 2)):
        a = np.float32(2.0 ** 5)
        below = np.nextafter(a, np.float32(0))
        for v, e in ((a, 5), (below, 4)):
            x = np.zeros((1, 32), np.float32)
            x[0, 3] = v
            _, s = bs.export(x, fmt)
            assert s[0, 0] == e - emax + 127, (fmt, v)
    # mxfp4: the predecessor of 32 has e(a) = 4, X = 4, and a / X just below 8 saturates to 6
    x = np.zeros((1, 32), np.float32)
    x[0, 0] = np.nextafter(np.float32(32), np.float32(0))
    assert bs.fake_quant(x, "mxfp4")[0, 0] == 24


def test_exponent_from_bits_subnormals_and_zero_block():
    assert bs.exponent(f32(2.0 ** -140, 3 * 2.0 ** -149, 1.0, 3.0, 2.0 ** -126, 0.0)).tolist() == \
        [-140, -148, 0, 1, -126, -150]
    sub = np.float32(2.0 ** -130)
    x = np.zeros((2, 32), np.float32)
    x[0, 0] = sub
    x[1, 0] = -0.0
    y = bs.fake_quant(x, "mxfp8")
    c, s = bs.export(x, "mxfp8")
    assert s[:, 0].tolist() == [0, 0]                                          # X = 2^-127
    assert y[0, 0] == sub                                                      # 2^-130 / 2^-127 = 0.125, on the grid
    assert np.signbit(y[1, 0]) and c[1, 0] == 0x80


def test_nan_and_inf_blocks():
    x = np.ones((1, 40), np.float32)
    x[0, 33] = np.inf
    y = bs.fake_quant(x, "mxfp8")
    c, s = bs.export(x, "mxfp8")
    assert np.all(np.isnan(y[0, 32:])) and not np.any(np.isnan(y[0, :32]))
    assert s.tolist() == [[127 - 8, 0xFF]] and np.all(c[0, 32:] == 0)          # a = 1: X = 2^-8
    x[0, 33] = np.nan
    y = bs.fake_quant(x, "nvfp4", w=np.float32(1))
    c, s = bs.export(x, "nvfp4", w=np.float32(1))
    assert np.all(np.isnan(y[0, 32:])) and s[0, 2] == 0x7F and s.shape == (1, 3)


def test_nvfp4_tensor_scale_rules():
    rng = np.random.default_rng(1)
    x = rng.standard_normal((3, 48)).astype(np.float32)
    x[1, :16] = 0                                                              # a zero block: +0
    w = np.float32(np.abs(x).max())
    y = bs.fake_quant(x, "nvfp4", w)
    assert np.all(y[1, :16] == 0) and not np.any(np.signbit(y[1, :16]))
    # the largest block reaches s_b = 448: a / 6 / (w / 2688) = 448
    _, s = bs.export(x, "nvfp4", w)
    assert bs.E4M3[s.max()] == 448
    yz = bs.fake_quant(x, "nvfp4", np.float32(0))
    assert np.all(yz == 0) and not np.any(np.signbit(yz))                      # w == 0: +0 everywhere
    assert np.all(np.isnan(bs.fake_quant(x, "nvfp4", np.float32(np.nan))))


def test_short_rows_and_odd_packing():
    x = np.arange(1, 8, dtype=np.float32).reshape(1, 7)
    c, s = bs.export(x, "mxfp4")
    assert c.shape == (1, 4) and s.shape == (1, 1) and (c[0, 3] >> 4) == 0   # zero pad nibble


def test_e4m3_rounding_equals_torch_cast():
    rng = np.random.default_rng(0)
    v = np.concatenate([
        rng.standard_normal(200000).astype(np.float32) * np.float32(100),
        (rng.standard_normal(50000) * 2.0 ** -8).astype(np.float32),            # the subnormal range
        np.array(bs.E4M3, np.float32), -np.array(bs.E4M3, np.float32),
        ((bs.E4M3[1:] + bs.E4M3[:-1]) / 2).astype(np.float32),                  # exact midpoints
        f32(447.9, 448, 463.9, -463.9)])
    v = v[np.abs(v) < 464]                                                     # torch saturates nothing
    ours = bs.cvt(v, bs.E4M3).astype(np.float32)
    ref = torch.from_numpy(v).to(torch.float8_e4m3fn).float().numpy()
    assert np.array_equal(ours.view(np.uint32), ref.view(np.uint32))
    # out of range: torch's cast gives NaN, the satfinite conversion 448
    assert torch.isnan(torch.tensor([500.0]).to(torch.float8_e4m3fn).float())[0]
    assert bs.cvt(f32(500, -1e9), bs.E4M3).tolist() == [448, -448]


def test_block_cabi_argument_errors_without_gpu():
    from qsparse_b200 import _native
    lib = _native.load_library()
    null = ctypes.c_void_p(0)
    buf = (ctypes.c_float * 64)()
    p = ctypes.cast(buf, ctypes.c_void_p)
    amax = ctypes.cast((ctypes.c_float * 1)(), ctypes.c_void_p)
    fwd, exp = lib.qsb_fq_block_fwd_dt, lib.qsb_block_export_dt
    assert fwd(null, 0, null, 2, 32, 0, null, null) == -1                    # null x / y
    assert fwd(p, 0, null, 2, 32, 0, null, null) == -1                       # null y
    assert fwd(p, 0, p, -1, 32, 0, null, null) == -1                         # negative sizes
    assert fwd(p, 0, p, 2, -32, 0, null, null) == -1
    assert fwd(p, 0, p, 2, 32, 3, null, null) == -1                          # bad fmt
    assert fwd(p, 0, p, 2, 32, -1, null, null) == -1
    assert fwd(p, 5, p, 2, 32, 0, null, null) == -1                          # bad dtype
    assert fwd(p, 0, p, 2, 32, 2, null, null) == -1                          # nvfp4 without w
    assert fwd(null, 0, null, 0, 32, 0, null, null) == 0                     # empty: no-op
    assert exp(p, 0, null, p, 2, 32, 0, null, null) == -1                    # null codes
    assert exp(p, 0, p, null, 2, 32, 1, null, null) == -1                    # null scales
    assert exp(p, 0, p, p, 2, 32, 7, amax, null) == -1
    assert exp(p, 0, p, p, 2, 32, 2, null, null) == -1
    assert exp(p, 0, p, p, -2, 32, 2, amax, null) == -1


def test_block_quantizer_host_checks():
    import qsparse_b200 as qs
    from qsparse_b200 import ops
    qs.set_qsparse_options(log_on_created=False)
    with pytest.raises(ValueError):
        qs.BlockScaledQuantizer("fp8")
    with pytest.raises(ValueError):
        qs.BlockScaledQuantizer("mxfp8", rows="first")
    with pytest.raises(ValueError, match="channelwise=-1"):
        qs.quantize(torch.nn.Linear(4, 4), callback=qs.BlockScaledQuantizer("nvfp4"), channelwise=1)
    with pytest.raises(ValueError, match="channelwise=-1"):
        qs.quantize(callback=qs.BlockScaledQuantizer("mxfp4"), channelwise=0)
    layer = qs.quantize(callback=qs.BlockScaledQuantizer("mxfp4"), channelwise=-1, timeout=1)
    assert layer.channelwise == -1
    with pytest.raises(ValueError, match="channelwise=-1"):
        qs.BlockScaledQuantizer("mxfp8").optimize(torch.zeros(2, 4), 8, channel_index=1)
    with pytest.raises(RuntimeError, match="CUDA-only"):
        qs.BlockScaledQuantizer("mxfp8").optimize(torch.zeros(2, 4), 8)
    with pytest.raises(RuntimeError, match="CUDA-only"):
        ops.fq_block_fwd(torch.zeros(2, 4), "mxfp8", 2, 4)
