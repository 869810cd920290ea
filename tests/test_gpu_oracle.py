"""GPU parity, part 2: CUDA kernels (through the C-ABI) against the CPU oracle on seeded
inputs — odd shapes, unaligned pointers, channels_last, element masks, big-ish sizes —
and size-independent properties at BASELINE.json's full sizes."""
import numpy as np
import pytest
import torch

from oracle import oracle as orc
from tests.conftest import bits_equal, ulp_diff

pytestmark = pytest.mark.gpu


def cu(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def npy(t):
    return t.detach().cpu().numpy()


def rnd(shape, seed, scale=1.0):
    rng = np.random.default_rng(seed)
    x = (rng.standard_normal(shape) * scale).astype(np.float32)
    f = x.reshape(-1)
    if f.size >= 16:
        f[rng.choice(f.size, 8, replace=False)] = [0.0, -0.0, 0.5, -0.5, 1.5, 2.5, 1e-40, -3.0]
    return x


SHAPES = [
    ((4, 6, 7, 7), 1),      # inner 49 (odd)
    ((3, 5, 56, 56), 1),    # inner 3136, row mode, rows misaligned to 32 B? (3136*4 % 32 == 0)
    ((2, 7, 9, 11), 1),     # inner 99
    ((64, 130), 1),         # [N, C], inner 1 (column mode)
    ((16, 4, 3, 3), 0),     # weights, channelwise=0, inner 36
    ((5, 3, 33), 2),        # channel = last axis
    ((2, 3, 1000), 1),      # inner 1000
    ((1, 2, 70001), 1),     # long rows, odd length
    ((64, 128), 1),         # channel-last, C % 8 == 0: group-resident kernel, row-lane column reduce
    ((33, 4096), 1),        # channel-last, more groups than one CTA covers
    ((1000, 8), 1),         # channel-last, one group
    ((5, 7, 24), 2),        # channel = last axis of a 3-D tensor
    ((64, 96, 7, 7), 1),    # 7x7 maps at scale: straddling vectors on the fast path, 4 short rows in flight
    ((8, 64, 14, 14), 1),   # inner 196
    ((6, 5, 16, 16), 1),    # inner 256: the short-row boundary
    ((3, 5, 257), 1),       # inner 257: just past it
]


@pytest.mark.parametrize("shape,ci", SHAPES)
def test_fakequant_channelwise_vs_oracle(shape, ci):
    from qsparse_b200.quantize import quantize_with_decimal, quantize_with_scaler, quantize_with_line
    x = rnd(shape, 11, 2.0)
    C = shape[ci]
    rng = np.random.default_rng(5)
    dec = rng.integers(-1, 9, C).astype(np.float32)
    sc = rng.uniform(0.01, 0.7, C).astype(np.float32)
    lines = np.stack([rng.uniform(-2, -0.1, C), rng.uniform(0.1, 2, C)], 1).astype(np.float32)
    xc = cu(x)
    assert bits_equal(npy(quantize_with_decimal(xc, 8, cu(dec), ci)), orc.fq_pow2_fwd(x, dec, ci))
    assert bits_equal(npy(quantize_with_scaler(xc, 8, cu(sc), ci)), orc.fq_scaler_fwd(x, sc, ci))
    for fzp in (True, False):
        assert bits_equal(npy(quantize_with_line(xc, 5, cu(lines), ci, False, fzp)),
                          orc.fq_line_fwd(x, lines, 5, ci, fzp))
    # per tensor
    assert bits_equal(npy(quantize_with_decimal(xc, 8, 4)), orc.fq_pow2_fwd(x, 4))
    assert bits_equal(npy(quantize_with_scaler(xc, 8, 0.0371)), orc.fq_scaler_fwd(x, np.float32(0.0371)))


@pytest.mark.parametrize("shape,ci", SHAPES)
def test_ste_backward_vs_oracle(shape, ci):
    from qsparse_b200 import ops
    from qsparse_b200._native import channel_layout
    g = rnd(shape, 12, 3.0)
    g.reshape(-1)[::97] = np.nan
    C = shape[ci]
    rng = np.random.default_rng(6)
    dec = rng.integers(2, 7, C).astype(np.float32)
    sc = rng.uniform(0.001, 0.05, C).astype(np.float32)
    for scale, is_dec in ((dec, True), (sc, False)):
        gc = cu(g).clone()
        ops.ste_bwd(gc, cu(scale), is_dec, 8, 1, channel_layout(shape, ci))
        ref, _ = orc.ste_bwd(g, scale, 8, ci, is_dec, True)
        assert bits_equal(npy(gc), ref), is_dec


def test_unaligned_and_channels_last():
    from qsparse_b200.quantize import quantize_with_decimal, quantize_with_scaler
    base = rnd((1 + 4 * 6 * 10 * 10,), 3, 2.0)
    xc = cu(base)[1:].view(4, 6, 10, 10)            # data pointer only 4-byte aligned
    x = base[1:].reshape(4, 6, 10, 10)
    dec = np.arange(6, dtype=np.float32)
    assert bits_equal(npy(quantize_with_decimal(xc, 8, cu(dec), 1)), orc.fq_pow2_fwd(x, dec, 1))
    assert bits_equal(npy(quantize_with_decimal(xc, 8, 3)), orc.fq_pow2_fwd(x, 3))
    xcl = cu(x).contiguous(memory_format=torch.channels_last)
    y = quantize_with_decimal(xcl, 8, cu(dec), 1)
    assert y.is_contiguous(memory_format=torch.channels_last)   # memory format follows the input (SURVEY Q6)
    assert bits_equal(npy(y), orc.fq_pow2_fwd(x, dec, 1))
    y = quantize_with_scaler(xcl, 8, 0.05)
    assert bits_equal(npy(y), orc.fq_scaler_fwd(x, np.float32(0.05)))
    # non-fp32 input: converted, result fp32 (SURVEY Q6)
    y = quantize_with_decimal(cu(x).half(), 8, 3)
    assert y.dtype == torch.float32
    assert bits_equal(npy(y), orc.fq_pow2_fwd(x.astype(np.float16).astype(np.float32), 3))


@pytest.mark.parametrize("shape,ci", SHAPES)
def test_reductions_vs_oracle(shape, ci):
    from qsparse_b200 import ops
    from qsparse_b200._native import channel_layout
    x = rnd(shape, 21, 1.5)
    for layout_ci in (ci, -1):
        st = ops.reduce_stats(cu(x), channel_layout(shape, layout_ci), absmax=True, minmax=True, abssum=True,
                              nnz=True)
        assert bits_equal(npy(st["absmax"]), orc.absmax(x, layout_ci))
        mn, mx = orc.minmax(x, layout_ci)
        assert np.array_equal(npy(st["min"]), mn) and np.array_equal(npy(st["max"]), mx)
        o, c, i = orc.layout(shape, layout_ci)
        xr = np.abs(x.astype(np.float64)).reshape(o, c, i)
        # 8-element fp32 pre-sums, then fp64: ~1e-7 relative of the exact sum (reduce.cu header)
        assert np.allclose(npy(st["abssum"]), xr.sum(axis=(0, 2)), rtol=3e-7, atol=0)
        assert np.array_equal(npy(st["nnz"]), (xr != 0).sum(axis=(0, 2)).astype(np.float64))
        assert npy(st["tensor_min"])[0] == x.min()
    # each single-statistic instantiation
    st = ops.reduce_stats(cu(x), channel_layout(shape, ci), absmax=True)
    assert bits_equal(npy(st["absmax"]), orc.absmax(x, ci))
    st = ops.reduce_stats(cu(x), channel_layout(shape, ci), minmax=True)
    assert np.array_equal(npy(st["min"]), orc.minmax(x, ci)[0])
    st = ops.reduce_stats(cu(x), channel_layout(shape, ci), abssum=True, absmax=True)
    assert bits_equal(npy(st["absmax"]), orc.absmax(x, ci))


@pytest.mark.parametrize("outer,C,inner,off", [(600, 96, 49, 0), (64, 300, 196, 3), (9, 20000, 16, 1),
                                               (4100, 8, 255, 5), (70, 1, 100, 2), (40000, 24, 1, 0)])
def test_short_row_reductions(outer, C, inner, off):
    """The tile kernel (16 <= inner <= 256): several tiles per CTA, ragged last tile, rows that start anywhere in a
    32-byte sector (a 4-byte-aligned view), more channels than slots; and the transposed finalize."""
    from qsparse_b200 import ops
    n = outer * C * inner
    base = rnd((n + off,), 31, 1.5)
    base[::1013] = 0.0
    x = base[off:].reshape(outer, C, inner)
    xc = cu(base)[off:].view(outer, C, inner)
    st = ops.reduce_stats(xc, (outer, C, inner), absmax=True, minmax=True, abssum=True, nnz=True)
    assert bits_equal(npy(st["absmax"]), np.abs(x).max(axis=(0, 2)))
    assert np.array_equal(npy(st["min"]), x.min(axis=(0, 2))) and np.array_equal(npy(st["max"]), x.max(axis=(0, 2)))
    xr = np.abs(x.astype(np.float64))
    assert np.allclose(npy(st["abssum"]), xr.sum(axis=(0, 2)), rtol=3e-7, atol=0)
    assert np.array_equal(npy(st["nnz"]), (xr != 0).sum(axis=(0, 2)).astype(np.float64))
    again = ops.reduce_stats(xc, (outer, C, inner), abssum=True, absmax=True)
    third = ops.reduce_stats(xc, (outer, C, inner), abssum=True, absmax=True)
    assert bits_equal(npy(again["abssum"]), npy(third["abssum"]))     # deterministic


def test_empty_and_single_element_inputs():
    """Degenerate sizes: an empty tensor passes through every functional entry point (the reference returns an empty
    tensor: all its ops are elementwise); one element goes through the scalar tail of every kernel."""
    from qsparse_b200 import ops
    from qsparse_b200.quantize import quantize_with_decimal, quantize_with_scaler, quantize_with_line
    e = torch.empty(0, device="cuda")
    for y in (quantize_with_decimal(e, 8, 4), quantize_with_scaler(e, 8, 0.1), quantize_with_line(e, 8, (-0.1, 0.9))):
        assert y.shape == (0,) and y.dtype == torch.float32
    e4 = torch.empty(0, 3, 5, 5, device="cuda")
    assert quantize_with_decimal(e4, 8, cu(np.array([1, 2, 3], np.float32)), 1).shape == (0, 3, 5, 5)
    assert ops.mask_apply(e, torch.empty(0, dtype=torch.bool, device="cuda"), (1, 1, 0)).shape == (0,)
    x1 = np.array([0.7391], np.float32)
    assert bits_equal(npy(quantize_with_decimal(cu(x1), 8, 4)), orc.fq_pow2_fwd(x1, 4))
    assert bits_equal(npy(quantize_with_scaler(cu(x1), 8, 0.013)), orc.fq_scaler_fwd(x1, np.float32(0.013)))
    lines = np.array([[-0.2, 0.9]], np.float32)
    assert bits_equal(npy(quantize_with_line(cu(x1), 8, (-0.2, 0.9))), orc.fq_line_fwd(x1, lines, 8, -1, True))
    st = ops.reduce_stats(cu(x1), (1, 1, 1), absmax=True, minmax=True, abssum=True, nnz=True)
    assert npy(st["absmax"])[0] == x1[0] and npy(st["min"])[0] == x1[0] and npy(st["max"])[0] == x1[0]
    assert npy(st["abssum"])[0] == np.float64(x1[0]) and npy(st["nnz"])[0] == 1.0
    assert npy(ops.kth_value(cu(x1), 0))[0] == x1[0]
    g = cu(np.array([500.0], np.float32))
    ops.ste_bwd(g, 0.0, True, 8, 0, (1, 1, 1))            # decimal 0, 8 bits: clamp to [-128, 127]
    assert npy(g)[0] == 127.0


@pytest.mark.parametrize("bits", [1, 2, 3, 12, 16, 24, 32])
def test_bit_width_extremes(bits):
    """The reference takes any bit width (its tests use 8 and 4): 2^bits - 1 is not representable in fp32 from 25
    bits on, the line quantizer's step underflows the fast-division range, the STE bounds reach 2^31."""
    from qsparse_b200 import ops
    from qsparse_b200.quantize import quantize_with_line
    x = rnd((3, 5, 41), 90 + bits, 2.0)
    x.reshape(-1)[::53] *= 1e6
    C = 5
    rng = np.random.default_rng(bits)
    lines = np.stack([rng.uniform(-2, -0.1, C), rng.uniform(0.1, 2, C)], 1).astype(np.float32)
    for fzp in (True, False):
        assert bits_equal(npy(quantize_with_line(cu(x), bits, cu(lines), 1, False, fzp)),
                          orc.fq_line_fwd(x, lines, bits, 1, fzp)), fzp
        assert bits_equal(npy(quantize_with_line(cu(x), bits, (-0.3, 1.1), -1, False, fzp)),
                          orc.fq_line_fwd(x, np.array([[-0.3, 1.1]], np.float32), bits, -1, fzp)), fzp
    g = rnd((3, 5, 41), 70 + bits, 3.0)
    g.reshape(-1)[::31] *= 1e9
    dec = rng.integers(-2, 7, C).astype(np.float32)
    sc = rng.uniform(0.001, 0.05, C).astype(np.float32)
    for scale, is_dec in ((dec, True), (sc, False)):
        gc = cu(g).clone()
        ops.ste_bwd(gc, cu(scale), is_dec, bits, 1, (3, 5, 41))
        ref, _ = orc.ste_bwd(g, scale, bits, 1, is_dec, True)
        assert bits_equal(npy(gc), ref), is_dec


def test_extreme_parameters_and_inputs():
    """Decimals / scales / lines far outside the useful range (overflowing 2^d, zero / negative / infinite / NaN
    scales, empty and inverted ranges) over inputs with +-0, +-inf, NaN, subnormals and huge values.  The oracle
    equals the unmodified reference (CPU) on all of these; the kernels must equal the oracle, per tensor (host
    parameter) and per channel (device parameters) — for the int32-based quantizers inside the documented parity
    domain |x * 2^d| < 2^31 (DESIGN 2, Q5: outside it `.int()` is INT_MIN on x86 and saturates on CUDA, in the
    reference as well)."""
    from qsparse_b200.quantize import quantize_with_decimal, quantize_with_scaler, quantize_with_line
    rng = np.random.default_rng(0)
    decs = [-40.0, -1.0, 0.0, 30.0, 100.0, 126.0, 130.0]
    scs = [1e-30, 3e37, -0.5, 0.0, float("inf"), float("nan"), 1e-42]
    lns = [(0.0, 0.0), (1.0, 1.0), (0.5, -0.5), (0.0, 1e-30), (-1e30, 1e30), (0.0, float("inf")), (-0.3, 0.7)]
    C = 7
    x = (rng.standard_normal((3, C, 330)) * 2).astype(np.float32)
    special = np.array([0.0, -0.0, np.inf, -np.inf, np.nan, 1e38, -1e38, 1e-40, -1e-40, 3e9, -3e9, 0.5], np.float32)
    x[:, :, :12] = special
    x[:, :, 12:40] *= np.float32(1e-12)                   # something inside the domain for the large decimals
    xc = cu(x)

    def in_domain(q):
        with np.errstate(all="ignore"):
            return np.isfinite(q) & (np.abs(q) < 2.0 ** 31)

    def check(got, exp, ok, what):
        assert bits_equal(np.where(ok, npy(got), 0), np.where(ok, exp, 0)), what

    with np.errstate(all="ignore"):
        dv, sv = np.array(decs, np.float32), np.array(scs, np.float32)
        check(quantize_with_decimal(xc, 8, cu(dv), 1), orc.fq_pow2_fwd(x, dv, 1),
              in_domain(x * (np.float32(2.0) ** dv).reshape(1, C, 1)), "decimal per channel")
        ok_s = in_domain(x / sv.reshape(1, C, 1))
        ok_s[:, [5], :] = False                           # a NaN scale: nothing is in the domain
        check(quantize_with_scaler(xc, 8, cu(sv), 1), orc.fq_scaler_fwd(x, sv, 1), ok_s, "scaler per channel")
        for d in decs:
            check(quantize_with_decimal(xc, 8, d), orc.fq_pow2_fwd(x, d), in_domain(x * np.float32(2.0) ** np.float32(d)),
                  ("decimal", d))
        for sc in scs[:5] + scs[6:]:
            check(quantize_with_scaler(xc, 8, sc), orc.fq_scaler_fwd(x, np.float32(sc)), in_domain(x / np.float32(sc)),
                  ("scaler", sc))
    lines = np.array(lns, np.float32)
    for fzp in (True, False):                             # no int32 in the line quantizer: the whole input range
        assert bits_equal(npy(quantize_with_line(xc, 8, cu(lines), 1, False, fzp)),
                          orc.fq_line_fwd(x, lines, 8, 1, fzp)), fzp
        for ln in lns:
            assert bits_equal(npy(quantize_with_line(xc, 8, ln, -1, False, fzp)),
                              orc.fq_line_fwd(x, np.array([ln], np.float32), 8, -1, fzp)), (ln, fzp)


def test_reduction_nan_propagates():
    from qsparse_b200 import ops
    x = rnd((4, 8, 100), 2)
    x[1, 3, 17] = np.nan
    st = ops.reduce_stats(cu(x), (4, 8, 100), absmax=True, minmax=True)
    am, mn = npy(st["absmax"]), npy(st["min"])
    assert np.isnan(am[3]) and np.isnan(mn[3]) and not np.isnan(np.delete(am, 3)).any()


@pytest.mark.parametrize("n", [2, 7, 64, 1000, 4097, 100003, 1 << 20, (1 << 22) + 5])
def test_kth_value_vs_sort(n):
    from qsparse_b200 import ops
    rng = np.random.default_rng(n)
    v = (rng.standard_normal(n) * rng.choice([1e-3, 1.0, 50.0], n)).astype(np.float32)
    if n >= 64:
        v[rng.choice(n, n // 8, replace=False)] = 0.25          # heavy ties
        v[rng.choice(n, 3, replace=False)] = [np.inf, -np.inf, -0.0]
    s = np.sort(v)
    vc = cu(v)
    for k in sorted({0, 1, n // 3, n // 2, n - 2, n - 1} & set(range(n))):
        got = npy(ops.kth_value(vc, k))[0]
        assert got == s[k], (n, k)
        got = npy(ops.kth_value(vc, k, take_abs=True))[0]
        assert got == np.sort(np.abs(v))[k], (n, k, "abs")
    if n >= 64:  # NaNs order last, like torch.sort
        v2 = v.copy()
        v2[:5] = np.nan
        assert np.isnan(npy(ops.kth_value(cu(v2), n - 1))[0])
        assert npy(ops.kth_value(cu(v2), n - 6))[0] == np.sort(v2)[n - 6]
    # unaligned base pointer
    if n > 8:
        got = npy(ops.kth_value(vc[1:], (n - 1) // 2))[0]
        assert got == np.sort(v[1:])[(n - 1) // 2]


@pytest.mark.parametrize("shape", [(8, 16, 3, 3), (37, 11), (3, 5, 7, 9)])
@pytest.mark.parametrize("sparsity", [0.0, 0.3, 0.5, 0.9])
def test_unstructured_mask_vs_oracle(shape, sparsity):
    from qsparse_b200 import calculate_mask_given_importance, ops
    imp = np.abs(rnd(shape, 31))
    m_ref, thr_ref = orc.mask_given_importance(imp, sparsity)
    assert np.array_equal(npy(calculate_mask_given_importance(cu(imp), sparsity)), m_ref)
    # fused build + apply
    x = rnd(shape, 32)
    mask = torch.empty(shape, dtype=torch.bool, device="cuda")
    thr = ops.kth_value(cu(imp), orc.kth_index(sparsity, imp.size))
    assert npy(thr)[0] == thr_ref
    y = ops.mask_build_apply(cu(imp), thr, cu(x), mask)
    assert np.array_equal(npy(mask), m_ref)
    assert bits_equal(npy(y), orc.mask_apply(x, m_ref.reshape(-1)))


@pytest.mark.parametrize("shape,mshape", [((4, 8, 5, 5), (1, 8, 1, 1)), ((3, 6, 7), (1, 6, 7)), ((5, 4, 3, 3), (5, 1, 1, 1)),
                                          ((2, 3, 6, 6), (2, 3, 6, 6)), ((6, 9), (1, 9))])
def test_mask_apply_and_fused_quant_vs_oracle(shape, mshape):
    from qsparse_b200 import ops
    from qsparse_b200.sparse import apply_mask
    x = rnd(shape, 41, 2.0)
    rng = np.random.default_rng(8)
    m = rng.random(mshape) > 0.4
    kind, layout = ops.mask_layout(shape, mshape)
    ci = {"element": -1}.get(kind, None)
    if kind == "channel":
        ci = [i for i, s in enumerate(mshape) if s != 1][0]
        o, c, i = layout
        ref = (x.reshape(o, c, i) * m.reshape(1, c, 1).astype(np.float32)).reshape(shape)
    else:
        ref = x * m.astype(np.float32)
    xc = cu(x).requires_grad_(True)
    y = apply_mask(xc, cu(m))
    assert bits_equal(npy(y), ref)                          # sign of zero kept (SURVEY Q8)
    g = rnd(shape, 42)
    y.backward(cu(g))
    gref = (g.reshape(layout) * m.reshape(1, layout[1], 1).astype(np.float32)).reshape(shape) if kind == "channel" \
        else g * m.astype(np.float32)
    assert bits_equal(npy(xc.grad), gref)
    # fused prune -> quantize forward / backward equals the two-step oracle
    mflat = cu(m.reshape(-1))
    yq = ops.fq_pow2_fwd(cu(x), 5.0, layout, mask=mflat)
    assert bits_equal(npy(yq), orc.fq_pow2_fwd(ref, 5))
    ys = ops.fq_scaler_fwd(cu(x), 0.043, layout, mask=mflat)
    assert bits_equal(npy(ys), orc.fq_scaler_fwd(ref, np.float32(0.043)))
    gc = cu(g).clone()
    _, gx = ops.ste_bwd(gc, 5.0, True, 8, 0, layout, mask=mflat, clamp_in_place=True, want_gx=True)
    gcl, _ = orc.ste_bwd(g, np.float32(5), 8, -1, True, False)
    assert bits_equal(npy(gc), gcl)
    gxr = (gcl.reshape(layout) * m.reshape(1, layout[1], 1).astype(np.float32)).reshape(shape) if kind == "channel" \
        else gcl * m.astype(np.float32)
    assert bits_equal(npy(gx), gxr)


def test_fused_param_step_vs_oracle():
    """qsb_prune_quant_params == magnitude EMA -> mask -> abs-max of kept -> scale EMA -> decimal."""
    from qsparse_b200 import ops
    C, shape = 64, (8, 64, 14, 14)
    mag = np.zeros(C, np.float32)
    scale = np.zeros(1, np.float32)
    mag_d = cu(mag)
    mask_d = torch.ones(C, dtype=torch.bool, device="cuda")
    scale_d = cu(scale)
    dec_d = torch.zeros(1, device="cuda")
    mask = np.ones(C, bool)
    for t in range(5):
        x = np.maximum(rnd(shape, 100 + t), 0) * np.linspace(0.2, 2.0, C, dtype=np.float32).reshape(1, C, 1, 1)
        st = ops.reduce_stats(cu(x), (8, C, 196), abssum=True, absmax=True)
        refresh = t > 0
        k = orc.kth_index(0.75, C)
        ops.prune_quant_params(mag_d, mask_d, scale_d, dec_d, st, 8 * 196.0, t, 1, refresh, k, 8, t, True)
        mag = orc.magnitude_ema(mag, orc.squeeze_mean_abs(x, (1, C, 1, 1)).reshape(-1), t)
        if refresh:
            mask, _ = orc.mask_given_importance(mag, 0.75)
        amax_kept = np.array([np.max(orc.absmax(x, 1) * mask)], np.float32)
        scale = orc.scale_ema(scale, amax_kept, 8, t)
        assert ulp_diff(npy(mag_d), mag).max() <= 8, t
        assert np.array_equal(npy(mask_d), mask), t
        assert bits_equal(npy(scale_d), scale), t
        assert bits_equal(npy(dec_d), orc.scale_to_decimal(scale)), t
        y = ops.fq_pow2_fwd(cu(x), dec_d, (8, C, 196), mask=mask_d)
        assert bits_equal(npy(y), orc.fq_pow2_fwd(x, npy(dec_d), 1, mask=mask))


def test_magnitude_ema_full_and_l0():
    from qsparse_b200 import ops
    x = rnd((3, 4, 50), 51)
    x[x < 0.3] = 0
    mag = np.abs(rnd((3, 4, 50), 52))
    md = cu(mag).clone()
    ops.magnitude_ema_full_(md, cu(x), 3)
    assert bits_equal(npy(md), orc.magnitude_ema(mag, np.abs(x), 3))
    md = cu(mag).clone()
    tmin = ops.reduce_stats(cu(x), (1, 1, x.size), nnz=True)["tensor_min"]
    ops.magnitude_ema_full_(md, cu(x), 3, tmin, True)     # min(x) == 0 -> indicator
    assert bits_equal(npy(md), orc.magnitude_ema(mag, (x != 0).astype(np.float32), 3))


# ------------------------------------------------------------------ properties at full size
def test_full_size_properties_config2():
    """[256,64,56,56] (BASELINE config 2): idempotence, integer grid, pruned channels zero,
    agreement with the oracle on a sampled sub-block."""
    from qsparse_b200 import ops
    torch.manual_seed(2)
    shape = (256, 64, 56, 56)
    x = torch.relu(torch.randn(shape, device="cuda"))
    layout = (256, 64, 3136)
    mask = (torch.arange(64, device="cuda") % 4 == 0)           # 75 % of the channels pruned
    dec = torch.tensor([5.0], device="cuda")
    y = ops.fq_pow2_fwd(x, dec, layout, mask=mask)
    assert torch.equal(ops.fq_pow2_fwd(y, dec, layout, mask=mask), y)          # idempotent
    q = y * 32.0
    assert torch.equal(q, q.round())                                           # on the 2^-5 grid
    assert torch.count_nonzero(y[:, ~mask]).item() == 0
    assert torch.equal(y[:, mask], ops.fq_pow2_fwd(x[:, mask].contiguous(), 5.0, (1, 1, 256 * 16 * 3136)))
    xs = x[7:9].contiguous()
    assert bits_equal(npy(ops.fq_pow2_fwd(xs, dec, (2, 64, 3136), mask=mask)),
                      orc.fq_pow2_fwd(npy(xs), 5, 1, mask=npy(mask)))
    st = ops.reduce_stats(x, layout, abssum=True, absmax=True)
    assert torch.equal(st["absmax"], x.abs().amax(dim=(0, 2, 3)))
    ref = x.double().abs().sum(dim=(0, 2, 3))
    assert torch.allclose(st["abssum"], ref, rtol=3e-7, atol=0)
    again = ops.reduce_stats(x, layout, abssum=True, absmax=True)
    assert torch.equal(again["abssum"], st["abssum"])        # deterministic: fixed summation order


def test_full_size_config2_step_vs_oracle_every_element():
    """The WHOLE [256,64,56,56] tensor of BASELINE config 2 through two fused training steps (one-launch
    statistics + parameter step, forward, backward) against the plain-C oracle on the identical tensor: all
    51,380,224 outputs and gradients bit for bit, mask / scale / decimal exact, magnitude within the documented
    mean tolerance."""
    from concurrent.futures import ThreadPoolExecutor
    from qsparse_b200 import ops
    torch.manual_seed(2)
    shape, layout, C = (256, 64, 56, 56), (256, 64, 3136), 64
    gen = torch.Generator(device="cuda").manual_seed(2)
    x = torch.relu(torch.randn(shape, device="cuda", generator=gen)) * torch.linspace(0.5, 1.5, C, device="cuda").view(
        1, C, 1, 1)
    g = torch.randn(shape, device="cuda", generator=gen) * 3
    xh, gh = npy(x), npy(g)
    mag = torch.zeros(C, device="cuda")
    mask = torch.ones(C, dtype=torch.bool, device="cuda")
    scale = torch.zeros(1, device="cuda")
    dec = torch.zeros(1, device="cuda")
    mag_ref, mask_ref, scale_ref = np.zeros(C, np.float32), np.ones(C, bool), np.zeros(1, np.float32)
    k = orc.kth_index(0.75, C)
    pool = ThreadPoolExecutor(8)
    parts = [slice(i * 32, (i + 1) * 32) for i in range(8)]
    for t in range(2):
        ops.reduce_prune_quant_step(x, layout, mag, mask, scale, dec, 256 * 3136.0, t, 1, t > 0, k, 8, t, True)
        y = ops.fq_pow2_fwd(x, dec, layout, mask=mask)
        _, gx = ops.ste_bwd(g, dec, True, 8, 0, layout, mask=mask, clamp_in_place=False, want_gx=True)
        mag_ref = orc.magnitude_ema(mag_ref, orc.squeeze_mean_abs(xh, (1, C, 1, 1)).reshape(-1), t)
        if t > 0:
            mask_ref, _ = orc.mask_given_importance(mag_ref, 0.75)
        scale_ref = orc.scale_ema(scale_ref, np.array([np.max(orc.absmax(xh, 1) * mask_ref)], np.float32), 8, t)
        dec_ref = orc.scale_to_decimal(scale_ref)
        assert np.array_equal(npy(mask), mask_ref) and bits_equal(npy(scale), scale_ref) and bits_equal(npy(dec), dec_ref)
        assert ulp_diff(npy(mag), mag_ref).max() <= 8
        yh, gxh = npy(y), npy(gx)
        y_ref = list(pool.map(lambda sl: orc.fq_pow2_fwd(xh[sl], dec_ref, 1, mask=mask_ref), parts))
        g_ref = list(pool.map(lambda sl: orc.ste_bwd(gh[sl].copy(), dec_ref, 8, 1, True, False, mask=mask_ref)[1], parts))
        for sl, yr, gr in zip(parts, y_ref, g_ref):
            assert np.array_equal(yh[sl].view(np.uint32), yr.view(np.uint32)), t
            assert np.array_equal(gxh[sl].view(np.uint32), gr.view(np.uint32)), t


def test_full_size_select_64M():
    """64 Mi-element importance (BASELINE config 4): exact threshold == torch.sort's, mask count."""
    from qsparse_b200 import calculate_mask_given_importance, ops
    torch.manual_seed(4)
    n = 1 << 26
    imp = (torch.randn(n, device="cuda") * 0.02).abs()
    for s in (0.5, 0.75):
        k = max(int(s * n - 1), 0) + 1
        thr = ops.kth_value(imp, k)
        ref = torch.sort(imp).values[k]
        assert thr.item() == ref.item()
        m = calculate_mask_given_importance(imp, s)
        assert torch.equal(m, imp >= ref)             # ties with the threshold are kept (SURVEY Q13)
        assert int((~m).sum().item()) <= k


def test_fast_division_is_exact():
    """The reciprocal-based division used by the scaler / line / EMA kernels must equal
    IEEE division bit for bit (2^31 operand pairs incl. rounding-boundary neighbours)."""
    from ctypes import c_int64, c_uint64
    from qsparse_b200 import _native as N
    lib = N.load_library()
    bad = torch.zeros(1, dtype=torch.int64, device="cuda")
    for seed in (1, 2, 3, 4):
        N.check(lib.qsb_selftest_fastdiv(c_int64(1 << 19), c_int64(1 << 10), c_uint64(seed), N.ptr(bad),
                                         N.stream_ptr(bad.device)), "selftest")
    assert bad.item() == 0


def test_scaler_line_dense_rounding_boundaries():
    """x placed on and next to every (k + 0.5) * s boundary: division + rint must agree with the oracle."""
    from qsparse_b200.quantize import quantize_with_scaler, quantize_with_line
    rng = np.random.default_rng(77)
    for s in (0.1, 0.037, 0.0123456, 1.7):
        k = np.arange(-300, 300, dtype=np.float32) + 0.5
        x = (k * np.float32(s)).astype(np.float32)
        xs = np.concatenate([x, np.nextafter(x, np.float32(10)), np.nextafter(x, np.float32(-10)),
                             rng.standard_normal(4096).astype(np.float32)])
        assert bits_equal(npy(quantize_with_scaler(cu(xs), 8, s)), orc.fq_scaler_fwd(xs, np.float32(s)))
        lines = np.array([[-3 * s, 250 * s]], np.float32)
        for fzp in (True, False):
            assert bits_equal(npy(quantize_with_line(cu(xs), 8, (float(lines[0, 0]), float(lines[0, 1])), -1, False, fzp)),
                              orc.fq_line_fwd(xs, lines, 8, -1, fzp))


@pytest.mark.parametrize("shape,C", [((8, 64, 14, 14), 64), ((4, 200, 9, 9), 200), ((16, 7, 70), 7), ((32, 48), 48)])
def test_fused_step_kernel_equals_separate_kernels(shape, C):
    """reduce_partials + prune_quant_step_params (finalize folded into the parameter kernel)
    must be bit-identical to reduce_stats + prune_quant_params."""
    from qsparse_b200 import ops
    from qsparse_b200._native import channel_layout
    layout = channel_layout(shape, 1)
    count = float(layout[0] * layout[2])
    st_a = dict(mag=torch.zeros(C, device="cuda"), mask=torch.ones(C, dtype=torch.bool, device="cuda"),
                scale=torch.zeros(1, device="cuda"), dec=torch.zeros(1, device="cuda"))
    st_b = {k: v.clone() for k, v in st_a.items()}
    st_c = {k: v.clone() for k, v in st_a.items()}          # graph mode: step index on the device
    counter = torch.zeros(1, dtype=torch.int64, device="cuda")
    k = orc.kth_index(0.5, C)
    for t in range(4):
        x = cu(np.maximum(rnd(shape, 300 + t), 0) * np.linspace(0.3, 1.7, C, dtype=np.float32).reshape(
            (1, C) + (1,) * (len(shape) - 2)))
        st = ops.reduce_stats(x, layout, abssum=True, absmax=True)
        ops.prune_quant_params(st_a["mag"], st_a["mask"], st_a["scale"], st_a["dec"], st, count, t, 1, t > 0, k, 8, t,
                               True)
        ws = ops.reduce_partials(x, layout)
        asum = torch.empty(C, dtype=torch.float64, device="cuda")
        amax = torch.empty(C, dtype=torch.float32, device="cuda")
        ops.prune_quant_step_params(st_b["mag"], st_b["mask"], st_b["scale"], st_b["dec"], ws, layout, count, t, 1,
                                    t > 0, k, 8, t, True, abssum_out=asum, absmax_out=amax)
        # the two kernels add the same partials in different (each fixed) orders: fp64 rounding only
        assert torch.allclose(asum, st["abssum"], rtol=1e-14, atol=0) and torch.equal(amax, st["absmax"]), t
        ws = ops.reduce_partials(x, layout)
        ops.prune_quant_step_params(st_c["mag"], st_c["mask"], st_c["scale"], st_c["dec"], ws, layout, count, 0, 1,
                                    1, k, 8, 0, True, step_counter=counter)
        assert counter.item() == t + 1
        for key in st_a:
            assert torch.equal(st_a[key], st_b[key]), (key, t)
            assert torch.equal(st_a[key], st_c[key]), (key, t, "graph mode")


@pytest.mark.parametrize("shape,C", [((8, 64, 56, 56), 64), ((8, 64, 14, 14), 64), ((4, 200, 9, 9), 200),
                                     ((16, 7, 70), 7), ((32, 48), 48), ((64, 1000), 1000), ((3, 1, 5000), 1),
                                     ((2, 1024, 300), 1024), ((5, 3, 1031), 3), ((2, 1, 9), 1), ((1, 1, 288), 1)])
def test_one_launch_step_equals_two_launch_step(shape, C):
    """qsb_reduce_prune_quant_step (the reduction's last-arriving CTA runs the parameter step) must be
    bit-identical to qsb_reduce_partials + qsb_prune_quant_step_params in every stage-1 mode (rows, columns,
    one channel), with the row-kernel variants and with / without the L2 keep hint; the arrival
    counter must be left at zero after every launch."""
    from qsparse_b200 import ops
    from qsparse_b200._native import channel_layout
    layout = channel_layout(shape, 1)
    count = float(layout[0] * layout[2])
    k = orc.kth_index(0.5, C)

    def fresh():
        return dict(mag=torch.zeros(C, device="cuda"), mask=torch.ones(C, dtype=torch.bool, device="cuda"),
                    scale=torch.zeros(1, device="cuda"), dec=torch.zeros(1, device="cuda"))

    xs = [cu(np.maximum(rnd(shape, 900 + t), 0) * np.linspace(0.3, 1.7, C, dtype=np.float32).reshape(
        (1, C) + (1,) * (len(shape) - 2))) for t in range(4)]
    try:
        for variant in (2, 0):
            ops.set_tuning(17, variant)
            ref = fresh()
            ref_stats = []
            for t, x in enumerate(xs):
                ws = ops.reduce_partials(x, layout)
                asum = torch.empty(C, dtype=torch.float64, device="cuda")
                amax = torch.empty(C, dtype=torch.float32, device="cuda")
                ops.prune_quant_step_params(ref["mag"], ref["mask"], ref["scale"], ref["dec"], ws, layout, count, t,
                                            1, t > 0 and C > 1, k, 8, t, True, abssum_out=asum, absmax_out=amax)
                ref_stats.append((asum, amax, {key: v.clone() for key, v in ref.items()}))
            for hint in (1, 0):
                ops.set_tuning(18, hint)
                st = fresh()
                stg = fresh()
                counter = torch.zeros(1, dtype=torch.int64, device="cuda")
                for t, x in enumerate(xs):
                    asum = torch.empty(C, dtype=torch.float64, device="cuda")
                    amax = torch.empty(C, dtype=torch.float32, device="cuda")
                    ops.reduce_prune_quant_step(x, layout, st["mag"], st["mask"], st["scale"], st["dec"], count, t, 1,
                                                t > 0 and C > 1, k, 8, t, True, abssum_out=asum, absmax_out=amax)
                    assert int(ops.arrival_counter(x.device)[0].item()) == 0
                    # (wide column-mode shapes take the three-launch form, whose parallel finalize adds the same
                    # partials in another fixed order: the fp64 sums then agree to the last bits, not bit for bit)
                    assert torch.allclose(asum, ref_stats[t][0], rtol=1e-13, atol=0), (variant, t)
                    assert torch.equal(amax, ref_stats[t][1]), (variant, t)
                    # local statistics row == the combined one on a single GPU
                    asum_l = torch.empty_like(asum)
                    amax_l = torch.empty_like(amax)
                    ops.reduce_prune_quant_step(x, layout, stg["mag"], stg["mask"], stg["scale"], stg["dec"], count, 0,
                                                1, 1 if C > 1 else 1 << 30, k if C > 1 else 0, 8, 0, True,
                                                abssum_out=asum_l, absmax_out=amax_l,
                                                stats_local=True, step_counter=counter)
                    assert counter.item() == t + 1
                    assert torch.equal(asum_l, asum) and torch.equal(amax_l, amax)
                    for key in st:
                        if key == "mag":
                            assert ulp_diff(npy(st[key]), npy(ref_stats[t][2][key])).max() <= 1, (key, t, variant, hint)
                        else:
                            assert torch.equal(st[key], ref_stats[t][2][key]), (key, t, variant, hint)
                        assert torch.equal(stg[key], st[key]), (key, t, variant, hint, "graph mode")
    finally:
        ops.set_tuning(17, -1)
        ops.set_tuning(18, 1)


def test_one_launch_step_oracle_three_steps():
    """the one-launch step against the plain-C oracle on the smoke shape (magnitude within the documented
    mean tolerance, mask / decimal exact)"""
    from qsparse_b200 import ops
    C, shape, layout = 16, (4, 16, 14, 14), (4, 16, 196)
    x = np.maximum(rnd(shape, 41), 0) * np.linspace(0.1, 2, C, dtype=np.float32).reshape(1, C, 1, 1)
    xd = cu(x)
    mag = torch.zeros(C, device="cuda")
    mask = torch.ones(C, dtype=torch.bool, device="cuda")
    scale = torch.zeros(1, device="cuda")
    dec = torch.zeros(1, device="cuda")
    mag_ref, mask_ref, scale_ref = np.zeros(C, np.float32), np.ones(C, bool), np.zeros(1, np.float32)
    k = orc.kth_index(0.75, C)
    for t in range(3):
        ops.reduce_prune_quant_step(xd, layout, mag, mask, scale, dec, 4 * 196.0, t, 1, t > 0, k, 8, t, True)
        mag_ref = orc.magnitude_ema(mag_ref, orc.squeeze_mean_abs(x, (1, C, 1, 1)).reshape(-1), t)
        if t > 0:
            mask_ref, _ = orc.mask_given_importance(mag_ref, 0.75)
        scale_ref = orc.scale_ema(scale_ref, np.array([np.max(orc.absmax(x, 1) * mask_ref)], np.float32), 8, t)
        assert np.array_equal(npy(mask), mask_ref)
        assert bits_equal(npy(scale), scale_ref)
        assert bits_equal(npy(dec), orc.scale_to_decimal(scale_ref))
        assert ulp_diff(npy(mag), mag_ref).max() <= 8


@pytest.mark.parametrize("shape", [(4000, 48), (300, 24, 5), (700, 1000)])
def test_fused_step_kernel_unaligned_column_mode(shape):
    """A 4-byte-aligned x makes the column reduction fall back to scalar columns; the partial layout that the
    parameter kernel re-derives (without seeing x) must still be the one the reduction wrote."""
    from qsparse_b200 import ops
    from qsparse_b200._native import channel_layout
    C = shape[1]
    layout = channel_layout(shape, 1)
    count = float(layout[0] * layout[2])
    n = int(np.prod(shape))
    base = cu(np.abs(rnd((n + 1,), 77)))
    k = orc.kth_index(0.5, C)
    res = []
    for x in (base[1:].view(shape), base[1:].clone().view(shape)):          # unaligned view, aligned copy
        st = dict(mag=torch.zeros(C, device="cuda"), mask=torch.ones(C, dtype=torch.bool, device="cuda"),
                  scale=torch.zeros(1, device="cuda"), dec=torch.zeros(1, device="cuda"))
        asum = torch.empty(C, dtype=torch.float64, device="cuda")
        amax = torch.empty(C, dtype=torch.float32, device="cuda")
        ws = ops.reduce_partials(x, layout)
        ops.prune_quant_step_params(st["mag"], st["mask"], st["scale"], st["dec"], ws, layout, count, 0, 1, True, k, 8,
                                    0, True, abssum_out=asum, absmax_out=amax)
        ref = ops.reduce_stats(x, layout, abssum=True, absmax=True)
        assert torch.equal(amax, ref["absmax"]) and torch.allclose(asum, ref["abssum"], rtol=1e-14, atol=0)
        assert torch.equal(amax, x.abs().amax(dim=tuple(i for i in range(len(shape)) if i != 1)))
        res.append((st, asum, amax))
    for key in res[0][0]:
        assert torch.equal(res[0][0][key], res[1][0][key]), key
    assert torch.equal(res[0][2], res[1][2])


@pytest.mark.parametrize("kind", ["normal", "all_equal", "half_zeros", "two_values", "with_nan"])
def test_kth_value_fast_route_and_fallback(kind):
    """n >= 2^22 takes the sampled-pivot route; data with heavy ties overflows the candidate buffer and
    must fall back to the full radix select on the device.  Both must equal torch.sort bit for bit."""
    from qsparse_b200 import ops
    n = (1 << 23) + 77
    g = torch.Generator(device="cuda").manual_seed(5)
    v = torch.randn(n, device="cuda", generator=g)
    if kind == "all_equal":
        v.fill_(0.125)
    elif kind == "half_zeros":
        v = torch.relu(v)
    elif kind == "two_values":
        v = (v > 0.3).float() * 2 - 0.5
    elif kind == "with_nan":
        v[::1000003] = float("nan")
    ref = torch.sort(v).values
    ref_abs = torch.sort(v.abs()).values
    for k in (0, 1, n // 7, n // 2, (3 * n) // 4, n - 2, n - 1):
        got = ops.kth_value(v, k)
        assert torch.equal(got.view(torch.int32), ref[k:k + 1].view(torch.int32)) or \
            (torch.isnan(got).item() and torch.isnan(ref[k]).item()), (kind, k)
        got = ops.kth_value(v, k, take_abs=True)
        assert torch.equal(got, ref_abs[k:k + 1]) or (torch.isnan(got).item() and torch.isnan(ref_abs[k]).item()), \
            (kind, k, "abs")
    ops.set_tuning(4, 0)          # 3-pass route only: same answers
    try:
        for k in (n // 2, n - 1):
            a = ops.kth_value(v, k)
            assert torch.equal(a.view(torch.int32), ref[k:k + 1].view(torch.int32)) or torch.isnan(a).item()
    finally:
        ops.set_tuning(4, 1)


# ----------------------------------------------------------------------------- K8 row-resident fused kernel
ROW_SHAPES = [(33, 8), (64, 288), (7, 1000), (130, 1024), (5, 2048), (48, 4096), (3, 8200), (2, 16384),
              (9, 4, 6, 12)]


@pytest.fixture(params=[0], ids=["registers"])
def row_variant(request):
    """the register-resident kernel for rows of 1 Ki .. 16 Ki elements"""
    yield request.param


@pytest.mark.parametrize("shape", ROW_SHAPES)
@pytest.mark.parametrize("kind", ["decimal", "scaler", "line"])
def test_row_quant_fused_vs_oracle_and_unfused(shape, kind, row_variant):
    """qsb_row_quant_fused == reduce -> EMA -> fake-quant (oracle, and our own three-kernel sequence), bit for
    bit, over several EMA steps; rows of every dispatch width (a warp per row, a CTA per row)."""
    from qsparse_b200 import ops
    rows = shape[0]
    bits = 4
    w_unf = None
    if kind == "line":
        w_fused = torch.zeros(rows, 2, device="cuda")
        w_orc = np.zeros((rows, 2), np.float32)
    else:
        w_fused = torch.zeros(rows, 1, device="cuda")
        w_orc = np.zeros((rows, 1), np.float32)
    w_unf = w_fused.clone()
    for step in range(3):
        x = rnd(shape, 100 + step, 0.02 * (step + 1))
        if step == 1:
            x.reshape(rows, -1)[0, :] = 0.0           # an all-zero row: scale 0 / step 0 -> 1e-4 paths
        xc = cu(x)
        assert ops.row_quant_supported(xc, rows)
        if kind == "line":
            t = step + 1
            y, _ = ops.row_quant_fused_(xc, w_fused, ops.ROW_LINE, bits, t, True)
            mn, mx = orc.minmax(x, 0)
            w_orc = orc.lines_ema(w_orc, mn, mx, t)
            y_orc = orc.fq_line_fwd(x, w_orc, bits, 0, True)
            st = ops.reduce_stats(xc, (1, rows, x.size // rows), minmax=True)
            ops.lines_ema_(w_unf, st["min"], st["max"], t)
            y_unf = ops.fq_line_fwd(xc, w_unf, bits, True, (1, rows, x.size // rows))
        else:
            t = step
            k = ops.ROW_DECIMAL if kind == "decimal" else ops.ROW_SCALER
            y, dec = ops.row_quant_fused_(xc, w_fused, k, bits, t)
            w_orc = orc.scale_ema(w_orc.reshape(-1), orc.absmax(x, 0), bits, t).reshape(rows, 1)
            st = ops.reduce_stats(xc, (1, rows, x.size // rows), absmax=True)
            ops.scale_ema_(w_unf, st["absmax"], bits, t)
            if kind == "decimal":
                d_orc = orc.scale_to_decimal(w_orc.reshape(-1))
                assert bits_equal(npy(dec), d_orc), step
                y_orc = orc.fq_pow2_fwd(x, d_orc, 0)
                y_unf = ops.fq_pow2_fwd(xc, ops.scale_to_decimal(w_unf).view(-1), (1, rows, x.size // rows))
            else:
                y_orc = orc.fq_scaler_fwd(x, w_orc.reshape(-1), 0)
                y_unf = ops.fq_scaler_fwd(xc, w_unf.view(-1), (1, rows, x.size // rows))
        assert bits_equal(npy(w_fused), w_orc), (kind, step, "param vs oracle")
        assert torch.equal(w_fused.view(torch.int32), w_unf.view(torch.int32)), (kind, step, "param vs unfused")
        assert bits_equal(npy(y), y_orc), (kind, step, "y vs oracle")
        assert torch.equal(y.view(torch.int32), y_unf.view(torch.int32)), (kind, step, "y vs unfused")


@pytest.mark.parametrize("shape", [(64, 4608), (300, 1152), (37, 256), (16, 16384)])
@pytest.mark.parametrize("kind", ["decimal", "scaler", "line"])
def test_row_quant_fused_masked_equals_mask_apply_then_row_quant(shape, kind):
    """K8 with an element mask == mask_apply followed by K8, bit for bit (values, parameters, decimals)"""
    from qsparse_b200 import ops
    code = {"decimal": ops.ROW_DECIMAL, "scaler": ops.ROW_SCALER, "line": ops.ROW_LINE}[kind]
    x = cu(rnd(shape, 21) * 0.05)
    mask = cu(np.random.default_rng(22).random(shape) > 0.6)
    wsz = 2 if kind == "line" else 1
    pa = torch.zeros(shape[0], wsz, device="cuda")
    pb = torch.zeros(shape[0], wsz, device="cuda")
    for t in range(3):
        tt = t + 1 if kind == "line" else t
        xm = ops.mask_apply(x, mask, (1, 1, x.numel()))
        ya, da = ops.row_quant_fused_(xm, pa, code, 4, tt)
        yb, db = ops.row_quant_fused_(x, pb, code, 4, tt, mask=mask)
        assert bits_equal(npy(ya), npy(yb)) and bits_equal(npy(pa), npy(pb)), (kind, t)
        if da is not None:
            assert bits_equal(npy(da), npy(db))
        x = x * 1.1


def test_row_quant_fused_nan_and_unsupported():
    from qsparse_b200 import ops
    x = rnd((4, 512), 3)
    x[2, 77] = np.nan
    xc = cu(x)
    w = torch.zeros(4, 2, device="cuda")
    ops.row_quant_fused_(xc, w, ops.ROW_LINE, 8, 1, True)
    wn = npy(w)
    assert np.isnan(wn[2]).all() and not np.isnan(np.delete(wn, 2, 0)).any()
    assert not ops.row_quant_supported(cu(rnd((4, 9), 1)), 4)         # rows are not whole vectors
    assert not ops.row_quant_supported(cu(rnd((2, 16392), 1)), 2)     # longer than 16 Ki
    with pytest.raises(RuntimeError):
        ops.row_quant_fused_(cu(rnd((4, 12), 1)), torch.zeros(4, 1, device="cuda"), ops.ROW_SCALER, 8, 0)


@pytest.mark.parametrize("cb_name", ["DecimalQuantizer", "ScalerQuantizer", "AdaptiveQuantizer"])
def test_weight_layer_fused_equals_unfused(cb_name):
    """quantize(nn.Linear, channelwise=0): the layer routed through K8 gives the same outputs, weights of the
    quantizer, gradients and counters as the reduce -> EMA -> quantize sequence (config 3 shape, 4 bits)."""
    import importlib
    import qsparse_b200 as q
    qz = importlib.import_module("qsparse_b200.quantize")   # the package attribute is the function
    outs = {}
    for fuse in (True, False):
        qz.FUSE_ROW_QUANTIZE = fuse
        try:
            torch.manual_seed(3)
            lin = torch.nn.Linear(512, 256).cuda()
            raw = lin.weight            # the leaf Parameter (lin.weight becomes a property below)
            layer = q.quantize(lin, bits=4, channelwise=0, timeout=1, callback=getattr(qz, cb_name)())
            layer.train()
            rec = []
            for step in range(4):
                xin = torch.randn(8, 512, device="cuda", generator=torch.Generator("cuda").manual_seed(step))
                with torch.no_grad():
                    raw.mul_(1.0 + 0.1 * step)
                y = layer(xin)
                y.square().mean().backward()
                rec.append((y.detach().clone(), raw.grad.detach().clone()))
                raw.grad = None
            sd = {k: v.detach().clone() for k, v in layer.state_dict().items()}
            outs[fuse] = (rec, sd)
        finally:
            qz.FUSE_ROW_QUANTIZE = True
    (ra, sa), (rb, sb) = outs[True], outs[False]
    assert sa.keys() == sb.keys()
    for k in sa:
        assert torch.equal(sa[k], sb[k]), k
    for (ya, ga), (yb, gb) in zip(ra, rb):
        assert torch.equal(ya, yb) and torch.equal(ga, gb)


def test_int64_indexing_4G_elements():
    """BASELINE config 5's largest size: 2^32 + 24 elements (element indices do not fit 32 bits).  The
    per-tensor and element-mask kernels, the STE backward, the per-channel window kernel and the
    reductions must address the whole tensor: checked on slices around 2^31, 2^32 and the end against
    the plain torch formula (bit-exact), plus an untouched-canary check past the end."""
    from qsparse_b200 import ops
    free, _ = torch.cuda.mem_get_info()
    n = (1 << 32) + 24
    if free < 60 * (1 << 30):
        pytest.skip("needs ~45 GB of free device memory")
    g = torch.Generator(device="cuda").manual_seed(5)
    buf = torch.empty(n + 64, device="cuda")
    x = buf[:n]
    for lo in range(0, n, 1 << 28):                       # fill in 1 GiB pieces (no 16 GB temporary)
        hi = min(lo + (1 << 28), n)
        x[lo:hi].normal_(generator=g)
    x[(1 << 32) + 3] = 77.25                              # the tensor's abs-max lives beyond 2^32
    ybuf = torch.full((n + 64,), -123.0, device="cuda")
    y = ybuf[:n]
    ops.fq_pow2_fwd(x, 4.0, (1, 1, n), out=y)
    spots = [0, (1 << 31) - 4096, (1 << 31), (1 << 32) - 4096, (1 << 32), n - 4096]

    def ref_q(v):
        return (v * 16.0).int().float() * 0.0625
    for s in spots:
        sl = slice(s, min(s + 4096, n))
        assert torch.equal(y[sl], ref_q(x[sl])), s
    assert torch.all(ybuf[n:] == -123.0)                  # nothing written past the end
    # element mask fused forward + backward
    mask = torch.empty(n, dtype=torch.bool, device="cuda")
    for lo in range(0, n, 1 << 28):
        hi = min(lo + (1 << 28), n)
        mask[lo:hi] = x[lo:hi] > -0.3
    ops.fq_pow2_fwd(x, 4.0, (1, 1, n), mask=mask, out=y)
    for s in spots:
        sl = slice(s, min(s + 4096, n))
        assert torch.equal(y[sl], ref_q(x[sl] * mask[sl])), s
    _, gx = ops.ste_bwd(x, 4.0, True, 8, 0, (1, 1, n), mask=mask, clamp_in_place=False, want_gx=True)
    for s in spots:
        sl = slice(s, min(s + 4096, n))
        want = torch.clamp(x[sl], -128 / 16.0, 127 / 16.0) * mask[sl]
        assert torch.equal(gx[sl], want), s
    del gx, mask
    # reductions: per tensor and per channel ([4, C = 8, inner]) over the whole 4G range
    st = ops.reduce_stats(x, (1, 1, n), absmax=True)
    assert st["absmax"].item() == 77.25
    inner = n // 32
    st = ops.reduce_stats(x[: 32 * inner], (4, 8, inner), absmax=True, minmax=True)
    view = x[: 32 * inner].view(4, 8, inner)
    assert torch.equal(st["max"], view.amax(dim=(0, 2))) and torch.equal(st["min"], view.amin(dim=(0, 2)))
    # per-channel decimals through the window kernel
    dec = torch.arange(8, device="cuda", dtype=torch.float32)
    ops.fq_pow2_fwd(x[: 32 * inner], dec, (4, 8, inner), out=y[: 32 * inner])
    yv = y[: 32 * inner].view(4, 8, inner)
    for o, c in ((0, 0), (1, 7), (3, 7), (2, 3)):
        d = float(c)
        seg = view[o, c, -2048:]
        assert torch.equal(yv[o, c, -2048:], (seg * 2.0 ** d).int().float() * 2.0 ** -d), (o, c)


def test_kth_value_batched_matches_single_and_sort():
    """several selects in one launch sequence (weight-set layers): mixed sizes (generic and sampled routes),
    an unaligned view, heavy ties, k at both ends."""
    from qsparse_b200 import ops
    g = torch.Generator(device="cuda").manual_seed(8)
    sizes = [2_359_296, 131_072, 100, 4097, 1 << 20, 300_001, 2_359_296, 65_536 * 3]
    vs = [torch.randn(s, device="cuda", generator=g) * 0.02 for s in sizes]
    vs[4] = torch.relu(vs[4])                       # half zeros
    vs[5] = torch.randn(300_002, device="cuda", generator=g)[1:]   # 4-byte aligned only
    vs[6] = torch.round(vs[6] * 512) / 512          # a coarse grid: heavy ties everywhere
    for frac in (0.5, 0.0, 0.999999, 0.75):
        ks = [min(int(frac * v.numel()), v.numel() - 1) for v in vs]
        for take_abs in (False, True):
            thr = ops.kth_value_batched(vs, ks, take_abs=take_abs)
            for i, (v, k) in enumerate(zip(vs, ks)):
                ref = torch.sort(v.abs() if take_abs else v).values[k]
                assert thr[i].item() == ref.item(), (frac, take_abs, i)
                assert ops.kth_value(v, k, take_abs=take_abs).item() == ref.item(), (frac, take_abs, i, "single")
    # more segments than one launch sequence holds
    many = [torch.randn(150_000 + 1000 * i, device="cuda", generator=g) for i in range(45)]
    ks = [m.numel() // 3 for m in many]
    thr = ops.kth_value_batched(many, ks)
    for i, (m, k) in enumerate(zip(many, ks)):
        assert thr[i].item() == torch.sort(m).values[k].item(), i


def test_multi_tensor_ema_and_mask_equal_single_tensor_calls():
    """one launch over a weight set == one launch per tensor (sizes with vector tails, a tile-multiple size,
    more tensors than one table holds; an unaligned tensor sends the whole call down the per-tensor path)."""
    from qsparse_b200 import ops
    g = torch.Generator(device="cuda").manual_seed(21)
    sizes = [455, 4096, 8192 + 3, 100_000, 7] + [1000 + 37 * i for i in range(50)]
    for unaligned in (False, True):
        xs = [torch.randn(s, device="cuda", generator=g) for s in sizes]
        if unaligned:
            xs[2] = torch.randn(sizes[2] + 1, device="cuda", generator=g)[1:]
        mags_a = [torch.rand(s, device="cuda", generator=g) for s in sizes]
        mags_b = [m.clone() for m in mags_a]
        ops.magnitude_ema_full_multi_(mags_a, xs, 3)
        for m, x in zip(mags_b, xs):
            ops.magnitude_ema_full_(m, x.contiguous(), 3)
        for a, b in zip(mags_a, mags_b):
            assert torch.equal(a, b)
        thr = torch.rand(len(sizes), device="cuda", generator=g) * 0.5
        masks_a = [torch.ones(s, dtype=torch.bool, device="cuda") for s in sizes]
        masks_b = [torch.ones(s, dtype=torch.bool, device="cuda") for s in sizes]
        outs_a = [torch.full((s,), 9.0, device="cuda") for s in sizes]
        ops.mask_build_apply_multi(mags_a, thr, xs, masks_a, outs_a)
        for i, (m, x, mk) in enumerate(zip(mags_b, xs, masks_b)):
            y = ops.mask_build_apply(m, thr[i:i + 1], x.contiguous(), mk)
            assert torch.equal(mk, masks_a[i]) and torch.equal(y, outs_a[i]), i
            assert torch.equal(mk, m >= thr[i])


# ----------------------------------------------------------------------------- integer export (SURVEY 8 f-3)
@pytest.mark.parametrize("shape,ci", [((4, 6, 7, 7), 1), ((16, 40), 0), ((3, 5, 33), 2), ((2, 3, 1000), -1)])
def test_quant_export_int8_codes_and_dequant(shape, ci):
    """codes == the numpy restatement of the reference's integer step; dequantised codes == the fake-quant
    output wherever the value is inside the bits-bit range; saturation outside."""
    from qsparse_b200 import ops
    from qsparse_b200.quantize import quantize_with_decimal, quantize_with_scaler, quantize_with_line
    bits = 6
    x = rnd(shape, 31, 1.5)
    C = shape[ci] if ci >= 0 else 1
    rng = np.random.default_rng(7)
    dec = rng.integers(2, 5, C).astype(np.float32)
    sc = rng.uniform(0.02, 0.2, C).astype(np.float32)
    lines = np.stack([rng.uniform(-2, -0.1, C), rng.uniform(0.1, 2, C)], 1).astype(np.float32)
    layout = (1, 1, x.size) if ci < 0 else tuple(orc.layout(shape, ci))
    bshape = [1] * len(shape)
    if ci >= 0:
        bshape[ci] = C
    xc = cu(x)
    lo_q, hi_q = -(1 << (bits - 1)), (1 << (bits - 1)) - 1
    # decimal
    q = npy(ops.quant_export_int8(xc, ops.EXPORT_DECIMAL, cu(dec), bits, layout))
    raw = np.trunc(x * np.float32(2.0) ** dec.reshape(bshape)).astype(np.int64)
    assert q.dtype == np.int8 and np.array_equal(q, np.clip(raw, lo_q, hi_q))
    inside = (raw >= lo_q) & (raw <= hi_q)
    fq = npy(quantize_with_decimal(xc, bits, cu(dec) if ci >= 0 else float(dec[0]), ci))
    deq = q.astype(np.float32) * np.float32(2.0) ** -dec.reshape(bshape)
    assert bits_equal(np.where(inside, deq, 0), np.where(inside, fq + np.float32(0), 0))
    assert inside.mean() < 1.0                                   # the saturation branch is exercised
    # scaler
    q = npy(ops.quant_export_int8(xc, ops.EXPORT_SCALER, cu(sc), bits, layout))
    raw = np.rint(x / sc.reshape(bshape)).astype(np.int64)
    assert np.array_equal(q, np.clip(raw, lo_q, hi_q))
    inside = (raw >= lo_q) & (raw <= hi_q)
    fq = npy(quantize_with_scaler(xc, bits, cu(sc) if ci >= 0 else float(sc[0]), ci))
    deq = q.astype(np.float32) * sc.reshape(bshape)
    assert bits_equal(np.where(inside, deq, 0), np.where(inside, fq + np.float32(0), 0))
    # line (float zero point): every code is in range by construction
    q = npy(ops.quant_export_int8(xc, ops.EXPORT_LINE, cu(lines), bits, layout))
    assert q.dtype == np.uint8 and q.max() <= (1 << bits) - 1
    lo, hi = lines[:, 0].reshape(bshape), lines[:, 1].reshape(bshape)
    step = (hi - lo) / np.float32(1 << bits)
    fq = npy(quantize_with_line(xc, bits, cu(lines), ci if ci >= 0 else -1, False, True))
    assert bits_equal(q.astype(np.float32) * step + lo, fq)


def test_export_integer_from_layers():
    import qsparse_b200 as q
    from qsparse_b200.quantize import export_integer
    x = cu(rnd((4, 10, 12, 12), 5, 0.5))
    for cb, key in ((q.DecimalQuantizer(), "decimal"), (q.ScalerQuantizer(), "scale"), (q.AdaptiveQuantizer(), "lines")):
        layer = q.quantize(bits=8, timeout=2, channelwise=1 if key == "lines" else -1, callback=cb)
        for _ in range(4):
            y = layer(x)
        out = export_integer(layer, x)
        if key == "decimal":
            deq = out["q"].float() * 2.0 ** -out["decimal"]
        elif key == "scale":
            deq = out["q"].float() * out["scale"]
        else:
            lo, hi = out["lines"][:, 0].view(1, -1, 1, 1), out["lines"][:, 1].view(1, -1, 1, 1)
            deq = out["q"].float() * ((hi - lo) / 256.0) + lo
        assert torch.equal(deq + 0.0, y + 0.0), key


@pytest.mark.parametrize("shape,ci,off", [((4, 6, 7, 7), 1, 0), ((16, 40), 0, 0), ((3, 5, 33), 2, 1), ((2, 3, 1001), -1, 0),
                                          ((7, 11, 1), 1, 3), ((64, 96, 14, 14), 1, 0)])
def test_quant_export_int4_packed(shape, ci, off):
    """two codes per byte == the low 4 bits of the int8 export of the same tensor at bits=4 (every layout incl.
    odd element counts, unaligned input, channel-last), and the layer-level pack / unpack round trip."""
    from qsparse_b200 import ops
    bits = 4
    n = int(np.prod(shape))
    base = rnd((n + off,), 33, 1.5)
    x = base[off:].reshape(shape)
    xc = cu(base)[off:].view(shape)
    C = shape[ci] if ci >= 0 else 1
    rng = np.random.default_rng(9)
    dec = rng.integers(0, 3, C).astype(np.float32)
    sc = rng.uniform(0.1, 0.5, C).astype(np.float32)
    lines = np.stack([rng.uniform(-2, -0.1, C), rng.uniform(0.1, 2, C)], 1).astype(np.float32)
    layout = (1, 1, x.size) if ci < 0 else tuple(orc.layout(shape, ci))
    for kind, param in ((ops.EXPORT_DECIMAL, dec), (ops.EXPORT_SCALER, sc), (ops.EXPORT_LINE, lines)):
        q8 = npy(ops.quant_export_int8(xc, kind, cu(param), bits, layout)).reshape(-1)
        q4 = npy(ops.quant_export_int8(xc, kind, cu(param), bits, layout, pack4=True))
        assert q4.dtype == np.uint8 and q4.shape == ((n + 1) // 2,)
        nib = np.stack([q4 & 0xF, q4 >> 4], 1).reshape(-1)
        assert np.array_equal(nib[:n], q8.view(np.uint8) & 0xF), kind
        assert n % 2 == 0 or nib[n] == 0
    # host scalars instead of device parameters
    q8 = npy(ops.quant_export_int8(xc, ops.EXPORT_SCALER, 0.3, bits, (1, 1, n))).reshape(-1)
    q4 = npy(ops.quant_export_int8(xc, ops.EXPORT_SCALER, 0.3, bits, (1, 1, n), pack4=True))
    assert np.array_equal(np.stack([q4 & 0xF, q4 >> 4], 1).reshape(-1)[:n], q8.view(np.uint8) & 0xF)


def test_export_integer_pack4_round_trip():
    import qsparse_b200 as q
    from qsparse_b200.quantize import export_integer, unpack_int4
    x = cu(rnd((4, 10, 12, 12), 5, 0.5))
    for cb in (q.DecimalQuantizer(), q.ScalerQuantizer(), q.AdaptiveQuantizer()):
        # channel-wise Decimal / Scaler estimation on a batch is the reference's crash domain (SURVEY Q10)
        layer = q.quantize(bits=4, timeout=2, channelwise=1 if isinstance(cb, q.AdaptiveQuantizer) else -1,
                           callback=cb)
        for _ in range(4):
            layer(x)
        plain, packed = export_integer(layer, x), export_integer(layer, x, pack4=True)
        assert packed["packed"] and packed["q"].numel() == x.numel() // 2
        assert torch.equal(unpack_int4(packed), plain["q"]), type(cb).__name__
    with pytest.raises(AssertionError):
        export_integer(q.quantize(bits=8, timeout=0, callback=q.ScalerQuantizer()), x, pack4=True)


# ----------------------------------------------------------------------------- K9 fused unstructured prune step
def _step_reference(mags, xs, ks, t):
    """EMA -> k-th value -> mask -> apply with the separate kernels (each pinned to the oracle elsewhere)"""
    from qsparse_b200 import ops
    thr, masks, outs = [], [], []
    for m, x, k in zip(mags, xs, ks):
        ops.magnitude_ema_full_(m, x, t)
        th = ops.kth_value(m, k)
        mk = torch.empty(x.shape, dtype=torch.bool, device=x.device)
        outs.append(ops.mask_build_apply(m, th, x, mk))
        masks.append(mk)
        thr.append(th)
    return torch.cat(thr), masks, outs


@pytest.mark.parametrize("kind", ["normal", "half_zero_weights", "grid", "sorted", "with_nan", "constant"])
def test_prune_step_fused_equals_separate_kernels(kind):
    """K9 == magnitude_ema_full + kth_value + mask_build_apply, bit for bit (magnitudes, thresholds, masks,
    outputs) over several steps, for sizes on both routes (sampled / generic), vector tails, heavy ties at the
    threshold (zeros, a value grid, a constant tensor), adversarial order and NaNs."""
    from qsparse_b200 import ops
    g = torch.Generator(device="cuda").manual_seed(12)
    sizes = [2_359_296, 131_072 + 5, 300_007, 999, 1 << 20]
    xs = [torch.randn(s, device="cuda", generator=g) * 0.02 for s in sizes]
    if kind == "half_zero_weights":
        xs = [torch.relu(x) for x in xs]
    elif kind == "grid":
        xs = [torch.round(x * 256) / 256 for x in xs]
    elif kind == "sorted":
        xs = [torch.sort(x).values for x in xs]
    elif kind == "with_nan":
        for x in xs:
            x[::1009] = float("nan")
    elif kind == "constant":
        xs = [torch.full_like(x, 0.125) for x in xs]
    mags_a = [torch.rand(s, device="cuda", generator=g) * 0.01 for s in sizes]
    mags_b = [m.clone() for m in mags_a]
    masks_a = [torch.ones(s, dtype=torch.bool, device="cuda") for s in sizes]
    outs_a = [torch.full((s,), 7.0, device="cuda") for s in sizes]
    for step, frac in enumerate((0.5, 0.75, 0.001, 0.98)):
        ks = [min(max(int(frac * s), 0), s - 1) for s in sizes]
        assert ops.prune_step_supported(mags_a, xs, masks_a, outs_a)
        thr_a = ops.prune_unstructured_step_batched_(mags_a, xs, masks_a, outs_a, ks, step)
        thr_b, masks_b, outs_b = _step_reference(mags_b, xs, ks, step)
        for i in range(len(sizes)):
            assert torch.equal(mags_a[i].view(torch.int32), mags_b[i].view(torch.int32)), (kind, step, i, "mag")
            ta, tb = thr_a[i], thr_b[i]
            assert (ta == tb).item() or (torch.isnan(ta) and torch.isnan(tb)).item(), (kind, step, i, ta, tb)
            assert torch.equal(masks_a[i], masks_b[i]), (kind, step, i, "mask")
            assert torch.equal(outs_a[i].view(torch.int32), outs_b[i].view(torch.int32)), (kind, step, i, "out")


@pytest.mark.parametrize("cb_name", ["DecimalQuantizer", "ScalerQuantizer"])
def test_per_tensor_layer_fused_equals_unfused(cb_name):
    """QuantizeLayer(channelwise=-1): the 3-launch step (partials, one parameter kernel, quantize) gives the same
    outputs, scale, counters and input gradients as reduce -> EMA -> [decimal] -> quantize (5 launches)."""
    import importlib
    import qsparse_b200 as q
    qz = importlib.import_module("qsparse_b200.quantize")
    outs = {}
    for fuse in (True, False):
        qz.FUSE_ROW_QUANTIZE = fuse
        try:
            layer = q.quantize(bits=8, channelwise=-1, timeout=2, callback=getattr(qz, cb_name)())
            layer.train()
            rec = []
            for step in range(6):
                g = torch.Generator("cuda").manual_seed(step)
                x = (torch.randn(16, 24, 20, 20, device="cuda", generator=g) * (0.3 + 0.2 * step)).requires_grad_(True)
                y = layer(x)
                (y * torch.randn(y.shape, device="cuda", generator=g) * 40).sum().backward()
                rec.append((y.detach().clone(), x.grad.clone()))
            sd = {k: v.detach().clone() for k, v in layer.state_dict().items()}
            outs[fuse] = (rec, sd, layer.callback.t)
        finally:
            qz.FUSE_ROW_QUANTIZE = True
    (ra, sa, ta), (rb, sb, tb) = outs[True], outs[False]
    assert ta == tb and sa.keys() == sb.keys()
    for k in sa:
        assert torch.equal(sa[k], sb[k]), k
    for i, ((ya, ga), (yb, gb)) in enumerate(zip(ra, rb)):
        assert torch.equal(ya, yb) and torch.equal(ga, gb), i


def test_prune_step_fused_many_small_tensors_and_repeat():
    """more tensors than one launch sequence holds (all on the generic route: too small to sample), plus the
    same call repeated on the same workspace (no stale state between calls)."""
    from qsparse_b200 import ops
    g = torch.Generator(device="cuda").manual_seed(77)
    sizes = [1000 + 257 * i for i in range(40)] + [200_000]
    xs = [torch.randn(s, device="cuda", generator=g) for s in sizes]
    mags_a = [torch.zeros(s, device="cuda") for s in sizes]
    mags_b = [torch.zeros(s, device="cuda") for s in sizes]
    masks_a = [torch.ones(s, dtype=torch.bool, device="cuda") for s in sizes]
    outs_a = [torch.empty(s, device="cuda") for s in sizes]
    for step in range(3):
        ks = [s // 2 for s in sizes]
        thr_a = ops.prune_unstructured_step_batched_(mags_a, xs, masks_a, outs_a, ks, step)
        thr_b, masks_b, outs_b = _step_reference(mags_b, xs, ks, step)
        assert torch.equal(thr_a, thr_b), step
        for i in range(len(sizes)):
            assert torch.equal(mags_a[i], mags_b[i]) and torch.equal(masks_a[i], masks_b[i]), (step, i)
            assert torch.equal(outs_a[i].view(torch.int32), outs_b[i].view(torch.int32)), (step, i)


# ----------------------------------------------------------------------------- extensions (SURVEY 8 f-4, north_star "percentile")
@pytest.mark.parametrize("shape,ci", [((64, 3, 7, 7), -1), ((1 << 22,), -1), ((48, 1152), 0), ((5, 4096), 0)])
@pytest.mark.parametrize("pct", [99.9, 50.0, 100.0])
def test_percentile_quantizer_statistic_vs_numpy(shape, ci, pct):
    """PercentileQuantizer.optimize: scale = sorted(|x|)[k] / 2^(bits-1) with the running mean of the abs-max
    estimators, against a numpy restatement; percentile = 100 equals DecimalQuantizer bit for bit."""
    import qsparse_b200 as q
    bits = 6
    est = q.PercentileQuantizer(percentile=pct)
    ref_w = None
    dq = q.DecimalQuantizer()
    w = wd = None
    for t in range(3):
        x = rnd(shape, 700 + t) * (1 + 0.3 * t)
        w = est.optimize(cu(x), bits, w, channel_index=ci)
        rows = np.abs(x).reshape(1, -1) if ci < 0 else np.abs(x).reshape(shape[0], -1)
        k = q.PercentileQuantizer.rank(pct, rows.shape[1])
        stat = np.sort(rows, axis=1)[:, k].astype(np.float32)
        ref_w = orc.scale_ema(np.zeros_like(stat) if ref_w is None else ref_w, stat, bits, t)
        assert bits_equal(npy(w).reshape(-1), ref_w), (pct, t)
        if pct == 100.0:
            wd = dq.optimize(cu(x), bits, wd, channel_index=ci)
            assert bits_equal(npy(w), npy(wd))
    # through a layer: forward + backward run, scale is what the estimator produced
    layer = q.quantize(bits=bits, channelwise=ci, timeout=1, callback=q.PercentileQuantizer(percentile=pct,
                                                                                           use_float_scaler=True))
    layer.batch_dimension = -1
    layer.train()
    xt = cu(rnd(shape, 710)).requires_grad_(True)
    layer(xt)
    y = layer(xt)
    y.sum().backward()
    # (a [1, 1] scale broadcasts a 1-D input's result to [1, n], like the reference's `input * toi`)
    assert y.numel() == xt.numel() and bool(torch.isfinite(y).all()) and xt.grad is not None


@pytest.mark.parametrize("C,wsz,groups", [(64, 1, 4), (1000, 1, 7), (96, 2, 5), (8, 1, 8)])
def test_group_mean_equals_reference_loop(C, wsz, groups):
    """qsb_group_mean == the reference's per-group `grouped[member] = grouped[member].mean(dim=0)` loop
    (quantize.py:361-366) to <= 1 ulp (it is the correctly rounded mean), exact for groups of equal values"""
    from qsparse_b200 import ops
    rng = np.random.default_rng(C)
    vals = (np.abs(rng.standard_normal((C, wsz))) * 0.05 + 1e-3).astype(np.float32)
    labels = rng.integers(0, groups, C)
    labels[:groups] = np.arange(groups)
    got = npy(ops.group_mean(cu(vals), torch.from_numpy(labels).cuda(), groups))
    ref = vals.copy()
    ref64 = vals.astype(np.float64)
    for g in range(groups):
        m = labels == g
        ref[m] = torch.from_numpy(vals[m]).mean(dim=0).numpy()
        exact = ref64[m].mean(axis=0).astype(np.float32)
        assert bits_equal(got[m], np.broadcast_to(exact, got[m].shape))
    assert ulp_diff(got, ref).max() <= 1
    same = np.full((C, wsz), 0.125, np.float32)
    assert bits_equal(npy(ops.group_mean(cu(same), torch.from_numpy(labels).cuda(), groups)), same)


def test_groupwise_quantizer_uses_device_group_mean():
    """DecimalQuantizer(group_num=...) after its group timeout: decimals equal the reference loop's"""
    import qsparse_b200 as q
    cb = q.DecimalQuantizer(group_num=3, group_timeout=0)
    cb.t = 1
    x = cu(rnd((24, 40), 31))
    scaler = cu((np.abs(rnd((24, 1), 32)) * 0.02 + 1e-3))
    y = cb(x, 8, scaler, channel_index=0)
    labels = cb.groups.cpu().numpy()
    grouped = npy(scaler).copy()
    for g in range(3):
        grouped[labels == g] = grouped[labels == g].mean(axis=0)
    exp = orc.fq_pow2_fwd(npy(x), orc.scale_to_decimal(grouped.reshape(-1)), 0)
    assert bits_equal(npy(y), exp)


# ----------------------------------------------------------------------------- warm-started select (pivot hints)
@pytest.mark.parametrize("kind", ["normal_abs", "relu", "grid", "signed"])
def test_kth_value_with_pivot_hints_stays_exact(kind):
    """A loop that asks for the same order statistic of a slowly drifting tensor: with a hint the pivots come from
    the previous answer (no sampler) from the third call on.  Every answer must still equal torch.sort's, through
    slow drift, an abrupt change of the data (the bracket misses: generic route on the device, hint widens), heavy
    ties and a change of sign."""
    from qsparse_b200 import ops
    n = (1 << 22) + 40
    g = torch.Generator(device="cuda").manual_seed(17)
    base = torch.randn(n, device="cuda", generator=g) * 0.02
    noise = torch.randn(n, device="cuda", generator=g) * 0.02
    take_abs = kind == "normal_abs"
    hint = ops.new_select_hints(1, base.device)
    states = []
    for t in range(12):
        v = base + noise * (0.01 * t)                       # slow drift
        if t in (6, 7):
            v = v * 3.0 + 0.01                              # abrupt change: the hinted bracket misses
        if kind == "relu":
            v = torch.relu(v)
        elif kind == "grid":
            v = torch.round(v * 64) / 64                    # heavy ties on a quantisation grid
        for k in ((n // 2,) if t else (n // 2,)):
            got = ops.kth_value(v, k, take_abs=take_abs, hint=hint)
            ref = torch.sort(v.abs() if take_abs else v).values[k]
            assert got.item() == ref.item(), (kind, t, got.item(), ref.item())
        states.append(int(hint[0, 0].item()))
    assert states[0] == 1 and 2 in states, states            # the warm route was actually taken
    # extreme ranks and a fresh hint per rank
    v = base.abs()
    for k in (0, 1, n - 2, n - 1):
        h = ops.new_select_hints(1, base.device)
        ref = torch.sort(v).values[k].item()
        for _ in range(4):
            assert ops.kth_value(v, k, hint=h).item() == ref, k


def test_prune_step_with_pivot_hints_equals_unhinted():
    """K9 over a set of layers for 10 steps with warm-started pivots == the same steps with sampled pivots, bit for
    bit (magnitudes, thresholds, masks, outputs), including a step at which the weights change abruptly."""
    from qsparse_b200 import ops
    from qsparse_b200.util import kth_rank
    rng = np.random.default_rng(23)
    shapes = [(256, 256, 3, 3), (512, 1024), (300_007,), (64, 32, 3, 3)]
    ws = [cu((rng.standard_normal(s) * 0.02).astype(np.float32)) for s in shapes]

    def fresh():
        return ([torch.zeros_like(w) for w in ws], [torch.ones(w.shape, dtype=torch.bool, device="cuda") for w in ws],
                [torch.empty_like(w) for w in ws])

    (ma, ka, oa), (mb, kb, ob) = fresh(), fresh()
    hints = ops.new_select_hints(len(ws), ws[0].device)
    ks = [kth_rank(0.6, w.numel()) for w in ws]
    used = 0
    for t in range(10):
        if t == 6:
            ws = [w * 1.7 for w in ws]
        else:
            ws = [w * 1.003 for w in ws]
        ta = ops.prune_unstructured_step_batched_(ma, ws, ka, oa, ks, t)
        tb = ops.prune_unstructured_step_batched_(mb, ws, kb, ob, ks, t, hints=hints)
        assert torch.equal(ta, tb), t
        for i in range(len(ws)):
            assert torch.equal(ma[i], mb[i]) and torch.equal(ka[i], kb[i]) and torch.equal(oa[i], ob[i]), (t, i)
            ref = torch.sort(ma[i].reshape(-1)).values[ks[i]]
            assert tb[i].item() == ref.item(), (t, i)
        used += int((hints[:, 0] == 2).sum().item())
    assert used > 0


@pytest.mark.parametrize("lay", [(256, 64, 3136), (8, 16, 196), (4, 200, 81), (32, 48, 1), (64, 1000, 1), (3, 1, 5000),
                                 (1, 4096, 4096), (2100, 8, 255), (1, 1, 1 << 22), (40, 3000, 7)])
def test_reduce_stats_matches_torch(lay):
    """ops.reduce_stats (stage 1, then a finalize launch) against torch on the same x, four statistic sets: max / min /
    nnz / the tensor minimum exact, sum|x| to the means contract of DESIGN §2 (fp32 pre-sums of 8 values, then fp64:
    within ~1e-7 of the exact sum)"""
    from qsparse_b200 import ops
    n = lay[0] * lay[1] * lay[2]
    g = torch.Generator(device="cuda").manual_seed(n % 1000)
    x = torch.randn(n, device="cuda", generator=g).view(lay)
    x.view(-1)[::97] = 0.0
    dims = (0, 2)
    ref = {"absmax": x.abs().amax(dim=dims), "min": x.amin(dim=dims), "max": x.amax(dim=dims),
           "abssum": x.double().abs().sum(dim=dims), "nnz": (x != 0).sum(dim=dims).double(),
           "tensor_min": x.min().reshape(1)}
    for kw, keys in (({"absmax": True, "minmax": True, "abssum": True, "nnz": True}, set(ref)),
                     ({"minmax": True}, {"min", "max"}), ({"absmax": True}, {"absmax"}),
                     ({"abssum": True, "absmax": True}, {"abssum", "absmax"})):
        res = ops.reduce_stats(x, lay, **kw)
        assert set(res) == keys, kw
        for key in keys:
            assert res[key].dtype == ref[key].dtype, (kw, key)
            if key == "abssum":
                assert torch.allclose(res[key], ref[key], rtol=1e-6, atol=0), (kw, key)
            else:
                assert torch.equal(res[key], ref[key]), (kw, key)


def test_fuzz_vs_oracle():
    """A short seeded slice of benchmarks/fuzz_vs_oracle.py: random ranks / shapes / channel axes / parameters / special
    values / alignments through every functional entry point, plus stateful step and row-quant flows, bit for bit
    against the oracle (12 600 cases and 1 538 flows of the full tool: profiles/r02_fuzz_vs_oracle.txt)."""
    import importlib.util
    from pathlib import Path
    spec = importlib.util.spec_from_file_location(
        "fuzz_vs_oracle", Path(__file__).resolve().parent.parent / "benchmarks" / "fuzz_vs_oracle.py")
    fz = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(fz)
    rng = np.random.default_rng(2026)
    for case in range(80):
        fz.one_case(rng, case)
    done = 0
    for case in range(24):
        done += fz.step_flow_case(rng, case) is not None
        done += fz.row_quant_case(rng, case) is not None
    assert done >= 30


def test_device_step_counter_forms_equal_host_index_forms():
    """The CUDA-graph forms of the running means — `qsb_scale_ema_at`, `qsb_lines_ema_at`, `qsb_row_quant_fused_at`
    (plain and masked, three kinds) and `qsb_prune_unstructured_step_batched_at` (small and sampled-route tensors,
    with pivot hints) — read their step index from device memory and must equal the host-index forms bit for bit,
    at index 0 and later ones, with non-zero offsets as well."""
    from qsparse_b200 import ops
    from qsparse_b200.util import kth_rank
    rng = np.random.default_rng(77)
    dev = torch.device("cuda")
    for t in (0, 1, 2, 7, 1000):
        for off in (0, 3):
            ctr = torch.full((1,), t - off, dtype=torch.int64, device=dev)
            w = cu(rng.uniform(0.01, 1, 37).astype(np.float32))
            amax = cu(rng.uniform(0, 9, 37).astype(np.float32))
            a, b = w.clone(), w.clone()
            ops.scale_ema_(a, amax, 8, t)
            ops.scale_ema_(b, amax, 8, off, t_dev=ctr)
            assert torch.equal(a.view(torch.int32), b.view(torch.int32)), ("scale", t, off)
            if t >= 1:
                lines = cu(rng.standard_normal((37, 2)).astype(np.float32))
                mn, mx = cu(rng.standard_normal(37).astype(np.float32)), cu(rng.standard_normal(37).astype(np.float32))
                a, b = lines.clone(), lines.clone()
                ops.lines_ema_(a, mn, mx, t)
                ops.lines_ema_(b, mn, mx, off, t_dev=ctr)
                assert torch.equal(a.view(torch.int32), b.view(torch.int32)), ("lines", t, off)
            x = cu((rng.standard_normal((48, 256)) * 0.3).astype(np.float32))
            m = cu(rng.random((48, 256)) > 0.4)
            for kind, width in ((ops.ROW_DECIMAL, 1), (ops.ROW_SCALER, 1), (ops.ROW_LINE, 2)):
                if kind == ops.ROW_LINE and t < 1:
                    continue
                for mask in (None, m):
                    p0 = cu(rng.uniform(0.01, 1, (48, width)).astype(np.float32))
                    pa, pb = p0.clone(), p0.clone()
                    ya, da = ops.row_quant_fused_(x, pa, kind, 4, t, True, mask=mask)
                    yb, db = ops.row_quant_fused_(x, pb, kind, 4, off, True, mask=mask, t_dev=ctr)
                    assert torch.equal(pa.view(torch.int32), pb.view(torch.int32)), ("row param", kind, t, off)
                    assert torch.equal(ya.view(torch.int32), yb.view(torch.int32)), ("row y", kind, t, off)
                    if da is not None:
                        assert torch.equal(da, db)
    # K9 over several steps: a sampled-route tensor (>= 2^22 elements) and small ones, hints on both sides
    shapes = [(1 << 22) + 24, (512, 1024), (64, 32, 3, 3)]
    ws = [cu((rng.standard_normal(s) * 0.02).astype(np.float32)) for s in shapes]

    def fresh():
        return ([torch.zeros_like(w) for w in ws], [torch.ones(w.shape, dtype=torch.bool, device="cuda") for w in ws],
                [torch.empty_like(w) for w in ws], ops.new_select_hints(len(ws), dev))

    (ma, ka, oa, ha), (mb, kb, ob, hb) = fresh(), fresh()
    ks = [kth_rank(0.6, w.numel()) for w in ws]
    ctr = torch.zeros(1, dtype=torch.int64, device=dev)
    for t in range(6):
        ws = [w * 1.002 for w in ws]
        ta = ops.prune_unstructured_step_batched_(ma, ws, ka, oa, ks, t, hints=ha)
        tb = ops.prune_unstructured_step_batched_(mb, ws, kb, ob, ks, 0, hints=hb, t_dev=ctr)
        ctr.add_(1)
        assert torch.equal(ta, tb), t
        for i in range(len(ws)):
            assert torch.equal(ma[i].view(torch.int32), mb[i].view(torch.int32)), (t, i, "magnitude")
            assert torch.equal(ka[i], kb[i]) and torch.equal(oa[i].view(torch.int32), ob[i].view(torch.int32)), (t, i)
