"""The structured prune -> pow2 quantize training step against the CPU oracle, on every route it takes.

Which code runs depends on the shape (the reduction plan, ``make_plan`` in reduce.cu, for a 148-SM B200) and on the
channel count:

  one       C <= 1024, C * fin_count <= 12288   stage 1 whose last-arriving CTA runs the step (step_epilogue.cuh)
  three     C <= 1024, C * fin_count >  12288   stage 1 -> parallel finalize -> prune_quant_step_kernel
  partials  1024 < C <= 2048                    reduce_partials + prune_quant_step_kernel
  params    2048 < C <= 4096                    reduce_stats (stage 1 -> finalize) + prune_quant_step_kernel on rows
  composed  C > 4096                            reduce_stats + EMA / k-th value / mask / abs-max / scale launches

(ops.structured_prune_quant_step picks among one, partials, params and composed by C; the partials entry point
itself takes up to 4096 channels, and the table covers that too.)

Every case names the route and the stage-1 kernel it is meant to reach, and a profiler recording of one step checks
that it does, so a dispatch change fails here instead of leaving a route untested.  The reference is the oracle's
restatement of the unfused layers (squeeze_mean_abs -> magnitude EMA -> calculate_mask_given_importance ->
scale EMA of max(absmax * mask) -> decimal -> fake quantize / STE), run on the CPU.

The inputs are small integers times powers of two, so every sum of |x| is exact in either summation order: the
magnitudes then match bit for bit, and ties between channels are real ties on both sides.
"""
import re

import numpy as np
import pytest
import torch

from oracle import oracle as orc
from tests.conftest import bits_equal, ulp_diff

pytestmark = pytest.mark.gpu

BITS = 8
STEPS = 4


# ----------------------------------------------------------------------------- inputs
def _k(sparsity, c):
    return orc.kth_index(sparsity, c)


def sparsity_for_k(which, c):
    """a sparsity whose threshold rank is 1, about C / 2 or C - 1"""
    return {"k1": 1.0 / c, "half": 0.5, "kC-1": (c - 0.5) / c}[which]


def make_x(layout, pattern, seed, sparsity):
    """float32 [outer, C, inner] of the named pattern (exactly summable values)"""
    o, c, i = layout
    rng = np.random.default_rng(seed)
    chan = np.random.default_rng(1234 + c)   # which channels are dead / tied: the same at every step
    x = rng.integers(-15, 16, size=(o, c, i)).astype(np.float32)
    x *= (2.0 ** (rng.integers(-2, 3, size=c))).astype(np.float32).reshape(1, c, 1)
    k = _k(sparsity, c) if sparsity < 1 else c - 1
    if pattern == "dead":
        # dead ReLU channels: exact-zero magnitudes, enough of them that rank k falls inside the zero block
        z = min(c, k + 1 + max(1, (c - k - 1) // 2))
        x[:, chan.permutation(c)[:z], :] = 0.0
    elif pattern == "dup":
        # duplicated channels: blocks of equal magnitude (also after the EMA), rank k strictly inside a block
        b = max(2, c // 8)
        while b > 2 and k % b == 0:
            b -= 1
        level = (1 + chan.permutation(c) // b).astype(np.float32) * 0.25
        x = np.sign(rng.integers(0, 2, size=(o, c, i)) - 0.5).astype(np.float32) * level.reshape(1, c, 1)
    elif pattern == "nan":
        x.reshape(-1)[rng.integers(x.size)] = np.nan
    elif pattern == "inf":
        x.reshape(-1)[rng.integers(x.size)] = np.inf
    elif pattern == "zero":
        x[:] = 0.0
    else:
        assert pattern == "rand", pattern
    return x


def make_g(shape, seed):
    rng = np.random.default_rng(10_000 + seed)
    return (rng.standard_normal(shape) * 4).astype(np.float32)


def to_device(x_np, shape, dtype, offset):
    """the array as a CUDA tensor of ``dtype``; ``offset``: a view one element into a larger buffer"""
    flat = torch.from_numpy(x_np.reshape(-1)).to(dtype)
    if not offset:
        return flat.cuda().view(shape)
    base = torch.zeros(flat.numel() + 1, dtype=dtype)
    base[1:] = flat
    return base.cuda()[1:].view(shape)


def refresh_schedule(mode):
    # mode 1 (running average): no refresh at t = 0, then every step; mode 2 (raw mean): every other step
    return [t > 0 for t in range(STEPS)] if mode == 1 else [t % 2 == 0 for t in range(STEPS)]


# ----------------------------------------------------------------------------- reference
def oracle_steps(xs, gs, sparsity, mode, refresh, summed_mean=False):
    """T steps of the unfused reference on host copies [outer, C, inner] (fp32).

    summed_mean: take the step's mean |x| as the kernels define it, the fp64 sum over outer and inner divided once
    by the count and rounded to fp32.  The oracle takes the mean one dimension at a time and rounds in between; the
    two agree bit for bit when outer is a power of two or inner is 1, and stay within the kernels' documented 8 ulp
    otherwise (checked here)."""
    c = xs[0].shape[1]
    mag = np.zeros(c, np.float32)
    mask = np.ones(c, bool)
    scale = np.zeros(1, np.float32)
    out = []
    for t, (x, g) in enumerate(zip(xs, gs)):
        m = orc.squeeze_mean_abs(x, (1, c, 1)).reshape(-1)
        if summed_mean:
            with np.errstate(invalid="ignore"):
                ms = (np.abs(x.astype(np.float64)).sum(axis=(0, 2)) / (x.shape[0] * x.shape[2])).astype(np.float32)
            fin = np.isfinite(m)
            assert np.array_equal(fin, np.isfinite(ms)) and ulp_diff(ms[fin], m[fin]).max(initial=0) <= 8
            m = ms
        if mode == 1:
            mag = orc.magnitude_ema(mag, m, t)
            imp = mag
        else:
            imp = m
        if refresh[t]:
            mask, _ = orc.mask_given_importance(imp, sparsity)
        amax = orc.absmax(x, 1)
        with np.errstate(invalid="ignore"):
            kept = np.max(amax * mask)              # x * mask: inf * 0 and NaN * 0 are NaN
        scale = orc.scale_ema(scale, np.array([kept], np.float32), BITS, t)
        dec = orc.scale_to_decimal(scale)
        y = orc.fq_pow2_fwd(x, dec, 1, mask=mask)
        _, gx = orc.ste_bwd(g, dec, BITS, 1, True, False, mask=mask)
        with np.errstate(invalid="ignore"):
            abssum = np.abs(x.astype(np.float64)).sum(axis=(0, 2))
        out.append(dict(imp=imp.copy(), mask=mask.copy(), scale=scale.copy(), dec=dec.copy(), y=y, gx=gx,
                        abssum=abssum, absmax=amax))
    return out


# ----------------------------------------------------------------------------- kernel routes (through ops)
class State:
    def __init__(self, c):
        dev = "cuda"
        self.mag = torch.zeros(c, device=dev)
        self.mask = torch.ones(c, dtype=torch.bool, device=dev)
        self.scale = torch.zeros(1, device=dev)
        self.dec = torch.zeros(1, device=dev)
        self.abssum = torch.full((c,), -1.0, dtype=torch.float64, device=dev)
        self.absmax = torch.full((c,), -1.0, device=dev)
        self.counter = torch.zeros(1, dtype=torch.int64, device=dev)


def run_step(route, xd, layout, st, t, mode, refresh, k, counter=False, interval=1):
    from qsparse_b200 import ops
    o, c, i = layout
    count = float(o * i)
    if route in ("one", "three"):
        if counter:
            # graph form: the step index comes from a device counter; refresh_mask carries the interval
            ops.reduce_prune_quant_step(xd, layout, st.mag, st.mask, st.scale, st.dec, count, 0, mode, interval,
                                        k, BITS, 0, True, abssum_out=st.abssum, absmax_out=st.absmax,
                                        step_counter=st.counter)
        else:
            ops.reduce_prune_quant_step(xd, layout, st.mag, st.mask, st.scale, st.dec, count, t, mode, refresh, k,
                                        BITS, t, True, abssum_out=st.abssum, absmax_out=st.absmax)
    elif route == "partials":
        ws = ops.reduce_partials(xd, layout)
        ops.prune_quant_step_params(st.mag, st.mask, st.scale, st.dec, ws, layout, count, t, mode, refresh, k,
                                    BITS, t, True, abssum_out=st.abssum, absmax_out=st.absmax)
    else:
        stats = ops.reduce_stats(xd, layout, abssum=True, absmax=True)
        st.abssum.copy_(stats["abssum"])
        st.absmax.copy_(stats["absmax"])
        ops.prune_quant_params(st.mag, st.mask, st.scale, st.dec, stats, count, t, mode, refresh, k, BITS, t, True)


def kernel_step_outputs(route, xd, gd, layout, st, t, mode, refresh, k, **kw):
    from qsparse_b200 import ops
    run_step(route, xd, layout, st, t, mode, refresh, k, **kw)
    y = ops.fq_pow2_fwd(xd, st.dec, layout, mask=st.mask)
    _, gx = ops.ste_bwd(gd.clone(), st.dec, True, BITS, 0, layout, mask=st.mask, want_gx=True)
    return dict(imp=(st.mag if mode == 1 else None), mask=st.mask.clone(), scale=st.scale.clone(),
                dec=st.dec.clone(), y=y, gx=gx, abssum=st.abssum.clone(), absmax=st.absmax.clone())


def check_step(got, ref, what, stats=True):
    h = lambda t: t.detach().cpu().numpy()
    assert np.array_equal(h(got["mask"]).astype(bool), ref["mask"]), ("mask", what)
    assert bits_equal(h(got["scale"]).reshape(-1), ref["scale"]), ("scale", what, h(got["scale"]), ref["scale"])
    assert bits_equal(h(got["dec"]).reshape(-1), ref["dec"]), ("decimal", what, h(got["dec"]), ref["dec"])
    if got["imp"] is not None:
        # exactly summable inputs: the magnitudes are bit-exact (the kernels' documented bound is 8 ulp)
        assert bits_equal(h(got["imp"]), ref["imp"]), ("magnitude", what)
    if stats:
        np.testing.assert_allclose(h(got["abssum"]), ref["abssum"], rtol=3e-7, equal_nan=True, err_msg=str(what))
        assert bits_equal(h(got["absmax"]), ref["absmax"]), ("absmax", what)
    if np.isfinite(ref["dec"]).all():
        # an inf / NaN scale gives a decimal of -inf: 2^-d overflows, outside the quantizers' parity domain
        # (SURVEY Q5); the parameters above are still compared on those steps
        assert bits_equal(h(got["y"]).reshape(ref["y"].shape), ref["y"]), ("y", what)
        assert bits_equal(h(got["gx"].float()).reshape(ref["gx"].shape), ref["gx"]), ("gx", what)


# ----------------------------------------------------------------------------- route table
# (id, shape, layout, route, stage-1 kernel, dtype, offset view, patterns)
# patterns: (data pattern, which rank, update_magnitude)
TIES = [("dead", "half", 1), ("dup", "half", 2)]
FULL = TIES + [("rand", "half", 1), ("nan", "half", 2), ("inf", "half", 1), ("zero", "half", 1),
               ("rand", "k1", 2), ("rand", "kC-1", 1), ("dup", "kC-1", 2), ("dead", "k1", 1)]
F32, BF16, F16 = torch.float32, torch.bfloat16, torch.float16

CASES = [
    # stage 1: column mode, 4 columns per thread
    ("col4-64x48", (64, 48), (64, 48, 1), "one", "cols4", F32, False, FULL),
    ("col4-32x200x7x7", (32, 200, 7, 7), (32, 200, 49), "three", "cols4", F32, False, FULL),
    ("col4-16x64x14x14", (16, 64, 14, 14), (16, 64, 196), "three", "cols4", F32, False, TIES),
    # column mode, one column per thread: C * inner not a multiple of 4, or a view one element in
    ("col1-16x63x5", (16, 63, 5), (16, 63, 5), "one", "cols1", F32, False, FULL),
    ("col1-64x48-offset", (64, 48), (64, 48, 1), "one", "cols1", F32, True, TIES),
    # the three-launch form (wide column mode)
    ("three-4096x1000", (4096, 1000), (4096, 1000, 1), "three", "cols4", F32, False, TIES + [("nan", "half", 1)]),
    # row mode, 4 loads in flight
    ("rows4-8x128x28x28", (8, 128, 28, 28), (8, 128, 784), "one", "rows4", F32, False, FULL),
    ("rows4-inner323", (4, 32, 323), (4, 32, 323), "one", "rows4", F32, False, TIES + [("nan", "half", 1)]),
    # row mode, 8 loads in flight
    ("rows8-4x64x56x56", (4, 64, 56, 56), (4, 64, 3136), "one", "rows8", F32, False, FULL),
    ("rows8-inner2053", (2, 32, 2053), (2, 32, 2053), "one", "rows8", F32, False, TIES + [("inf", "half", 2)]),
    # 16-bit input, aligned and one element in (2-byte aligned: element loads / scalar columns)
    ("bf16-rows8", (4, 64, 56, 56), (4, 64, 3136), "one", "rows8", BF16, False, TIES + [("nan", "half", 1)]),
    ("bf16-rows8-offset", (4, 64, 56, 56), (4, 64, 3136), "one", "rows8-elem", BF16, True, TIES),
    ("bf16-rows4-offset", (4, 32, 323), (4, 32, 323), "one", "rows4-elem", BF16, True, TIES),
    ("bf16-col4", (64, 48), (64, 48, 1), "one", "cols4", BF16, False, TIES),
    ("bf16-col1-offset", (64, 48), (64, 48, 1), "one", "cols1", BF16, True, TIES),
    ("fp16-rows4", (8, 128, 28, 28), (8, 128, 784), "one", "rows4", F16, False, TIES + [("inf", "half", 2)]),
    ("fp16-rows4-offset", (8, 128, 28, 28), (8, 128, 784), "one", "rows4-elem", F16, True, TIES),
    ("fp16-rows8-offset", (2, 32, 2053), (2, 32, 2053), "one", "rows8-elem", F16, True, TIES),
    ("fp16-col4", (32, 200, 7, 7), (32, 200, 49), "three", "cols4", F16, False, TIES),
    ("fp16-col1-offset", (16, 64, 14, 14), (16, 64, 196), "three", "cols1", F16, True, TIES),
    ("f32-rows8-offset", (2, 32, 2053), (2, 32, 2053), "one", "rows8", F32, True, TIES),
    ("f32-rows4-offset", (4, 32, 323), (4, 32, 323), "one", "rows4", F32, True, TIES),
]
# channel counts at the steps of the tail's threads per channel (32 ... 1 at C = 9, 17, 33, 65, 129, 257) and at
# the route limits, as [16, C] with the channel last (column mode); the partials entry point up to its own limit
for _c, _route in [(2, "one"), (8, "one"), (9, "one"), (16, "one"), (17, "one"), (33, "one"), (65, "one"),
                   (129, "one"), (256, "one"), (257, "one"), (1000, "one"), (1024, "one"), (1025, "partials"),
                   (2048, "partials"), (2049, "params"), (4096, "params"), (2049, "partials"), (4096, "partials")]:
    _id = f"C{_c}-{_route}" if _c > 2048 else f"C{_c}"     # above 2048 channels both routes are covered
    CASES.append((_id, (16, _c), (16, _c, 1), _route, "cols4" if _c % 4 == 0 else "cols1", F32, False,
                  FULL if _c in (9, 257, 1024, 1025, 2049, 4096) else TIES))
# more channels than the fused tail holds, in row mode (the partials / params routes read row-mode partials too)
CASES += [
    ("C1025-rows4", (2, 1025, 320), (2, 1025, 320), "partials", "rows4", F32, False, TIES),
    ("C2049-rows4-params", (2, 2049, 320), (2, 2049, 320), "params", "rows4", F32, False, TIES),
    ("C2048-bf16-offset", (16, 2048), (16, 2048, 1), "partials", "cols1", BF16, True, TIES),
]

STAGE1 = {
    "cols4": r"reduce_cols_kernel<\d+, 4, ",
    "cols1": r"reduce_cols_kernel<\d+, 1, ",
    "rows4": r"reduce_rows_kernel<\d+, 4, 4, [^>]*, (float|__half|__nv_half|__nv_bfloat16), true>",
    "rows8": r"reduce_rows_kernel<\d+, 8, 2, [^>]*, (float|__half|__nv_half|__nv_bfloat16), true>",
    "rows4-elem": r"reduce_rows_kernel<\d+, 4, 4, [^>]*, false>",
    "rows8-elem": r"reduce_rows_kernel<\d+, 8, 2, [^>]*, false>",
}
# the kernels of one step call beyond stage 1, and the total launch count
ROUTE_KERNELS = {
    "one": ([r"StepTail"], 1),
    "three": ([r"prune_quant_step_kernel", r"reduce_finalize"], 3),
    "partials": ([r"prune_quant_step_kernel"], 2),
    "params": ([r"prune_quant_step_kernel", r"reduce_finalize"], 3),
}


def recorded_kernels(fn):
    """names of the CUDA kernels of the qsb namespace that ``fn`` launches (torch.profiler, CUDA activity)"""
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    names = []
    for e in prof.events():
        if e.device_type == torch.autograd.DeviceType.CUDA and "qsb::" in e.name:
            names.append(e.name)
    return names


def check_route(route, stage1, names, what):
    assert names, ("no kernel recorded", what)
    extra, launches = ROUTE_KERNELS[route]
    assert len(names) == launches, (what, names)
    assert any(re.search(STAGE1[stage1], n) for n in names), (what, stage1, names)
    for pat in extra:
        assert any(re.search(pat, n) for n in names), (what, pat, names)
    if route == "one":
        assert not any("prune_quant_step_kernel" in n for n in names), (what, names)
    if route == "partials":
        assert not any("reduce_finalize" in n for n in names), (what, names)


@pytest.mark.parametrize("case", CASES, ids=[c[0] for c in CASES])
def test_step_route_matches_oracle(case):
    from qsparse_b200 import ops
    cid, shape, layout, route, stage1, dtype, offset, patterns = case
    c = layout[1]
    # the route: record one step (after a warm-up call that creates the arrival counter and loads modules)
    xw = to_device(make_x(layout, "rand", 99, 0.5), shape, dtype, offset)
    assert (xw.data_ptr() % 16 != 0) == offset
    run_step(route, xw, layout, State(c), 1, 1, True, _k(0.5, c))
    names = recorded_kernels(lambda: run_step(route, xw, layout, State(c), 1, 1, True, _k(0.5, c)))
    check_route(route, stage1, names, cid)

    for p_i, (pattern, which, mode) in enumerate(patterns):
        sparsity = sparsity_for_k(which, c)
        k = _k(sparsity, c)
        refresh = refresh_schedule(mode)
        xs = [make_x(layout, pattern if t > 0 or pattern not in ("nan", "inf") else "rand", 7 * p_i + t, sparsity)
              for t in range(STEPS)]
        gs = [make_g(layout, 7 * p_i + t) for t in range(STEPS)]
        xds = [to_device(x, shape, dtype, offset) for x in xs]
        ref = oracle_steps([xd.float().cpu().numpy().reshape(layout) for xd in xds], gs, sparsity, mode, refresh)
        st = State(c)
        st_ctr = State(c) if route in ("one", "three") else None
        interval = 1 if mode == 1 else 2
        for t in range(STEPS):
            gd = torch.from_numpy(gs[t]).cuda()
            what = (cid, pattern, which, mode, t)
            got = kernel_step_outputs(route, xds[t], gd, layout, st, t, mode, refresh[t], k)
            check_step(got, ref[t], what)
            assert int(ops.arrival_counter(xds[t].device).abs().sum()) == 0, what
            if st_ctr is not None:
                # the device-step-counter form equals the host-index form bit for bit
                got_c = kernel_step_outputs(route, xds[t], gd, layout, st_ctr, t, mode, refresh[t], k, counter=True,
                                            interval=interval)
                for key in ("mask", "scale", "dec", "y", "gx", "abssum", "absmax"):
                    assert torch.equal(got[key].view(-1).cpu().view(torch.uint8),
                                       got_c[key].view(-1).cpu().view(torch.uint8)), (key, what)
                assert torch.equal(st.mag.cpu().view(torch.int32), st_ctr.mag.cpu().view(torch.int32)), what
                assert int(st_ctr.counter.item()) == t + 1, what


@pytest.mark.parametrize("route,layout", [("one", (16, 64, 1)), ("three", (512, 256, 1)), ("partials", (16, 1025, 1)),
                                          ("params", (16, 2049, 1)), ("params", (16, 4097, 1))])
def test_sparsity_one_is_rejected_without_writing(route, layout):
    """k = C (sparsity 1.0): the reference raises IndexError; the kernels return QSB_E_BADARG and write no mask"""
    o, c, i = layout
    xd = to_device(make_x(layout, "rand", 3, 0.5), (o, c * i), torch.float32, False)
    st = State(c)
    st.mask.copy_(torch.arange(c, device="cuda") % 3 == 0)
    before = st.mask.clone()
    with pytest.raises(RuntimeError, match="bad argument"):
        run_step(route, xd, layout, st, 1, 1, True, c)
    torch.cuda.synchronize()
    assert torch.equal(st.mask, before)
    with pytest.raises(IndexError):
        orc.mask_given_importance(np.arange(c, dtype=np.float32), 1.0)


@pytest.mark.parametrize("c", [64, 2049, 4096, 4097])
def test_params_takes_no_statistics_it_does_not_use(c):
    """prune_quant_params with the magnitude kept (update_magnitude 0) takes no abssum and any count, and without a
    scale update no absmax: the mask then comes from the stored magnitude (ties included), the scale stays"""
    from qsparse_b200 import ops
    st = State(c)
    mag = np.abs(make_x((1, c, 1), "dup", 5, 0.5).reshape(-1))
    st.mag.copy_(torch.from_numpy(mag))
    st.scale.fill_(3.0)
    k = _k(0.5, c)
    ops.prune_quant_params(st.mag, st.mask, st.scale, st.dec, {}, 0.0, 1, 0, True, k, BITS, 1, False)
    mask, _ = orc.mask_given_importance(mag, 0.5)
    scale = np.array([3.0], np.float32)
    assert np.array_equal(st.mask.cpu().numpy(), mask.astype(bool))
    assert bits_equal(st.mag.cpu().numpy(), mag)
    assert bits_equal(st.scale.cpu().numpy(), scale)
    assert bits_equal(st.dec.cpu().numpy(), orc.scale_to_decimal(scale))
    # the scale update on the stored mask, from absmax alone
    amax = np.abs(make_x((1, c, 1), "rand", 6, 0.5).reshape(-1))
    ops.prune_quant_params(st.mag, st.mask, st.scale, st.dec, {"absmax": torch.from_numpy(amax).cuda()}, 0.0, 1, 0,
                           False, k, BITS, 1, True)
    scale = orc.scale_ema(scale, np.array([np.max(amax * mask)], np.float32), BITS, 1)
    assert np.array_equal(st.mask.cpu().numpy(), mask.astype(bool))
    assert bits_equal(st.scale.cpu().numpy(), scale)
    assert bits_equal(st.dec.cpu().numpy(), orc.scale_to_decimal(scale))


# ----------------------------------------------------------------------------- module level
MODULE_CHANNELS = [64, 1024, 1025, 2048, 2049, 4096, 4097, 8192]


@pytest.mark.parametrize("c", MODULE_CHANNELS)
def test_prune_quantize_module_matches_oracle(c):
    """fused.PruneQuantize on [512, C] (channels last), 4 training steps, forward and backward, at and across
    every channel limit of its routes"""
    from qsparse_b200.fused import PruneQuantize
    layout = (512, c, 1)
    sparsity = 0.5
    m = PruneQuantize(sparsity, BITS, channel_index=1).cuda().train()
    patterns = ["rand", "dup", "nan" if c in (64, 4097, 8192) else "dead", "rand"]
    xs = [make_x(layout, patterns[t] if t > 0 else "rand", 100 + t, sparsity) for t in range(STEPS)]
    gs = [make_g(layout, 100 + t) for t in range(STEPS)]
    ref = oracle_steps(xs, gs, sparsity, 1, refresh_schedule(1))
    for t in range(STEPS):
        x = torch.from_numpy(xs[t].reshape(512, c)).cuda().requires_grad_(True)
        y = m(x)
        y.backward(torch.from_numpy(gs[t].reshape(512, c)).cuda())
        got = dict(imp=m.magnitude.data, mask=m.mask.data, scale=m.scale.data, dec=m.decimal, y=y.detach(),
                   gx=x.grad)
        check_step(got, ref[t], (c, t), stats=False)
    assert m.t_prune == STEPS


@pytest.mark.parametrize("c", [64, 4097])
def test_prune_quantize_sparsity_one_raises_index_error(c):
    from qsparse_b200.fused import PruneQuantize
    m = PruneQuantize(1.0, BITS, channel_index=1).cuda().train()
    x = torch.from_numpy(make_x((32, c, 1), "rand", 0, 0.5).reshape(32, c)).cuda()
    m(x)                                   # step 0 has no refresh
    before = m.mask.data.clone()
    with pytest.raises(IndexError):
        m(x)
    assert torch.equal(m.mask.data, before) and m.t_prune == 1


def _site(fuse):
    import torch.nn as nn

    from qsparse_b200 import DecimalQuantizer, fuse_prune_quantize, prune, quantize
    site = nn.Sequential(nn.Sequential(nn.Identity(), prune(sparsity=0.5, dimensions={1}, start=1, interval=1,
                                                            repetition=1)),
                         quantize(bits=BITS, channelwise=-1, timeout=1, callback=DecimalQuantizer())).cuda()
    return fuse_prune_quantize(site) if fuse else site


@pytest.mark.parametrize("c", MODULE_CHANNELS)
def test_fused_site_equals_unfused(c):
    """a converted prune -> quantize site with the fusion pass against the same site with fusion off
    (no fusion pass, the callback's own fused step off): outputs, gradients and all state bit for bit"""
    import importlib
    sp = importlib.import_module("qsparse_b200.sparse")
    from qsparse_b200.fused import FusedPruneQuantSequential
    layout = (512, c, 1)
    xs = [make_x(layout, ["rand", "dup", "dead", "rand", "nan", "rand"][t], 200 + t, 0.5) for t in range(6)]
    res = {}
    for fuse in (True, False):
        sp.FUSE_PRUNE_STEP = fuse
        try:
            site = _site(fuse).train()
            rec = []
            for t, xn in enumerate(xs):
                x = torch.from_numpy(xn.reshape(512, c)).cuda().requires_grad_(True)
                y = site(x)
                y.backward(torch.from_numpy(make_g(layout, t).reshape(512, c)).cuda())
                rec.append([y.detach().clone(), x.grad.clone()] + [v.clone() for v in site.state_dict().values()])
            res[fuse] = rec
            if fuse:
                fused = sum(mm.fused_steps for mm in site.modules() if isinstance(mm, FusedPruneQuantSequential))
                assert (fused > 0) == (c <= 2048), (c, fused)
        finally:
            sp.FUSE_PRUNE_STEP = True
    for t, (a, b) in enumerate(zip(res[True], res[False])):
        assert len(a) == len(b)
        for i, (u, v) in enumerate(zip(a, b)):
            assert u.dtype == v.dtype and u.shape == v.shape, (c, t, i)
            assert torch.equal(u.contiguous().view(-1).cpu().view(torch.uint8),
                               v.contiguous().view(-1).cpu().view(torch.uint8)), (c, t, i)
