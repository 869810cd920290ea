"""The structured prune -> AdaptiveQuantizer (line) training step against the CPU oracle and against the unfused
layers, on every route it takes:

  one       C <= 1024, C * fin_count <= 12288   stage 1 (sum|x|, min / max x) whose last-arriving CTA runs the step
  three     C <= 1024, C * fin_count >  12288   stage 1 -> parallel finalize -> prune_quant_step_kernel<true>
  partials  1024 < C <= 2048                    reduce_line_partials + prune_quant_step_kernel<true>

The reference chains squeeze_mean_abs -> magnitude EMA -> calculate_mask_given_importance, then the (min, max) of
x * mask -> lines EMA (t from 1) -> line fake-quantize with the float zero point, and gx = g * mask.  The inputs are
small integers times powers of two (exact sums).  The oracle keeps the first of two equal zeros it meets, so its
lines are compared by value (+0 == -0); the bits of the lines are compared with the unfused GPU sequence
mask_apply -> reduce_stats(minmax) -> lines_ema_, which the fused and the unfused site alternate with.
"""
import copy
import re

import numpy as np
import pytest
import torch
import torch.nn as nn

from oracle import oracle as orc
from tests.conftest import bits_equal
from tests.test_gpu_prune_quant_step_routes import make_g, recorded_kernels, sparsity_for_k, to_device
from tests.test_gpu_prune_quant_step_routes import make_x as make_x_base

pytestmark = pytest.mark.gpu

BITS = 8
STEPS = 4
F32, BF16, F16 = torch.float32, torch.bfloat16, torch.float16


# ----------------------------------------------------------------------------- inputs
def make_x(layout, pattern, seed, sparsity):
    """the patterns of the pow2 route test, and four whose pruned channels have a fixed sign: all negative ("neg"),
    all positive ("pos"), only +0 / -0 ("pm0"), and a post-ReLU tensor whose pruned channels mix small positive
    values with -0 ("relu": the per-tensor min is then a zero of either sign)"""
    if pattern not in ("neg", "pos", "pm0", "relu"):
        return make_x_base(layout, pattern, seed, sparsity)
    o, c, i = layout
    rng = np.random.default_rng(seed)
    small = np.random.default_rng(4321 + c).permutation(c)[:orc.kth_index(sparsity, c)]   # pruned on a refresh
    x = rng.integers(1, 16, size=(o, c, i)).astype(np.float32)
    if pattern == "relu":
        x[rng.random(x.shape) < 0.2] = 0.0
    else:
        x *= np.where(rng.random(x.shape) < 0.5, -1.0, 1.0).astype(np.float32)
    s = rng.integers(1, 4, size=(o, len(small), i)).astype(np.float32) * 0.125
    if pattern == "neg":
        s = -s
    elif pattern == "pm0":
        s = np.where(rng.random(s.shape) < 0.5, np.float32(-0.0), np.float32(0.0)).astype(np.float32)
    elif pattern == "relu":
        s[rng.random(s.shape) < 0.3] = np.float32(-0.0)
    x[:, small, :] = s
    return x


def refresh_schedule(mode):
    return [t > 0 for t in range(STEPS)] if mode == 1 else [t % 2 == 0 for t in range(STEPS)]


# ----------------------------------------------------------------------------- reference
def oracle_line_steps(xs, gs, sparsity, mode, refresh, per_channel):
    c = xs[0].shape[1]
    mag = np.zeros(c, np.float32)
    mask = np.ones(c, bool)
    lines = np.zeros((c if per_channel else 1, 2), np.float32)
    out = []
    for t, (x, g) in enumerate(zip(xs, gs)):
        m = orc.squeeze_mean_abs(x, (1, c, 1)).reshape(-1)
        if mode == 1:
            mag = orc.magnitude_ema(mag, m, t)
            imp = mag
        else:
            imp = m
        if refresh[t]:
            mask, _ = orc.mask_given_importance(imp, sparsity)
        mn, mx = orc.minmax(orc.mask_apply(x, mask, 1), 1 if per_channel else -1)
        lines = orc.lines_ema(lines, mn, mx, t + 1)
        y = orc.fq_line_fwd(x, lines, BITS, 1, True, mask=mask)
        gx = orc.mask_apply(g, mask, 1)
        with np.errstate(invalid="ignore"):
            abssum = np.abs(x.astype(np.float64)).sum(axis=(0, 2))
        out.append(dict(imp=imp.copy(), mask=mask.copy(), lines=lines.copy(), y=y, gx=gx, abssum=abssum,
                        minmax=orc.minmax(x, 1)))
    return out


# ----------------------------------------------------------------------------- kernel routes (through ops)
class State:
    def __init__(self, c, n_lines):
        dev = "cuda"
        self.mag = torch.zeros(c, device=dev)
        self.mask = torch.ones(c, dtype=torch.bool, device=dev)
        self.lines = torch.zeros(n_lines, 2, device=dev)
        self.abssum = torch.full((c,), -1.0, dtype=torch.float64, device=dev)
        self.mn = torch.full((c,), -1.0, device=dev)
        self.mx = torch.full((c,), -1.0, device=dev)
        self.counter = torch.zeros(1, dtype=torch.int64, device=dev)


def run_step(route, xd, layout, st, t, mode, refresh, k, counter=False, interval=1):
    from qsparse_b200 import ops
    o, c, i = layout
    count = float(o * i)
    outs = dict(abssum_out=st.abssum, min_out=st.mn, max_out=st.mx)
    if route in ("one", "three"):
        if counter:
            # graph form: step index and call index from the device counter, refresh_mask carries the interval
            ops.reduce_prune_line_step(xd, layout, st.mag, st.mask, st.lines, count, 0, mode, interval, k, 1,
                                       step_counter=st.counter, **outs)
        else:
            ops.reduce_prune_line_step(xd, layout, st.mag, st.mask, st.lines, count, t, mode, refresh, k, t + 1,
                                       **outs)
    else:
        ws = ops.reduce_line_partials(xd, layout)
        if counter:
            ops.prune_line_step_params(st.mag, st.mask, st.lines, ws, layout, count, 0, mode, interval, k, 1,
                                       step_counter=st.counter, **outs)
        else:
            ops.prune_line_step_params(st.mag, st.mask, st.lines, ws, layout, count, t, mode, refresh, k, t + 1,
                                       **outs)


def kernel_step_outputs(route, xd, gd, layout, st, t, mode, refresh, k, **kw):
    from qsparse_b200 import ops
    run_step(route, xd, layout, st, t, mode, refresh, k, **kw)
    y = ops.fq_line_fwd(xd, st.lines, BITS, True, layout, mask=st.mask)
    gx = ops.mask_apply(gd, st.mask, layout, out_dtype=xd.dtype)
    return dict(imp=(st.mag if mode == 1 else None), mask=st.mask.clone(), lines=st.lines.clone(), y=y, gx=gx,
                abssum=st.abssum.clone(), mn=st.mn.clone(), mx=st.mx.clone())


def unfused_lines_(lines, xd, mask, layout, t):
    """the unfused AdaptiveQuantizer.optimize on the PruneLayer's fp32 output: bit for bit what the fused step
    must write"""
    from qsparse_b200 import ops
    xm = ops.mask_apply(xd, mask, layout, out_dtype=torch.float32)
    st = ops.reduce_stats(xm, layout if lines.shape[0] > 1 else (1, 1, xm.numel()), minmax=True)
    ops.lines_ema_(lines, st["min"], st["max"], t)


def check_step(got, ref, what, dtype=torch.float32):
    h = lambda t: t.detach().cpu().numpy()
    assert np.array_equal(h(got["mask"]).astype(bool), ref["mask"]), ("mask", what)
    if got["imp"] is not None:
        assert bits_equal(h(got["imp"]), ref["imp"]), ("magnitude", what)
    assert np.array_equal(h(got["lines"]), ref["lines"], equal_nan=True), ("lines", what, h(got["lines"]),
                                                                            ref["lines"])
    np.testing.assert_allclose(h(got["abssum"]), ref["abssum"], rtol=3e-7, equal_nan=True, err_msg=str(what))
    assert np.array_equal(h(got["mn"]), ref["minmax"][0], equal_nan=True), ("min", what)
    assert np.array_equal(h(got["mx"]), ref["minmax"][1], equal_nan=True), ("max", what)
    if np.isfinite(ref["lines"]).all():
        assert bits_equal(h(got["y"]).reshape(ref["y"].shape), ref["y"]), ("y", what)
    gx_ref = torch.from_numpy(ref["gx"]).to(dtype).float().numpy()      # written in x's dtype
    assert bits_equal(h(got["gx"].float()).reshape(ref["gx"].shape), gx_ref), ("gx", what)


# ----------------------------------------------------------------------------- route table
SIGNS = [("pm0", "half", 1), ("relu", "half", 2), ("neg", "half", 1), ("dead", "half", 1)]
FULL = SIGNS + [("dup", "half", 2), ("rand", "half", 1), ("nan", "half", 2), ("inf", "half", 1), ("zero", "half", 1),
                ("pos", "half", 2), ("rand", "k1", 2), ("rand", "kC-1", 1), ("dup", "kC-1", 2), ("relu", "k1", 1)]

CASES = [
    ("col4-64x48", (64, 48), (64, 48, 1), "one", "cols4", F32, False, FULL),
    ("col4-32x200x7x7", (32, 200, 7, 7), (32, 200, 49), "three", "cols4", F32, False, FULL),
    ("col1-16x63x5", (16, 63, 5), (16, 63, 5), "one", "cols1", F32, False, FULL),
    ("col1-64x48-offset", (64, 48), (64, 48, 1), "one", "cols1", F32, True, SIGNS),
    ("three-4096x1000", (4096, 1000), (4096, 1000, 1), "three", "cols4", F32, False, SIGNS + [("nan", "half", 1)]),
    ("rows4-8x128x28x28", (8, 128, 28, 28), (8, 128, 784), "one", "rows4", F32, False, FULL),
    ("rows4-inner323", (4, 32, 323), (4, 32, 323), "one", "rows4", F32, False, SIGNS),
    ("rows8-4x64x56x56", (4, 64, 56, 56), (4, 64, 3136), "one", "rows8", F32, False, FULL),
    ("rows8-inner2053", (2, 32, 2053), (2, 32, 2053), "one", "rows8", F32, False, SIGNS + [("inf", "half", 2)]),
    ("f32-rows8-offset", (2, 32, 2053), (2, 32, 2053), "one", "rows8", F32, True, SIGNS),
    ("bf16-rows8", (4, 64, 56, 56), (4, 64, 3136), "one", "rows8", BF16, False, SIGNS + [("nan", "half", 1)]),
    ("bf16-rows8-offset", (4, 64, 56, 56), (4, 64, 3136), "one", "rows8-elem", BF16, True, SIGNS),
    ("bf16-col4", (64, 48), (64, 48, 1), "one", "cols4", BF16, False, SIGNS),
    ("bf16-col1-offset", (64, 48), (64, 48, 1), "one", "cols1", BF16, True, SIGNS),
    ("fp16-rows4", (8, 128, 28, 28), (8, 128, 784), "one", "rows4", F16, False, SIGNS + [("inf", "half", 2)]),
    ("fp16-rows4-offset", (4, 32, 323), (4, 32, 323), "one", "rows4-elem", F16, True, SIGNS),
    ("fp16-col4", (32, 200, 7, 7), (32, 200, 49), "three", "cols4", F16, False, SIGNS),
    ("fp16-col1-offset", (16, 64, 14, 14), (16, 64, 196), "three", "cols1", F16, True, SIGNS),
]
for _c, _route in [(2, "one"), (9, "one"), (257, "one"), (1024, "one"), (1025, "partials"), (2048, "partials")]:
    CASES.append((f"C{_c}", (16, _c), (16, _c, 1), _route, "cols4" if _c % 4 == 0 else "cols1", F32, False,
                  FULL if _c in (9, 1024, 1025, 2048) else SIGNS))
CASES += [
    ("C1025-rows4", (2, 1025, 320), (2, 1025, 320), "partials", "rows4", F32, False, SIGNS),
    ("C2048-bf16-offset", (16, 2048), (16, 2048, 1), "partials", "cols1", BF16, True, SIGNS),
]

STAGE1 = {
    "cols4": r"reduce_cols_kernel<6, 4, ",
    "cols1": r"reduce_cols_kernel<6, 1, ",
    "rows4": r"reduce_rows_kernel<6, 4, 4, [^>]*, (float|__half|__nv_half|__nv_bfloat16), true>",
    "rows8": r"reduce_rows_kernel<6, 8, 2, [^>]*, (float|__half|__nv_half|__nv_bfloat16), true>",
    "rows4-elem": r"reduce_rows_kernel<6, 4, 4, [^>]*, false>",
    "rows8-elem": r"reduce_rows_kernel<6, 8, 2, [^>]*, false>",
}
ROUTE_KERNELS = {
    "one": ([r"StepTail"], 1),
    "three": ([r"prune_quant_step_kernel<true>", r"reduce_finalize"], 3),
    "partials": ([r"prune_quant_step_kernel<true>"], 2),
}


def check_route(route, stage1, names, what):
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
def test_line_step_route_matches_oracle(case):
    from qsparse_b200 import ops
    cid, shape, layout, route, stage1, dtype, offset, patterns = case
    c = layout[1]
    k0 = orc.kth_index(0.5, c)
    xw = to_device(make_x(layout, "rand", 99, 0.5), shape, dtype, offset)
    assert (xw.data_ptr() % 16 != 0) == offset
    run_step(route, xw, layout, State(c, c), 1, 1, True, k0)
    names = recorded_kernels(lambda: run_step(route, xw, layout, State(c, c), 1, 1, True, k0))
    check_route(route, stage1, names, cid)

    for p_i, (pattern, which, mode) in enumerate(patterns):
        sparsity = sparsity_for_k(which, c)
        k = orc.kth_index(sparsity, c)
        refresh = refresh_schedule(mode)
        xs = [make_x(layout, pattern if t > 0 or pattern not in ("nan", "inf") else "rand", 7 * p_i + t, sparsity)
              for t in range(STEPS)]
        gs = [make_g(layout, 7 * p_i + t) for t in range(STEPS)]
        xds = [to_device(x, shape, dtype, offset) for x in xs]
        xf = [xd.float().cpu().numpy().reshape(layout) for xd in xds]
        for per_channel in (False, True):
            n_lines = c if per_channel else 1
            ref = oracle_line_steps(xf, gs, sparsity, mode, refresh, per_channel)
            st, st_ctr = State(c, n_lines), State(c, n_lines)
            lines_unf = torch.zeros(n_lines, 2, device="cuda")
            interval = 1 if mode == 1 else 2
            for t in range(STEPS):
                gd = torch.from_numpy(gs[t]).cuda()
                what = (cid, pattern, which, mode, per_channel, t)
                got = kernel_step_outputs(route, xds[t], gd, layout, st, t, mode, refresh[t], k)
                check_step(got, ref[t], what, dtype)
                unfused_lines_(lines_unf, xds[t], st.mask, layout, t + 1)
                assert torch.equal(lines_unf.view(torch.int32), st.lines.view(torch.int32)), (
                    "lines vs unfused", what, lines_unf.cpu(), st.lines.cpu())
                assert int(ops.arrival_counter(xds[t].device).abs().sum()) == 0, what
                # the device-step-counter form equals the host-index form bit for bit
                got_c = kernel_step_outputs(route, xds[t], gd, layout, st_ctr, t, mode, refresh[t], k, counter=True,
                                            interval=interval)
                for key in ("mask", "lines", "y", "gx", "abssum", "mn", "mx"):
                    assert torch.equal(got[key].reshape(-1).cpu().view(torch.uint8),
                                       got_c[key].reshape(-1).cpu().view(torch.uint8)), (key, what)
                assert torch.equal(st.mag.cpu().view(torch.int32), st_ctr.mag.cpu().view(torch.int32)), what
                assert int(st_ctr.counter.item()) == t + 1, what


@pytest.mark.parametrize("route,layout", [("one", (16, 64, 1)), ("three", (512, 256, 1)), ("partials", (16, 1025, 1))])
def test_line_step_sparsity_one_is_rejected_without_writing(route, layout):
    o, c, i = layout
    xd = to_device(make_x(layout, "rand", 3, 0.5), (o, c * i), torch.float32, False)
    st = State(c, c)
    st.mask.copy_(torch.arange(c, device="cuda") % 3 == 0)
    before, lines = st.mask.clone(), st.lines.clone()
    with pytest.raises(RuntimeError, match="bad argument"):
        run_step(route, xd, layout, st, 1, 1, True, c)
    torch.cuda.synchronize()
    assert torch.equal(st.mask, before) and torch.equal(st.lines, lines)


def test_line_step_routes_by_channel_count():
    """one ladder for both forms: a device counter above 1024 channels is not capturable, above 2048 there is no
    line route"""
    from qsparse_b200 import graphs, ops
    for c, exc in [(1025, graphs.NotCapturable), (2049, graphs.NotCapturable)]:
        st = State(c, 1)
        x = torch.zeros(16, c, device="cuda")
        with pytest.raises(exc):
            ops.structured_prune_line_step(x, (16, c, 1), st.mag, st.mask, st.lines, 16.0, 0, 1, 1, 0, 1,
                                           step_counter=st.counter)
    st = State(2049, 1)
    with pytest.raises(ValueError):
        ops.structured_prune_line_step(torch.zeros(16, 2049, device="cuda"), (16, 2049, 1), st.mag, st.mask,
                                       st.lines, 16.0, 1, 1, True, 0, 1)


# ----------------------------------------------------------------------------- sites
def _line_model(c, channelwise, fuse, sparsity=0.5):
    from qsparse_b200 import AdaptiveQuantizer, fuse_prune_quantize, prune, quantize
    torch.manual_seed(c)
    site = nn.Sequential(nn.Sequential(nn.Identity(), prune(sparsity=sparsity, dimensions={1}, start=1, interval=1,
                                                            repetition=2)),
                         quantize(bits=BITS, channelwise=channelwise, timeout=2, callback=AdaptiveQuantizer()))
    model = nn.Sequential(nn.Linear(16, c), site).cuda()
    return fuse_prune_quantize(model) if fuse else model


def _bits(t):
    return t.detach().contiguous().view(-1).cpu().view(torch.uint8)


# training steps 0-5, an eval step, training steps 6-7: warm-up (prune n = 0), the sparsity ramp (n = 1, 2), the
# quantizer's timeout (its first estimate at step 2), then steady steps — fused from training step 3 on
SITE_STEPS = ["train"] * 6 + ["eval"] + ["train"] * 2
SITE_FUSED = 5


@pytest.mark.parametrize("autocast", [False, True], ids=["fp32", "bf16-autocast"])
@pytest.mark.parametrize("channelwise", [-1, 1], ids=["per-tensor", "per-channel"])
@pytest.mark.parametrize("c", [2, 64, 1024, 1025, 2048, 2049])
def test_line_site_equals_unfused(c, channelwise, autocast):
    from qsparse_b200.fused import FusedPruneQuantSequential
    rng = np.random.default_rng(c)
    xs = [torch.from_numpy(rng.integers(-8, 9, size=(64, 16)).astype(np.float32) * 0.25) for _ in SITE_STEPS]
    gs = [torch.from_numpy(rng.standard_normal((64, c)).astype(np.float32)) for _ in SITE_STEPS]
    res = {}
    for fuse in (True, False):
        model = _line_model(c, channelwise, fuse)
        opt = torch.optim.SGD(model.parameters(), lr=0.05)
        rec = []
        for kind, x, g in zip(SITE_STEPS, xs, gs):
            model.train(kind == "train")
            x = x.cuda().requires_grad_(True)
            g = g.cuda()
            g0 = g.clone()
            opt.zero_grad(set_to_none=True)
            with torch.autocast("cuda", dtype=torch.bfloat16, enabled=autocast):
                y = model(x)
            y.backward(g)
            assert torch.equal(_bits(g), _bits(g0)), "grad_output was written"
            if kind == "train":
                opt.step()
            rec.append([y.detach().clone(), x.grad.clone()] + [v.clone() for v in model.state_dict().values()])
        res[fuse] = rec
        if fuse:
            fused = sum(m.fused_steps for m in model.modules() if isinstance(m, FusedPruneQuantSequential))
            assert fused == (SITE_FUSED if c <= 2048 else 0), (c, fused)
    for t, (a, b) in enumerate(zip(res[True], res[False])):
        assert len(a) == len(b)
        for i, (u, v) in enumerate(zip(a, b)):
            assert u.dtype == v.dtype and u.shape == v.shape, (c, t, i)
            assert torch.equal(_bits(u), _bits(v)), (c, channelwise, autocast, t, i)


@pytest.mark.parametrize("channelwise", [-1, 1])
def test_line_site_sparsity_one_raises_index_error(channelwise):
    model = _line_model(64, channelwise, True)
    x = torch.randn(64, 16, device="cuda")
    for _ in range(4):
        model(x)
    p = model[1][0][1]
    p._cur_sparsity.data.fill_(1.0)
    p._s_mirror.wrote(p._cur_sparsity, 1.0)
    before, lines = p.mask.data.clone(), model[1][1].weight.data.clone()
    with pytest.raises(IndexError):
        model(x)
    assert torch.equal(p.mask.data, before) and torch.equal(model[1][1].weight.data, lines)


# ----------------------------------------------------------------------------- graph mode
class _Affine(nn.Module):
    """x * w + b per channel: elementwise, so its gradients are the same bits in a graph and eagerly"""

    def __init__(self, c):
        super().__init__()
        self.w = nn.Parameter(torch.linspace(0.5, 1.5, c).view(1, c, 1, 1))
        self.b = nn.Parameter(torch.linspace(-0.25, 0.25, c).view(1, c, 1, 1))

    def forward(self, x):
        return x * self.w + self.b


def _graph_net():
    from qsparse_b200 import AdaptiveQuantizer, fuse_prune_quantize, prune, quantize

    def site(channelwise):
        return nn.Sequential(nn.Sequential(nn.ReLU(), prune(sparsity=0.5, dimensions={1}, start=1, interval=1,
                                                            repetition=1)),
                             quantize(bits=BITS, channelwise=channelwise, timeout=1, callback=AdaptiveQuantizer()))
    net = nn.Sequential(_Affine(16), site(-1), _Affine(16), site(1)).cuda()
    return fuse_prune_quantize(net)


def test_line_sites_graphed_equal_eager():
    """a net with a per-tensor and a per-channel Adaptive site: 3 warm-up steps and 5 replays of the step captured
    by GraphedTrainStep equal 8 eager steps in every parameter, line, mask and magnitude and in the device and host
    counters; after sync_host() the next eager steps agree too"""
    from qsparse_b200 import graphs
    from qsparse_b200.fused import FusedPruneQuantSequential
    rng = np.random.default_rng(5)
    xs = [torch.from_numpy(rng.standard_normal((8, 16, 8, 8)).astype(np.float32)).cuda() for _ in range(10)]
    ys = [torch.from_numpy(rng.standard_normal((8, 16, 8, 8)).astype(np.float32)).cuda() for _ in range(10)]
    base = _graph_net().train()
    for i in range(4):                              # into the steady state, eagerly
        (base(xs[i]) * ys[i]).sum().backward()
    nets = [copy.deepcopy(base), copy.deepcopy(base)]
    opts = [torch.optim.SGD(n.parameters(), lr=0.01) for n in nets]
    sx, sy = xs[0].clone(), ys[0].clone()

    def step(net, opt):
        opt.zero_grad(set_to_none=True)
        loss = (net(sx) * sy).sum()
        loss.backward()
        opt.step()
        return loss.detach().clone()

    def counters(net):
        """host counters and mirrors, and the device counters they mirror"""
        from qsparse_b200.quantize import AdaptiveQuantizer, QuantizeLayer
        from qsparse_b200.sparse import MagnitudePruningCallback, PruneLayer
        out = []
        for m in net.modules():
            if isinstance(m, QuantizeLayer):
                out += [int(m._t_mirror.get(m._n_updates)), int(m._n_updates.item())]
            elif isinstance(m, PruneLayer):
                out += [int(m._n_mirror.get(m._n_updates)), int(m._n_updates.item())]
            elif isinstance(m, MagnitudePruningCallback):
                out += [int(m._t()), int(m.t.item())]
            elif isinstance(m, AdaptiveQuantizer):
                out += [graphs.host_index(m)]
            elif isinstance(m, FusedPruneQuantSequential):
                out += [m.fused_steps]
        return out

    # eager
    eager = []
    for i in range(4, 12):
        sx.copy_(xs[i % 10]); sy.copy_(ys[i % 10])
        eager.append(step(nets[1], opts[1]))
    # graphed: three warm-up steps on their own batches, then replays
    feed = iter(range(4, 7))

    class _Step:
        n = 0

        def __call__(self):
            self.n += 1
            if self.n <= 3:
                j = next(feed)
                sx.copy_(xs[j]); sy.copy_(ys[j])
            return step(nets[0], opts[0])
    gs = graphs.GraphedTrainStep(nets[0], _Step(), warmup=3)
    replayed = []
    for i in range(7, 12):
        sx.copy_(xs[i % 10]); sy.copy_(ys[i % 10])
        replayed.append(gs.replay().clone())
    gs.sync_host()
    assert torch.equal(_bits(torch.stack(eager[3:])), _bits(torch.stack(replayed)))
    sa, sb = nets[0].state_dict(), nets[1].state_dict()
    assert sorted(sa) == sorted(sb)
    bad = [k for k in sa if not torch.equal(_bits(sa[k]), _bits(sb[k]))]
    assert not bad, bad
    assert counters(nets[0]) == counters(nets[1])
    assert all(m.fused_steps > 0 for m in nets[0].modules() if isinstance(m, FusedPruneQuantSequential))
    # back to eager steps
    for net, opt in zip(nets, opts):
        for i in range(2):
            sx.copy_(xs[i]); sy.copy_(ys[i])
            step(net, opt)
    sa, sb = nets[0].state_dict(), nets[1].state_dict()
    bad = [k for k in sa if not torch.equal(_bits(sa[k]), _bits(sb[k]))]
    assert not bad, bad
    assert counters(nets[0]) == counters(nets[1])
