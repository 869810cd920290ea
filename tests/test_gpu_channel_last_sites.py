"""Converted prune -> quantize sites on channel-last activations: a contiguous tensor pruned along an axis other than
1 (``[B, T, H]`` with ``dimensions={2}``, ``[N, H, W, C]`` with ``dimensions={3}``) and a 4-D channels_last feature
map pruned along its channels.  The fusion pass walks both in memory order, as [rows, C, 1] (column mode), with no
copy of x or of grad_output, and keeps x's memory format for y and gx.

  twins         fused site against the same site with fusion off, over warm-up, ramp, timeout, eval and steady steps:
                y, x.grad, grad_output and every state_dict entry bit for bit (exact-sum inputs)
  oracle        one fused step on seeded normal inputs against oracle/oracle.py on the [outer, C, inner] view
  launch list   a fused step runs the step kernel(s), one forward and one backward, and no copy
  graph mode    GraphedTrainStep replays equal eager steps, also on the three-launch column form
  PruneQuantize channels_last and [..., C] inputs against the permuted contiguous input
"""
import copy
import re

import numpy as np
import pytest
import torch
import torch.nn as nn

from oracle import oracle as orc
from tests.conftest import bits_equal, ulp_diff
from tests.test_gpu_prune_line_step import SITE_FUSED, SITE_STEPS
from tests.test_gpu_prune_quant_step_routes import recorded_kernels

pytestmark = pytest.mark.gpu

BITS = 8
ROWS = 64

# name -> (shape for C channels, prune axis, channels_last)
LAYOUTS = {
    "BTH-d2": (lambda c: (4, 16, c), 2, False),
    "NHWC-d3": (lambda c: (4, 4, 4, c), 3, False),
    "NCHW-cl-d1": (lambda c: (4, c, 4, 4), 1, True),
}
QUANTIZERS = ["decimal", "scaler", "adaptive", "adaptive-channel"]
CHANNELS = [8, 64, 768, 1020, 1024, 1025, 2048, 2049]


def _fmt(layout):
    return torch.channels_last if LAYOUTS[layout][2] else torch.contiguous_format


def _device(a, layout, dtype=torch.float32):
    return torch.from_numpy(a).to(dtype).cuda().contiguous(memory_format=_fmt(layout))


def _site(layout, quant, fuse, start=1, repetition=2, timeout=2, pre=None):
    from qsparse_b200 import AdaptiveQuantizer, DecimalQuantizer, ScalerQuantizer, fuse_prune_quantize, prune, quantize
    _, d, _ = LAYOUTS[layout]
    cb = {"decimal": DecimalQuantizer, "scaler": ScalerQuantizer}.get(quant, AdaptiveQuantizer)()
    site = nn.Sequential(nn.Sequential(pre if pre is not None else nn.Identity(),
                                       prune(sparsity=0.5, dimensions={d}, start=start, interval=1,
                                             repetition=repetition)),
                         quantize(bits=BITS, channelwise=d if quant == "adaptive-channel" else -1, timeout=timeout,
                                  callback=cb)).cuda()
    return fuse_prune_quantize(site) if fuse else site


def _bits(t):
    return t.detach().contiguous().view(-1).cpu().view(torch.uint8)


def _fused_count(model):
    from qsparse_b200.fused import FusedPruneQuantSequential
    return sum(m.fused_steps for m in model.modules() if isinstance(m, FusedPruneQuantSequential))


# ----------------------------------------------------------------------------- twins
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16], ids=["fp32", "bf16-autocast"])
@pytest.mark.parametrize("quant", QUANTIZERS)
@pytest.mark.parametrize("layout", list(LAYOUTS))
@pytest.mark.parametrize("c", CHANNELS)
def test_channel_last_site_equals_unfused(c, layout, quant, dtype):
    shape = LAYOUTS[layout][0](c)
    fmt = _fmt(layout)
    rng = np.random.default_rng(c)
    # small integers times powers of two: every sum is exact, whatever order the two routes reduce in
    xs = [rng.integers(-8, 9, size=shape).astype(np.float32) * 0.25 for _ in SITE_STEPS]
    gs = [rng.standard_normal(shape).astype(np.float32) * 4 for _ in SITE_STEPS]
    res = {}
    for fuse in (True, False):
        model = _site(layout, quant, fuse)
        rec = []
        for kind, xn, gn in zip(SITE_STEPS, xs, gs):
            model.train(kind == "train")
            x = _device(xn, layout, dtype).requires_grad_(True)
            g = _device(gn, layout)
            grads = []
            x.register_hook(grads.append)           # the input gradient as the site returns it
            before = _fused_count(model)
            with torch.autocast("cuda", dtype=torch.bfloat16, enabled=dtype != torch.float32):
                y = model(x)
            y.backward(g)
            if fuse and _fused_count(model) > before:
                what = (c, layout, quant, kind)
                assert y.is_contiguous(memory_format=fmt), what
                assert grads[0].is_contiguous(memory_format=fmt) and grads[0].dtype == dtype, what
            rec.append([y.detach().clone(), x.grad.clone(), g.clone()] + [v.clone() for v in model.state_dict().values()])
        res[fuse] = rec
        if fuse:
            assert _fused_count(model) == (SITE_FUSED if c <= 2048 else 0), (c, _fused_count(model))
    for t, (a, b) in enumerate(zip(res[True], res[False])):
        assert len(a) == len(b)
        for i, (u, v) in enumerate(zip(a, b)):
            assert u.dtype == v.dtype and u.shape == v.shape, (c, t, i)
            assert torch.equal(_bits(u), _bits(v)), (c, layout, quant, dtype, t, i)


# ----------------------------------------------------------------------------- oracle
def _to_ocl(a, layout):
    """the [outer, C, inner] view of a logical-order array"""
    shape_of, d, _ = LAYOUTS[layout]
    c = a.shape[d]
    return a.reshape(int(np.prod(a.shape[:d])), c, -1)


@pytest.mark.parametrize("quant", ["decimal", "adaptive-channel"])
@pytest.mark.parametrize("layout", list(LAYOUTS))
def test_fused_channel_last_step_matches_oracle(layout, quant):
    from qsparse_b200 import graphs
    c = 96
    shape = LAYOUTS[layout][0](c)
    rng = np.random.default_rng(11)
    site = _site(layout, quant, True, repetition=1, timeout=1).train()
    p, q = site[0][1], site[1]
    for _ in range(4):                                     # into the steady state
        site(_device(rng.standard_normal(shape).astype(np.float32), layout))
    n0 = _fused_count(site)
    assert n0 > 0
    mag0 = p.callback.magnitude.detach().cpu().numpy().reshape(-1)
    weight0 = q.weight.detach().cpu().numpy()
    t_prune = p.callback._t()
    t_quant = graphs.host_index(q.callback)
    sparsity = float(p._cur_sparsity.item())

    xn = rng.standard_normal(shape).astype(np.float32)
    gn = rng.standard_normal(shape).astype(np.float32)
    x = _device(xn, layout).requires_grad_(True)
    g = _device(gn, layout)
    y = site(x)
    y.backward(g)
    assert _fused_count(site) == n0 + 1

    xo, go = _to_ocl(xn, layout), _to_ocl(gn, layout)
    mag = orc.magnitude_ema(mag0, orc.squeeze_mean_abs(xo, (1, c, 1)).reshape(-1), t_prune)
    mask, _ = orc.mask_given_importance(mag, sparsity)
    if quant == "decimal":
        scale = orc.scale_ema(weight0.reshape(-1), np.array([np.max(orc.absmax(xo, 1) * mask)], np.float32), BITS,
                              t_quant)
        dec = orc.scale_to_decimal(scale)
        y_ref = orc.fq_pow2_fwd(xo, dec, 1, mask=mask)
        _, gx_ref = orc.ste_bwd(go, dec, BITS, 1, True, False, mask=mask)
        assert bits_equal(q.weight.detach().cpu().numpy().reshape(-1), scale)
    else:
        mn, mx = orc.minmax(orc.mask_apply(xo, mask, 1), 1)
        lines = orc.lines_ema(weight0, mn, mx, t_quant + 1)
        y_ref = orc.fq_line_fwd(xo, lines, BITS, 1, True, mask=mask)
        gx_ref = orc.mask_apply(go, mask, 1)
        assert np.array_equal(q.weight.detach().cpu().numpy(), lines)
    got_mask = p.mask.detach().cpu().numpy().reshape(-1)
    assert np.array_equal(got_mask, mask.astype(bool))
    assert ulp_diff(p.callback.magnitude.detach().cpu().numpy().reshape(-1), mag).max() <= 4
    h = lambda t: _to_ocl(t.detach().float().cpu().numpy(), layout)   # the tensor in logical order
    assert bits_equal(h(y), y_ref)
    assert bits_equal(h(x.grad), gx_ref)


# ----------------------------------------------------------------------------- launch list
@pytest.mark.parametrize("c", [768, 1020])
@pytest.mark.parametrize("quant", ["decimal", "adaptive"])
@pytest.mark.parametrize("layout", list(LAYOUTS))
def test_fused_channel_last_step_launches(layout, quant, c):
    """one fused step: the one-launch step kernel, one forward and one backward map kernel (the channel-resident
    lastdim kernel when C % 8 == 0, the MODE 2 walk otherwise) and no copy of x, y or g"""
    shape = LAYOUTS[layout][0](c)
    rng = np.random.default_rng(3)
    site = _site(layout, quant, True, repetition=1, timeout=1).train()
    x = _device(rng.standard_normal(shape).astype(np.float32), layout).requires_grad_(True)
    g = _device(rng.standard_normal(shape).astype(np.float32), layout)
    for _ in range(4):
        site(x).backward(g)
    n0 = _fused_count(site)
    assert n0 > 0
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        site(x).backward(g)
        torch.cuda.synchronize()
    assert _fused_count(site) == n0 + 1
    names = [e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]
    assert not [n for n in names if re.search(r"copy|contiguous", n, re.IGNORECASE)], names
    qsb = [n for n in names if "qsb::" in n]
    assert len(qsb) == 3, qsb
    assert any("StepTail" in n for n in qsb), qsb
    maps = [n for n in qsb if "map_" in n]
    assert len(maps) == 2, qsb
    kernel = "map_lastdim_kernel" if c % 8 == 0 else "map_chan_kernel"
    assert all(kernel in n for n in maps), (kernel, maps)


# ----------------------------------------------------------------------------- graph mode
class _Net(nn.Module):
    """Linear -> GELU -> site on the hidden axis -> Linear, and channels_last conv -> ReLU -> site on the channels"""

    def __init__(self, hidden):
        super().__init__()
        self.inp = nn.Linear(32, hidden)
        self.tok = _site("BTH-d2", "decimal", False, repetition=1, timeout=1, pre=nn.GELU())
        self.out = nn.Linear(hidden, 32)
        self.conv = nn.Conv2d(8, 16, 3, padding=1)
        self.img = _site("NCHW-cl-d1", "adaptive-channel", False, repetition=1, timeout=1, pre=nn.ReLU())

    def forward(self, x, z):
        return self.out(self.tok(self.inp(x))), self.img(self.conv(z))


@pytest.mark.parametrize("hidden", [64, 256], ids=["one-launch", "three-launch"])
def test_channel_last_sites_graphed_equal_eager(hidden):
    """3 warm-up steps and 5 replays of the captured step equal 8 eager steps in every parameter, mask, magnitude,
    scale, line and counter; [512, 256] takes the three-launch column form of the step"""
    from qsparse_b200 import fuse_prune_quantize, graphs
    from qsparse_b200.quantize import AdaptiveQuantizer, QuantizeLayer
    from qsparse_b200.sparse import MagnitudePruningCallback, PruneLayer
    det = torch.backends.cudnn.deterministic, torch.backends.cudnn.benchmark
    torch.backends.cudnn.deterministic, torch.backends.cudnn.benchmark = True, False
    try:
        torch.manual_seed(0)
        rng = np.random.default_rng(5)
        f = lambda *s: torch.from_numpy(rng.standard_normal(s).astype(np.float32)).cuda()
        data = [(f(4, 128, 32), f(4, 128, 32), f(8, 8, 8, 8).contiguous(memory_format=torch.channels_last),
                 f(8, 16, 8, 8).contiguous(memory_format=torch.channels_last)) for _ in range(10)]
        base = fuse_prune_quantize(_Net(hidden).cuda().to(memory_format=torch.channels_last)).train()
        for i in range(4):                          # into the steady state, eagerly
            a, b = base(data[i][0], data[i][2])
            ((a * data[i][1]).sum() + (b * data[i][3]).sum()).backward()
        a, b = base(data[4][0], data[4][2])
        assert b.is_contiguous(memory_format=torch.channels_last)
        names = recorded_kernels(lambda: base.tok(base.inp(data[4][0])))
        assert any("reduce_finalize" in n for n in names) == (hidden == 256), names
        del a, b
        nets = [copy.deepcopy(base), copy.deepcopy(base)]
        opts = [torch.optim.SGD(n.parameters(), lr=0.01) for n in nets]
        static = [t.clone() for t in data[0]]

        def step(net, opt):
            opt.zero_grad(set_to_none=True)
            a, b = net(static[0], static[2])
            loss = (a * static[1]).sum() + (b * static[3]).sum()
            loss.backward()
            opt.step()
            return loss.detach().clone()

        def feed(i):
            for s, t in zip(static, data[i % 10]):
                s.copy_(t)

        def counters(net):
            out = []
            for m in net.modules():
                if isinstance(m, (QuantizeLayer, PruneLayer)):
                    mirror = m._t_mirror if isinstance(m, QuantizeLayer) else m._n_mirror
                    out += [int(mirror.get(m._n_updates)), int(m._n_updates.item())]
                elif isinstance(m, MagnitudePruningCallback):
                    out += [int(m._t()), int(m.t.item())]
                elif isinstance(m, AdaptiveQuantizer):
                    out += [graphs.host_index(m)]
            return out + [_fused_count(net)]

        eager = []
        for i in range(5, 13):
            feed(i)
            eager.append(step(nets[1], opts[1]))
        warm = iter(range(5, 8))

        class _Step:
            n = 0

            def __call__(self):
                self.n += 1
                if self.n <= 3:
                    feed(next(warm))
                return step(nets[0], opts[0])
        gs = graphs.GraphedTrainStep(nets[0], _Step(), warmup=3)
        replayed = []
        for i in range(8, 13):
            feed(i)
            replayed.append(gs.replay().clone())
        gs.sync_host()
        assert torch.equal(_bits(torch.stack(eager[3:])), _bits(torch.stack(replayed)))
        sa, sb = nets[0].state_dict(), nets[1].state_dict()
        assert sorted(sa) == sorted(sb)
        bad = [k for k in sa if not torch.equal(_bits(sa[k]), _bits(sb[k]))]
        assert not bad, bad
        assert counters(nets[0]) == counters(nets[1])
        assert _fused_count(nets[0]) > _fused_count(base) + 3
    finally:
        torch.backends.cudnn.deterministic, torch.backends.cudnn.benchmark = det


# ----------------------------------------------------------------------------- PruneQuantize
@pytest.mark.parametrize("case", ["channels_last", "last-axis"])
def test_prune_quantize_channel_last_inputs(case):
    """channels_last [N, C, H, W] (channel_index 1) and contiguous [B, T, C] (channel_index 2) against the same values
    permuted to a contiguous tensor, over 4 training steps: y, gx and state bit for bit, y and gx in x's format"""
    from qsparse_b200.fused import PruneQuantize
    c = 48
    rng = np.random.default_rng(7)
    if case == "channels_last":
        shape, ci, fmt = (4, c, 6, 5), 1, torch.channels_last
        perm, ref_ci = (0, 2, 3, 1), 3                  # NHWC: the same memory order as channels_last NCHW
    else:
        shape, ci, fmt = (4, 10, c), 2, torch.contiguous_format
        perm, ref_ci = (0, 2, 1), 1
    mods = [PruneQuantize(0.5, BITS, channel_index=ci).cuda().train(),
            PruneQuantize(0.5, BITS, channel_index=ref_ci).cuda().train()]
    for t in range(4):
        xn = rng.integers(-8, 9, size=shape).astype(np.float32) * 0.25
        gn = rng.standard_normal(shape).astype(np.float32)
        x = torch.from_numpy(xn).cuda().contiguous(memory_format=fmt).requires_grad_(True)
        grads = []
        x.register_hook(grads.append)
        y = mods[0](x)
        y.backward(torch.from_numpy(gn).cuda().contiguous(memory_format=fmt))
        assert y.is_contiguous(memory_format=fmt) and grads[0].is_contiguous(memory_format=fmt), t
        xr = torch.from_numpy(xn).cuda().permute(perm).contiguous().requires_grad_(True)
        yr = mods[1](xr)
        yr.backward(torch.from_numpy(gn).cuda().permute(perm).contiguous())
        assert torch.equal(_bits(y.permute(perm)), _bits(yr)), t
        assert torch.equal(_bits(x.grad.permute(perm)), _bits(xr.grad)), t
        for name in ("magnitude", "mask", "scale"):
            assert torch.equal(_bits(getattr(mods[0], name)), _bits(getattr(mods[1], name))), (name, t)
