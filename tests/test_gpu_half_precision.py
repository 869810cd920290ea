"""bf16 / fp16 activations read natively by the prune / quantize kernels.

Every case runs the same call twice: on the 16-bit tensor itself, and on ``x.float()`` inside the autograd graph
(the route the package took before it read 16-bit values: an fp32 copy in front of the kernels, autograd's cast
of the fp32 input gradient behind them).  Outputs, input gradients (compared as int16 bit patterns), dtypes,
the in-place clamp of grad_output and every piece of layer state must be equal.
"""
import contextlib
import ctypes
import io

import pytest
import torch
import torch.nn as nn

HALF = [torch.bfloat16, torch.float16]


def bits(t):
    t = t.detach()
    if t.dtype in (torch.bfloat16, torch.float16):
        return t.contiguous().view(torch.int16).cpu()
    if t.dtype == torch.float32:
        return t.contiguous().view(torch.int32).cpu()
    return t.cpu()


def same(a, b, what=""):
    assert a.dtype == b.dtype, (what, a.dtype, b.dtype)
    assert a.shape == b.shape, (what, a.shape, b.shape)
    assert torch.equal(bits(a), bits(b)), what


def make_x(shape, dtype, seed=0, specials=True, channels_last=False):
    g = torch.Generator(device="cpu").manual_seed(seed)
    x = torch.randn(shape, generator=g) * 3
    if specials:
        flat = x.view(-1)
        n = flat.numel()
        tiny = torch.finfo(dtype).tiny
        vals = [float("nan"), float("inf"), -float("inf"), -0.0, 0.0, tiny / 4, -tiny / 2, 1e-30]
        for i, v in enumerate(vals):
            flat[(i * 7919) % n] = v
    x = x.to(dtype).cuda()
    if channels_last:
        x = x.contiguous(memory_format=torch.channels_last)
    return x


def run_both(fn, x, g):
    """(y, gx, g_after) of fn on the 16-bit leaf and on its fp32 copy inside the graph"""
    outs = []
    for upcast in (False, True):
        xl = x.detach().clone().requires_grad_(True)
        y = fn(xl.float() if upcast else xl)
        gg = g.clone()
        y.backward(gg)
        outs.append((y.detach(), xl.grad, gg))
    return outs


SHAPES = [
    ((32, 64, 56, 56), 1, False),   # long rows
    ((16, 32, 7, 7), 1, False),
    ((16, 32, 14, 14), 1, False),
    ((4096, 768), 1, False),        # channel-last
    ((8, 32, 14, 14), 1, True),     # channels_last 4-D
    ((3, 5, 7, 9), -1, False),      # per tensor, size not a multiple of 8
    ((6, 13, 11), 1, False),        # per channel, rows not a multiple of 8
]


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", HALF)
@pytest.mark.parametrize("shape,ci,cl", SHAPES)
def test_fake_quantizers(dtype, shape, ci, cl):
    from qsparse_b200.quantize import quantize_with_decimal, quantize_with_line, quantize_with_scaler
    x = make_x(shape, dtype, channels_last=cl)
    g = torch.randn(x.shape, device="cuda") * 8
    if cl:
        g = g.contiguous(memory_format=torch.channels_last)
    C = x.shape[ci] if ci >= 0 else 1
    dec = torch.arange(C, device="cuda", dtype=torch.float32) % 5 + 1 if ci >= 0 else 4
    sc = torch.rand(C, device="cuda") * 0.2 + 0.01 if ci >= 0 else 0.05
    lines = torch.stack([-torch.rand(C, device="cuda"), torch.rand(C, device="cuda")], 1) if ci >= 0 else (-1.0, 2.0)
    fns = [lambda t: quantize_with_decimal(t, 8, dec, ci),
           lambda t: quantize_with_scaler(t, 6, sc, ci),
           lambda t: quantize_with_line(t, 8, lines, ci)]
    for i, fn in enumerate(fns):
        (y, gx, ga), (y_ref, gx_ref, ga_ref) = run_both(fn, x, g)
        same(y, y_ref, ("y", i))
        assert y.dtype == torch.float32
        same(gx, gx_ref, ("gx", i))
        assert gx.dtype == dtype
        same(ga, ga_ref, ("grad_output", i))


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", HALF)
def test_unaligned_view(dtype):
    """a view at an odd element offset (2-byte aligned): statistics, quantize, gradient"""
    from qsparse_b200 import ops
    from qsparse_b200.quantize import quantize_with_decimal
    base = make_x((1 + 8 * 64 * 33 * 33,), dtype)
    x = base[1:].view(8, 64, 33, 33)
    assert x.data_ptr() % 4 == 2
    lay = (8, 64, 33 * 33)
    a = ops.reduce_stats(x, lay, absmax=True, minmax=True, abssum=True)
    b = ops.reduce_stats(x.float(), lay, absmax=True, minmax=True, abssum=True)
    for k in a:
        assert torch.equal(bits(a[k]), bits(b[k])), k
    x2 = base[1:].view(16, 2 * 33 * 33 * 16)
    lay2 = (16, 1, x2.shape[1])
    a = ops.reduce_stats(x2, lay2, absmax=True, abssum=True)
    b = ops.reduce_stats(x2.float(), lay2, absmax=True, abssum=True)
    for k in a:
        assert torch.equal(bits(a[k]), bits(b[k])), k
    g = torch.randn(x.shape, device="cuda")
    dec = torch.arange(64, device="cuda", dtype=torch.float32) % 4 + 2
    (y, gx, ga), (y_ref, gx_ref, ga_ref) = run_both(lambda t: quantize_with_decimal(t, 8, dec, 1), x, g)
    same(y, y_ref, "y")
    same(gx, gx_ref, "gx")


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", HALF)
def test_gradient_rounding(dtype):
    """bf16 ties round to even like autograd's cast; fp16 overflows to inf; NaN through mask apply"""
    from qsparse_b200.quantize import quantize_with_scaler
    from qsparse_b200.sparse import apply_mask
    x = make_x((4, 16, 8, 8), dtype, specials=False)
    # fp32 values exactly halfway between two bf16 (and fp16) neighbours, plus values beyond fp16's range
    ties = torch.tensor([1 + 2 ** -8, 1 + 3 * 2 ** -8, -(1 + 2 ** -8), 1 + 2 ** -11, 1 + 3 * 2 ** -11,
                         70000.0, -1e5, 65520.0], device="cuda")
    g = ties.repeat(x.numel() // ties.numel()).view(x.shape)
    (y, gx, ga), (y_ref, gx_ref, ga_ref) = run_both(lambda t: quantize_with_scaler(t, 8, 1000.0, -1), x, g)
    same(gx, gx_ref, "gx")
    same(ga, ga_ref, "grad_output")
    if dtype == torch.float16:
        assert torch.isinf(gx.float()).any()
    mask = torch.tensor([True, False] * 8, device="cuda").view(1, 16, 1, 1)
    gn = g.clone()
    gn.view(-1)[::5] = float("nan")
    (y, gx, _), (y_ref, gx_ref, _) = run_both(lambda t: apply_mask(t, mask), x, gn)
    same(y, y_ref, "masked y")
    assert y.dtype == torch.float32
    same(gx, gx_ref, "masked gx")


def _site(cb_cls, seed):
    from qsparse_b200 import fuse_prune_quantize, prune, quantize
    torch.manual_seed(seed)
    m = nn.Sequential(nn.Sequential(nn.Identity(), prune(sparsity=0.5, dimensions={1}, start=6, interval=5,
                                                          repetition=3)),
                      quantize(bits=8, channelwise=-1, timeout=3, callback=cb_cls())).cuda()
    fuse_prune_quantize(m)
    return m


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", HALF)
@pytest.mark.parametrize("cb", ["decimal", "scaler"])
def test_fused_site_ramp(dtype, cb):
    """a fused prune -> quantize site through a sparsity ramp: native vs a forward pre-hook x.float()"""
    from qsparse_b200 import DecimalQuantizer, ScalerQuantizer
    from qsparse_b200.fused import FusedPruneQuantSequential
    cls = DecimalQuantizer if cb == "decimal" else ScalerQuantizer
    a, b = _site(cls, 0), _site(cls, 0)
    b.register_forward_pre_hook(lambda mod, inp: (inp[0].float(),))
    for step in range(30):
        x = make_x((16, 32, 14, 14), dtype, seed=step, specials=False) * (1 + step / 10)
        g = torch.randn(x.shape, device="cuda")
        outs = []
        for m in (a, b):
            xl = x.detach().clone().requires_grad_(True)
            y = m(xl)
            y.backward(g.clone())
            outs.append((y.detach(), xl.grad))
        # warm-up steps pass x through unchanged (in its own dtype); every prune / quantize step returns fp32
        same(outs[0][0].float(), outs[1][0], ("y", step))
        same(outs[0][1], outs[1][1], ("gx", step))
        sa, sb = a.state_dict(), b.state_dict()
        assert sa.keys() == sb.keys()
        for k in sa:
            same(sa[k], sb[k], (k, step))
    fa = [m.fused_steps for m in a.modules() if isinstance(m, FusedPruneQuantSequential)]
    fb = [m.fused_steps for m in b.modules() if isinstance(m, FusedPruneQuantSequential)]
    assert fa == fb and fa[0] > 10, (fa, fb)


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", HALF)
def test_prune_quantize_module(dtype):
    from qsparse_b200.fused import PruneQuantize
    a, b = PruneQuantize(0.5, 8, mutate_grad_output=True), PruneQuantize(0.5, 8, mutate_grad_output=True)
    for step in range(6):
        x = make_x((32, 64, 28, 28), dtype, seed=step, specials=False)
        g = torch.randn(x.shape, device="cuda")
        res = []
        for m, up in ((a, False), (b, True)):
            xl = x.detach().clone().requires_grad_(True)
            y = m(xl.float() if up else xl)
            gg = g.clone()
            y.backward(gg)
            res.append((y.detach(), xl.grad, gg))
        for i, name in enumerate(("y", "gx", "grad_output")):
            same(res[0][i], res[1][i], (name, step))
        for name in ("magnitude", "mask", "scale", "decimal"):
            same(getattr(a, name), getattr(b, name), (name, step))


@pytest.mark.gpu
def test_no_fp32_copy():
    """one native forward of a 64 MB bf16 tensor allocates its fp32 output and nothing the size of x in fp32"""
    from qsparse_b200.quantize import quantize_with_decimal
    x = torch.randn(32 * 1024 * 1024, device="cuda").to(torch.bfloat16).view(64, 512, 1024)
    quantize_with_decimal(x, 8, 5, -1)
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    base = torch.cuda.memory_allocated()
    y = quantize_with_decimal(x, 8, 5, -1)
    torch.cuda.synchronize()
    grown = torch.cuda.max_memory_allocated() - base
    assert grown <= y.numel() * 4 + (2 << 20), grown


def test_bad_dtype_code_without_gpu():
    """a dtype code other than QSB_DTYPE_* is rejected before any CUDA call"""
    from qsparse_b200 import _native
    lib = _native.load_library()
    p = ctypes.c_void_p(16)
    bad = -1
    assert lib.qsb_fq_pow2_fwd_dt(p, 3, p, None, 1, 0.0, None, 0, 1, 1, 8, None) == bad
    assert lib.qsb_fq_scaler_fwd_dt(p, -1, p, None, 1, 0.1, None, 0, 1, 1, 8, None) == bad
    assert lib.qsb_fq_line_fwd_dt(p, 7, p, None, 1, 0.0, 1.0, 8, 1, None, 0, 1, 1, 8, None) == bad
    assert lib.qsb_ste_bwd_dt(p, p, p, 5, None, 1, 0.0, 1, 8, 0, None, 0, 1, 1, 8, None) == bad
    assert lib.qsb_mask_apply_dt(p, 0, p, 9, p, 1, 1, 1, 8, None) == bad
    assert lib.qsb_reduce_stats_dt(p, 4, 1, 1, 1, 8, p, None, None, None, None, None, p, 1 << 20, None) == bad
    assert lib.qsb_reduce_partials_dt(p, 3, 1, 1, 8, p, 1 << 20, None) == bad
    assert lib.qsb_reduce_prune_quant_step_dt(p, 3, 1, 2, 8, p, 1 << 20, p, p, p, p, p, None, 1, 8.0, 0, 1, 0, 0, 8,
                                              0, 1, None, None, 0, None, None, None) == bad


# ----------------------------------------------------------------------------- training under autocast
def _deterministic():
    import qsparse_b200 as qs
    qs.set_qsparse_options(log_on_created=False)
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.deterministic = True
    torch.backends.cudnn.benchmark = False


def _upcast_sites(model):
    """a forward pre-hook ``x.float()`` on every prune / quantize site: the route taken before 16-bit reads"""
    from qsparse_b200.fused import FusedPruneQuantSequential, PruneQuantize
    from qsparse_b200.quantize import QuantizeLayer
    from qsparse_b200.sparse import PruneLayer
    for m in model.modules():
        if isinstance(m, (PruneLayer, QuantizeLayer, FusedPruneQuantSequential, PruneQuantize)):
            m.register_forward_pre_hook(lambda mod, inp: (inp[0].float(),) + tuple(inp[1:]))


def _train(model, opt, xs, ys, steps, graph_from=None, loss_fn=None):
    """`steps` bf16-autocast training steps on batches xs[i], ys[i]; from step `graph_from` on, three warm-up steps
    on their own batches and then replays of ONE captured step (``GraphedTrainStep``).  Returns the losses of the
    eager and replayed steps (not the warm-up ones), the state, the fused-step counts and the host counters."""
    from qsparse_b200 import graphs
    F = torch.nn.functional
    loss_fn = loss_fn or F.nll_loss
    sx, sy = xs[0].clone(), ys[0].clone()
    model.train()

    def step():
        opt.zero_grad(set_to_none=True)
        # no cast cache: a captured graph must re-cast the weights that the optimizer updates in place
        with torch.autocast("cuda", dtype=torch.bfloat16, cache_enabled=False):
            loss = loss_fn(model(sx), sy)
        loss.backward()
        opt.step()
        return loss.detach().clone()

    losses = []
    i = 0
    while i < steps:
        if graph_from is not None and i == graph_from:
            feed = iter(range(i, i + 3))

            class _Two:
                n = 0

                def __call__(self):
                    self.n += 1
                    if self.n <= 3:
                        j = next(feed)
                        sx.copy_(xs[j]); sy.copy_(ys[j])
                    return step()
            gs = graphs.GraphedTrainStep(model, _Two(), warmup=3)
            i += 3
            while i < steps:
                sx.copy_(xs[i]); sy.copy_(ys[i])
                losses.append(gs.replay().clone())
                i += 1
            gs.sync_host()
            break
        sx.copy_(xs[i]); sy.copy_(ys[i])
        losses.append(step())
        i += 1
    state = {k: v.clone() for k, v in model.state_dict().items()}
    fused = [m.fused_steps for m in model.modules() if hasattr(m, "fused_steps")]
    host = [graphs.host_index(m) for m in model.modules() if hasattr(m, "optimize") and hasattr(m, "t")]
    return torch.stack(losses), state, fused, host


def _same_state(a, b):
    assert sorted(a) == sorted(b)
    bad = [k for k in a if a[k].dtype != b[k].dtype or not torch.equal(bits(a[k]), bits(b[k]))]
    assert not bad, bad


@pytest.mark.gpu
@pytest.mark.parametrize("fuse", [False, True])
@pytest.mark.parametrize("kind", ["DecimalQuantizer", "ScalerQuantizer"])
def test_config1_mnist_autocast(kind, fuse):
    """The converted config-1 MNIST net trained under bf16 autocast: its activation sites see bf16.  60 eager steps
    equal, loss for loss and in every parameter, mask, scale and magnitude, the same net whose sites upcast their
    input with a pre-hook; then 3 warm-up steps and 7 replays of the step captured by GraphedTrainStep equal 70
    eager steps."""
    from benchmarks.configs import _c1_convert, _c1_net
    import qsparse_b200 as qs
    _deterministic()
    dev = torch.device("cuda:0")

    def setup(upcast=False):
        torch.manual_seed(0)
        model = _c1_convert(torch, qs, _c1_net(torch), kind, fuse).to(dev)
        for m in model.modules():           # dropout off: its RNG draws differ between the runs
            if isinstance(m, nn.Dropout):
                m.p = 0.0
        if upcast:
            _upcast_sites(model)
        gen = torch.Generator(device=dev).manual_seed(11)
        xs = torch.randn(70, 64, 1, 28, 28, device=dev, generator=gen)
        ys = torch.randint(0, 10, (70, 64), device=dev, generator=gen)
        return model, torch.optim.SGD(model.parameters(), lr=0.01), xs, ys

    seen = []
    model, opt, xs, ys = setup()
    from qsparse_b200.quantize import QuantizeLayer
    for m in model.modules():
        if isinstance(m, QuantizeLayer) and m.channelwise < 0:
            m.register_forward_pre_hook(lambda mod, inp: seen.append(inp[0].dtype))
    nat_losses, nat_state, nat_fused, _ = _train(model, opt, xs, ys, 60)
    assert torch.bfloat16 in seen                 # the native kernels really saw 16-bit activations
    up_losses, up_state, up_fused, _ = _train(*setup(upcast=True), 60)
    assert torch.equal(nat_losses, up_losses)
    _same_state(nat_state, up_state)
    assert nat_fused == up_fused
    if fuse:
        assert all(f > 0 for f in nat_fused), nat_fused

    ref_losses, ref_state, ref_fused, ref_host = _train(*setup(), 70)
    got_losses, got_state, got_fused, got_host = _train(*setup(), 70, graph_from=60)
    assert torch.equal(ref_losses[:60], got_losses[:60]) and torch.equal(ref_losses[63:], got_losses[60:])
    _same_state(ref_state, got_state)
    assert ref_fused == got_fused and ref_host == got_host


@pytest.mark.gpu
@pytest.mark.parametrize("fuse", [False, True])
def test_graphed_activation_routes_autocast(fuse):
    """Under bf16 autocast, GraphedTrainStep captures every activation route that reads 16-bit values — Decimal
    estimation through ``optimize`` + ``forward`` (a subclass is not fused), per-channel Adaptive (min / max) estimation, a stand-alone structured prune layer, a
    per-tensor Decimal layer, PruneQuantize — and 12 eager steps + 3 warm-up + 5 replays equal 20 eager steps; the
    eager steps also equal the upcast-hook route."""
    import qsparse_b200 as qs
    from qsparse_b200.fused import PruneQuantize
    from qsparse_b200.quantize import AdaptiveQuantizer, DecimalQuantizer
    _deterministic()
    dev = torch.device("cuda:0")
    F = torch.nn.functional

    class PlainDecimal(DecimalQuantizer):
        """not the stock class: the layer runs optimize() (abs-max reduction) and forward() separately"""

    class Net(nn.Module):
        def __init__(self):
            super().__init__()
            self.c1 = nn.Conv2d(3, 16, 3, padding=1)
            self.dq = qs.quantize(bits=8, channelwise=-1, timeout=2, callback=PlainDecimal())
            self.c2 = nn.Conv2d(16, 16, 3, padding=1)
            self.aq = qs.quantize(bits=8, channelwise=1, timeout=2, callback=AdaptiveQuantizer())
            self.c3 = nn.Conv2d(16, 32, 3, padding=1)
            self.p = qs.prune(sparsity=0.5, dimensions={1}, start=2, interval=1, repetition=2)
            self.tq = qs.quantize(bits=8, channelwise=-1, timeout=3, callback=DecimalQuantizer())
            self.c4 = nn.Conv2d(32, 32, 3, padding=1)
            self.pq = PruneQuantize(0.5, 8)
            self.fc = nn.Linear(32 * 8 * 8, 10)

        def forward(self, x):
            x = self.dq(F.relu(self.c1(x)))
            x = self.aq(F.relu(self.c2(x)))
            x = self.tq(self.p(F.relu(self.c3(x))))
            x = self.pq(F.relu(self.c4(x)))
            return self.fc(x.flatten(1))

    def setup(upcast=False):
        torch.manual_seed(5)
        with contextlib.redirect_stdout(io.StringIO()):
            model = Net().to(dev)
            if fuse:
                qs.fuse_prune_quantize(model)
        if upcast:
            _upcast_sites(model)
        gen = torch.Generator(device=dev).manual_seed(9)
        xs = torch.randn(20, 16, 3, 8, 8, device=dev, generator=gen)
        ys = torch.randint(0, 10, (20, 16), device=dev, generator=gen)
        return model, torch.optim.SGD(model.parameters(), lr=0.05), xs, ys

    ce = F.cross_entropy
    with contextlib.redirect_stdout(io.StringIO()):
        nat = _train(*setup(), 20, loss_fn=ce)
        up = _train(*setup(upcast=True), 20, loss_fn=ce)
        got = _train(*setup(), 20, graph_from=12, loss_fn=ce)
    assert torch.equal(nat[0], up[0])
    _same_state(nat[1], up[1])
    assert torch.equal(nat[0][:12], got[0][:12]) and torch.equal(nat[0][15:], got[0][12:])
    _same_state(nat[1], got[1])
    assert nat[2] == got[2] and nat[3] == got[3]
