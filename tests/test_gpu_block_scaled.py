"""Block-scaled FP8 / FP4 fake quantization (MXFP8, MXFP4, NVFP4) on the GPU, bit for bit against the numpy
restatement in oracle/block_scaled.py: the forward and the packed export over fp32 / bf16 / fp16 inputs, short
and odd rows, unaligned views, channels_last tensors, conv weights split on their leading axis, special values,
element indices past 2^31; then the quantizer inside layers, the fusion pass and CUDA graphs."""
import copy

import numpy as np
import pytest
import torch
import torch.nn as nn

from oracle import block_scaled as bs
from oracle import oracle as orc

pytestmark = pytest.mark.gpu

FMTS = ["mxfp8", "mxfp4", "nvfp4"]
DTYPES = [torch.float32, torch.bfloat16, torch.float16]
LENGTHS = [1, 7, 16, 31, 32, 33, 56, 4096, 4100]


def same_bits(a, b):
    """fp32 arrays equal bit for bit (-0 != +0); NaN matches NaN whatever its payload"""
    a, b = np.ascontiguousarray(a, np.float32), np.ascontiguousarray(b, np.float32)
    assert a.shape == b.shape, (a.shape, b.shape)
    ok = (a.view(np.uint32) == b.view(np.uint32)) | (np.isnan(a) & np.isnan(b))
    if not ok.all():
        i = np.flatnonzero(~ok.reshape(-1))[:5]
        raise AssertionError(f"{(~ok).sum()} mismatches, first at {i}: {a.reshape(-1)[i]} vs {b.reshape(-1)[i]}")


def make_rows(rows, L, dtype, seed, specials=True):
    """[rows, L] values whose magnitudes spread over many binades, with zero blocks, +-0, subnormals, NaN and +-inf
    sprinkled in (each special only once per tensor, so most blocks stay finite)"""
    rng = np.random.default_rng(seed)
    x = rng.standard_normal((rows, L)) * np.exp2(rng.integers(-12, 12, size=(rows, 1)))
    x = x.astype(np.float32).reshape(-1)
    n = x.size
    if specials and n >= 64:
        pos = rng.choice(n, size=32, replace=False)
        x[pos[:8]] = 0.0
        x[pos[8:12]] = -0.0
        tiny = np.float32(torch.finfo(dtype).tiny)
        x[pos[12:20]] = tiny * np.float32(0.375) * np.sign(rng.standard_normal(8)).astype(np.float32)
        x[pos[20]] = np.nan
        x[pos[21]] = np.inf
        x[pos[22]] = -np.inf
        b0 = int(rng.integers(0, n // 16)) * 16
        x[b0:b0 + 32] = 0.0                                            # a zero block (any block size)
        b1 = int(rng.integers(0, n // 16)) * 16
        x[b1:b1 + 16] = tiny * np.float32(0.5) * rng.standard_normal(16).astype(np.float32)  # subnormal block
    t = torch.from_numpy(x.reshape(rows, L)).to(dtype)
    return t


def w_of(x32: np.ndarray) -> np.float32:
    """nvfp4's tensor abs-max: a bit below the finite max, so some block scales saturate"""
    f = x32[np.isfinite(x32)]
    return np.float32(np.abs(f).max() * np.float32(0.75)) if f.size else np.float32(1)


def block_layer(fmt, x, w=None, rows="last"):
    """an initialised QuantizeLayer with this callback and nvfp4's w set"""
    import qsparse_b200 as qs
    layer = qs.quantize(bits=8, channelwise=-1, timeout=1, callback=qs.BlockScaledQuantizer(fmt, rows=rows))
    layer._allocate(x)
    if w is not None:
        layer.weight.data.fill_(float(w))
    return layer


def check_all(layer, x, x2d_ref, w, channels_last=False):
    """forward, export and dequantize of one layer on x against the numpy restatement of the [R, L] rows"""
    from qsparse_b200.quantize import dequantize_block_scaled, export_block_scaled
    fmt = layer.callback.fmt
    y = layer.callback(x, 8, layer.weight, channel_index=-1)
    assert y.dtype == torch.float32 and y.shape == x.shape
    y_rows = y.permute(0, 2, 3, 1) if channels_last else y
    same_bits(y_rows.reshape(x2d_ref.shape).cpu().numpy(), bs.fake_quant(x2d_ref, fmt, w))
    e = export_block_scaled(layer, x)
    codes, scales = bs.export(x2d_ref, fmt, w)
    assert np.array_equal(e["codes"].cpu().numpy(), codes)
    assert np.array_equal(e["scales"].cpu().numpy(), scales)
    same_bits(dequantize_block_scaled(e).cpu().numpy(), y.cpu().numpy())
    return y


@pytest.mark.parametrize("dtype", DTYPES, ids=lambda d: str(d).split(".")[1])
@pytest.mark.parametrize("fmt", FMTS)
@pytest.mark.parametrize("L", LENGTHS)
def test_rows_vs_reference(fmt, dtype, L):
    for seed, rows in enumerate((1, 5, 64)):
        x = make_rows(rows, L, dtype, seed).cuda()
        ref = x.float().cpu().numpy()
        layer = block_layer(fmt, x, w_of(ref))
        check_all(layer, x, ref, w_of(ref))


@pytest.mark.parametrize("dtype", DTYPES, ids=lambda d: str(d).split(".")[1])
@pytest.mark.parametrize("fmt", FMTS)
@pytest.mark.parametrize("L", [32, 56, 4096, 33])
def test_views_offset_by_one_element(fmt, dtype, L):
    rows = 24
    flat = make_rows(1, rows * L + 1, dtype, 7).reshape(-1).cuda()
    x = flat[1:].view(rows, L)
    assert x.data_ptr() % 16 != 0
    ref = x.float().cpu().numpy()
    check_all(block_layer(fmt, x, w_of(ref)), x, ref, w_of(ref))


@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16], ids=["float32", "bfloat16"])
@pytest.mark.parametrize("fmt", FMTS)
def test_channels_last_activation(fmt, dtype):
    x = make_rows(4 * 7 * 9, 40, dtype, 3).reshape(4, 7, 9, 40).permute(0, 3, 1, 2).cuda()
    assert x.is_contiguous(memory_format=torch.channels_last) and not x.is_contiguous()
    ref = bs.rows_view(x.float().cpu().numpy(), "last", channels_last=True)
    y = check_all(block_layer(fmt, x, w_of(ref)), x, ref, w_of(ref), channels_last=True)
    assert y.is_contiguous(memory_format=torch.channels_last)


@pytest.mark.parametrize("fmt", FMTS)
def test_leading_rows_on_a_conv_weight(fmt):
    w = (torch.randn(64, 48, 3, 3, generator=torch.Generator().manual_seed(1)) * 0.05).cuda()
    ref = bs.rows_view(w.cpu().numpy(), "leading")
    assert ref.shape == (64, 432)
    check_all(block_layer(fmt, w, w_of(ref), rows="leading"), w, ref, w_of(ref))


def test_nvfp4_tensor_scale_specials():
    """w = 0 gives +0 everywhere, a NaN w NaN everywhere, both in the forward and through the export"""
    x = make_rows(8, 64, torch.float32, 11, specials=False).cuda()
    ref = x.cpu().numpy()
    for w in (np.float32(0), np.float32(np.nan), np.float32(1e-30), np.float32(3e38)):
        check_all(block_layer("nvfp4", x, w), x, ref, w)


@pytest.mark.parametrize("case", ["float32-aligned", "bfloat16-odd-rows"])
def test_element_indices_past_2_31(case):
    """a tensor of more than 2^31 elements: the rows around element 2^31 and the last rows equal the reference"""
    from qsparse_b200 import ops
    dtype, L, fmt = (torch.float32, 4096, "nvfp4") if case == "float32-aligned" else (torch.bfloat16, 4100, "mxfp4")
    rows = (1 << 31) // L + 3
    g = torch.Generator(device="cuda").manual_seed(0)
    x = torch.randn(rows, L, device="cuda", dtype=dtype, generator=g)
    w = torch.full((1,), 3.0, device="cuda")
    r0 = (1 << 31) // L
    sel = [r0 - 1, r0, r0 + 1, rows - 1]
    ref = x[sel].float().cpu().numpy()
    y = ops.fq_block_fwd(x, fmt, rows, L, w)
    same_bits(y[sel].cpu().numpy(), bs.fake_quant(ref, fmt, np.float32(3)))
    del y
    codes, scales = ops.block_export(x, fmt, rows, L, w)
    c_ref, s_ref = bs.export(ref, fmt, np.float32(3))
    assert np.array_equal(codes[sel].cpu().numpy(), c_ref)
    assert np.array_equal(scales[sel].cpu().numpy(), s_ref)
    del x, codes, scales
    torch.cuda.empty_cache()


# ----------------------------------------------------------------------------- layers
def test_nvfp4_layers_train_eval_state_and_grad():
    """an activation layer and a quantized Linear: the timeout, the w EMA (DecimalQuantizer's at one bit) against
    the reference over several steps, eval on the stored w, the state_dict keys and the identity backward"""
    import qsparse_b200 as qs
    qs.set_qsparse_options(log_on_created=False)
    torch.manual_seed(0)
    act = qs.quantize(bits=8, channelwise=-1, timeout=2, callback=qs.BlockScaledQuantizer("nvfp4")).cuda()
    lin = qs.quantize(nn.Linear(64, 48), bits=4, channelwise=-1, timeout=1,
                      callback=qs.BlockScaledQuantizer("nvfp4")).cuda()
    w_act, t_act = np.zeros(1, np.float32), 0
    w_lin, t_lin = np.zeros(1, np.float32), 0
    raw_w = lin._parameters["weight"]
    for step in range(6):
        x = (torch.randn(16, 64) * (step + 1)).cuda().requires_grad_()
        y = act(x)
        if step < 2:
            assert y is x
        else:
            xn = x.detach().cpu().numpy()
            w_act = orc.scale_ema(w_act, np.abs(xn).max(keepdims=True), 1, t_act)
            t_act += 1
            same_bits(act.weight.detach().cpu().numpy().reshape(-1), w_act)
            same_bits(y.detach().cpu().numpy(), bs.fake_quant(xn, "nvfp4", w_act[0]))
        g = torch.randn_like(y)
        y.backward(g)
        assert torch.equal(x.grad.view(torch.int32), g.view(torch.int32))
        wq = lin.weight                                  # the weight's QuantizeLayer runs on every read
        if step >= 1:
            wn = raw_w.detach().cpu().numpy()
            w_lin = orc.scale_ema(w_lin, np.abs(wn).max(keepdims=True), 1, t_lin)
            t_lin += 1
            same_bits(wq.detach().cpu().numpy(), bs.fake_quant(wn, "nvfp4", w_lin[0]))
    assert sorted(act.state_dict()) == ["_n_updates", "weight"] and tuple(act.weight.shape) == (1, 1)
    act.eval()
    x = torch.randn(16, 64).cuda()
    before = act.weight.detach().clone()
    same_bits(act(x).cpu().numpy(), bs.fake_quant(x.cpu().numpy(), "nvfp4", w_act[0]))
    assert torch.equal(act.weight, before)


@pytest.mark.parametrize("fmt", ["mxfp8", "mxfp4"])
def test_mx_layer_only_counts(fmt):
    import qsparse_b200 as qs
    qs.set_qsparse_options(log_on_created=False)
    layer = qs.quantize(bits=8, channelwise=-1, timeout=1, callback=qs.BlockScaledQuantizer(fmt)).cuda()
    for step in range(4):
        x = torch.randn(8, 96).cuda()
        y = layer(x)
        if step >= 1:
            same_bits(y.cpu().numpy(), bs.fake_quant(x.cpu().numpy(), fmt))
    assert layer.callback.t == 3 and float(layer.weight) == 0.0


def _pq_net(fmt):
    import qsparse_b200 as qs
    return nn.Sequential(
        nn.Linear(64, 128),
        nn.Sequential(nn.Sequential(nn.Identity(), qs.prune(sparsity=0.5, dimensions={1}, start=1, interval=1,
                                                            repetition=2)),
                      qs.quantize(bits=8, channelwise=-1, timeout=2, callback=qs.BlockScaledQuantizer(fmt))),
        qs.quantize(nn.Linear(128, 32), bits=4, channelwise=-1, timeout=1, callback=qs.BlockScaledQuantizer("nvfp4")),
        qs.quantize(bits=8, channelwise=-1, timeout=1, callback=qs.BlockScaledQuantizer("mxfp8")),
    ).cuda()


def test_fusion_pass_leaves_block_scaled_sites_unfused():
    """fuse_prune_quantize keeps working on a model with these callbacks; their sites never take the fused step and
    compute what the unconverted model computes"""
    import qsparse_b200 as qs
    from qsparse_b200.fused import FusedPruneQuantSequential
    qs.set_qsparse_options(log_on_created=False)
    torch.manual_seed(0)
    plain = _pq_net("nvfp4")
    fused = qs.fuse_prune_quantize(copy.deepcopy(plain))
    sites = [m for m in fused.modules() if isinstance(m, FusedPruneQuantSequential)]
    assert sites
    for step in range(6):
        x = torch.randn(32, 64).cuda()
        a, b = plain(x), fused(x)
        assert torch.equal(a.view(torch.int32), b.view(torch.int32)), step
        a.sum().backward()
        b.sum().backward()
    assert all(m.fused_steps == 0 for m in sites)
    for (ka, va), (kb, vb) in zip(sorted(plain.state_dict().items()), sorted(fused.state_dict().items())):
        assert ka == kb and torch.equal(va, vb), ka


def test_graphed_steps_equal_eager_steps():
    import qsparse_b200 as qs
    from qsparse_b200 import graphs
    qs.set_qsparse_options(log_on_created=False)
    torch.manual_seed(0)
    rng = np.random.default_rng(3)
    # a batch of 64: the prune step of a [batch, 128] activation is capturable from 64 rows per channel on
    data = [(torch.from_numpy(rng.standard_normal((64, 64)).astype(np.float32)).cuda(),
             torch.from_numpy(rng.standard_normal((64, 32)).astype(np.float32)).cuda()) for _ in range(12)]
    base = qs.fuse_prune_quantize(_pq_net("mxfp4")).train()
    for i in range(4):                                   # past every timeout and the prune schedule, eagerly
        (base(data[i][0]) * data[i][1]).sum().backward()
    nets = [copy.deepcopy(base), copy.deepcopy(base)]
    opts = [torch.optim.SGD(n.parameters(), lr=0.01) for n in nets]
    static = [t.clone() for t in data[0]]

    def step(net, opt):
        opt.zero_grad(set_to_none=True)
        loss = (net(static[0]) * static[1]).sum()
        loss.backward()
        opt.step()
        return loss.detach().clone()

    def feed(i):
        for s, t in zip(static, data[i % 12]):
            s.copy_(t)

    eager = []
    for i in range(4, 12):
        feed(i)
        eager.append(step(nets[1], opts[1]))
    warm = iter(range(4, 7))

    class _Step:
        n = 0

        def __call__(self):
            self.n += 1
            if self.n <= 3:
                feed(next(warm))
            return step(nets[0], opts[0])
    gs = graphs.GraphedTrainStep(nets[0], _Step(), warmup=3)
    replayed = []
    for i in range(7, 12):
        feed(i)
        replayed.append(gs.replay().clone())
    gs.sync_host()
    assert torch.equal(torch.stack(eager[3:]).view(torch.int32), torch.stack(replayed).view(torch.int32))
    sa, sb = nets[0].state_dict(), nets[1].state_dict()
    assert sorted(sa) == sorted(sb)
    bad = [k for k in sa if not torch.equal(sa[k], sb[k])]
    assert not bad, bad
    cbs = [[m.t for m in n.modules() if isinstance(m, qs.BlockScaledQuantizer)] for n in nets]
    assert cbs[0] == cbs[1]
