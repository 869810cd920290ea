"""oracle/torch_eager.py (the reference's ATen op sequence restated as plain torch ops — the
"PyTorch-eager on the same B200" baseline of bench.py) against the outputs the unmodified reference
(mlzxy/qsparse v2.0.1) produced on CPU tensors, recorded in tests/golden/ by oracle/gen_golden.py and
oracle/gen_golden_config1.py.  Every comparison is bit-exact.  Most compare with a recorded array directly;
where the recordings hold no array for a combined step, the expected value is derived from recorded
arrays, as the docstring of that test says."""
import numpy as np
import torch

from tests.conftest import ROOT, bits_equal


def _t(a):
    return torch.from_numpy(np.array(a, copy=True))


def test_prune_quantize_step_matches_reference_layers(golden):
    """PruneQuantizeEager, the step bench.py times as the PyTorch-eager baseline of config 2.

    Against raw recordings: the mask and magnitude of every step of the reference's six-step channel-prune
    run (`cb/struct`), and the first step's forward, backward and in-place clamped grad_output.
    Against derived values: on every step of that run, y, the averaged scale and gx must equal
    EagerQuantizeLayer (DecimalQuantizer, pinned to the reference's `layer/q_dec` run in
    test_mnist_eager_net_matches_reference_converted_net) applied to the reference's recorded masked
    output `cb/struct_out`, with its gradient times the recorded mask; y and gx must be zero on every
    channel the recorded mask prunes.  max|x| is 128 on every step of that run, so its averaged scale never
    moves; a second, seeded run with a growing input scale checks y, mask, the averaged scale and gx against
    EagerPruneLayer -> EagerQuantizeLayer (both pinned to the reference's layer runs in that test)."""
    from oracle.torch_eager import EagerPruneLayer, EagerQuantizeLayer, PruneQuantizeEager
    g = golden
    xs = g["cb/struct_x"]
    C = xs.shape[2]
    eager = PruneQuantizeEager(C, "cpu", sparsity=0.5, bits=8)
    q = EagerQuantizeLayer(bits=8, timeout=1, kind="decimal").train()
    q(torch.zeros(1, C, 1, 1))          # the pass-through call before the quantizer's timeout
    gen = torch.Generator().manual_seed(0)
    n_pruned = n_clamped = n_kept = 0
    for t in range(len(xs)):
        y = eager.forward(_t(xs[t]))
        mask_ref = g["cb/struct_mask"][t]
        assert np.array_equal(eager.mask.numpy(), mask_ref), t
        assert bits_equal(eager.magnitude, g["cb/struct_mag"][t]), t
        out_ref = _t(g["cb/struct_out"][t]).requires_grad_(True)
        y_ref = q(out_ref)
        assert bits_equal(y, y_ref.detach()), t
        assert bits_equal(eager.weight, q.weight.detach()), t
        grad = torch.randn(xs.shape[1:], generator=gen) * 100     # the clamp bound is 128 here
        gx = eager.backward(grad.clone())
        y_ref.backward(grad.clone())
        assert bits_equal(gx, out_ref.grad * _t(mask_ref)), t
        pruned = ~mask_ref.reshape(-1)
        assert not y[:, pruned].any() and not gx[:, pruned].any(), t
        n_pruned += int(pruned.sum())
        n_clamped += int((out_ref.grad != grad).sum())
        n_kept += int((out_ref.grad == grad).sum())
    assert n_pruned > 0 and n_clamped > 0 and n_kept > 0      # the run prunes channels, clamps some gradients
    # the running average of the scale over steps at 75 % sparsity
    C = 12
    prune = EagerPruneLayer(sparsity=0.75, start=0, interval=1, repetition=1).train()    # 75 % from step 0
    q = EagerQuantizeLayer(bits=8, timeout=1, kind="decimal").train()
    q(torch.zeros(1, C, 1, 1))
    eager = PruneQuantizeEager(C, "cpu", sparsity=0.75, bits=8)
    channel_scale = torch.linspace(0.2, 2.0, C).view(1, C, 1, 1)
    weights = set()
    for t in range(5):
        x = torch.relu(torch.randn(6, C, 9, 9, generator=gen)) * channel_scale * (1 + t)
        xin = x.clone().requires_grad_(True)
        y_ref = q(prune(xin))
        y = eager.forward(x.clone())
        assert torch.equal(eager.mask, prune.mask), t
        assert bits_equal(y, y_ref.detach()), t
        assert bits_equal(eager.weight, q.weight.detach()), t
        grad = torch.randn(x.shape, generator=gen) * 30
        gx = eager.backward(grad.clone())
        y_ref.backward(grad.clone())
        assert bits_equal(gx, xin.grad), t
        weights.add(float(q.weight))
    assert len(weights) == 5 and not eager.mask.all()
    # quantize half: the first step (mask still all ones, DecimalQuantizer weight = max|x| / 2^(bits-1)) is
    # quantize_with_decimal forward and backward; the scale of x selects the decimal (128 -> 0, 4 -> 5, 256 -> -1)
    x4, gr = g["pow2/x"], g["bwd/g"]
    assert np.abs(x4).max() == 128
    for scale, d in ((1.0, 0), (1 / 32, 5), (2.0, -1)):
        eager = PruneQuantizeEager(x4.shape[1], "cpu", sparsity=0.75, bits=8)
        y = eager.forward(_t(x4 * np.float32(scale)))
        assert float((1 / eager.weight).log2().round()) == d
        if d == 0:
            assert bits_equal(y, g["pow2/y_d0"])
        go = _t(gr)
        gx = eager.backward(go)
        if d != 0:
            assert bits_equal(gx, g[f"bwd/pow2_b8_d{d}_f0_gx"]), d
            assert bits_equal(go, g[f"bwd/pow2_b8_d{d}_f0_go"]), d      # grad_output clamped in place


def test_weight_line_quant_matches_reference_layer(golden):
    from oracle.torch_eager import WeightLineQuantEager
    g = golden
    # AdaptiveQuantizer.optimize, channel_index=0, not batched: the running average of per-row [min, max]
    xs = g["dq/xs"]
    eager = WeightLineQuantEager(bits=4)
    for t in range(len(xs)):
        eager.forward(_t(xs[t]))
        assert bits_equal(eager.lines, g["aq/lines_ci0_b0"][t]), t
    # LineQuantization forward in training: quantize(bits=8, channelwise=1, AdaptiveQuantizer()) on a batch of
    # one after its timeout, with the channel axis moved to the front
    x = _t(g["layer/x"]).transpose(0, 1)
    eager = WeightLineQuantEager(bits=8)
    for t in range(3):
        y = eager.forward(x).transpose(0, 1)
        assert bits_equal(y, g["layer/q_adp_out"][3 + t]), t
    assert bits_equal(eager.lines, g["layer/q_adp_weight"])


def test_unstructured_prune_matches_reference_callback(golden):
    from oracle.torch_eager import UnstructuredPruneEager
    g = golden
    xs = g["cb/unstruct_x"]                  # MagnitudePruningCallback() with a full-size mask, 50 %
    eager = UnstructuredPruneEager(_t(xs[0]), 0.5)
    for t in range(len(xs)):
        ye = eager.forward(_t(xs[t]))
        assert bits_equal(ye, g["cb/unstruct_out"][t]), t
        assert np.array_equal(eager.mask.numpy(), g["cb/unstruct_mask"][t]), t
        assert bits_equal(eager.magnitude, g["cb/unstruct_mag"][t]), t


def test_mnist_eager_net_matches_reference_converted_net(golden):
    """build_mnist_eager (the config-1 GPU-eager baseline of bench.py) trains step for step like the
    reference's convert()'ed net on CPU: identical losses for all 60 recorded steps (warm-up, quantization
    start at 10, pruning start at 20 and the ramp points), and its prune / quantize layers reproduce the
    reference's layer-level runs."""
    import torch.nn.functional as F
    from oracle.gen_golden_config1 import STEPS, data
    from oracle.torch_eager import EagerPruneLayer, EagerQuantizeLayer, build_mnist_eager
    g = golden
    x = _t(g["layer/x"])
    for kind, key in (("decimal", "layer/q_dec"), ("scaler", "layer/q_scl")):
        q = EagerQuantizeLayer(bits=8, timeout=3, kind=kind).train()
        outs = np.stack([q(x.clone()).detach().numpy() for _ in range(6)])
        assert bits_equal(outs, g[key + "_out"]) and bits_equal(q.weight.detach(), g[key + "_weight"]), kind
    p = EagerPruneLayer(sparsity=0.5, start=2, interval=2, repetition=3).train()
    px = _t(g["layer/px"])
    for t in range(12):
        assert bits_equal(p(px.clone()), g["layer/p_out"][t]), t
        assert np.array_equal(p.mask.numpy(), g["layer/p_mask"][t]), t

    ref = np.load(ROOT / "tests" / "golden" / "config1_mnist.npz")
    threads = torch.get_num_threads()
    # the reference ran with 8 intra-op threads; CPU convolution splits its sums by thread, and a different
    # split changes the last bits of the losses within the first few steps.  The comparison also assumes
    # that oneDNN picks convolution kernels that round alike on every host CPU: if these losses differ on
    # one host only, look there first.
    torch.set_num_threads(8)
    try:
        for kind in ("scaler", "decimal"):
            mine = build_mnist_eager(kind)
            mine.train()
            opt = torch.optim.Adadelta([p for p in mine.parameters() if p.requires_grad], lr=1.0)
            losses = []
            for step in range(STEPS):
                xb, yb = data(step)
                opt.zero_grad()
                loss = F.nll_loss(mine(xb), yb)
                loss.backward()
                opt.step()
                losses.append(loss.item())
            np.testing.assert_array_equal(np.array(losses), ref[f"{kind}/loss"], err_msg=kind)
    finally:
        torch.set_num_threads(threads)
