"""TEST / BENCH INFRASTRUCTURE — not part of the product (only tests/ and bench.py's baseline legs import it).

The reference's own ATen op sequence for the hot path, restated as plain eager torch ops in the
same order, so it can run on CUDA tensors on the GPU box (where /root/reference does not exist)
as the "PyTorch-eager on the same B200" baseline BASELINE.md asks for.  Every function cites the
reference lines whose ops it repeats.  No qsparse_b200 kernel is involved: this is what a user of
mlzxy/qsparse gets on a B200 today, and the bar the hand-written kernels have to beat.
"""
from __future__ import annotations

import torch


def squeeze_tensor_to_shape(x, shape):
    """ref qsparse/util.py:92-98: one `mean(i, keepdim=True)` per squeezed axis, in axis order"""
    for i, (sx, sm) in enumerate(zip(x.shape, shape)):
        if sx != sm:
            x = x.mean(i, keepdim=True)
    return x


def calculate_mask_given_importance(importance, sparsity):
    """ref qsparse/util.py:113-117: full sort, threshold = values[idx + 1], mask = importance >= thr"""
    values = importance.flatten().sort()[0]
    n = len(values)
    idx = max(int(sparsity * n - 1), 0)
    return importance >= values[idx + 1]


class PruneQuantizeEager:
    """`Sequential(PruneLayer(dimensions={1}, MagnitudePruningCallback()), QuantizeLayer(bits,
    channelwise=-1, DecimalQuantizer()))` in its steady state (pruning started, quantizer past its
    timeout), forward + backward, as the reference executes it (ref qsparse/sparse.py:82-122,
    qsparse/quantize.py:30-77,312-349,501-508).  Host synchronisations (`.item()`) are kept where
    the reference has them."""

    def __init__(self, channels, device, sparsity=0.75, bits=8):
        self.sparsity, self.bits = sparsity, bits
        self.t = torch.zeros(1, dtype=torch.int64, device=device)          # callback.t (nn.Parameter)
        self.magnitude = torch.zeros(1, channels, 1, 1, device=device)
        self.mask = torch.ones(1, channels, 1, 1, dtype=torch.bool, device=device)
        self.weight = torch.zeros(1, 1, device=device)                     # QuantizeLayer.weight
        self.tq = 0                                                        # DecimalQuantizer.t (python int)
        self.n_updates = torch.zeros(1, dtype=torch.int32, device=device)  # QuantizeLayer._n_updates

    @torch.no_grad()
    def forward(self, x):
        # ---- MagnitudePruningCallback.forward (sparse.py:100-122) ----
        t_item = self.t.item()                                             # sparse.py:108 (host sync)
        # update_magnitude (sparse.py:82-89)
        xa = squeeze_tensor_to_shape(x.abs(), self.magnitude.shape)        # abs + 3 means
        t = self.t.item()                                                  # sparse.py:88 (host sync)
        self.magnitude[:] = (t * self.magnitude + xa) / (t + 1)
        if t_item > 0:
            # prune_and_update_mask (sparse.py:58-66)
            self.mask[:] = calculate_mask_given_importance(self.magnitude, self.sparsity)
        out = x * self.mask                                                # sparse.py:66 / :116
        self.t += 1
        # ---- QuantizeLayer.forward (quantize.py:495-518): t = _n_updates.item(), optimize, callback ----
        _ = self.n_updates.item()                                          # quantize.py:496 (host sync)
        # DecimalQuantizer.optimize (quantize.py:327-349), channel_index == -1
        a = out.abs().view(1, -1)
        new_weight = (a.max(dim=1).values / (2 ** (self.bits - 1))).view(1, 1)
        if self.tq == 0:
            self.weight = new_weight
        else:
            self.weight[:] = (self.tq * self.weight + new_weight) / (self.tq + 1)
        self.tq += 1
        # DecimalQuantizer.quantize (quantize.py:312-325)
        decimal = (1 / self.weight).nan_to_num(posinf=1, neginf=1).log2().round()
        # DecimalQuantization.forward (quantize.py:43-63)
        limit = 2.0 ** (self.bits - 1)
        tof = 2.0 ** -decimal
        toi = 2.0 ** decimal
        q = (out * toi).int()
        q.float().clamp_(-limit, limit - 1)                                # quantize.py:59-62 (result discarded)
        y = q.float() * tof
        self.n_updates += 1
        self._saved = (limit, tof)
        return y

    @torch.no_grad()
    def backward(self, grad_output):
        limit, tof = self._saved
        # DecimalQuantization.backward (quantize.py:67-77)
        v = grad_output.clamp_((-limit) * tof, (limit - 1) * tof)
        v[v != grad_output] = 0
        # backward of `x * mask` (sparse.py:66)
        return v * self.mask


class WeightLineQuantEager:
    """config 3: `quantize(nn.Linear(4096, 4096), bits=4, channelwise=0, timeout=1,
    callback=AdaptiveQuantizer())`, the training access of `.weight`
    (ref qsparse/quantize.py:140-185 LineQuantization, :393-430 AdaptiveQuantizer.optimize)."""

    def __init__(self, bits=4):
        self.bits = bits
        self.lines = None
        self.t = 0

    @torch.no_grad()
    def forward(self, w):
        x = w.contiguous().view(-1, w[0].numel())                           # channel_index == 0, not batched
        lb = x.min(dim=1).values
        ub = x.max(dim=1).values
        sample = torch.cat([lb.view(-1, 1), ub.view(-1, 1)], dim=1)
        self.t += 1
        self.lines = sample if self.lines is None else (self.lines * (self.t - 1) + sample) / self.t
        # LineQuantization.forward, training (float zero point), quantize.py:148-181
        lines = self.lines
        shape = [1] * w.dim()
        shape[0] = -1
        lo, hi = lines[:, 0].view(shape), lines[:, 1].view(shape)
        xc = torch.clamp(w, lo, hi)
        step = (hi - lo) / (2 ** self.bits)
        step[step == 0] = 0.0001
        qa = ((xc - lo) / step).round()
        qa.clamp_(0, 2 ** self.bits - 1)
        return qa * step + lo


class UnstructuredPruneEager:
    """config 4: `MagnitudePruningCallback(running_average=True)` with a full-size mask on one weight tensor
    (ref qsparse/sparse.py:58-66,82-89, qsparse/util.py:103-117)."""

    def __init__(self, like, sparsity):
        self.sparsity = sparsity
        self.magnitude = torch.zeros_like(like)
        self.mask = torch.ones(like.shape, dtype=torch.bool, device=like.device)
        self.t = 0

    @torch.no_grad()
    def forward(self, w):
        xa = w.abs()
        self.magnitude[:] = (self.t * self.magnitude + xa) / (self.t + 1)
        if self.t > 0:
            self.mask[:] = calculate_mask_given_importance(self.magnitude, self.sparsity)
        self.t += 1
        return w * self.mask


@torch.no_grad()
def masked_pow2_fwd_bwd(x, g, mask, decimal, bits=8):
    """config 5: `quantize_with_decimal(x * mask, bits, decimal)` forward and its backward
    (ref qsparse/quantize.py:43-77 and the `x * mask` of sparse.py:116)."""
    limit = 2.0 ** (bits - 1)
    tof, toi = 2.0 ** -decimal, 2.0 ** decimal
    out = x * mask
    q = (out * toi).int()
    q.float().clamp_(-limit, limit - 1)
    y = q.float() * tof
    v = g.clamp_((-limit) * tof, (limit - 1) * tof)
    v[v != g] = 0
    return y, v * mask


# ---------------------------------------------------------------------------------------------------------
# config 1: the reference's LAYERS as eager nn.Modules (control flow of qsparse/quantize.py:473-518 and
# qsparse/sparse.py:99-122,215-273 incl. their `.item()` host syncs), so that the converted MNIST net of
# examples/mnist.py can be timed on the GPU box without the reference tree.  Checked step for step against the
# reference's recorded run in tests/test_torch_eager_vs_reference.py.
# ---------------------------------------------------------------------------------------------------------
import torch.nn as nn
import torch.nn.functional as F


class _DecimalFn(torch.autograd.Function):
    """ref qsparse/quantize.py:30-77"""

    @staticmethod
    def forward(ctx, input, bits, decimal):
        limit = 2.0 ** (bits - 1)
        tof = 2.0 ** -decimal
        toi = 2.0 ** decimal
        ctx.save_for_backward(torch.tensor(limit), tof)
        q = (input * toi).int()
        q.float().clamp_(-limit, limit - 1)
        return q.float() * tof

    @staticmethod
    def backward(ctx, grad_output):
        limit, tof = ctx.saved_tensors
        v = grad_output.clamp_((-limit) * tof, (limit - 1) * tof)
        v[v != grad_output] = 0
        return v, None, None


class _ScalerFn(torch.autograd.Function):
    """ref qsparse/quantize.py:86-131"""

    @staticmethod
    def forward(ctx, input, bits, scaler):
        limit = 2.0 ** (bits - 1)
        ctx.save_for_backward(torch.tensor(limit), scaler)
        q = (input / scaler).round().int()
        q.float().clamp_(-limit, limit - 1)
        return q.float() * scaler

    @staticmethod
    def backward(ctx, grad_output):
        limit, scaler = ctx.saved_tensors
        v = grad_output.clamp_((-limit) * scaler, (limit - 1) * scaler)
        v[v != grad_output] = 0
        return v, None, None


class EagerQuantizeLayer(nn.Module):
    """per-tensor (channelwise = -1) QuantizeLayer with a Decimal / Scaler quantizer"""

    def __init__(self, bits=8, timeout=10, kind="scaler"):
        super().__init__()
        self.bits, self.timeout, self.kind = bits, timeout, kind
        self.cb_t = 0
        self._quantized = False

    def forward(self, x):
        if not hasattr(self, "_n_updates"):
            self.weight = nn.Parameter(torch.zeros(1, 1).to(x.device), requires_grad=False)
            self._n_updates = nn.Parameter(torch.zeros(1, dtype=torch.int).to(x.device), requires_grad=False)
        t = self._n_updates.item()
        out = x
        if self.timeout > 0:
            if t >= self.timeout:
                if self.training:
                    with torch.no_grad():
                        a = x.abs().view(1, -1)
                        new_weight = (a.max(dim=1).values / (2 ** (self.bits - 1))).view(1, 1)
                    if self.cb_t == 0:
                        self.weight.data[:] = new_weight
                    else:
                        self.weight.data[:] = (self.cb_t * self.weight + new_weight) / (self.cb_t + 1)
                    self.cb_t += 1
                    self._quantized = True
                if self._quantized:
                    if self.kind == "decimal":
                        d = (1 / self.weight).nan_to_num(posinf=1, neginf=1).log2().round()
                        out = _DecimalFn.apply(x, self.bits, d)
                    else:
                        out = _ScalerFn.apply(x, self.bits, self.weight)
            if self.training:
                self._n_updates += 1
        return out


class EagerPruneLayer(nn.Module):
    """structured channel prune (dimensions = {1}), MagnitudePruningCallback(running_average=True)"""

    def __init__(self, sparsity=0.5, start=20, interval=10, repetition=4):
        super().__init__()
        self.sparsity, self.start, self.interval, self.repetition = sparsity, start, interval, repetition
        self.schedules = [start + interval * i for i in range(repetition)]
        self.rampup_interval = interval
        self._n = nn.Parameter(torch.tensor(-1, dtype=torch.int), requires_grad=False)
        self.t = nn.Parameter(torch.full((1,), -1), requires_grad=False)

    def forward(self, x):
        if self._n.dim() == 0:
            shape = [1 if i != 1 else s for i, s in enumerate(x.shape)]
            self.mask = nn.Parameter(torch.ones(*shape, dtype=torch.bool).to(x.device), requires_grad=False)
            self._n = nn.Parameter(torch.zeros(1, dtype=torch.int).to(x.device), requires_grad=False)
            self._cur = nn.Parameter(torch.zeros(1).to(x.device), requires_grad=False)
            self.t = nn.Parameter(self.t.data.to(x.device), requires_grad=False)
        if (self._n.item() in self.schedules) and self.training:
            ratio = (1.0 - (self._n.item() - self.start + self.rampup_interval) / (self.interval * self.repetition)) ** 3
            self._cur[0] = self.sparsity * (1 - ratio)
            _ = self._cur.item()                                          # the reference logs it (sparse.py:258)
        if not self.training:
            return x * self.mask
        n_updates = self._n.item()
        if n_updates >= self.start:
            sparsity = self._cur.item()
            if self.t.item() == -1:                                        # callback.initted
                self.magnitude = nn.Parameter(torch.zeros(*self.mask.shape, device=x.device), requires_grad=False)
                self.t.data[:] = 0
            t_item = self.t.item()
            with torch.no_grad():
                xa = squeeze_tensor_to_shape(x.abs(), self.magnitude.shape)
                t = self.t.item()
                self.magnitude.data[:] = (t * self.magnitude + xa) / (t + 1)
            if sparsity >= 0 and t_item > 0:
                self.mask.data[:] = calculate_mask_given_importance(self.magnitude, sparsity)
            out = x * self.mask
            self.t += 1
        else:
            out = x
        self._n += 1
        return out


class _QuantizedWeightLayer(nn.Module):
    """`quantize(layer)`: the layer runs with quantize_layer(weight) (ref qsparse/imitation.py)"""

    def __init__(self, layer, kind):
        super().__init__()
        self.layer = layer
        self.q = EagerQuantizeLayer(8, 10, kind)

    def forward(self, x):
        w = self.q(self.layer.weight)
        if isinstance(self.layer, nn.Conv2d):
            return F.conv2d(x, w, self.layer.bias, self.layer.stride, self.layer.padding)
        return F.linear(x, w, self.layer.bias)


def build_mnist_eager(kind="scaler"):
    """the converted Net of BASELINE config 1 (oracle/gen_golden_config1.py::build) with eager reference layers:
    input quantize; conv/linear weights quantized; ReLU -> prune -> quantize after the first two ReLUs, ReLU ->
    quantize after the third."""
    torch.manual_seed(1)
    conv1, bn1 = nn.Conv2d(1, 32, 3, 1), nn.BatchNorm2d(32)
    conv2, bn2 = nn.Conv2d(32, 64, 3, 1), nn.BatchNorm2d(64)
    fc1, bn3, fc2 = nn.Linear(9216, 128), nn.BatchNorm1d(128), nn.Linear(128, 10)

    def site(prune):
        mods = [nn.ReLU()] + ([EagerPruneLayer()] if prune else []) + [EagerQuantizeLayer(8, 10, kind)]
        return nn.Sequential(*mods)

    class Net(nn.Module):
        def __init__(self):
            super().__init__()
            self.inq = EagerQuantizeLayer(8, 10, kind)
            self.conv_part = nn.Sequential(_QuantizedWeightLayer(conv1, kind), bn1, site(True),
                                           _QuantizedWeightLayer(conv2, kind), bn2, site(True), nn.MaxPool2d(2))
            self.linear_part = nn.Sequential(nn.Flatten(), _QuantizedWeightLayer(fc1, kind), bn3, site(False),
                                             _QuantizedWeightLayer(fc2, kind))

        def forward(self, x):
            return F.log_softmax(self.linear_part(self.conv_part(self.inq(x))), dim=1)

    return Net()
