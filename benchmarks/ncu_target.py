"""Short workload for ncu captures: a few fused prune->quantize training steps on the
config-2 tensor plus one config-3 and one config-4 pass."""
import sys
from pathlib import Path

import torch

sys.path.insert(0, str(Path(__file__).resolve().parent.parent))
from qsparse_b200 import ops  # noqa: E402

dev = torch.device("cuda:0")
torch.manual_seed(2)
shape, layout = (256, 64, 56, 56), (256, 64, 3136)
x = torch.relu(torch.randn(shape, device=dev))
g = torch.randn(shape, device=dev)
y = torch.empty_like(x)
mag = torch.zeros(64, device=dev)
mask = torch.ones(64, dtype=torch.bool, device=dev)
scale = torch.zeros(1, device=dev)
dec = torch.zeros(1, device=dev)
steps = int(sys.argv[1]) if len(sys.argv) > 1 else 3
for t in range(steps):
    ws = ops.reduce_partials(x, layout)
    ops.prune_quant_step_params(mag, mask, scale, dec, ws, layout, 256 * 3136.0, t, 1, t > 0, 48, 8, t, True)
    ops.fq_pow2_fwd(x, dec, layout, mask=mask, out=y)
    gc = g.clone()
    ops.ste_bwd(gc, dec, True, 8, 0, layout, mask=mask, clamp_in_place=False, want_gx=True)
# dense variants for the roofline (no read skipping)
ops.fq_pow2_fwd(x, dec, (1, 1, x.numel()), out=y)
ops.ste_bwd(g, dec, True, 8, 0, (1, 1, x.numel()))
w = torch.randn(4096, 4096, device=dev) * 0.02
st = ops.reduce_stats(w, (1, 4096, 4096), minmax=True)
lines = torch.zeros(4096, 2, device=dev)
ops.lines_ema_(lines, st["min"], st["max"], 1)
ops.fq_line_fwd(w, lines, 4, True, (1, 4096, 4096))
n4 = 1 << 26
wt = torch.randn(n4, device=dev) * 0.02
magf = wt.abs()
ops.magnitude_ema_full_(magf, wt, 3)
thr = ops.kth_value(magf, n4 // 2)
mk = torch.empty(n4, dtype=torch.bool, device=dev)
ops.mask_build_apply(magf, thr, wt, mk)
# config 3 through the row-resident fused kernel
lines2 = torch.zeros(4096, 2, device=dev)
ops.row_quant_fused_(w, lines2, ops.ROW_LINE, 4, 1, True)
sc2 = torch.zeros(4096, 1, device=dev)
ops.row_quant_fused_(w, sc2, ops.ROW_SCALER, 4, 0)
# config 4 as a weight set: multi-tensor EMA, batched select, multi-tensor mask build + apply
del wt, magf, mk
from qsparse_b200 import parallel  # noqa: E402
shapes = [(512, 512, 3, 3)] * 28 + [(256, 4096)]
wset = [torch.randn(s, device=dev) * 0.02 for s in shapes]
mags = [v.abs() * 0.9 for v in wset]
masks = [torch.ones(v.shape, dtype=torch.bool, device=dev) for v in wset]
outs = [torch.empty_like(v) for v in wset]
parallel.prune_weight_set_step(wset, mags, masks, outs, 3, 0.5)
torch.cuda.synchronize()
print("done")
