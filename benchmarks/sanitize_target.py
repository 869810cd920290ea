"""Small invocations of every kernel family for compute-sanitizer (memcheck / racecheck / synccheck):
    compute-sanitizer --tool racecheck python benchmarks/sanitize_target.py
"""
import sys
from pathlib import Path

import torch

sys.path.insert(0, str(Path(__file__).resolve().parent.parent))
from qsparse_b200 import ops, parallel  # noqa: E402

dev = torch.device("cuda:0")
g = torch.Generator(device=dev).manual_seed(1)
# select: sampled route (n >= 2^22), generic route, batched, ties
v = torch.randn((1 << 22) + 5, device=dev, generator=g)
for k in (0, v.numel() // 2, v.numel() - 1):
    ops.kth_value(v, k)
    ops.kth_value(v, k, take_abs=True)
ops.kth_value(torch.relu(v), v.numel() // 3)
ops.kth_value(v[: 100003], 5000)
ops.kth_value(v[1: 70001], 5000)
vs = [torch.randn(s, device=dev, generator=g) for s in (200_000, 131_072, 999, 300_000)]
ops.kth_value_batched(vs, [s.numel() // 2 for s in vs])
# row-resident kernels: warp per row, CTA per row
for shape in ((33, 8), (64, 288), (130, 1024), (48, 4096), (3, 8200), (2, 16384)):
    x = torch.randn(shape, device=dev, generator=g)
    for kind, w in ((ops.ROW_LINE, 2), (ops.ROW_SCALER, 1), (ops.ROW_DECIMAL, 1)):
        ops.row_quant_fused_(x, torch.zeros(shape[0], w, device=dev), kind, 4, 1 if kind == ops.ROW_LINE else 0)
# multi-tensor EMA / mask, weight-set step
shapes = [(64, 32, 3, 3), (40, 1000), (7, 13, 5), (256, 64, 3, 3)]
ws = [torch.randn(s, device=dev, generator=g) for s in shapes]
mags = [torch.zeros_like(w) for w in ws]
masks = [torch.ones(w.shape, dtype=torch.bool, device=dev) for w in ws]
outs = [torch.empty_like(w) for w in ws]
for t in range(2):
    parallel.prune_weight_set_step(ws, mags, masks, outs, t, 0.5)
# K9 fused prune step: sampled route (ties, NaN), generic route for the small tensors
xs9 = [torch.randn(s, device=dev, generator=g) * 0.02 for s in (300_000, 131_072 + 5, 999)]
xs9[0] = torch.relu(xs9[0])
xs9[1][::1009] = float("nan")
mg9 = [torch.zeros_like(x) for x in xs9]
mk9 = [torch.ones(x.shape, dtype=torch.bool, device=dev) for x in xs9]
ot9 = [torch.empty_like(x) for x in xs9]
for t in range(2):
    ops.prune_unstructured_step_batched_(mg9, xs9, mk9, ot9, [x.numel() // 2 for x in xs9], t)
# fused training step pieces + maps + export
x = torch.relu(torch.randn(8, 16, 14, 14, device=dev, generator=g))
layout = (8, 16, 196)
mag = torch.zeros(16, device=dev)
mask = torch.ones(16, dtype=torch.bool, device=dev)
scale, dec = torch.zeros(1, device=dev), torch.zeros(1, device=dev)
for t in range(2):
    wsp = ops.reduce_partials(x, layout)
    ops.prune_quant_step_params(mag, mask, scale, dec, wsp, layout, 8 * 196.0, t, 1, t > 0, 8, 8, t, True)
    y = ops.fq_pow2_fwd(x, dec, layout, mask=mask)
    ops.ste_bwd(torch.randn_like(x), dec, True, 8, 0, layout, mask=mask, clamp_in_place=False, want_gx=True)
ops.reduce_stats(x, layout, abssum=True, absmax=True, minmax=True)
ops.fq_line_fwd(x, torch.tensor([[-0.1, 0.9]] * 16, device=dev), 8, True, layout)
ops.fq_scaler_fwd(x, 0.037, (1, 1, x.numel()))
ops.quant_export_int8(x, ops.EXPORT_DECIMAL, 4.0, 8, (1, 1, x.numel()))
ops.quant_export_int8(x, ops.EXPORT_LINE, torch.tensor([[-0.1, 0.9]] * 16, device=dev), 8, layout)
# short-row / channel-last layouts: column reduction (4-byte-aligned views), transposed finalize, row-lane column
# reduction, group-resident channel-last maps, straddling vectors, packed int4 export
for lay, off in (((300, 24, 196), 0), ((40, 96, 64), 3), ((9, 700, 100), 1), ((2100, 8, 255), 5), ((5000, 24, 1), 0),
                 ((600, 1000, 1), 0), ((64, 96, 49), 0)):
    n_ = lay[0] * lay[1] * lay[2]
    xb = torch.randn(n_ + off, device=dev, generator=g)
    xl = xb[off:].view(lay)
    ops.reduce_stats(xl, lay, abssum=True, absmax=True, minmax=True, nnz=True)
    ops.reduce_stats(xl, lay, minmax=True)
    decl = torch.full((lay[1],), 4.0, device=dev)
    lin = torch.tensor([[-0.5, 0.5]] * lay[1], device=dev)
    ops.fq_pow2_fwd(xl, decl, lay)
    ops.fq_line_fwd(xl, lin, 8, True, lay)
    ops.ste_bwd(xl.clone(), decl, True, 8, 0, lay)
    ops.quant_export_int8(xl, ops.EXPORT_LINE, lin, 4, lay, pack4=True)
    ops.quant_export_int8(xl, ops.EXPORT_SCALER, 0.3, 4, (1, 1, n_), pack4=True)
# ---- round 2 ----
# one-launch training step (reduction + last-arriving CTA's parameter step) in every stage-1 mode, both row
# variants, with / without the L2 keep hint, host step index and device step counter, local statistics output
for lay in ((8, 16, 3136), (8, 16, 196), (4, 200, 81), (32, 48, 1), (64, 1000, 1), (3, 1, 5000), (2, 1024, 300)):
    C = lay[1]
    xs_ = torch.relu(torch.randn(lay, device=dev, generator=g))
    for variant in (2, 0, -1):
        ops.set_tuning(17, variant)
        for hint_ in (1, 0):
            ops.set_tuning(18, hint_)
            mag_ = torch.zeros(C, device=dev)
            mask_ = torch.ones(C, dtype=torch.bool, device=dev)
            sc_, de_ = torch.zeros(1, device=dev), torch.zeros(1, device=dev)
            ctr = torch.zeros(1, dtype=torch.int64, device=dev)
            asum = torch.empty(C, dtype=torch.float64, device=dev)
            amax = torch.empty(C, dtype=torch.float32, device=dev)
            tm = torch.full((8,), torch.iinfo(torch.int64).max, dtype=torch.int64, device=dev)
            for t in range(3):
                ops.reduce_prune_quant_step(xs_, lay, mag_, mask_, sc_, de_, float(lay[0] * lay[2]), t, 1,
                                            t > 0 and C > 1, C // 2 if C > 1 else 0, 8, t, True, abssum_out=asum,
                                            absmax_out=amax, stats_local=(t == 1), timing=tm)
                ops.reduce_prune_quant_step(xs_, lay, mag_, mask_, sc_, de_, float(lay[0] * lay[2]), 0, 1,
                                            1 if C > 1 else 1 << 30, C // 2 if C > 1 else 0, 8, 0, True,
                                            step_counter=ctr)
ops.set_tuning(17, -1)
ops.set_tuning(18, 1)
# the stand-alone parameter step on finalized rows (host-buffer pipeline form)
st_ = ops.reduce_stats(x, layout, abssum=True, absmax=True)
ops.prune_quant_rows_step_params(mag, mask, scale, dec, st_, 8 * 196.0, 2, 1, True, 8, 8, 2, True)
# K8 with an element mask, group mean, packed int4 on the map skeleton (aligned, n % 8 == 0)
for shape in ((64, 4608), (37, 256), (16, 16384)):
    xr = torch.randn(shape, device=dev, generator=g) * 0.05
    mk = torch.rand(shape, device=dev, generator=g) > 0.5
    for kind, w in ((ops.ROW_LINE, 2), (ops.ROW_SCALER, 1), (ops.ROW_DECIMAL, 1)):
        ops.row_quant_fused_(xr, torch.zeros(shape[0], w, device=dev), kind, 4, 1 if kind == ops.ROW_LINE else 0, mask=mk)
ops.group_mean(torch.rand(96, 2, device=dev), torch.randint(0, 5, (96,), device=dev), 5)
xa = torch.randn(8, 16, 196, device=dev, generator=g)
ops.quant_export_int8(xa, ops.EXPORT_DECIMAL, torch.full((16,), 3.0, device=dev), 4, (8, 16, 196), pack4=True)
ops.quant_export_int8(xa, ops.EXPORT_LINE, torch.tensor([[-0.5, 0.5]] * 16, device=dev), 4, (8, 16, 196), pack4=True)
# warm-started select and fused prune step (hint states 0 -> 1 -> 2, then a miss)
hint = ops.new_select_hints(1, dev)
vv = torch.randn((1 << 22) + 8, device=dev, generator=g)
for t in range(5):
    ops.kth_value(vv * (1 + 0.001 * t) if t != 3 else vv * 4 + 1, vv.numel() // 2, hint=hint)
hints9 = ops.new_select_hints(len(xs9), dev)
for t in range(2, 6):
    ops.prune_unstructured_step_batched_(mg9, xs9, mk9, ot9, [x_.numel() // 2 for x_ in xs9], t, hints=hints9)
# device-step-counter (CUDA-graph) forms of the running means, with offsets, and a captured + replayed sequence
ctr = torch.full((1,), 2, dtype=torch.int64, device=dev)
ops.scale_ema_(torch.rand(37, device=dev), torch.rand(37, device=dev), 8, 1, t_dev=ctr)
ops.lines_ema_(torch.rand(37, 2, device=dev), torch.rand(37, device=dev), torch.rand(37, device=dev), 1, t_dev=ctr)
xr = torch.randn(37, 256, device=dev, generator=g) * 0.05
mk = torch.rand(37, 256, device=dev, generator=g) > 0.5
for kind, w in ((ops.ROW_LINE, 2), (ops.ROW_SCALER, 1), (ops.ROW_DECIMAL, 1)):
    ops.row_quant_fused_(xr, torch.zeros(37, w, device=dev), kind, 4, 1, t_dev=ctr)
    ops.row_quant_fused_(xr, torch.zeros(37, w, device=dev), kind, 4, 1, mask=mk, t_dev=ctr)
for t in range(2):
    ops.prune_unstructured_step_batched_(mg9, xs9, mk9, ot9, [x_.numel() // 2 for x_ in xs9], 0, hints=hints9, t_dev=ctr)
    ctr.add_(1)
side = torch.cuda.Stream()
side.wait_stream(torch.cuda.current_stream())
wq, pq = torch.zeros(37, 1, device=dev), torch.rand(37, device=dev)
with torch.cuda.stream(side):
    ops.row_quant_fused_(xr, wq, ops.ROW_SCALER, 4, 0, t_dev=ctr)
    ops.scale_ema_(pq, torch.rand(37, device=dev), 8, 0, t_dev=ctr)
torch.cuda.current_stream().wait_stream(side)
gr = torch.cuda.CUDAGraph()
with torch.cuda.graph(gr):
    ops.row_quant_fused_(xr, wq, ops.ROW_SCALER, 4, 0, t_dev=ctr)
    ops.scale_ema_(pq, pq.clone(), 8, 0, t_dev=ctr)
    ctr.add_(1)
for _ in range(3):
    gr.replay()
torch.cuda.synchronize()
print("sanitize target done")
