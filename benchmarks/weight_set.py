"""BASELINE config 4 as a weight SET: 28 x [512,512,3,3] + remainder = 64 Mi elements, one unstructured
running-average prune step per layer (EMA 12 + select 4 + mask/apply 13 = 29 B/elem), eager and as one
captured CUDA graph.  Development tool.

    python benchmarks/weight_set.py
"""
import json
import sys
from pathlib import Path

import torch

sys.path.insert(0, str(Path(__file__).resolve().parent.parent))
from qsparse_b200 import parallel  # noqa: E402

dev = torch.device("cuda:0")
torch.manual_seed(4)
total = 1 << 26
shapes = [(512, 512, 3, 3)] * 28
rest = total - sum(512 * 512 * 9 for _ in shapes)
shapes.append((rest // 4096, 4096))
ws = [torch.randn(s, device=dev) * 0.02 for s in shapes]
mags = [w.abs() * 0.9 for w in ws]
masks = [torch.ones(w.shape, dtype=torch.bool, device=dev) for w in ws]
outs = [torch.empty_like(w) for w in ws]
n = sum(w.numel() for w in ws)
flush = torch.zeros(128 * 1024 * 1024, device=dev)
flush_rd = torch.zeros(96 * 1024 * 1024, device=dev)


def step():
    parallel.prune_weight_set_step(ws, mags, masks, outs, 3, 0.5)


def timed(fn, iters=8):
    for _ in range(3):
        fn()
    ts = []
    for _ in range(iters):
        flush.add_(1.0)
        flush_rd.max()
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        fn()
        e.record()
        e.synchronize()
        ts.append(s.elapsed_time(e) * 1e3)
    ts.sort()
    return ts[len(ts) // 2]


t_eager = timed(step)
side = torch.cuda.Stream()
side.wait_stream(torch.cuda.current_stream())
with torch.cuda.stream(side):
    step()
torch.cuda.current_stream().wait_stream(side)
g = torch.cuda.CUDAGraph()
with torch.cuda.graph(g):
    step()
t_graph = timed(g.replay)
for name, t in (("eager", t_eager), ("cuda_graph", t_graph)):
    print(json.dumps(dict(kernel="c4_weight_set_step", mode=name, layers=len(ws), elems=n, us=round(t, 1),
                          gbs=round(29 * n / t / 1e3, 1), frac_of_copy_peak=round(29 * n / t / 1e3 / 6457.4, 3))))
