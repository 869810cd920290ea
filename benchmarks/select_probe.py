"""k-th value probe: correctness against torch.sort on several distributions and CUDA-event
timing of qsb_kth_value (development tool).

    python benchmarks/select_probe.py [log2n] [--time-only]
"""
import json
import sys
from pathlib import Path

import torch

sys.path.insert(0, str(Path(__file__).resolve().parent.parent))
from qsparse_b200 import ops  # noqa: E402

log2n = int(sys.argv[1]) if len(sys.argv) > 1 and sys.argv[1].isdigit() else 26
n = 1 << log2n
torch.manual_seed(4)
dev = torch.device("cuda:0")
base = torch.randn(n, device=dev) * 0.02
flush = torch.zeros(128 * 1024 * 1024, device=dev)
flush_rd = torch.zeros(96 * 1024 * 1024, device=dev)


def timed(fn, iters=10):
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
    return ts[len(ts) // 2], ts[0]


def cases():
    yield "abs_normal", base.abs(), False
    yield "signed_normal", base, False
    yield "signed_take_abs", base, True
    yield "relu (half zeros)", torch.relu(base), False
    yield "grid_256 (8-bit values)", torch.round(base * 1024).clamp(-128, 127) / 1024, False
    yield "grid_64k", torch.round(base * 2 ** 18) / 2 ** 18, False
    yield "sorted", torch.sort(base).values, False
    u = torch.rand(n, device=dev)
    yield "uniform", u, False
    yield "bimodal gap", torch.where(u > 0.5, u + 100.0, u), False


for name, v, take_abs in cases():
    ref = None
    if "--time-only" not in sys.argv:
        ref = torch.sort(v.abs() if take_abs else v).values
    for frac in (0.5, 0.75, 0.001):
        k = int(frac * n)
        ok = None
        if ref is not None:
            got = ops.kth_value(v, k, take_abs=take_abs)
            ok = bool((got == ref[k]).item())
        med = timed(lambda: ops.kth_value(v, k, take_abs=take_abs))[0]
        print(json.dumps(dict(case=name, frac=frac, ok=ok, us_32k=round(med, 2), gbs=round(4 * n / med / 1e3, 1))),
              flush=True)
    del ref
