"""bf16 activations through the fused prune -> quantize training step: native 16-bit reads vs the fp32 copy.

    python benchmarks/half_step.py [--steps 50] [--warmup 10] [--rounds 5] [--shape N,C,H,W] [--out DIR]

Default shape: bench.py's config 2, x [256, 64, 56, 56] in bf16, fp32 gradient, 75 % channel sparsity, 8-bit pow2.
Its 3136-element rows take the 8-loads-per-lane statistics kernel; rows of 257 .. 2047 elements (e.g.
``--shape 256,128,28,28``) take the 4-load variant.
Two arms, each one CUDA graph of a whole training step (forward + backward), replayed alternately in the same
process and timed with CUDA events around the replays, as bench.py does:

  native   the site reads the bf16 x and writes gx in bf16
  upcast   the same site behind a forward pre-hook ``x.float()``: the route the package took before it read
           16-bit values (an fp32 copy of x, and autograd's cast of the fp32 gx)

Two routes are timed: ``fused.PruneQuantize`` and a converted site (``FusedPruneQuantSequential``, which also
clamps grad_output in place).  The outputs of the two arms are checked bit for bit before timing.  Bytes per
element are a model from shapes (x 2 B, y 4 B, g 4 B, gx 2 B; the pruned channels' 75 % of x is not read by
the forward); GB/s is that model over the measured step time, beside the HBM copy peak of 6 457 GB/s that
profiles/ measured on this card.  Prints one JSON line.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
from pathlib import Path

import torch
import torch.nn as nn

sys.path.insert(0, str(Path(__file__).resolve().parent.parent))

SHAPE = (256, 64, 56, 56)
COPY_PEAK_GBS = 6457.0


def card():
    name = torch.cuda.get_device_name(0)
    try:
        pl = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader"], capture_output=True,
                            text=True, timeout=30).stdout.strip().splitlines()[0]
    except Exception:  # noqa: BLE001 - the power limit is reported when it can be read
        pl = "unknown"
    return name, pl


def byte_model(route: str, native: bool, keep: float):
    """B/elem dense (every channel kept) and actual (the forward skips pruned channels), per training step"""
    xb = 2 if native else 4
    copy = 0 if native else 2 + 4          # x.float(): read bf16, write fp32
    cast = 0 if native else 4 + 2          # autograd's cast of gx: read fp32, write bf16
    gc = 4 if route == "site" else 0       # the converted site also writes the clamped grad_output back
    gxb = 2 if native else 4
    stats = xb                             # statistics pass reads all of x
    dense = copy + stats + xb + 4 + 4 + gc + gxb + cast
    actual = copy + stats + xb * keep + 4 + 4 + gc + gxb + cast
    return dense, actual


def make_arm(route: str, native: bool):
    from qsparse_b200 import DecimalQuantizer, fuse_prune_quantize, prune, quantize
    from qsparse_b200.fused import PruneQuantize
    torch.manual_seed(0)
    if route == "prune_quantize":
        m = PruneQuantize(0.75, 8).cuda()
    else:
        m = nn.Sequential(nn.Sequential(nn.Identity(), prune(sparsity=0.75, dimensions={1}, start=1, interval=1,
                                                              repetition=1)),
                          quantize(bits=8, channelwise=-1, timeout=1, callback=DecimalQuantizer())).cuda()
        fuse_prune_quantize(m)
    if not native:
        m.register_forward_pre_hook(lambda mod, inp: (inp[0].float(),))
    return m


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--shape", default=",".join(map(str, SHAPE)))
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    shape = tuple(int(v) for v in a.shape.split(","))
    assert len(shape) == 4, "--shape N,C,H,W"
    if not torch.cuda.is_available():
        raise SystemExit("half_step.py measures on the GPU; no CUDA device found")
    from qsparse_b200 import GraphedTrainStep
    n = 1
    for s in shape:
        n *= s
    gen = torch.Generator(device="cuda").manual_seed(0)
    x_src = (torch.randn(shape, device="cuda", generator=gen) *
             torch.linspace(0.1, 2.0, shape[1], device="cuda").view(1, -1, 1, 1)).to(torch.bfloat16)
    g_src = torch.randn(shape, device="cuda", generator=gen)
    result = {"shape": list(shape), "dtype": "bfloat16", "n": n}
    name, pl = card()
    result.update(card=name, power_limit=pl, copy_peak_gbs=COPY_PEAK_GBS, steps=a.steps, rounds=a.rounds)
    for route in ("prune_quantize", "site"):
        arms = {}
        for native in (True, False):
            m = make_arm(route, native)
            x = x_src.clone().requires_grad_(True)
            g = g_src.clone()
            box = {}

            def step(m=m, x=x, g=g, box=box):
                y = m(x)
                box["y"], (box["gx"],) = y, torch.autograd.grad(y, x, g)

            for _ in range(4):            # reach the steady state (fused steps) before capture
                step()
            gs = GraphedTrainStep(m, step, warmup=3)
            arms[native] = (gs, box)
        for native in (True, False):      # equal outputs after the same number of steps
            arms[native][0].replay()
        torch.cuda.synchronize()
        yn, gxn = arms[True][1]["y"], arms[True][1]["gx"]
        yu, gxu = arms[False][1]["y"], arms[False][1]["gx"]
        equal = bool(torch.equal(yn.view(torch.int32), yu.view(torch.int32)) and gxn.dtype == gxu.dtype and
                     torch.equal(gxn.view(torch.int16), gxu.view(torch.int16)))
        times = {True: [], False: []}
        for _ in range(a.warmup):
            for native in (True, False):
                arms[native][0].replay()
        for _ in range(a.rounds):
            for native in (True, False):
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                for _ in range(a.steps):
                    arms[native][0].replay()
                e1.record()
                e1.synchronize()
                times[native].append(e0.elapsed_time(e1) * 1e3 / a.steps)
        keep = 0.25
        r = {"outputs_bit_equal": equal}
        for native in (True, False):
            t = sorted(times[native])[len(times[native]) // 2]
            dense, actual = byte_model(route, native, keep)
            arm = "native" if native else "upcast"
            r[arm] = {"step_us": round(t, 2), "step_us_all": [round(v, 2) for v in times[native]],
                      "B_per_elem_dense": dense, "B_per_elem_actual": actual,
                      "GBps": round(actual * n / (t * 1e-6) / 1e9, 1),
                      "fraction_of_copy_peak": round(actual * n / (t * 1e-6) / 1e9 / COPY_PEAK_GBS, 3)}
        r["speedup"] = round(r["upcast"]["step_us"] / r["native"]["step_us"], 3)
        result[route] = r
        del arms
        torch.cuda.empty_cache()
    line = json.dumps(result)
    print(line)
    if a.out:
        os.makedirs(a.out, exist_ok=True)
        Path(a.out, "half_step_" + "x".join(map(str, shape)) + ".json").write_text(line + "\n")


if __name__ == "__main__":
    # everything on a side stream: autograd then never makes the legacy default stream wait on the capture
    with torch.cuda.stream(torch.cuda.Stream()):
        main()
