"""A converted prune -> AdaptiveQuantizer activation site: the fused line step vs the same site unfused.

    python benchmarks/prune_line_step.py [--steps 50] [--warmup 10] [--rounds 5] [--shape N,C,H,W] [--out DIR]

Site: ``Sequential(Sequential(Identity, prune(75 %, dimensions={1})), quantize(8 bits, AdaptiveQuantizer))`` on x
[256, 64, 56, 56] (bench.py's config 2 activation), with per-tensor (``channelwise=-1``) and per-channel
(``channelwise=1``) lines, for fp32 x and for bf16 x with an fp32 gradient.  Two arms per case, each one CUDA graph
of the site's forward + backward (``GraphedTrainStep``), replayed alternately in one process and timed with CUDA
events around the replays:

  fused    the site after ``fuse_prune_quantize``: statistics launch whose last CTA runs the parameter step, the
           masked line forward, gx = g * mask
  unfused  the same site without the fusion pass: prune step, x * mask, min / max of it, lines EMA, line forward,
           identity backward, g * mask

Before timing, both arms have run the same steps on the same inputs: their outputs, input gradients and every
``state_dict`` entry are compared bit for bit.  Bytes per element are a model counted from the code (fp32 x: 20
fused, 32 unfused; bf16 x: 14 and 26).  The forward of both arms reads the pruned channels.  x is 51 MB in fp32
and a step also writes y and gx of that size, more than the 126 MB L2 holds.  Prints one JSON line with the card
name and its power limit.
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
BYTES = {("fused", torch.float32): 20, ("unfused", torch.float32): 32,
         ("fused", torch.bfloat16): 14, ("unfused", torch.bfloat16): 26}


def card():
    name = torch.cuda.get_device_name(0)
    try:
        pl = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader"], capture_output=True,
                            text=True, timeout=30).stdout.strip().splitlines()[0]
    except Exception:  # noqa: BLE001 - the power limit is reported when it can be read
        pl = "unknown"
    return name, pl


def make_site(fuse: bool, channelwise: int):
    from qsparse_b200 import AdaptiveQuantizer, fuse_prune_quantize, prune, quantize
    torch.manual_seed(0)
    m = nn.Sequential(nn.Sequential(nn.Identity(), prune(sparsity=0.75, dimensions={1}, start=1, interval=1,
                                                          repetition=1)),
                      quantize(bits=8, channelwise=channelwise, timeout=1, callback=AdaptiveQuantizer())).cuda()
    return fuse_prune_quantize(m) if fuse else m


def _bits(t):
    return t.detach().contiguous().view(-1).view(torch.uint8)


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
        raise SystemExit("prune_line_step.py measures on the GPU; no CUDA device found")
    from qsparse_b200 import GraphedTrainStep
    from qsparse_b200.fused import FusedPruneQuantSequential
    n = 1
    for s in shape:
        n *= s
    gen = torch.Generator(device="cuda").manual_seed(0)
    x32 = torch.relu(torch.randn(shape, device="cuda", generator=gen) *
                     torch.linspace(0.1, 2.0, shape[1], device="cuda").view(1, -1, 1, 1))
    g_src = torch.randn(shape, device="cuda", generator=gen)
    name, pl = card()
    result = {"shape": list(shape), "n": n, "sparsity": 0.75, "bits": 8, "card": name, "power_limit": pl,
              "steps": a.steps, "rounds": a.rounds, "cases": {}}
    for dtype in (torch.float32, torch.bfloat16):
        for channelwise in (-1, 1):
            arms = {}
            for arm in ("fused", "unfused"):
                m = make_site(arm == "fused", channelwise)
                x = x32.to(dtype).clone().requires_grad_(True)
                g = g_src.clone()
                box = {}

                def step(m=m, x=x, g=g, box=box):
                    # keep no output that carries an autograd graph across steps (GraphedTrainStep captures)
                    y = m(x)
                    (gx,) = torch.autograd.grad(y, x, g)
                    box["y"], box["gx"] = y.detach(), gx

                for _ in range(4):            # past warm-up and timeout before capture
                    step()
                arms[arm] = (GraphedTrainStep(m, step, warmup=3), box, m)
            for arm in arms:
                arms[arm][0].replay()
                arms[arm][0].sync_host()
            torch.cuda.synchronize()
            (_, bf, mf), (_, bu, mu) = arms["fused"], arms["unfused"]
            sf, su = mf.state_dict(), mu.state_dict()
            equal = (torch.equal(_bits(bf["y"]), _bits(bu["y"])) and bf["gx"].dtype == bu["gx"].dtype and
                     torch.equal(_bits(bf["gx"]), _bits(bu["gx"])) and sorted(sf) == sorted(su) and
                     all(torch.equal(_bits(sf[k]), _bits(su[k])) for k in sf))
            fused_steps = sum(mm.fused_steps for mm in mf.modules() if isinstance(mm, FusedPruneQuantSequential))
            times = {arm: [] for arm in arms}
            for _ in range(a.warmup):
                for arm in arms:
                    arms[arm][0].replay()
            for _ in range(a.rounds):
                for arm in arms:
                    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    e0.record()
                    for _ in range(a.steps):
                        arms[arm][0].replay()
                    e1.record()
                    e1.synchronize()
                    times[arm].append(e0.elapsed_time(e1) * 1e3 / a.steps)
            r = {"outputs_gx_state_bit_equal": bool(equal), "fused_steps_before_timing": int(fused_steps)}
            for arm in arms:
                t = sorted(times[arm])[len(times[arm]) // 2]
                b = BYTES[(arm, dtype)]
                r[arm] = {"step_us": round(t, 2), "step_us_all": [round(v, 2) for v in times[arm]],
                          "B_per_elem": b, "GBps": round(b * n / (t * 1e-6) / 1e9, 1)}
            r["speedup"] = round(r["unfused"]["step_us"] / r["fused"]["step_us"], 3)
            key = f"{'fp32' if dtype == torch.float32 else 'bf16'}-{'per_tensor' if channelwise < 0 else 'per_channel'}"
            result["cases"][key] = r
            del arms
            torch.cuda.empty_cache()
    line = json.dumps(result)
    print(line)
    if a.out:
        os.makedirs(a.out, exist_ok=True)
        with open(os.path.join(a.out, "prune_line_step.json"), "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
