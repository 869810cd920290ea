"""Converted prune -> DecimalQuantizer sites on channel-last activations: the fused step vs the same site unfused.

    python benchmarks/channel_last_step.py [--steps 50] [--warmup 10] [--rounds 5] [--out DIR]

Site: ``Sequential(Sequential(Identity, prune(75 %, dimensions={d})), quantize(8 bits, DecimalQuantizer, per
tensor))``, one training step = forward + ``autograd.grad`` of x.  Cases:

  cl-fp32 / cl-bf16   x [256, 64, 56, 56] channels_last, d = 1 (a convnet activation; fp32, and bf16 as under
                      autocast)
  bth768-bf16         x [32, 1024, 768] bf16, d = 2 (32768 tokens x 768 hidden, pruned along the hidden axis)
  bth2048-bf16        x [8, 1024, 2048] bf16, d = 2 (8192 tokens x 2048 hidden)

The gradient g is fp32 (y is fp32) in x's memory format.  Two arms per case:

  fused    the site after ``fuse_prune_quantize``: the step kernel(s) on x's memory, y = Q(x * mask), gx = clamp(g) * mask
  unfused  the same site without the fusion pass (the prune callback's fused structured step, x * mask, abs-max, the
           quantize forward, the STE backward, g * mask), with the copies it makes of a channels_last x and g

Each arm is timed with CUDA events around ``--steps`` eager steps, and around as many replays of the step captured
by ``GraphedTrainStep`` where the step is capturable (up to 1024 channels; bth2048 is eager only), alternating the
arms, ``--rounds`` times; the median is reported.  Before timing, the two arms have run the same steps on the same
inputs: y, gx and every ``state_dict`` entry are compared bit for bit.

Bytes per element come from each arm's launch list, recorded with torch.profiler for one eager step, under this
model (every element read or written once per kernel that touches it): a reduction reads x; a qsb map kernel reads
its input and writes each output its op writes (the STE backward writes grad_output in place and gx); a torch copy
kernel reads and writes its tensor; step / finalize kernels and counter updates count 0.  The model counts the
pruned channels of the pow2 forward as read (the kernel skips them), so it is an upper bound for that kernel.

Prints one JSON line with the card name and its power limit.
"""
from __future__ import annotations

import argparse
import json
import os
import re
import subprocess
import sys
from pathlib import Path

import torch
import torch.nn as nn

sys.path.insert(0, str(Path(__file__).resolve().parent.parent))

CASES = {
    "cl-fp32": ((256, 64, 56, 56), 1, torch.float32, torch.channels_last),
    "cl-bf16": ((256, 64, 56, 56), 1, torch.bfloat16, torch.channels_last),
    "bth768-bf16": ((32, 1024, 768), 2, torch.bfloat16, torch.contiguous_format),
    "bth2048-bf16": ((8, 1024, 2048), 2, torch.bfloat16, torch.contiguous_format),
}
GRAPH_MAX_CHANNELS = 1024      # a device step counter is taken by the one-launch step route only


def card():
    name = torch.cuda.get_device_name(0)
    try:
        pl = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader"], capture_output=True,
                            text=True, timeout=30).stdout.strip().splitlines()[0]
    except Exception:  # noqa: BLE001 - the power limit is reported when it can be read
        pl = "unknown"
    return name, pl


def make_site(fuse: bool, d: int):
    from qsparse_b200 import DecimalQuantizer, fuse_prune_quantize, prune, quantize
    torch.manual_seed(0)
    m = nn.Sequential(nn.Sequential(nn.Identity(), prune(sparsity=0.75, dimensions={d}, start=1, interval=1,
                                                          repetition=1)),
                      quantize(bits=8, channelwise=-1, timeout=1, callback=DecimalQuantizer())).cuda()
    return fuse_prune_quantize(m) if fuse else m


def _bits(t):
    return t.detach().contiguous().view(-1).view(torch.uint8)


_SIZE = {"float": 4, "__nv_bfloat16": 2, "__half": 2, "__nv_half": 2}


def kernel_bytes(name: str) -> int:
    """bytes per element of x that one launch of this kernel moves, under the model in the module docstring"""
    if "qsb::" in name:
        if "reduce_rows_kernel" in name or "reduce_cols_kernel" in name:
            t = re.search(r"\b(float|__nv_bfloat16|__half|__nv_half)\b", name)
            return _SIZE[t.group(1)] if t else 4
        io = re.search(r"MapIOT<([\w:]+), ([\w:]+), ([\w:]+)>", name)
        if io is None:
            return 0                                       # finalize / parameter step: per channel
        ti, to0, to1 = (_SIZE.get(s.split("::")[-1], 4) for s in io.groups())
        ste = re.search(r"SteOp<\d+, (true|false), (true|false)>", name)
        if ste:
            return ti + (to0 if ste.group(1) == "true" else 0) + (to1 if ste.group(2) == "true" else 0)
        if "MaskApplyOp" in name or re.search(r"(Pow2|Scaler|Line)Op<", name):
            return ti + to0
        return 0
    if "copy" in name.lower():
        half = "BFloat16" in name or "Half" in name
        full = "float" in name
        return 6 if half and full else 4 if half else 8
    return 0


def launch_list(step):
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        step()
        torch.cuda.synchronize()
    return [e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]


def time_arms(runs, steps, warmup, rounds):
    """median us per step of each callable, alternating them, CUDA events around `steps` calls"""
    for _ in range(warmup):
        for fn in runs.values():
            fn()
    times = {k: [] for k in runs}
    for _ in range(rounds):
        for k, fn in runs.items():
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(steps):
                fn()
            e1.record()
            e1.synchronize()
            times[k].append(e0.elapsed_time(e1) * 1e3 / steps)
    return {k: (sorted(v)[len(v) // 2], [round(u, 2) for u in v]) for k, v in times.items()}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--cases", default=",".join(CASES))
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("channel_last_step.py measures on the GPU; no CUDA device found")
    from qsparse_b200 import GraphedTrainStep
    from qsparse_b200.graphs import NotCapturable
    from qsparse_b200.fused import FusedPruneQuantSequential
    name, pl = card()
    result = {"card": name, "power_limit": pl, "sparsity": 0.75, "bits": 8, "steps": a.steps, "rounds": a.rounds,
              "cases": {}}
    for key in a.cases.split(","):
        shape, d, dtype, fmt = CASES[key]
        n = 1
        for s in shape:
            n *= s
        gen = torch.Generator(device="cuda").manual_seed(0)
        scale = torch.linspace(0.1, 2.0, shape[d], device="cuda").view([-1 if i == d else 1 for i in range(len(shape))])
        x_src = (torch.relu(torch.randn(shape, device="cuda", generator=gen)) * scale).to(dtype)
        g_src = torch.randn(shape, device="cuda", generator=gen)
        arms = {}
        for arm in ("fused", "unfused"):
            m = make_site(arm == "fused", d).train()
            x = x_src.clone(memory_format=fmt).requires_grad_(True)
            g = g_src.clone(memory_format=fmt)
            box = {}

            def step(m=m, x=x, g=g, box=box):
                # keep no output that carries an autograd graph across steps (GraphedTrainStep captures)
                y = m(x)
                (gx,) = torch.autograd.grad(y, x, g)
                box["y"], box["gx"] = y.detach(), gx

            for _ in range(4):            # past warm-up and timeout
                step()
            arms[arm] = dict(m=m, step=step, box=box, x=x, g=g)
        # the same steps on the same inputs: results equal before anything is timed
        bf, bu = arms["fused"]["box"], arms["unfused"]["box"]
        sf, su = arms["fused"]["m"].state_dict(), arms["unfused"]["m"].state_dict()
        equal = (torch.equal(_bits(bf["y"]), _bits(bu["y"])) and bf["gx"].dtype == bu["gx"].dtype and
                 torch.equal(_bits(bf["gx"]), _bits(bu["gx"])) and sorted(sf) == sorted(su) and
                 all(torch.equal(_bits(sf[k]), _bits(su[k])) for k in sf))
        fused_steps = sum(mm.fused_steps for mm in arms["fused"]["m"].modules()
                          if isinstance(mm, FusedPruneQuantSequential))
        r = {"shape": list(shape), "prune_axis": d, "dtype": str(dtype).replace("torch.", ""),
             "channels_last": fmt == torch.channels_last, "n": n, "outputs_gx_state_bit_equal": bool(equal),
             "fused_steps_before_timing": int(fused_steps),
             "y_gx_in_x_format": bool(bf["y"].is_contiguous(memory_format=fmt) and
                                      bf["gx"].is_contiguous(memory_format=fmt))}
        for arm, v in arms.items():
            names = launch_list(v["step"])
            b = sum(kernel_bytes(k) for k in names)
            r[arm] = {"launches": len(names), "qsb_launches": sum("qsb::" in k for k in names),
                      "copy_launches": sum("copy" in k.lower() for k in names), "B_per_elem": b}
        eager = time_arms({arm: v["step"] for arm, v in arms.items()}, a.steps, a.warmup, a.rounds)
        for arm in arms:
            t, all_t = eager[arm]
            r[arm]["eager_step_us"], r[arm]["eager_step_us_all"] = round(t, 2), all_t
            r[arm]["eager_GBps"] = round(r[arm]["B_per_elem"] * n / (t * 1e-6) / 1e9, 1)
        r["eager_speedup"] = round(eager["unfused"][0] / eager["fused"][0], 3)
        if shape[d] <= GRAPH_MAX_CHANNELS:
            try:
                graphs = {arm: GraphedTrainStep(v["m"], v["step"], warmup=3) for arm, v in arms.items()}
            except NotCapturable as e:
                graphs = None
                r["graph"] = f"not capturable: {e}"
        else:
            graphs = None
            r["graph"] = f"not capturable: {shape[d]} channels > {GRAPH_MAX_CHANNELS}"
        if graphs is not None:
            replay = time_arms({arm: gs.replay for arm, gs in graphs.items()}, a.steps, a.warmup, a.rounds)
            for arm in arms:
                t, all_t = replay[arm]
                r[arm]["graph_step_us"], r[arm]["graph_step_us_all"] = round(t, 2), all_t
                r[arm]["graph_GBps"] = round(r[arm]["B_per_elem"] * n / (t * 1e-6) / 1e9, 1)
            r["graph_speedup"] = round(replay["unfused"][0] / replay["fused"][0], 3)
            del graphs
        result["cases"][key] = r
        del arms
        torch.cuda.empty_cache()
    line = json.dumps(result)
    print(line)
    if a.out:
        os.makedirs(a.out, exist_ok=True)
        with open(os.path.join(a.out, "channel_last_step.json"), "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
