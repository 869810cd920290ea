"""Rates of the block-scaled FP8 / FP4 kernels (qsb_fq_block_fwd_dt, qsb_block_export_dt) next to the pow2 forward.

Workloads: [256, 64, 56, 56] fp32 (205 MB; rows of 56, so every row ends in a short block) and [32768, 4096] in fp32
and bf16 (long rows).  Every tensor is larger than the 126 MB L2.  Each arm is warmed up, then timed with CUDA events
around `--iters` back-to-back launches into preallocated outputs.  Rates are the modelled bytes over kernel time:
  forward  n * (input element size + 4)
  export   n * input element size + code bytes (n for E4M3, rows * ceil(L / 2) for E2M1) + rows * ceil(L / B)
  pow2     n * (input element size + 4)          (qsb_fq_pow2_fwd_dt, per tensor: the reference streaming rate)
and their fraction of the 6457 GB/s copy peak measured on B200 (DESIGN §4).  One JSON line per arm, the GPU name and
power limit in every line.

  python benchmarks/block_scaled.py [--iters 50] [--out profiles/block_scaled.jsonl]
"""
from __future__ import annotations

import argparse
import json
import subprocess
import sys
from ctypes import c_double, c_int, c_int64
from pathlib import Path

import torch

sys.path.insert(0, str(Path(__file__).resolve().parent.parent))
from qsparse_b200 import _native as N  # noqa: E402
from qsparse_b200 import ops  # noqa: E402

COPY_PEAK_GBS = 6457.0
WORKLOADS = [("[256,64,56,56] fp32", (256 * 64 * 56, 56), torch.float32),
             ("[32768,4096] fp32", (32768, 4096), torch.float32),
             ("[32768,4096] bf16", (32768, 4096), torch.bfloat16)]


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        name, power = (s.strip() for s in out[torch.cuda.current_device()].split(","))
    except Exception:  # noqa: BLE001  nvidia-smi missing: the name still comes from torch
        name, power = torch.cuda.get_device_name(), "unknown"
    return name, power


def time_us(fn, iters):
    for _ in range(5):
        fn()
    start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    start.record()
    for _ in range(iters):
        fn()
    end.record()
    end.synchronize()
    return start.elapsed_time(end) * 1000.0 / iters


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=50)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("needs a CUDA device")
    lib = N.load_library()
    name, power = gpu_info()
    lines = []
    for label, (rows, L), dtype in WORKLOADS:
        x = torch.randn(rows, L, device="cuda").to(dtype)
        n, es = x.numel(), x.element_size()
        stream = N.stream_ptr(x.device)
        y = torch.empty(rows, L, device="cuda")
        w = x.abs().amax().float().reshape(1)
        dt = c_int(N.dtype_code(x))

        def pow2():
            N.check(lib.qsb_fq_pow2_fwd_dt(N.ptr(x), dt, N.ptr(y), None, c_int64(1), c_double(4.0), None, c_int(0),
                                           c_int64(1), c_int64(1), c_int64(n), stream), "pow2")
        arms = [("pow2", None, pow2, n * (es + 4))]
        for fmt, (code, B) in ops.BLOCK_FORMATS.items():
            codes = torch.empty(rows, L if fmt == "mxfp8" else (L + 1) // 2, dtype=torch.uint8, device="cuda")
            scales = torch.empty(rows, (L + B - 1) // B, dtype=torch.uint8, device="cuda")

            def fwd(code=code):
                N.check(lib.qsb_fq_block_fwd_dt(N.ptr(x), dt, N.ptr(y), c_int64(rows), c_int64(L), c_int(code),
                                                N.ptr(w), stream), "fwd")

            def export(code=code, codes=codes, scales=scales):
                N.check(lib.qsb_block_export_dt(N.ptr(x), dt, N.ptr(codes), N.ptr(scales), c_int64(rows), c_int64(L),
                                                c_int(code), N.ptr(w), stream), "export")
            arms.append(("forward", fmt, fwd, n * (es + 4)))
            arms.append(("export", fmt, export, n * es + codes.numel() + scales.numel()))
        for kind, fmt, fn, nbytes in arms:
            us = time_us(fn, args.iters)
            gbs = nbytes / us / 1e3
            line = dict(workload=label, kind=kind, fmt=fmt, us=round(us, 2), modelled_bytes=nbytes,
                        gb_per_s=round(gbs, 1), copy_peak_fraction=round(gbs / COPY_PEAK_GBS, 3), gpu=name,
                        power_limit=power, iters=args.iters)
            print(json.dumps(line), flush=True)
            lines.append(line)
        del x, y
        torch.cuda.empty_cache()
    if args.out:
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        Path(args.out).write_text("".join(json.dumps(line) + "\n" for line in lines))


if __name__ == "__main__":
    main()
