"""BASELINE.json configurations 3, 4 and 5 for bench.py (`python bench.py --config N`), same JSON schema
as the headline configuration (roofline, cpu_baseline, e2e, clocks, gpu_launches).

  3  channel-wise 4-bit weight quantization of a [4096, 4096] linear weight, adaptive (min/max) scale
     estimation: one training access of the weight = estimate -> EMA -> line fake-quant
     (ref qsparse/quantize.py:140-185, 393-430).  Weights are replicated under data parallelism: at
     N > 1 every rank runs the same access ("replicas only", no collective).
  4  unstructured magnitude prune (running-average statistics, exact k-th value mask) of a 64 Mi
     element conv weight set (28 x [512,512,3,3] + remainder), one step = EMA + threshold + mask + apply
     per layer (ref qsparse/sparse.py:58-66,82-89, util.py:103-117).  N > 1: replicated one-pass step
     (no communication) and, reported beside it, the layer-sharded select + one all-reduce of thresholds.
  5  element-wise fused prune(mask) + pow2 fake-quant forward and backward over flat tensors of
     2^20 .. 2^32 elements (ref qsparse/quantize.py:43-77 + sparse.py:116); N GPUs each on its own
     shard (weak: n per GPU fixed; --strong: n / N per GPU), no collective.

Timing: CUDA events on the launching stream around every step, a clean-line L2 flush (512 MB write +
384 MB read) between steps whenever the step's tensors fit the 126 MB L2, max over ranks.
"""
from __future__ import annotations

import json
import os
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent
L2_BYTES = 126 * 1024 * 1024


def _dist():
    import torch.distributed as dist
    return dist if (dist.is_available() and dist.is_initialized()) else None


class Flusher:
    def __init__(self, torch, dev):
        self.w = torch.zeros(128 * 1024 * 1024, device=dev)   # 512 MB written ...
        self.r = torch.zeros(96 * 1024 * 1024, device=dev)    # ... then 384 MB read: L2 holds clean lines

    def __call__(self):
        self.w.add_(1.0)
        self.r.max()


def timed(torch, fn, steps, warmup, flush=None, world=1, dev=None):
    """ms per step (sum of per-step CUDA-event intervals; the flush sits outside them), max over ranks"""
    dist = _dist()
    for _ in range(max(warmup, 3)):
        fn()
    torch.cuda.synchronize()
    if dist:
        dist.barrier()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    for s, e in ev:
        if flush is not None:
            flush()
        s.record()
        fn()
        e.record()
    torch.cuda.synchronize()
    ms = sum(s.elapsed_time(e) for s, e in ev) / steps
    if dist:
        t = torch.tensor([ms], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = t.item()
        dist.barrier()
    return ms


def back_to_back(torch, fn, steps, warmup, world=1, dev=None):
    """ms per step of `steps` calls issued back to back (one event pair around all of them)"""
    dist = _dist()
    for _ in range(max(warmup, 3)):
        fn()
    torch.cuda.synchronize()
    if dist:
        dist.barrier()
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s.record()
    for _ in range(steps):
        fn()
    e.record()
    torch.cuda.synchronize()
    ms = s.elapsed_time(e) / steps
    if dist:
        t = torch.tensor([ms], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = t.item()
        dist.barrier()
    return ms


def _prof():
    p = ROOT / "profiles" / "roofline_traffic.json"
    try:
        return json.loads(p.read_text())
    except Exception:
        return {}


def _base(metric, value, world, args, ms, cfg, n_units, clocks, scaling="weak"):
    return {"metric": metric, "value": round(value, 2), "unit": "GB/s", "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": round(ms, 5), "higher_is_better": True, "scaling": scaling,
            "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": cfg,
            "elems_per_s": round(n_units / (ms * 1e-3), 1), "clocks": clocks}


# ============================================================================= config 3
C3_SHAPE = (4096, 4096)
C3_BITS = 4
C3_METRIC = "channelwise 4-bit weight quantize (adaptive estimate + line fake-quant) HBM GB/s"


def c3_config():
    return {"workload": "config[2]: [4096,4096] fp32 linear weight, bits=4, channelwise=0, AdaptiveQuantizer: one training "
                        "access = per-row min/max -> EMA -> line fake-quant, fused in ONE row-resident launch "
                        "(8 B/elem: one read + one write; the reference's algorithm re-reads the tensor: 12 B/elem)",
            "shape_per_gpu": list(C3_SHAPE), "bits": C3_BITS, "parallelism": "replicas only (weights are replicated under "
            "data parallelism; no collective)", "l2": "67 MB tensor fits the 126 MB L2: clean-line flush (512 MB write + "
            "384 MB read) between timed steps; the L2-warm figure is reported beside it"}


def run_c3(args, env):
    import torch
    import qsparse_b200 as q
    from qsparse_b200 import ops
    world, rank, dev = env["world"], env["rank"], env["dev"]
    peak, peak_src = env["peak"]
    n = C3_SHAPE[0] * C3_SHAPE[1]
    torch.manual_seed(3)
    w = torch.randn(C3_SHAPE, device=dev) * 0.02
    lines = torch.zeros(C3_SHAPE[0], 2, device=dev)
    state = {"t": 1}

    def step():
        ops.row_quant_fused_(w, lines, ops.ROW_LINE, C3_BITS, state["t"], True)
        state["t"] += 1

    flush = Flusher(torch, dev)
    sampler = env["sampler_cls"](dev.index)
    if rank == 0:
        sampler.start()
        time.sleep(0.2)
    steps = min(args.steps, 400)
    ms = timed(torch, step, steps, args.warmup, flush, world, dev)
    ms_warm = back_to_back(torch, step, steps, args.warmup, world, dev)
    t_soak = time.perf_counter()
    while time.perf_counter() - t_soak < 0.6:
        for _ in range(50):
            step()
        torch.cuda.synchronize()
    clocks = sampler.stop() if rank == 0 else None
    # the three-launch route of the same access (what the un-fused path costs)
    lines3 = torch.zeros_like(lines)
    wy = torch.empty_like(w)

    def step3():
        st_ = ops.reduce_stats(w, (1, C3_SHAPE[0], C3_SHAPE[1]), minmax=True)
        ops.lines_ema_(lines3, st_["min"], st_["max"], 2)
        ops.fq_line_fwd(w, lines3, C3_BITS, True, (1, C3_SHAPE[0], C3_SHAPE[1]), out=wy)
    ms3 = timed(torch, step3, min(steps, 100), 3, flush, world, dev)

    # module API: quantize(nn.Linear, bits=4, channelwise=0, timeout=1, AdaptiveQuantizer()).weight in training
    q.set_qsparse_options(log_on_created=False)
    lin = torch.nn.Linear(C3_SHAPE[1], C3_SHAPE[0], bias=False).to(dev)
    with torch.no_grad():
        lin.weight.copy_(w)
    ql = q.quantize(lin, bits=C3_BITS, channelwise=0, timeout=1, callback=q.AdaptiveQuantizer()).train()
    with torch.no_grad():
        _ = ql.weight
        _ = ql.weight

        def mod_step():
            return ql.weight
        ms_mod = timed(torch, mod_step, min(steps, 100), 3, flush, world, dev)
        yq = ql.weight
    # parity against the raw kernel on the same EMA state is covered by tests; here: same shape, finite
    assert yq.shape == w.shape and bool(torch.isfinite(yq).all().item())

    # e2e: pinned host weight in, quantized weight out, through the module API
    hw = torch.empty(C3_SHAPE, dtype=torch.float32).pin_memory()
    hw.copy_(w)
    hy = torch.empty(C3_SHAPE, dtype=torch.float32).pin_memory()
    e2e_steps = max(4, min(args.steps, 20))

    def e2e_step():
        with torch.no_grad():
            lin.weight.copy_(hw, non_blocking=True)
            hy.copy_(ql.weight, non_blocking=True)
    for _ in range(2):
        e2e_step()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        e2e_step()
    torch.cuda.synchronize()
    e2e_s = (time.perf_counter() - t0) / e2e_steps
    dist = _dist()
    if dist:
        t = torch.tensor([e2e_s], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_s = t.item()

    gpu_eager = cpu = None
    if world == 1 and not args.no_gpu_eager:
        from oracle.torch_eager import WeightLineQuantEager
        eg = WeightLineQuantEager(C3_BITS)
        ms_e = timed(torch, lambda: eg.forward(w), 20, 3, flush, 1, dev)
        gpu_eager = {"what": "the reference's eager ATen sequence (min, max, cat, EMA, clamp, sub, div, round, clamp_, mul, add)",
                     "ms_per_step": round(ms_e, 4), "value": round(8 * n / (ms_e * 1e-3) / 1e9, 2), "unit": "GB/s",
                     "speedup_of_this_repo": round(ms_e / ms, 2)}
    if world == 1 and not args.no_cpu_baseline:
        cpu = cpu_c3(env["host_threads"], 5)
    prof = _prof()
    value = world * 8 * n / (ms * 1e-3) / 1e9
    line = _base(C3_METRIC, value, world, args, ms, c3_config(), world * n, clocks)
    line["steps"] = steps
    line.update({
        "frac_of_measured_hbm_peak": round(value / world / peak, 4),
        "value_actual": round(value, 2),
        "value_on_reference_algorithm_bytes": round(world * 12 * n / (ms * 1e-3) / 1e9, 2),
        "bytes_per_elem": {"algorithmic": 8, "actual": 8, "reference_algorithm": 12},
        "l2_warm": {"ms_per_step": round(ms_warm, 5), "value": round(world * 8 * n / (ms_warm * 1e-3) / 1e9, 2)},
        "three_launch_route": {"ms_per_step": round(ms3, 5), "what": "reduce_stats(minmax) + lines_ema + fq_line_fwd (12 B/elem)"},
        "module_api": {"api": "quantize(nn.Linear, bits=4, channelwise=0, timeout=1, AdaptiveQuantizer()).weight",
                       "ms_per_step": round(ms_mod, 5), "value": round(world * 8 * n / (ms_mod * 1e-3) / 1e9, 2)},
        "launch_mode": "eager, one launch per step (row_quant_kernel)",
        "gpu_launches": steps,
        "e2e": {"value": round(world * 8 * n / e2e_s / 1e9, 3), "unit": "GB/s", "h2d_bytes_per_step": 4 * n * world,
                "d2h_bytes_per_step": 4 * n * world, "ms_per_step": round(e2e_s * 1e3, 3), "steps": e2e_steps,
                "api": "pinned host weight -> layer.weight.copy_ -> quantize(...).weight (module API) -> pinned host"},
        "roofline": {"bound": "hbm", "kernel": "row_quant_kernel<LINE> (row-resident estimate + EMA + line fake-quant)",
                     "achieved": round(8 * n / (ms * 1e-3) / 1e9, 1), "peak": peak, "peak_source": peak_src, "unit": "GB/s",
                     "frac": round(8 * n / (ms * 1e-3) / 1e9 / peak, 4), "traffic": prof.get("row_quant_line_dram_bytes_per_launch"),
                     "algorithmic_bytes_per_launch": 8 * n, "avg_launch_us": round(ms * 1e3, 2)},
        "gpu_eager_baseline": gpu_eager, "cpu_baseline": cpu,
    })
    return line


def cpu_c3(threads, steps):
    import numpy as np
    from concurrent.futures import ThreadPoolExecutor
    from oracle import oracle as orc
    rng = np.random.default_rng(3)
    w = (rng.standard_normal(C3_SHAPE, dtype=np.float32) * np.float32(0.02))
    rows = C3_SHAPE[0]
    threads = max(1, min(threads, rows))
    sl = [slice(i * rows // threads, (i + 1) * rows // threads) for i in range(threads)]
    pool = ThreadPoolExecutor(threads)
    lines = np.zeros((rows, 2), np.float32)
    st = {"t": 1}

    def part(s):
        mn, mx = orc.minmax(w[s], 0)
        lines[s] = orc.lines_ema(lines[s], mn, mx, st["t"])
        return orc.fq_line_fwd(w[s], lines[s], C3_BITS, 0, True)

    def step():
        list(pool.map(part, sl))
        st["t"] += 1
    step()
    t0 = time.perf_counter()
    for _ in range(steps):
        step()
    dt = (time.perf_counter() - t0) / steps
    n = w.size
    return {"value": round(8 * n / dt / 1e9, 3), "unit": "GB/s", "cores": threads, "kind": "port", "steps": steps,
            "sample": f"{steps} accesses of the full [4096,4096] weight, row-sliced over the threads, {dt*1e3:.1f} ms/step",
            "elems_per_s": round(n / dt, 1), "ms_per_step": round(dt * 1e3, 3)}


# ============================================================================= config 4
C4_TOTAL = 1 << 26
C4_METRIC = "unstructured magnitude prune step (EMA + k-th value mask + apply) HBM GB/s"


def c4_shapes():
    shapes = [(512, 512, 3, 3)] * 28
    rest = C4_TOTAL - sum(512 * 512 * 9 for _ in shapes)
    shapes.append((rest // 4096, 4096))
    return shapes


def c4_config(sparsity):
    return {"workload": f"config[3]: 64 Mi-element conv weight set (28 x [512,512,3,3] + [256,4096]), unstructured magnitude "
                        f"prune at sparsity {sparsity:g}, running-average statistics, exact k-th value threshold per layer: "
                        "EMA 12 + select 4 + mask/apply 13 = 29 B/elem in the reference's algorithm; here ONE streaming "
                        "pass (~17.5 B/elem of traffic) + candidate passes + fix-up",
            "elements": C4_TOTAL, "layers": 29, "sparsity": sparsity,
            "parallelism": "weights are replicated under data parallelism: every rank runs the one-pass step on all "
                           "layers (no communication; thresholds are exact, so ranks agree bit for bit); the layer-sharded "
                           "select + all-reduce route is timed beside it",
            "l2": "268 MB per tensor kind exceeds the 126 MB L2; no flush"}


def run_c4(args, env):
    import torch
    from qsparse_b200 import ops, parallel
    from qsparse_b200.util import kth_rank
    world, rank, dev = env["world"], env["rank"], env["dev"]
    peak, peak_src = env["peak"]
    sparsity = 0.5 if args.sparsity is None else args.sparsity
    torch.manual_seed(4)
    ws = [torch.randn(s, device=dev) * 0.02 for s in c4_shapes()]
    mags = [w.abs() * 0.9 for w in ws]
    masks = [torch.ones(w.shape, dtype=torch.bool, device=dev) for w in ws]
    outs = [torch.empty_like(w) for w in ws]
    n = sum(w.numel() for w in ws)
    state = {"t": 3}
    hints = ops.new_select_hints(len(ws), dev)      # warm-started pivots, kept across the steps of the loop

    def step():
        parallel.prune_weight_set_step(ws, mags, masks, outs, state["t"], sparsity, hints=hints)
        state["t"] += 1

    def step_cold():
        parallel.prune_weight_set_step(ws, mags, masks, outs, state["t"], sparsity)
        state["t"] += 1

    def step_sharded():
        parallel.prune_weight_set_step(ws, mags, masks, outs, state["t"], sparsity, shard_by_layer=True)
        state["t"] += 1

    sampler = env["sampler_cls"](dev.index)
    if rank == 0:
        sampler.start()
        time.sleep(0.2)
    steps = min(args.steps, 200)
    ms = back_to_back(torch, step, steps, args.warmup, world, dev)
    t_soak = time.perf_counter()
    while time.perf_counter() - t_soak < 0.6:
        for _ in range(10):
            step()
        torch.cuda.synchronize()
    clocks = sampler.stop() if rank == 0 else None
    ms_cold = back_to_back(torch, step_cold, min(steps, 50), 3, world, dev)
    ms_sh = back_to_back(torch, step_sharded, min(steps, 50), 3, world, dev)
    # graph: the whole step as one captured CUDA graph (launch-gap free)
    side = torch.cuda.Stream(device=dev)
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        parallel.prune_weight_set_step(ws, mags, masks, outs, 3, sparsity)
    torch.cuda.current_stream().wait_stream(side)
    gr = torch.cuda.CUDAGraph()
    with torch.cuda.graph(gr):
        parallel.prune_weight_set_step(ws, mags, masks, outs, 3, sparsity, hints=hints)
    ms_graph = back_to_back(torch, gr.replay, min(steps, 100), 3, world, dev)

    # correctness inside the bench: masks equal torch.sort's threshold on two layers; ranks agree bit for bit
    ok = True
    for i in (0, 28):
        kk = kth_rank(sparsity, mags[i].numel())
        thr = torch.sort(mags[i].reshape(-1)).values[kk]
        ok = ok and bool(torch.equal(masks[i], mags[i] >= thr)) and bool(torch.equal(outs[i], ws[i] * masks[i]))
    dist = _dist()
    ranks_equal = None
    if dist:
        digest = torch.stack([m.view(torch.uint8).sum(dtype=torch.int64) for m in masks])
        got = [torch.empty_like(digest) for _ in range(world)]
        dist.all_gather(got, digest)
        ranks_equal = all(torch.equal(got[0], g_) for g_ in got)
        ok = ok and ranks_equal

    # module API: MagnitudePruningCallback per layer (the reference's own call)
    from qsparse_b200.sparse import MagnitudePruningCallback
    cbs = [MagnitudePruningCallback(running_average=True).train() for _ in ws]
    cmasks = [torch.nn.Parameter(torch.ones(w.shape, dtype=torch.bool, device=dev), requires_grad=False) for w in ws]

    def mod_step():
        with torch.no_grad():
            for cb, w, m in zip(cbs, ws, cmasks):
                cb(w, sparsity, m)
    ms_mod = back_to_back(torch, mod_step, min(steps, 20), 3, world, dev)
    del cbs, cmasks
    # the same through prune()-wrapped modules with the model-level batched step (WeightSetPruner)
    import qsparse_b200 as q

    class _W(torch.nn.Module):
        def __init__(self, w):
            super().__init__()
            self.weight = torch.nn.Parameter(w.clone(), requires_grad=False)

    q.set_qsparse_options(log_on_created=False)
    mods = torch.nn.ModuleList([q.prune(_W(w), sparsity=sparsity, dimensions=set(range(w.dim())), start=0, interval=1,
                                        repetition=1) for w in ws]).train()
    pruner = q.WeightSetPruner(mods)

    def batched_mod_step():
        with torch.no_grad():
            pruner.step()
            for m in mods:
                m.weight
    for _ in range(3):
        batched_mod_step()
    ms_bmod = back_to_back(torch, batched_mod_step, min(steps, 50), 3, world, dev)
    ms_gbmod = None
    try:    # the batched step + the 29 module accesses as ONE CUDA graph
        gsb = q.GraphedTrainStep(mods, batched_mod_step, warmup=3)
        ms_gbmod = back_to_back(torch, gsb.replay, min(steps, 100), 3, world, dev)
        gsb.sync_host()
        del gsb
    except Exception:
        ms_gbmod = None
    del pruner
    # ... and with the per-layer module accesses of one step captured into ONE CUDA graph (GraphedTrainStep: the
    # one-pass kernels read the step index from each callback's own `t` Parameter)
    ms_gmod = None
    try:
        def access_all():
            with torch.no_grad():
                for m in mods:
                    m.weight
        gs = q.GraphedTrainStep(mods, access_all, warmup=3)
        ms_gmod = back_to_back(torch, gs.replay, min(steps, 100), 3, world, dev)
        gs.sync_host()
    except Exception as exc:       # reported, not fatal: the line then carries no graphed figure
        ms_gmod = None
        graph_note = f"{type(exc).__name__}: {exc}"
    del mods

    # e2e: pinned host weights in, pruned weights + masks out
    hws = [torch.empty(w.shape, dtype=torch.float32).pin_memory() for w in ws]
    hos = [torch.empty(w.shape, dtype=torch.float32).pin_memory() for w in ws]
    for h, w in zip(hws, ws):
        h.copy_(w)
    e2e_steps = max(2, min(args.steps, 6))

    def e2e_step():
        for w, h in zip(ws, hws):
            w.copy_(h, non_blocking=True)
        step()
        for h, o in zip(hos, outs):
            h.copy_(o, non_blocking=True)
    e2e_step()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        e2e_step()
    torch.cuda.synchronize()
    e2e_s = (time.perf_counter() - t0) / e2e_steps
    if dist:
        t = torch.tensor([e2e_s], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_s = t.item()
    del hws, hos

    gpu_eager = cpu = None
    if world == 1 and not args.no_gpu_eager:
        from oracle.torch_eager import UnstructuredPruneEager
        egs = [UnstructuredPruneEager(w, sparsity) for w in ws]
        for e_ in egs:
            e_.t = 3

        def eager_step():
            for e_, w in zip(egs, ws):
                e_.forward(w)
        ms_e = back_to_back(torch, eager_step, 5, 2, 1, dev)
        gpu_eager = {"what": "the reference's eager ATen sequence per layer (abs, mul, add, div, copy, flatten, sort, ge, copy, mul)",
                     "ms_per_step": round(ms_e, 4), "value": round(29 * n / (ms_e * 1e-3) / 1e9, 2), "unit": "GB/s",
                     "speedup_of_this_repo": round(ms_e / ms, 2)}
        del egs
    if world == 1 and not args.no_cpu_baseline:
        cpu = cpu_c4(env["host_threads"], sparsity)
    prof = _prof()
    value = world * 29 * n / (ms * 1e-3) / 1e9
    traffic_bpe = 17.5
    line = _base(C4_METRIC, value, world, args, ms, c4_config(sparsity), world * n, clocks)
    line["steps"] = steps
    line.update({
        "frac_of_measured_hbm_peak": round(value / world / peak, 4),
        "value_actual": round(world * traffic_bpe * n / (ms * 1e-3) / 1e9, 2),
        "frac_actual": round(traffic_bpe * n / (ms * 1e-3) / 1e9 / peak, 4),
        "bytes_per_elem": {"algorithmic": 29, "actual": traffic_bpe,
                           "note": "value is quoted on the reference algorithm's 29 B/elem (SURVEY 8d); the one-pass step "
                                   "really moves ~17.5 B/elem (R w, R mag, W mag, W y, 1 B W mask + candidates): value_actual"},
        "masks_equal_sort_threshold": ok, "ranks_bit_equal": ranks_equal,
        "sampled_pivots_every_step": {"ms_per_step": round(ms_cold, 5), "value": round(world * 29 * n / (ms_cold * 1e-3) / 1e9, 2),
                                      "what": "the same step without the pivot hints (a 32 Ki-element sample per layer and "
                                              "step): what the first two steps of a loop, or a one-off call, cost"},
        "pivot_hint_states": [int(v) for v in hints[:, 0].tolist()],
        "cuda_graph": {"ms_per_step": round(ms_graph, 5), "value": round(world * 29 * n / (ms_graph * 1e-3) / 1e9, 2)},
        "layer_sharded_select": {"ms_per_step": round(ms_sh, 5), "value": round(world * 29 * n / (ms_sh * 1e-3) / 1e9, 2),
                                 "what": "replicated multi-tensor EMA + per-rank batched select on owned layers + all-reduce "
                                         "of 29 thresholds + replicated multi-tensor mask/apply"},
        "module_api": {"api": "MagnitudePruningCallback(running_average=True)(w, sparsity, mask) per layer",
                       "ms_per_step": round(ms_mod, 5), "value": round(world * 29 * n / (ms_mod * 1e-3) / 1e9, 2)},
        "module_api_one_cuda_graph": (None if ms_gmod is None else
                                      {"api": "the 29 prune()-wrapped modules' weight accesses of one step as ONE CUDA graph "
                                              "(qsparse_b200.GraphedTrainStep)", "ms_per_step": round(ms_gmod, 5),
                                       "value": round(world * 29 * n / (ms_gmod * 1e-3) / 1e9, 2)}),
        "module_api_batched_one_cuda_graph": (None if ms_gbmod is None else
                                              {"api": "WeightSetPruner.step() + the 29 module accesses captured into ONE CUDA "
                                                      "graph (qsparse_b200.GraphedTrainStep)",
                                               "ms_per_step": round(ms_gbmod, 5),
                                               "value": round(world * 29 * n / (ms_gbmod * 1e-3) / 1e9, 2)}),
        "module_api_batched": {"api": "WeightSetPruner(model).step() + every prune()-wrapped module's .weight",
                               "ms_per_step": round(ms_bmod, 5),
                               "value": round(world * 29 * n / (ms_bmod * 1e-3) / 1e9, 2)},
        "launch_mode": "eager (sampler, streaming pass, 3 candidate passes, fix-up, gated full pass)",
        "gpu_launches": 7 * steps,
        "e2e": {"value": round(world * 29 * n / e2e_s / 1e9, 3), "unit": "GB/s", "h2d_bytes_per_step": 4 * n * world,
                "d2h_bytes_per_step": 4 * n * world, "ms_per_step": round(e2e_s * 1e3, 3), "steps": e2e_steps,
                "api": "pinned host weights -> device -> parallel.prune_weight_set_step -> pruned weights to pinned host"},
        "roofline": {"bound": "hbm", "kernel": "step_partition_kernel (EMA + provisional mask + apply + candidate append, one pass)",
                     "achieved": round(traffic_bpe * n / (ms * 1e-3) / 1e9, 1), "peak": peak, "peak_source": peak_src,
                     "unit": "GB/s", "frac": round(traffic_bpe * n / (ms * 1e-3) / 1e9 / peak, 4),
                     "traffic": prof.get("step_partition_dram_bytes_per_launch"),
                     "algorithmic_bytes_per_launch": int(traffic_bpe * n), "avg_launch_us": round(ms * 1e3, 2),
                     "note": "whole-step time over the streaming pass's bytes: the sampler, candidate passes and fix-up "
                             "(~25 % of the step) are charged to it"},
        "gpu_eager_baseline": gpu_eager, "cpu_baseline": cpu,
    })
    return line


def cpu_c4(threads, sparsity):
    """bounded sample: `threads` layers of [512,512,3,3] (one per thread): EMA + sort-based mask + apply"""
    import numpy as np
    from concurrent.futures import ThreadPoolExecutor
    from oracle import oracle as orc
    layers = max(1, min(threads, 8))
    rng = np.random.default_rng(4)
    ws = [(rng.standard_normal((512, 512, 3, 3), dtype=np.float32) * np.float32(0.02)) for _ in range(layers)]
    mags = [np.abs(w) * np.float32(0.9) for w in ws]
    pool = ThreadPoolExecutor(layers)

    def one(i):
        mags[i] = orc.magnitude_ema(mags[i].reshape(-1), np.abs(ws[i]).reshape(-1), 3).reshape(ws[i].shape)
        mask, _ = orc.mask_given_importance(mags[i].reshape(-1), sparsity)
        return orc.mask_apply(ws[i].reshape(-1), mask.reshape(-1), -1)

    t0 = time.perf_counter()
    list(pool.map(one, range(layers)))
    dt = time.perf_counter() - t0
    n = sum(w.size for w in ws)
    return {"value": round(29 * n / dt / 1e9, 3), "unit": "GB/s", "cores": layers, "kind": "port", "steps": 1,
            "sample": f"one step over {layers} of the 29 layers ([512,512,3,3] each, one per thread; qsort-based threshold), "
                      f"{dt:.1f} s", "elems_per_s": round(n / dt, 1)}


# ============================================================================= config 5
C5_METRIC = "elementwise fake-quant+prune fwd/bwd HBM GB/s"


def c5_config(strong, sizes):
    return {"workload": "config[4]: flat fp32 tensors, fused prune (element mask given) + 8-bit pow2 fake-quant forward "
                        "(R x, R mask, W y = 9 B/elem) and backward (R g, R mask, W gx = 9 B/elem), 2^20 .. 2^32 elements",
            "log2_sizes": sizes, "headline_size": "2^30 elements per GPU" if not strong else "2^32 elements over all GPUs",
            "parallelism": "independent shards, no collective (" + ("strong: total fixed" if strong else "weak: n per GPU fixed") + ")",
            "l2": "clean-line flush between timed launches for tensors that fit the 126 MB L2 (n <= 2^24)"}


def run_c5(args, env):
    import torch
    from qsparse_b200 import ops
    world, rank, dev = env["world"], env["rank"], env["dev"]
    peak, peak_src = env["peak"]
    sizes = [20, 22, 24, 26, 28, 30, 32]
    headline = 32 if args.strong else 30
    dec = torch.tensor([5.0], device=dev)
    flush = Flusher(torch, dev)
    sampler = env["sampler_cls"](dev.index)
    if rank == 0:
        sampler.start()
        time.sleep(0.2)
    sweep = []
    head = None
    for p in sizes:
        n_total = 1 << p
        n5 = n_total // world if args.strong else n_total
        if n5 < 1024:
            continue
        x5 = torch.empty(n5, device=dev)
        m5 = torch.empty(n5, dtype=torch.bool, device=dev)
        gen = torch.Generator(device=dev).manual_seed(5 + rank)
        for lo in range(0, n5, 1 << 28):              # fill in 1 GiB pieces: no 16 GB temporaries at 2^32
            hi = min(lo + (1 << 28), n5)
            x5[lo:hi].normal_(generator=gen)
            m5[lo:hi] = torch.rand(hi - lo, device=dev, generator=gen) > 0.5
        y5 = torch.empty_like(x5)
        lay = (1, 1, n5)
        fl = flush if n5 * 4 <= L2_BYTES * 2 else None
        steps = max(5, min(args.steps, 200 if p <= 26 else (40 if p <= 30 else 10)))

        def fwd():
            ops.fq_pow2_fwd(x5, dec, lay, mask=m5, out=y5)

        def bwd():
            ops.ste_bwd(x5, dec, True, 8, 0, lay, mask=m5, clamp_in_place=False, want_gx=True)

        def both():
            fwd()
            bwd()
        ms_f = timed(torch, fwd, steps, 3, fl, world, dev)
        ms_b = timed(torch, bwd, steps, 3, fl, world, dev)
        rec = {"log2n": p, "n_per_gpu": n5, "fwd_us": round(ms_f * 1e3, 2), "bwd_us": round(ms_b * 1e3, 2),
               "fwd_gbs": round(world * 9 * n5 / (ms_f * 1e-3) / 1e9, 1), "bwd_gbs": round(world * 9 * n5 / (ms_b * 1e-3) / 1e9, 1),
               "fwd_frac": round(9 * n5 / (ms_f * 1e-3) / 1e9 / peak, 4), "bwd_frac": round(9 * n5 / (ms_b * 1e-3) / 1e9 / peak, 4)}
        if p == headline:
            ms_h = back_to_back(torch, both, steps, 3, world, dev)
            # property at full size: idempotence of the fake-quantizer on its own output, masked zeros are +0
            fwd()
            y_again = ops.fq_pow2_fwd(y5, dec, lay, mask=m5)
            head_n = min(n5, 1 << 22)
            prop = bool(torch.equal(y_again, y5)) and bool((y5[:head_n][~m5[:head_n]] == 0).all().item())
            head = dict(n5=n5, ms=ms_h, steps=steps, prop=prop, ms_f=ms_f, ms_b=ms_b)
            del y_again
        sweep.append(rec)
        del x5, y5, m5
        torch.cuda.empty_cache()
    clocks = sampler.stop() if rank == 0 else None
    n5, ms = head["n5"], head["ms"]

    # e2e at 2^26 per GPU: pinned host x, g, mask in; y, gx out, through the autograd functional API
    from qsparse_b200.quantize import quantize_with_decimal
    ne = 1 << 26
    hx = torch.randn(ne).pin_memory()
    hg = torch.randn(ne).pin_memory()
    hm = (torch.rand(ne) > 0.5).pin_memory()
    hy = torch.empty(ne).pin_memory()
    hgx = torch.empty(ne).pin_memory()
    e2e_steps = max(4, min(args.steps, 10))

    def e2e_step():
        xd = hx.to(dev, non_blocking=True).requires_grad_(True)
        md = hm.to(dev, non_blocking=True)
        gd = hg.to(dev, non_blocking=True)
        yd = quantize_with_decimal(xd * md, 8, 5)
        yd.backward(gd)
        hy.copy_(yd.detach(), non_blocking=True)
        hgx.copy_(xd.grad, non_blocking=True)
    e2e_step()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        e2e_step()
    torch.cuda.synchronize()
    e2e_s = (time.perf_counter() - t0) / e2e_steps
    dist = _dist()
    if dist:
        t = torch.tensor([e2e_s], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_s = t.item()
    del hx, hg, hm, hy, hgx

    gpu_eager = cpu = None
    if world == 1 and not args.no_gpu_eager:
        from oracle.torch_eager import masked_pow2_fwd_bwd
        n_e = 1 << 28
        xe = torch.randn(n_e, device=dev)
        ge = torch.randn(n_e, device=dev)
        me = torch.rand(n_e, device=dev) > 0.5
        ms_e = back_to_back(torch, lambda: masked_pow2_fwd_bwd(xe, ge, me, dec), 5, 2, 1, dev)
        ours_e = next(r for r in sweep if r["log2n"] == 28)
        ours_ms = (ours_e["fwd_us"] + ours_e["bwd_us"]) / 1e3
        gpu_eager = {"what": "the reference's eager ATen sequence (mul, pow, mul, int, float, clamp_, float, mul | clamp_, ne, "
                             "index_put_, mul) at 2^28 elements",
                     "ms_per_step": round(ms_e, 4), "value": round(18 * n_e / (ms_e * 1e-3) / 1e9, 2), "unit": "GB/s",
                     "speedup_of_this_repo": round(ms_e / ours_ms, 2)}
        del xe, ge, me
    if world == 1 and not args.no_cpu_baseline:
        cpu = cpu_c5(env["host_threads"])
    value = world * 18 * n5 / (ms * 1e-3) / 1e9
    line = _base(C5_METRIC, value, world, args, ms, c5_config(args.strong, sizes), world * n5, clocks,
                 scaling="strong" if args.strong else "weak")
    line["steps"] = head["steps"]
    best = head["ms_f"]
    line.update({
        "frac_of_measured_hbm_peak": round(value / world / peak, 4),
        "value_actual": round(value, 2), "bytes_per_elem": {"algorithmic": 18, "actual": 18},
        "sweep": sweep, "full_size_property_ok": head["prop"],
        "launch_mode": "eager, forward + backward kernel per step",
        "gpu_launches": 2 * head["steps"],
        "e2e": {"value": round(world * 18 * ne / e2e_s / 1e9, 3), "unit": "GB/s", "h2d_bytes_per_step": 9 * ne * world,
                "d2h_bytes_per_step": 8 * ne * world, "ms_per_step": round(e2e_s * 1e3, 3), "steps": e2e_steps,
                "api": "pinned host x, g, mask -> device -> quantize_with_decimal(x * mask, 8, 5) + autograd backward "
                       "(functional API) -> y, gx to pinned host; 2^26 elements per GPU"},
        "roofline": {"bound": "hbm", "kernel": "map_kernel<Pow2Op<ELEMENT mask>> (y = Q(x*mask), 9 B/elem)",
                     "achieved": round(9 * n5 / (best * 1e-3) / 1e9, 1), "peak": peak, "peak_source": peak_src, "unit": "GB/s",
                     "frac": round(9 * n5 / (best * 1e-3) / 1e9 / peak, 4), "traffic": _prof().get("c5_fwd_dram_bytes_per_launch"),
                     "algorithmic_bytes_per_launch": 9 * n5, "avg_launch_us": round(best * 1e3, 2)},
        "gpu_eager_baseline": gpu_eager, "cpu_baseline": cpu,
    })
    return line


def cpu_c5(threads):
    import numpy as np
    from concurrent.futures import ThreadPoolExecutor
    from oracle import oracle as orc
    n = 1 << 26
    threads = max(1, threads)
    rng = np.random.default_rng(5)
    x = rng.standard_normal(n, dtype=np.float32)
    g = rng.standard_normal(n, dtype=np.float32)
    m = rng.random(n, dtype=np.float32) > 0.5
    sl = [slice(i * n // threads, (i + 1) * n // threads) for i in range(threads)]
    pool = ThreadPoolExecutor(threads)
    dec = np.array([5.0], np.float32)

    def part(s):
        orc.fq_pow2_fwd(x[s], dec, -1, mask=m[s])
        orc.ste_bwd(g[s], dec, 8, -1, True, False, mask=m[s])

    list(pool.map(part, sl))
    steps = 5
    t0 = time.perf_counter()
    for _ in range(steps):
        list(pool.map(part, sl))
    dt = (time.perf_counter() - t0) / steps
    return {"value": round(18 * n / dt / 1e9, 3), "unit": "GB/s", "cores": threads, "kind": "port", "steps": steps,
            "sample": f"{steps} forward+backward passes over 2^26 elements, sliced over the threads, {dt*1e3:.0f} ms/step",
            "elems_per_s": round(n / dt, 1)}


# ============================================================================= config 1
C1_METRIC = "MNIST-net training steps/s (8-bit quantize + 50% channel prune, batch 64)"
C1_BATCH = 64


def c1_config(kind):
    return {"workload": "config[0]: the CNN of examples/mnist.py (conv 1-32-64, fc 9216-128-10, BatchNorm), batch 64 of "
                        "synthetic MNIST-shaped data, converted with prune(sparsity=0.5, dimensions={1}, start=20, "
                        "interval=10, repetition=4) on the first two ReLU outputs and quantize(bits=8, channelwise=-1, "
                        f"timeout=10, callback={kind}) on the input, 4 weights and 3 activations; one step = forward + "
                        "nll_loss + backward + Adadelta step, in the steady state (after step 60)",
            "batch": C1_BATCH, "quantizer": kind,
            "parallelism": "replicas only (launch-bound: every tensor is < 6 MB)",
            "l2": "every tensor fits the L2: this configuration measures launch / host overhead, not bandwidth"}


def _c1_net(torch):
    nn, F = torch.nn, torch.nn.functional

    class Net(nn.Module):
        """topology of examples/mnist.py:17-44"""

        def __init__(self):
            super().__init__()
            self.conv_part = nn.Sequential(
                nn.Conv2d(1, 32, 3, 1), nn.BatchNorm2d(32), nn.ReLU(),
                nn.Conv2d(32, 64, 3, 1), nn.BatchNorm2d(64), nn.ReLU(),
                nn.MaxPool2d(2), nn.Dropout(0.0))
            self.linear_part = nn.Sequential(
                nn.Flatten(), nn.Linear(9216, 128), nn.BatchNorm1d(128), nn.ReLU(), nn.Dropout(0.0), nn.Linear(128, 10))

        def forward(self, x):
            return F.log_softmax(self.linear_part(self.conv_part(x)), dim=1)

    torch.manual_seed(1)
    return Net()


def _c1_convert(torch, q, net, kind, fuse):
    nn = torch.nn
    cb = {"ScalerQuantizer": q.ScalerQuantizer, "DecimalQuantizer": q.DecimalQuantizer}[kind]
    net = q.convert(net, q.prune(sparsity=0.5, dimensions={1}, start=20, interval=10, repetition=4),
                    activation_layers=[nn.ReLU], excluded_activation_layer_indexes=[(nn.ReLU, [-1])], log=False)
    return q.convert(net, q.quantize(bits=8, channelwise=-1, timeout=10, callback=cb()),
                     activation_layers=[nn.ReLU], weight_layers=[nn.Conv2d, nn.Linear], input=True, log=False,
                     fuse=fuse)


def _c1_time(torch, model, dev, steps, warm, host_batches=None):
    """(wall ms/step, CUDA-event ms/step, losses) of `steps` training steps after `warm` warm-up steps"""
    F = torch.nn.functional
    model.train()
    opt = torch.optim.Adadelta([p for p in model.parameters() if p.requires_grad], lr=1.0)
    g = torch.Generator(device=dev).manual_seed(11)
    x = torch.randn(C1_BATCH, 1, 28, 28, device=dev, generator=g)
    y = torch.randint(0, 10, (C1_BATCH,), device=dev, generator=g)

    def step(i):
        if host_batches is not None:
            hx, hy = host_batches[i % len(host_batches)]
            xb, yb = hx.to(dev, non_blocking=True), hy.to(dev, non_blocking=True)
        else:
            xb, yb = x, y
        opt.zero_grad(set_to_none=True)
        loss = F.nll_loss(model(xb), yb)
        loss.backward()
        opt.step()
        return loss

    for i in range(warm):
        step(i)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0 = time.perf_counter()
    e0.record()
    last = None
    for i in range(steps):
        last = step(i)
        if host_batches is not None:
            last = last.item()         # the step's result is read back every step on the e2e path
    e1.record()
    torch.cuda.synchronize()
    wall = (time.perf_counter() - t0) / steps * 1e3
    return wall, e0.elapsed_time(e1) / steps, float(last)


def _c1_time_graph(torch, q, model, dev, steps, warm):
    """(CUDA-event ms/step, loss) of the steady-state training step captured into ONE CUDA graph
    (qsparse_b200.GraphedTrainStep; for the plain net: a bare torch.cuda.graph capture)"""
    F = torch.nn.functional
    model.train()
    opt = torch.optim.Adadelta([p for p in model.parameters() if p.requires_grad], lr=1.0, capturable=True)
    g = torch.Generator(device=dev).manual_seed(11)
    x = torch.randn(C1_BATCH, 1, 28, 28, device=dev, generator=g)
    y = torch.randint(0, 10, (C1_BATCH,), device=dev, generator=g)

    def step():
        opt.zero_grad(set_to_none=True)
        loss = F.nll_loss(model(x), y)
        loss.backward()
        opt.step()
        return loss

    for _ in range(warm):
        step()
    torch.cuda.synchronize()
    gs = q.GraphedTrainStep(model, step, warmup=3)
    for _ in range(10):
        gs.replay()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0 = time.perf_counter()
    e0.record()
    for _ in range(steps):
        gs.replay()
    e1.record()
    torch.cuda.synchronize()
    wall = (time.perf_counter() - t0) / steps * 1e3
    gs.sync_host()
    return wall, e0.elapsed_time(e1) / steps, float(gs.result)


def run_c1(args, env):
    import io
    import contextlib
    import torch
    import qsparse_b200 as q
    world, rank, dev = env["world"], env["rank"], env["dev"]
    peak, peak_src = env["peak"]
    q.set_qsparse_options(log_on_created=False)
    torch.backends.cudnn.benchmark = False
    kind = "DecimalQuantizer" if getattr(args, "c1_decimal", False) else "ScalerQuantizer"
    steps = max(50, min(args.steps, 300))
    warm = 70
    sampler = env["sampler_cls"](dev.index)
    if rank == 0:
        sampler.start()
    res = {}
    with contextlib.redirect_stdout(io.StringIO()), contextlib.redirect_stderr(io.StringIO()):
        res["plain_net_no_qsparse"] = _c1_time(torch, _c1_net(torch).to(dev), dev, steps, warm)
        fused = _c1_convert(torch, q, _c1_net(torch), kind, True).to(dev)
        res["fused"] = _c1_time(torch, fused, dev, steps, warm)
        res["unfused"] = _c1_time(torch, _c1_convert(torch, q, _c1_net(torch), kind, False).to(dev), dev, steps, warm)
        res["fused_one_cuda_graph"] = _c1_time_graph(torch, q, _c1_convert(torch, q, _c1_net(torch), kind, True).to(dev),
                                                     dev, steps, warm)
        res["plain_net_one_cuda_graph"] = _c1_time_graph(torch, q, _c1_net(torch).to(dev), dev, steps, warm)
        hb = [(torch.randn(C1_BATCH, 1, 28, 28).pin_memory(), torch.randint(0, 10, (C1_BATCH,)).pin_memory())
              for _ in range(8)]
        e2e_model = _c1_convert(torch, q, _c1_net(torch), kind, True).to(dev)
        res["e2e"] = _c1_time(torch, e2e_model, dev, steps, warm, host_batches=hb)
    clocks = sampler.stop() if rank == 0 else None
    from qsparse_b200.fused import FusedPruneQuantSequential
    fused_steps = [m.fused_steps for m in fused.modules() if isinstance(m, FusedPruneQuantSequential)]
    gpu_eager = cpu = None
    if world == 1 and not args.no_gpu_eager:
        from oracle.torch_eager import build_mnist_eager
        eg = build_mnist_eager("decimal" if kind == "DecimalQuantizer" else "scaler").to(dev)
        w_e, ev_e, _ = _c1_time(torch, eg, dev, steps, warm)
        gpu_eager = {"what": "the same converted net with the reference's layers restated as eager torch modules "
                             "(oracle/torch_eager.py::build_mnist_eager, equal to the reference step for step on CPU)",
                     "ms_per_step": round(w_e, 4), "cuda_event_ms_per_step": round(ev_e, 4),
                     "value": round(1e3 / w_e, 2), "unit": "steps/s",
                     "speedup_of_this_repo": round(w_e / res["fused"][0], 2),
                     "speedup_of_this_repo_as_one_cuda_graph": round(w_e / res["fused_one_cuda_graph"][0], 2)}
    if world == 1 and not args.no_cpu_baseline:
        from oracle.torch_eager import build_mnist_eager
        cpu_dev = torch.device("cpu")
        torch.set_num_threads(env["host_threads"])
        egc = build_mnist_eager("decimal" if kind == "DecimalQuantizer" else "scaler")
        F = torch.nn.functional
        opt = torch.optim.Adadelta([p for p in egc.parameters() if p.requires_grad], lr=1.0)
        xc, yc = torch.randn(C1_BATCH, 1, 28, 28), torch.randint(0, 10, (C1_BATCH,))
        egc.train()

        def cstep():
            opt.zero_grad()
            F.nll_loss(egc(xc), yc).backward()
            opt.step()
        for _ in range(62):
            cstep()
        t0 = time.perf_counter()
        for _ in range(40):
            cstep()
        dt = (time.perf_counter() - t0) / 40
        cpu = {"value": round(1 / dt, 2), "unit": "steps/s", "cores": env["host_threads"], "kind": "port",
               "sample": f"40 steady-state training steps of the eager restatement on CPU tensors, {dt*1e3:.1f} ms/step",
               "ms_per_step": round(dt * 1e3, 3)}
    wall, evms, loss = res["fused_one_cuda_graph"]      # the headline: the step as ONE CUDA graph
    hot_elems = C1_BATCH * (28 * 28 + 32 * 26 * 26 + 64 * 24 * 24 + 128) + 32 * 9 + 64 * 32 * 9 + 128 * 9216 + 1280
    hot_bytes = 20 * hot_elems
    line = _base(C1_METRIC, world * 1e3 / wall, world, args, wall, c1_config(kind), world * C1_BATCH, clocks)
    line["unit"] = "steps/s"
    line["steps"] = steps
    line.update({
        "loss_after_timed_steps": loss, "fused_steps_per_site": fused_steps,
        "variants_ms_per_step": {k: {"wall": round(v[0], 4), "cuda_events": round(v[1], 4)} for k, v in res.items()},
        "qsparse_overhead_ms_per_step": {"fused": round(res["fused"][0] - res["plain_net_no_qsparse"][0], 4),
                                         "unfused": round(res["unfused"][0] - res["plain_net_no_qsparse"][0], 4),
                                         "one_cuda_graph": round(res["fused_one_cuda_graph"][0]
                                                                 - res["plain_net_one_cuda_graph"][0], 4)},
        "launch_mode": "ONE CUDA graph per training step (qsparse_b200.GraphedTrainStep over the module API: 10 prune / "
                       "quantize layers per step, fusion pass applied to the two prune->quantize activation sites); the "
                       "eager module API is variants_ms_per_step.fused",
        "eager_module_api": {"ms_per_step": round(res["fused"][0], 4), "value": round(world * 1e3 / res["fused"][0], 2),
                             "unit": "steps/s"},
        "cuda_graph": {"what": "the same steady-state training step (forward, backward, Adadelta step) captured into ONE "
                               "CUDA graph by qsparse_b200.GraphedTrainStep: step indices live on the device, replays "
                               "are bit-equal to eager steps (tests/test_gpu_configs.py)",
                       "ms_per_step": round(res["fused_one_cuda_graph"][0], 4),
                       "value": round(world * 1e3 / res["fused_one_cuda_graph"][0], 2), "unit": "steps/s",
                       "plain_net_ms_per_step": round(res["plain_net_one_cuda_graph"][0], 4)},
        "gpu_launches": None,
        "e2e": {"value": round(world * 1e3 / res["e2e"][0], 2), "unit": "steps/s", "h2d_bytes_per_step": C1_BATCH * (784 * 4 + 8),
                "d2h_bytes_per_step": 4, "ms_per_step": round(res["e2e"][0], 4), "steps": steps,
                "api": "pinned host batch -> device -> converted model forward / backward / optimizer step -> loss.item()"},
        "roofline": {"bound": "hbm", "kernel": "(launch-bound configuration) all prune / quantize tensors of one step",
                     "achieved": round(hot_bytes / (wall * 1e-3) / 1e9, 2), "peak": peak, "peak_source": peak_src,
                     "unit": "GB/s", "frac": round(hot_bytes / (wall * 1e-3) / 1e9 / peak, 5), "traffic": None,
                     "algorithmic_bytes_per_launch": hot_bytes,
                     "note": "20 B/elem over the 1.5 M activation + 1.2 M weight elements the operators touch per step, "
                             "divided by the WHOLE training step's wall time: this configuration is bound by kernel-launch "
                             "and Python overhead, the roofline fraction is reported for completeness"},
        "gpu_eager_baseline": gpu_eager, "cpu_baseline": cpu,
    })
    return line


# ============================================================================= dispatch
def run_ours(args, env):
    return {1: run_c1, 3: run_c3, 4: run_c4, 5: run_c5}[args.config](args, env)


def run_reference(args):
    threads = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    if args.config == 1:
        import torch
        from oracle.torch_eager import build_mnist_eager
        F = torch.nn.functional
        torch.set_num_threads(threads)
        net = build_mnist_eager("scaler").train()
        opt = torch.optim.Adadelta([p for p in net.parameters() if p.requires_grad], lr=1.0)
        xc, yc = torch.randn(C1_BATCH, 1, 28, 28), torch.randint(0, 10, (C1_BATCH,))

        def cstep():
            opt.zero_grad()
            F.nll_loss(net(xc), yc).backward()
            opt.step()
        for _ in range(62):
            cstep()
        n = max(5, min(args.steps, 40))
        t0 = time.perf_counter()
        for _ in range(n):
            cstep()
        dt = (time.perf_counter() - t0) / n
        cpu = {"value": round(1 / dt, 2), "unit": "steps/s", "cores": threads, "kind": "port", "steps": n,
               "ms_per_step": round(dt * 1e3, 3),
               "sample": f"{n} steady-state training steps of the eager restatement of the reference's layers on CPU tensors"}
        metric, cfg = C1_METRIC, c1_config("ScalerQuantizer")
    elif args.config == 3:
        cpu = cpu_c3(threads, max(1, min(args.steps, 10)))
        metric, cfg = C3_METRIC, c3_config()
    elif args.config == 4:
        sp = 0.5 if args.sparsity is None else args.sparsity
        cpu = cpu_c4(threads, sp)
        metric, cfg = C4_METRIC, c4_config(sp)
    else:
        cpu = cpu_c5(threads)
        metric, cfg = C5_METRIC, c5_config(args.strong, [20, 22, 24, 26, 28, 30, 32])
    v = cpu["value"]
    return {"impl": "reference", "metric": metric, "value": v, "unit": cpu["unit"], "n_gpus": args.gpus, "steps": cpu["steps"],
            "warmup": args.warmup, "ms_per_step": cpu.get("ms_per_step"), "higher_is_better": True,
            "scaling": "strong" if (args.config == 5 and args.strong) else "weak", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic", "config": cfg, "cpu_baseline": cpu,
            "e2e": {"value": v, "unit": cpu["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "note": "oracle/ (plain-C restatement of the reference, pinned to its golden vectors) on the host cores"}
