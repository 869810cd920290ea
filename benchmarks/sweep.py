"""Per-kernel bandwidth sweep on one B200 (development tool, not the graded bench).

    python benchmarks/sweep.py [--out gpurun_out/sweep.jsonl] [--quick]

Times every hot-path kernel with CUDA events on the launching stream; between timed
launches a 512 MB buffer is rewritten to flush the 126 MB L2.  GB/s = algorithmic bytes
(SURVEY §8d table) / time.
"""
import argparse
import json
import sys
from pathlib import Path

import torch

sys.path.insert(0, str(Path(__file__).resolve().parent.parent))
from qsparse_b200 import ops  # noqa: E402

PEAK = 6457.4  # MEASURED_PEAKS.json hbm_gbs (copy)


def timeit(fn, iters=12, warmup=3, flush=None):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(iters):
        if flush is not None:
            flush[0].add_(1.0)
            flush[1].max()
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        fn()
        e.record()
        e.synchronize()
        ts.append(s.elapsed_time(e) * 1e3)
    ts.sort()
    return ts[len(ts) // 2], ts[0]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default="gpurun_out/sweep.jsonl")
    ap.add_argument("--quick", action="store_true")
    args = ap.parse_args()
    Path(args.out).parent.mkdir(parents=True, exist_ok=True)
    out = open(args.out, "w")
    dev = torch.device("cuda:0")
    flush = torch.zeros(128 * 1024 * 1024, device=dev)  # 512 MB, rewritten between launches
    flush_rd = torch.zeros(96 * 1024 * 1024, device=dev)  # 384 MB, read after the write so that the
    # L2 holds CLEAN lines when the timed kernel starts (dirty lines would be written
    # back during the measurement and charge up to 126 MB of DRAM writes to it)
    torch.manual_seed(2)

    def report(name, nbytes, fn, **extra):
        med, best = timeit(fn, flush=(flush, flush_rd))
        rec = dict(kernel=name, us_median=round(med, 2), us_best=round(best, 2), gbs_median=round(nbytes / med / 1e3, 1),
                   gbs_best=round(nbytes / best / 1e3, 1), frac_of_copy_peak=round(nbytes / med / 1e3 / PEAK, 3), **extra)
        print(json.dumps(rec), flush=True)
        out.write(json.dumps(rec) + "\n")
        out.flush()

    # ---------------- config 2: [256, 64, 56, 56]
    shape, layout = (256, 64, 56, 56), (256, 64, 3136)
    n = 256 * 64 * 3136
    x = torch.relu(torch.randn(shape, device=dev))
    g = torch.randn(shape, device=dev)
    y = torch.empty_like(x)
    gx = torch.empty_like(x)
    dec1 = torch.tensor([5.0], device=dev)
    decC = torch.full((64,), 5.0, device=dev)
    mask75 = (torch.arange(64, device=dev) % 4 == 0)
    mask0 = torch.ones(64, dtype=torch.bool, device=dev)
    emask = torch.rand(shape, device=dev) > 0.5

    report("torch_copy", 8 * n, lambda: y.copy_(x))
    report("fq_pow2_tensor", 8 * n, lambda: ops.fq_pow2_fwd(x, dec1, (1, 1, n), out=y))
    report("ste_bwd_inplace", 8 * n, lambda: ops.ste_bwd(g, dec1, True, 8, 0, (1, 1, n)))
    report("fq_pow2_chdec", 8 * n, lambda: ops.fq_pow2_fwd(x, decC, layout, out=y))
    report("fq_pow2_chmask0", 8 * n, lambda: ops.fq_pow2_fwd(x, dec1, layout, mask=mask0, out=y))
    report("fq_pow2_chmask75", 8 * n, lambda: ops.fq_pow2_fwd(x, dec1, layout, mask=mask75, out=y),
           note="dense-algorithmic bytes; 75% of reads skipped")
    report("fq_pow2_emask", 9 * n, lambda: ops.fq_pow2_fwd(x, dec1, (1, 1, n), mask=emask, out=y))
    report("fq_scaler_tensor", 8 * n, lambda: ops.fq_scaler_fwd(x, 0.037, (1, 1, n), out=y))
    report("fq_line_tensor", 8 * n, lambda: ops.fq_line_fwd(x, (-0.1, 0.9), 8, True, (1, 1, n), out=y))
    lines64 = torch.tensor([[-0.1, 0.9]] * 64, device=dev)
    report("fq_line_ch", 8 * n, lambda: ops.fq_line_fwd(x, lines64, 8, True, layout, out=y))

    def bwd_fused():
        lib_gx = ops.N.load_library()
        from ctypes import c_double, c_int, c_int64
        ops.N.check(lib_gx.qsb_ste_bwd(ops.N.ptr(g), ops.N.ptr(None), ops.N.ptr(gx), ops.N.ptr(dec1), c_int64(1),
                                       c_double(0), c_int(1), c_int(8), c_int(0), ops.N.ptr(mask75), c_int(1),
                                       c_int64(256), c_int64(64), c_int64(3136), ops.N.stream_ptr(dev)), "ste")
    report("ste_bwd_fused_gx", 8 * n, bwd_fused)
    report("export_int8_pow2_ch", 5 * n, lambda: ops.quant_export_int8(x, ops.EXPORT_DECIMAL, decC, 8, layout),
           note="4 B read + 1 B written per element")
    report("export_int4_pow2_ch", 4.5 * n,
           lambda: ops.quant_export_int8(x, ops.EXPORT_DECIMAL, decC, 4, layout, pack4=True),
           note="4 B read + half a byte written per element")
    report("mask_apply_ch", 8 * n, lambda: ops.mask_apply(x, mask75, layout, out=y))
    report("reduce_abssum_absmax_ch", 4 * n, lambda: ops.reduce_stats(x, layout, abssum=True, absmax=True))
    report("reduce_absmax_tensor", 4 * n, lambda: ops.reduce_stats(x, (1, 1, n), absmax=True))
    report("reduce_minmax_ch", 4 * n, lambda: ops.reduce_stats(x, layout, minmax=True))
    report("torch_absmax_tensor", 4 * n, lambda: x.abs().max())
    report("torch_amax_ch", 4 * n, lambda: x.amax(dim=(0, 2, 3)))

    # reduce -> params -> apply, then backward: the fused training step (20 B/elem)
    mag = torch.zeros(64, device=dev)
    mask = torch.ones(64, dtype=torch.bool, device=dev)
    scale = torch.zeros(1, device=dev)
    dec = torch.zeros(1, device=dev)
    state = dict(t=0)

    def step():
        st = ops.reduce_stats(x, layout, abssum=True, absmax=True)
        ops.prune_quant_params(mag, mask, scale, dec, st, 256 * 3136.0, state["t"], 1, state["t"] > 0, 48, 8,
                               state["t"], True)
        ops.fq_pow2_fwd(x, dec, layout, mask=mask, out=y)
        bwd_fused()
        state["t"] += 1
    report("fused_train_step", 20 * n, step)

    # the reference-API route of config 2 (iii): MagnitudePruningCallback with a channel mask, refresh every step
    import importlib
    sp = importlib.import_module("qsparse_b200.sparse")
    for fuse in (True, False):
        sp.FUSE_PRUNE_STEP = fuse
        cb = sp.MagnitudePruningCallback(running_average=True)
        cb.train()
        pmask = torch.nn.Parameter(torch.ones(1, 64, 1, 1, dtype=torch.bool, device=dev), requires_grad=False)
        with torch.no_grad():
            cb(x, 0.75, pmask)
            report("prune_callback_structured_step", 12 * n, lambda: cb(x, 0.75, pmask),
                   route="3 launches (partials, parameter kernel, apply)" if fuse else "9 launches")
    sp.FUSE_PRUNE_STEP = True
    # config 2 (ii): QuantizeLayer(bits=8, channelwise=-1, DecimalQuantizer) training forward, 12 B/elem
    import qsparse_b200 as q
    qz = importlib.import_module("qsparse_b200.quantize")
    for fuse in (True, False):
        qz.FUSE_ROW_QUANTIZE = fuse
        ql = q.quantize(bits=8, channelwise=-1, timeout=1, callback=q.DecimalQuantizer())
        ql.train()
        with torch.no_grad():
            ql(x)
            ql(x)
            report("quantize_layer_tensor_step", 12 * n, lambda: ql(x),
                   route="3 launches (partials, parameter kernel, quantize)" if fuse else "5 launches")
    qz.FUSE_ROW_QUANTIZE = True
    del emask
    # ---------------- config 3: [4096, 4096] channelwise=0
    w = torch.randn(4096, 4096, device=dev) * 0.02
    wy = torch.empty_like(w)
    nw = w.numel()
    lines = torch.zeros(4096, 2, device=dev)
    report("c3_reduce_minmax", 4 * nw, lambda: ops.reduce_stats(w, (1, 4096, 4096), minmax=True))
    st = ops.reduce_stats(w, (1, 4096, 4096), minmax=True)
    ops.lines_ema_(lines, st["min"], st["max"], 1)
    report("c3_line_fwd", 8 * nw, lambda: ops.fq_line_fwd(w, lines, 4, True, (1, 4096, 4096), out=wy))

    def c3_access():      # the real weight access: reduce -> EMA -> line quant, back to back (W stays in L2)
        st_ = ops.reduce_stats(w, (1, 4096, 4096), minmax=True)
        ops.lines_ema_(lines, st_["min"], st_["max"], 2)
        ops.fq_line_fwd(w, lines, 4, True, (1, 4096, 4096), out=wy)
    report("c3_weight_access", 12 * nw, c3_access)
    # the same access through the row-resident fused kernel: one launch, 8 B/elem of traffic.  Reported
    # against the 12 B/elem of the reference's algorithm too (what the two-launch path is measured on).
    lines2 = torch.zeros(4096, 2, device=dev)
    report("c3_weight_access_fused", 8 * nw, lambda: ops.row_quant_fused_(w, lines2, ops.ROW_LINE, 4, 2, True),
           note="8 B/elem actual traffic")
    report("c3_weight_access_fused_alg12", 12 * nw,
           lambda: ops.row_quant_fused_(w, lines2, ops.ROW_LINE, 4, 2, True), note="12 B/elem dense-algorithmic")
    sc2 = torch.zeros(4096, 1, device=dev)
    report("c3_weight_access_fused_scaler", 8 * nw, lambda: ops.row_quant_fused_(w, sc2, ops.ROW_SCALER, 4, 1))
    report("c3_weight_access_fused_decimal", 8 * nw, lambda: ops.row_quant_fused_(w, sc2, ops.ROW_DECIMAL, 4, 1))

    # ---------------- config 4: 64 Mi unstructured
    n4 = 1 << 26
    wt = torch.randn(n4, device=dev) * 0.02
    magf = wt.abs() * 0.9
    yb = torch.empty_like(wt)
    mk = torch.empty(n4, dtype=torch.bool, device=dev)
    report("c4_ema_full", 12 * n4, lambda: ops.magnitude_ema_full_(magf, wt, 3))
    report("c4_kth_value", 4 * n4, lambda: ops.kth_value(magf, n4 // 2), route="sampled pivots, ~1 pass")
    hint = ops.new_select_hints(1, dev)
    report("c4_kth_value_hinted", 4 * n4, lambda: ops.kth_value(magf, n4 // 2, hint=hint),
           route="pivots from the previous answer (warm start), ~1 pass")
    ops.set_tuning(4, 0)
    report("c4_kth_value_3pass", 4 * n4, lambda: ops.kth_value(magf, n4 // 2), route="3-pass radix select")
    ops.set_tuning(4, 1)
    thr = ops.kth_value(magf, n4 // 2)
    report("c4_mask_build_apply", 13 * n4, lambda: ops.mask_build_apply(magf, thr, wt, mk, out=yb))
    report("c4_torch_sort", 4 * n4, lambda: torch.sort(magf))
    # the whole step (EMA + select + mask/apply) as three kernels' worth of calls, and in one pass (K9)
    state = {"t": 3}

    def c4_three_stage():
        ops.magnitude_ema_full_(magf, wt, state["t"])
        th = ops.kth_value(magf, n4 // 2)
        ops.mask_build_apply(magf, th, wt, mk, out=yb)
    report("c4_prune_step_3stage", 29 * n4, c4_three_stage, note="EMA 12 + select 4 + mask/apply 13 B/elem")
    report("c4_prune_step_fused", 29 * n4,
           lambda: ops.prune_unstructured_step_batched_([magf], [wt], [mk], [yb], [n4 // 2], state["t"]),
           note="K9: one streaming pass, ~17.5 B/elem of traffic; GB/s on the reference's 29 B/elem")
    hint9 = ops.new_select_hints(1, dev)
    report("c4_prune_step_fused_hinted", 29 * n4,
           lambda: ops.prune_unstructured_step_batched_([magf], [wt], [mk], [yb], [n4 // 2], state["t"], hints=hint9),
           note="K9 with warm-started pivots")
    del wt, magf, yb, mk, x, g, y

    # ---------------- config 5: flat sweep, fused prune(element mask) + pow2 quant fwd, bwd
    for p in ([22, 26] if args.quick else [20, 22, 24, 26, 28, 30, 32]):
        n5 = 1 << p
        x5 = torch.empty(n5, device=dev)
        m5 = torch.empty(n5, dtype=torch.bool, device=dev)
        for lo in range(0, n5, 1 << 28):              # fill in 1 GiB pieces: no 16 GB temporaries at 2^32
            hi = min(lo + (1 << 28), n5)
            x5[lo:hi].normal_()
            m5[lo:hi] = torch.rand(hi - lo, device=dev) > 0.5
        y5 = torch.empty_like(x5)
        report("c5_fused_fwd", 9 * n5, lambda: ops.fq_pow2_fwd(x5, dec1, (1, 1, n5), mask=m5, out=y5), log2n=p)
        report("c5_fused_bwd", 9 * n5, lambda: ops.ste_bwd(x5, dec1, True, 8, 0, (1, 1, n5), mask=m5,
                                                           clamp_in_place=False, want_gx=True), log2n=p)
        report("c5_plain_fwd", 8 * n5, lambda: ops.fq_pow2_fwd(x5, dec1, (1, 1, n5), out=y5), log2n=p)
        del x5, y5, m5
    out.close()


if __name__ == "__main__":
    main()
