"""The host-buffer training step of the C-ABI (qsb_host_prune_quant_step / _submit / qsb_host_ctx_wait) against the
CPU oracle, and the parameter step on several statistics rows.

The host step uploads x and g chunk by chunk, reduces each x chunk into its own statistics row, combines the rows in
chunk order in one parameter step (qsb_prune_quant_rows_step_params), then applies the forward and the backward per
chunk and downloads y and gx.  It is the oracle's running-average form (update_magnitude 1): the mask is refreshed
whenever t_prune > 0 and the scale EMA runs at t_quant, so with t_prune = t_quant = t the reference is
``oracle_steps(xs, gs, sparsity, 1, refresh, summed_mean=True)`` with refresh = [t > 0 ...]: the mean |x| as the
kernels take it, the whole fp64 sum divided once by the count.

The inputs are the exactly summable patterns of test_gpu_prune_quant_step_routes, so every chunking sums to the
same fp64 value and magnitude, mask, scale, decimal, y and gx match the oracle bit for bit at every step.
"""
import ctypes
from ctypes import byref, c_int, c_int64, c_void_p

import numpy as np
import pytest
import torch

from oracle import oracle as orc
from tests.conftest import bits_equal, ulp_diff
from tests.test_gpu_prune_quant_step_routes import (
    BITS, FULL, TIES, State, _k, check_step, make_g, make_x, oracle_steps, refresh_schedule, sparsity_for_k)

BADARG, UNSUPPORTED = -1, -4
SENTINEL = np.array([0x7FA5A5A5], np.uint32).view(np.float32)[0]    # a NaN no step writes
STEPS_HOST = 6        # two rounds of two slots, then a third round that submits into busy slots


def _lib():
    from qsparse_b200 import _native as N
    return N.load_library()


def refresh_for(n):
    """refresh_schedule(1) (no refresh at t = 0, then every step) for n steps"""
    sched = refresh_schedule(1)
    return sched[:n] + [True] * (n - len(sched))


# ----------------------------------------------------------------------------- host buffers and the context
class HostBufs:
    """x, g in and y, gx out of one step: pinned torch tensors, or plain (pageable) numpy arrays"""

    def __init__(self, x, g, pinned=True):
        if pinned:
            self.arrs = [torch.from_numpy(np.ascontiguousarray(a)).pin_memory() for a in (x, g, x, g)]
            self.np = [a.numpy() for a in self.arrs]
        else:
            self.np = [np.array(a, np.float32, order="C", copy=True) for a in (x, g, x, g)]
        self.reset()

    def reset(self):
        for a in self.np[2:]:
            a.fill(SENTINEL)

    def ptrs(self):
        return [a.ctypes.data for a in self.np]

    def y(self):
        return self.np[2].copy()

    def gx(self):
        return self.np[3].copy()


class HostCtx:
    def __init__(self, max_elems, max_channels, n_chunks):
        from qsparse_b200 import _native as N
        self.lib = _lib()
        self.ctx = c_void_p()
        N.check(self.lib.qsb_host_ctx_create(byref(self.ctx), c_int64(max_elems), c_int64(max_channels),
                                             c_int(n_chunks)), "qsb_host_ctx_create")

    def submit(self, slot, bufs, st, layout, t_prune, k, t_quant=None, stream=None, sync=False, ptrs=None,
               state=None):
        from qsparse_b200 import _native as N
        o, c, i = layout
        x, g, y, gx = bufs.ptrs() if ptrs is None else ptrs
        mag, mask, scale, dec = (N.ptr(st.mag), N.ptr(st.mask), N.ptr(st.scale), N.ptr(st.dec)) \
            if state is None else state
        t_quant = t_prune if t_quant is None else t_quant
        stream = torch.cuda.current_stream().cuda_stream if stream is None else stream
        args = (x, g, y, gx, mag, mask, scale, dec, o, c, i, t_prune, k, BITS, t_quant, None, 1, stream or None)
        if sync:
            return self.lib.qsb_host_prune_quant_step(self.ctx, *args)
        return self.lib.qsb_host_prune_quant_step_submit(self.ctx, slot, *args)

    def wait(self, slot):
        assert self.lib.qsb_host_ctx_wait(self.ctx, slot) == 0

    def destroy(self):
        if self.ctx:
            assert self.lib.qsb_host_ctx_destroy(self.ctx) == 0
            self.ctx = c_void_p()


def host_got(st, bufs):
    return dict(imp=st.mag, mask=st.mask.clone(), scale=st.scale.clone(), dec=st.dec.clone(),
                y=torch.from_numpy(bufs.y()), gx=torch.from_numpy(bufs.gx()))


def unwritten(a):
    return int((a.view(np.uint32) == SENTINEL.view(np.uint32)).sum())


def check_out(bufs, ref, what):
    """y and gx of one step (the layer state may already hold a later step's)"""
    assert unwritten(bufs.y()) == 0 and unwritten(bufs.gx()) == 0, ("not written", what)
    if np.isfinite(ref["dec"]).all():
        assert bits_equal(bufs.y(), ref["y"]), ("y", what)
        assert bits_equal(bufs.gx(), ref["gx"]), ("gx", what)


def sequence(layout, pattern, which, seed, n):
    c = layout[1]
    sparsity = sparsity_for_k(which, c)
    xs = [make_x(layout, pattern if t > 0 or pattern not in ("nan", "inf") else "rand", seed + t, sparsity)
          for t in range(n)]
    gs = [make_g(layout, seed + t) for t in range(n)]
    return sparsity, xs, gs


def run_api(api, ctx, bufs, layout, k, refs, what):
    """one sequence through one form of the API, checked step by step"""
    st = State(layout[1])
    for b in bufs:
        b.reset()
    n = len(bufs)
    if api == "sync":
        for t in range(n):
            assert ctx.submit(0, bufs[t], st, layout, t, k, sync=True) == 0
            check_step(host_got(st, bufs[t]), refs[t], what + (api, t), stats=False)
    elif api == "alternate":
        for t in range(n):
            assert ctx.submit(t % 2, bufs[t], st, layout, t, k) == 0
            ctx.wait(t % 2)
            check_step(host_got(st, bufs[t]), refs[t], what + (api, t), stats=False)
    else:
        assert api == "in-flight"
        # t on slot 0 and t + 1 on slot 1, then wait on both ...
        assert ctx.submit(0, bufs[0], st, layout, 0, k) == 0
        assert ctx.submit(1, bufs[1], st, layout, 1, k) == 0
        ctx.wait(0)
        ctx.wait(1)
        check_out(bufs[0], refs[0], what + (api, 0))
        check_step(host_got(st, bufs[1]), refs[1], what + (api, 1), stats=False)
        # ... then every submit goes into a slot whose previous step nobody waited for (the implicit wait)
        for t in range(2, n):
            assert ctx.submit(t % 2, bufs[t], st, layout, t, k) == 0
        ctx.wait(0)
        ctx.wait(1)
        for t in range(2, n):
            check_out(bufs[t], refs[t], what + (api, t))
        check_step(host_got(st, bufs[n - 1]), refs[n - 1], what + (api, n - 1), stats=False)


# ----------------------------------------------------------------------------- chunking table
MODE1_FULL = [(p, w) for p, w, _ in FULL]
MODE1_TIES = [(p, w) for p, w, _ in TIES]
# (id, layout, n_chunks, patterns)
HOST_CASES = [
    ("even-1", (16, 64, 196), 1, MODE1_TIES),
    ("even-8", (16, 64, 196), 8, MODE1_TIES),
    ("short-last", (13, 64, 196), 8, MODE1_FULL),              # 7 chunks of 2 rows, the last of 1
    ("chunks>rows-3", (3, 64, 196), 8, MODE1_TIES),
    ("chunks>rows-1", (1, 64, 3136), 8, MODE1_TIES),
    ("col-mode", (64, 48, 1), 8, MODE1_FULL),
    ("odd-inner", (5, 257, 2053), 4, MODE1_FULL),
    ("256-chunks", (256, 7, 1), 256, MODE1_TIES),
    ("256->150-chunks", (300, 9, 1), 256, MODE1_FULL),           # 2 rows a chunk: 150 chunks
    ("big-col-chunk", (4096, 1000, 1), 8, MODE1_TIES),
    ("C2049", (2, 2049, 320), 3, MODE1_FULL),
    ("C4096", (16, 4096, 1), 3, MODE1_TIES),
]


@pytest.mark.gpu
@pytest.mark.parametrize("case", HOST_CASES, ids=[c[0] for c in HOST_CASES])
def test_host_step_matches_oracle(case):
    """sync call, submit / wait on alternating slots, and two steps in flight with implicit waits: each gives the
    oracle's sequence.  Every step has its own host buffers, so a slot or staging mix-up changes the result."""
    cid, layout, n_chunks, patterns = case
    o, c, i = layout
    ctx = HostCtx(o * c * i, c, n_chunks)
    try:
        for p_i, (pattern, which) in enumerate(patterns):
            sparsity, xs, gs = sequence(layout, pattern, which, 7 * p_i, STEPS_HOST)
            refs = oracle_steps(xs, gs, sparsity, 1, refresh_for(STEPS_HOST), summed_mean=True)
            bufs = [HostBufs(x, g) for x, g in zip(xs, gs)]
            for api in ("sync", "alternate", "in-flight"):
                run_api(api, ctx, bufs, layout, _k(sparsity, c), refs, (cid, pattern, which))
    finally:
        ctx.destroy()


@pytest.mark.gpu
def test_host_step_one_channel():
    """one channel: the only rank a refresh takes is k = 0 (the oracle's k = 1 is out of range, see
    test_host_step_refuses_bad_arguments), which keeps the channel: the oracle's mask of ones"""
    layout = (8, 1, 64)
    ctx = HostCtx(8 * 64, 1, 4)
    try:
        for p_i, pattern in enumerate(["rand", "zero", "dead"]):
            _, xs, gs = sequence(layout, pattern, "half", 50 + p_i, STEPS_HOST)
            refs = oracle_steps(xs, gs, 0.5, 1, [False] * STEPS_HOST, summed_mean=True)
            bufs = [HostBufs(x, g) for x, g in zip(xs, gs)]
            for api in ("sync", "alternate", "in-flight"):
                run_api(api, ctx, bufs, layout, 0, refs, ("C1", pattern))
    finally:
        ctx.destroy()


@pytest.mark.gpu
def test_host_step_pageable_buffers_give_the_pinned_bits():
    layout, n_chunks = (13, 64, 196), 8
    c = layout[1]
    ctx = HostCtx(int(np.prod(layout)), c, n_chunks)
    try:
        sparsity, xs, gs = sequence(layout, "dup", "half", 70, 4)
        refs = oracle_steps(xs, gs, sparsity, 1, refresh_for(4), summed_mean=True)
        k = _k(sparsity, c)
        outs = {}
        for pinned in (True, False):
            bufs = [HostBufs(x, g, pinned=pinned) for x, g in zip(xs, gs)]
            run_api("sync", ctx, bufs, layout, k, refs, ("pageable" if not pinned else "pinned",))
            outs[pinned] = [(b.y(), b.gx()) for b in bufs]
        for (y0, g0), (y1, g1) in zip(outs[True], outs[False]):
            assert y0.tobytes() == y1.tobytes() and g0.tobytes() == g1.tobytes()
    finally:
        ctx.destroy()


# ----------------------------------------------------------------------------- the context's life
@pytest.mark.gpu
def test_host_step_grows_its_workspace_with_a_step_in_flight():
    """a second layer whose per-chunk reduction needs a larger workspace, submitted while the first layer's step
    is still in flight on the other slot: the workspace is regrown and both layers match the oracle"""
    small, big, n_chunks = (16, 64, 196), (4096, 1000, 1), 8
    lib = _lib()
    need_small = lib.qsb_reduce_workspace_bytes(small[0] // n_chunks, small[1], small[2])
    need_big = lib.qsb_reduce_workspace_bytes(big[0] // n_chunks, big[1], big[2])
    assert (need_big + 255) // 256 > (need_small + 255) // 256      # the regrow branch runs
    ctx = HostCtx(int(max(np.prod(small), np.prod(big))), 1000, n_chunks)
    try:
        seqs = {}
        for name, layout in (("small", small), ("big", big)):
            sparsity, xs, gs = sequence(layout, "dup", "half", 80 if name == "small" else 90, 4)
            refs = oracle_steps(xs, gs, sparsity, 1, refresh_for(4), summed_mean=True)
            seqs[name] = (layout, _k(sparsity, layout[1]), refs,
                          [HostBufs(x, g) for x, g in zip(xs, gs)], State(layout[1]))
        for t in range(4):
            for slot, name in enumerate(("small", "big")):
                layout, k, refs, bufs, st = seqs[name]
                assert ctx.submit(slot, bufs[t], st, layout, t, k) == 0
            for slot, name in enumerate(("small", "big")):
                layout, k, refs, bufs, st = seqs[name]
                ctx.wait(slot)
                check_step(host_got(st, bufs[t]), refs[t], ("grow", name, t), stats=False)
    finally:
        ctx.destroy()


def _state_from_ref(ref):
    return (torch.from_numpy(ref["imp"].copy()).cuda(), torch.from_numpy(ref["mask"].copy()).cuda(),
            torch.from_numpy(ref["scale"].copy()).cuda())


@pytest.mark.gpu
def test_host_step_runs_after_the_callers_stream():
    """the layer state is overwritten on the caller's stream behind a short device-side delay; the step,
    ordered after that stream, sees the new state"""
    layout, n_chunks = (16, 64, 196), 8
    c = layout[1]
    ctx = HostCtx(int(np.prod(layout)), c, n_chunks)
    try:
        sp_a, xs_a, gs_a = sequence(layout, "rand", "half", 100, 2)
        sp_b, xs_b, gs_b = sequence(layout, "dup", "half", 110, 3)
        refs_b = oracle_steps(xs_b, gs_b, sp_b, 1, refresh_for(3), summed_mean=True)
        st = State(c)
        for t in range(2):                         # the state of another sequence
            assert ctx.submit(0, HostBufs(xs_a[t], gs_a[t]), st, layout, t, _k(sp_a, c), sync=True) == 0
        new = _state_from_ref(refs_b[1])
        bufs = HostBufs(xs_b[2], gs_b[2])
        side = torch.cuda.Stream()
        torch.cuda.synchronize()
        with torch.cuda.stream(side):
            torch.cuda._sleep(20_000_000)          # ~10 ms of spinning: the submit below returns long before
            st.mag.copy_(new[0])
            st.mask.copy_(new[1])
            st.scale.copy_(new[2])
        assert ctx.submit(0, bufs, st, layout, 2, _k(sp_b, c), stream=side.cuda_stream) == 0
        ctx.wait(0)
        torch.cuda.synchronize()
        check_step(host_got(st, bufs), refs_b[2], ("caller stream",), stats=False)
    finally:
        ctx.destroy()


@pytest.mark.gpu
def test_host_ctx_destroy_completes_steps_in_flight():
    layout, n_chunks = (13, 64, 196), 8
    c = layout[1]
    sparsity, xs, gs = sequence(layout, "dead", "half", 120, 2)
    refs = oracle_steps(xs, gs, sparsity, 1, refresh_for(2), summed_mean=True)
    bufs = [HostBufs(x, g) for x, g in zip(xs, gs)]
    st = State(c)
    ctx = HostCtx(int(np.prod(layout)), c, n_chunks)
    try:
        for t in range(2):
            assert ctx.submit(t, bufs[t], st, layout, t, _k(sparsity, c)) == 0
    finally:
        ctx.destroy()
    check_out(bufs[0], refs[0], ("destroy", 0))
    check_step(host_got(st, bufs[1]), refs[1], ("destroy", 1), stats=False)


# ----------------------------------------------------------------------------- parity with the resident step
@pytest.mark.gpu
@pytest.mark.parametrize("layout", [(32, 64, 3136), (16, 2049, 49)], ids=["C64", "C2049"])
def test_host_step_matches_resident_step_on_gaussian_data(layout):
    """Gaussian data (sums not exact): mask, scale, decimal, y and gx equal the resident route's.  The host step
    sums fp64 chunk rows and the resident step its own partials, so a step's mean may round 1 ulp apart, and the
    running average carries that on: at most t + 1 ulp at step t."""
    from qsparse_b200 import ops
    o, c, i = layout
    rng = np.random.default_rng(130)
    xs = [rng.standard_normal(layout).astype(np.float32) * (1 + np.arange(c, dtype=np.float32) % 7).reshape(1, c, 1)
          for _ in range(4)]
    gs = [make_g(layout, 130 + t) for t in range(4)]
    k = _k(0.5, c)
    ctx = HostCtx(o * c * i, c, 8)
    st_h, st_r = State(c), State(c)
    try:
        for t in range(4):
            bufs = HostBufs(xs[t], gs[t])
            assert ctx.submit(0, bufs, st_h, layout, t, k, sync=True) == 0
            xd, gd = torch.from_numpy(xs[t]).cuda(), torch.from_numpy(gs[t]).cuda()
            ops.structured_prune_quant_step(xd, layout, st_r.mag, st_r.mask, st_r.scale, st_r.dec, float(o * i), t,
                                            1, t > 0, k, BITS, t, True)
            y = ops.fq_pow2_fwd(xd, st_r.dec, layout, mask=st_r.mask)
            _, gx = ops.ste_bwd(gd.clone(), st_r.dec, True, BITS, 0, layout, mask=st_r.mask, want_gx=True)
            what = (layout, t)
            assert torch.equal(st_h.mask, st_r.mask), what
            assert torch.equal(st_h.dec, st_r.dec), what
            assert torch.equal(st_h.scale, st_r.scale), what
            # one rounding of the step's mean apart per step, carried on by the running average
            assert ulp_diff(st_h.mag.cpu().numpy(), st_r.mag.cpu().numpy()).max() <= t + 1, what
            assert bufs.y().tobytes() == y.cpu().numpy().tobytes(), ("y",) + what
            assert bufs.gx().tobytes() == gx.cpu().numpy().tobytes(), ("gx",) + what
    finally:
        ctx.destroy()


# ----------------------------------------------------------------------------- arguments refused before any work
def recorded_work(fn):
    """copies and qsb:: kernels that ``fn`` puts on the device (torch.profiler, CUDA activity)"""
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        out = fn()
        torch.cuda.synchronize()
    work = [e.name for e in prof.events()
            if e.device_type == torch.autograd.DeviceType.CUDA and ("qsb::" in e.name or "emcpy" in e.name)]
    return out, work


BAD_ARGS = [
    # (id, what to change, expected code)
    ("null-ctx", dict(ctx=None), BADARG),
    ("slot-1", dict(slot=-1), BADARG),
    ("slot2", dict(slot=2), BADARG),
    ("null-x", dict(host=0), BADARG),
    ("null-gx", dict(host=3), BADARG),
    ("zero-outer", dict(layout=(0, 64, 196)), BADARG),
    ("zero-channels", dict(layout=(16, 0, 196)), BADARG),
    ("zero-inner", dict(layout=(16, 64, 0)), BADARG),
    ("channels>max", dict(layout=(1, 128, 98)), BADARG),
    ("elems>max", dict(layout=(17, 64, 196)), BADARG),
    ("k=C", dict(k=64), BADARG),
    ("k=-1", dict(k=-1), BADARG),
    ("C4097", dict(layout=(2, 4097, 1), wide=True), UNSUPPORTED),
    ("null-mask", dict(state=1), BADARG),
    ("null-scale", dict(state=2), BADARG),
    ("null-magnitude", dict(state=0), BADARG),
    ("null-decimal", dict(state=3), BADARG),
]


@pytest.mark.gpu
@pytest.mark.parametrize("case", BAD_ARGS, ids=[b[0] for b in BAD_ARGS])
def test_host_step_refuses_bad_arguments_before_any_work(case):
    """the code comes back before any copy or launch: the layer state and the host outputs stay as they were, and
    the call records no memcpy and no qsb:: kernel (a copy left running after an error return races the caller
    freeing or refilling its buffers)"""
    from qsparse_b200 import _native as N
    cid, change, code = case
    layout = (16, 64, 196)
    wide = change.get("wide", False)
    ctx = HostCtx(int(np.prod(layout)) if not wide else 2 * 8192, 64 if not wide else 8192, 8)
    bad_layout = change.get("layout", layout)
    c = max(bad_layout[1], 1)
    try:
        xb = make_x((16, 64, 196) if not wide else (2, 4097, 1), "rand", 140, 0.5)
        bufs = HostBufs(xb, make_g(xb.shape, 140))
        st = State(c)
        st.mag.copy_(torch.arange(c, device="cuda", dtype=torch.float32))
        st.mask.copy_(torch.arange(c, device="cuda") % 3 == 0)
        st.scale.fill_(5.0)
        st.dec.fill_(-3.0)
        before = [v.clone() for v in (st.mag, st.mask, st.scale, st.dec)]
        ptrs = bufs.ptrs()
        if "host" in change:
            ptrs[change["host"]] = None
        state = [N.ptr(st.mag), N.ptr(st.mask), N.ptr(st.scale), N.ptr(st.dec)]
        if "state" in change:
            state[change["state"]] = None
        k = change.get("k", _k(0.5, c))
        if "ctx" in change:
            ctx_saved, ctx.ctx = ctx.ctx, c_void_p()
        try:
            rc, work = recorded_work(lambda: ctx.submit(change.get("slot", 0), None, st, bad_layout, 1, k,
                                                        ptrs=ptrs, state=state))
        finally:
            if "ctx" in change:
                ctx.ctx = ctx_saved
        assert rc == code, (cid, rc)
        for a, b in zip(before, (st.mag, st.mask, st.scale, st.dec)):
            assert torch.equal(a, b), cid
        assert unwritten(bufs.y()) == xb.size and unwritten(bufs.gx()) == xb.size, cid
        assert work == [], (cid, work)
        ctx.wait(0)
        ctx.wait(1)
    finally:
        ctx.destroy()


@pytest.mark.gpu
def test_host_step_takes_any_rank_without_a_refresh():
    """at t_prune = 0 the mask is not refreshed, so k = C is accepted (as on the resident routes)"""
    layout = (16, 64, 196)
    c = layout[1]
    sparsity, xs, gs = sequence(layout, "rand", "half", 150, 1)
    refs = oracle_steps(xs, gs, sparsity, 1, [False], summed_mean=True)
    ctx = HostCtx(int(np.prod(layout)), c, 8)
    try:
        st = State(c)
        bufs = HostBufs(xs[0], gs[0])
        rc, work = recorded_work(lambda: ctx.submit(0, bufs, st, layout, 0, c, sync=True))
        assert rc == 0
        # what the refusals above must not record: a step's copies and kernels
        assert any("emcpy" in w for w in work) and any("qsb::" in w for w in work), work
        check_step(host_got(st, bufs), refs[0], ("k=C at t=0",), stats=False)
    finally:
        ctx.destroy()


def test_host_api_null_context_without_gpu():
    """argument errors of the host entry points need no GPU"""
    lib = _lib()
    assert lib.qsb_host_ctx_wait(None, 0) == BADARG
    assert lib.qsb_host_ctx_destroy(None) == 0
    one = ctypes.c_float(0.0)
    p = ctypes.addressof(one)
    assert lib.qsb_host_prune_quant_step_submit(None, 0, p, p, p, p, p, p, p, p, 1, 1, 1, 0, 0, BITS, 0, None, 1,
                                                None) == BADARG
    assert lib.qsb_host_prune_quant_step(None, p, p, p, p, p, p, p, p, 1, 1, 1, 0, 0, BITS, 0, None, 1,
                                         None) == BADARG


# ----------------------------------------------------------------------------- several statistics rows
def row_stride(c, padded):
    """bytes a row [C doubles | C floats] takes, or that rounded up to 256 bytes plus 256 more"""
    return ((c * 12 + 255) // 256) * 256 + 256 if padded else c * 12


def stat_rows(x, c, stride):
    """one statistics row per outer row of x [n_rows, C, inner]: sum|x| (fp64, exact for these inputs) and max|x|"""
    n = x.shape[0]
    buf = np.zeros(n * stride, np.uint8)
    for r in range(n):
        row = buf[r * stride:(r + 1) * stride]
        with np.errstate(invalid="ignore"):
            row[:c * 8].view(np.float64)[:] = np.abs(x[r].astype(np.float64)).sum(axis=1)
        row[c * 8:c * 12].view(np.float32)[:] = orc.absmax(x[r:r + 1], 1)
    dev = torch.from_numpy(buf).cuda()
    return {"abssum": dev[:c * 8].view(torch.float64), "absmax": dev[c * 8:c * 12].view(torch.float32)}


def rows_x(n_rows, c, inner, t, seed, special):
    """exactly summable x [n_rows, C, inner]; ``special``: at t >= 1 an inf in row 0's channels 0 and C - 1 and a NaN
    in the last row's channel 0 (one row's sum holds an inf, a later row's absmax a NaN in the same channel)"""
    x = make_x((n_rows, c, inner), "dup" if t % 2 else "rand", seed + t, 0.5)
    if special and t >= 1:
        x[0, 0, 0] = np.inf
        x[0, c - 1, inner - 1] = np.inf
        x[-1, 0, 0] = np.nan
    return x


ROWS_STEPS = 3
# (n_rows, C, inner, padded stride, NaN / inf rows); kernel route: C <= 4096
ROWS_CASES = [(n, c, 4 if n < 4096 else 1, True, n >= 2) for n in (1, 2, 7, 4096) for c in (2, 1024, 2049, 4096)
              if (n, c) != (4096, 4096)]
ROWS_CASES += [(7, 1024, 3, False, True), (2, 2, 5, False, False)]       # rows packed back to back
# the composed route (C > 4096) loops over the rows on the host: a few rows
ROWS_CASES += [(n, c, 2, True, n >= 2) for n in (1, 2, 7) for c in (4097, 6000)]


# prune_quant_rows_step_params is the one-CTA kernel only (C <= 4096)
ROWS_RUNS = [(case, entry) for case in ROWS_CASES for entry in ("params", "rows_step")
             if entry == "params" or case[1] <= 4096]


@pytest.mark.gpu
@pytest.mark.parametrize("case,entry", ROWS_RUNS,
                         ids=[f"rows{n}-C{c}-{'pad' if p else 'tight'}{'-naninf' if s else ''}-{e}"
                              for (n, c, _, p, s), e in ROWS_RUNS])
def test_step_on_statistics_rows_matches_oracle(case, entry):
    """ops.prune_quant_params(n_rows, row_stride_bytes) and ops.prune_quant_rows_step_params on one statistics row
    per outer row: the rows combine into the oracle's step on the whole tensor (fp64 sums, NaN-propagating maxima)"""
    from qsparse_b200 import ops
    n_rows, c, inner, padded, special = case
    xs = [rows_x(n_rows, c, inner, t, 160 + n_rows, special) for t in range(ROWS_STEPS)]
    refs = oracle_steps(xs, [np.zeros_like(x) for x in xs], 0.5, 1, refresh_for(ROWS_STEPS), summed_mean=True)
    stride = row_stride(c, padded)
    k = _k(0.5, c)
    st = State(c)
    fn = ops.prune_quant_params if entry == "params" else ops.prune_quant_rows_step_params
    for t in range(ROWS_STEPS):
        stats = stat_rows(xs[t], c, stride)
        fn(st.mag, st.mask, st.scale, st.dec, stats, float(n_rows * inner), t, 1, t > 0, k, BITS, t, True,
           n_rows=n_rows, row_stride_bytes=stride)
        h = lambda v: v.cpu().numpy()
        what = (case, entry, t)
        assert np.array_equal(h(st.mask), refs[t]["mask"]), ("mask",) + what
        assert bits_equal(h(st.mag), refs[t]["imp"]), ("magnitude",) + what
        assert bits_equal(h(st.scale), refs[t]["scale"]), ("scale",) + what
        assert bits_equal(h(st.dec), refs[t]["dec"]), ("decimal",) + what
    if special:
        assert np.isnan(refs[-1]["imp"][0]) and np.isnan(refs[-1]["scale"]).all()


@pytest.mark.gpu
@pytest.mark.parametrize("c,entry", [(64, "params"), (64, "rows_step"), (4096, "params"), (4096, "rows_step"),
                                     (4097, "params")])
@pytest.mark.parametrize("n_rows", [0, 4097])
def test_step_refuses_a_bad_row_count_without_writing(n_rows, c, entry):
    """at most 4096 rows, at least one, on the kernel and on the composed route alike; nothing is written"""
    from qsparse_b200 import ops
    stride = row_stride(c, True)
    stats = stat_rows(make_x((1, c, 1), "rand", 170, 0.5), c, stride)
    st = State(c)
    st.mag.copy_(torch.arange(c, device="cuda", dtype=torch.float32))
    st.mask.copy_(torch.arange(c, device="cuda") % 3 == 0)
    st.scale.fill_(5.0)
    st.dec.fill_(-3.0)
    before = [v.clone() for v in (st.mag, st.mask, st.scale, st.dec)]
    fn = ops.prune_quant_params if entry == "params" else ops.prune_quant_rows_step_params
    with pytest.raises(RuntimeError, match="bad argument"):
        fn(st.mag, st.mask, st.scale, st.dec, stats, 4.0, 1, 1, True, _k(0.5, c), BITS, 1, True, n_rows=n_rows,
           row_stride_bytes=stride)
    torch.cuda.synchronize()
    for a, b in zip(before, (st.mag, st.mask, st.scale, st.dec)):
        assert torch.equal(a, b)
