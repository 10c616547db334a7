"""BASELINE config #4 microbench: fused backward-warp + photometric/EPE fwd and bwd at 8x2x436x1024,
plus the plain warp / splat kernels.  Prints achieved GB/s against the algorithmic bytes
(SURVEY.md section 8d: fwd 40 B/px, bwd 60 B/px)."""
import json
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from opticalflowdiffusion_b200 import _lib  # noqa: E402


def _timeit(fn, iters=50, warmup=10, flush=None, clean=None):
    """Median device time of fn() between two CUDA events on the launching stream.  flush: a buffer larger than L2 that is
    WRITTEN before every launch (cold inputs; L2 is left full of dirty lines whose write-back then competes with the kernel for
    DRAM).  clean: a second buffer that is READ after the write, so that the kernel starts with cold inputs and an L2 of clean
    lines (nothing to write back).  All iterations are enqueued before the one synchronisation at the end: the 70 us flush in
    front of every timed launch keeps the stream busy, so the events bracket the kernels' execution (what ncu's
    gpu__time_duration reports, profiles/r2_warp_launch_table.txt) and not the host's launch latency -- with a
    synchronisation per iteration every number carried ~6 us of it (backwarp_fwd: 41.0 us against 35.1 us under ncu)."""
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    evs = []
    for _ in range(iters):
        if flush is not None:
            flush.zero_()
        if clean is not None:
            clean.sum(dtype=torch.int64)
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        fn()
        e.record()
        evs.append((s, e))
    torch.cuda.synchronize()
    ts = sorted(s.elapsed_time(e) * 1e-3 for s, e in evs)
    return ts[len(ts) // 2]


def measure(iters=50, warmup=10):
    lib = _lib.load(check_device=True)
    B, C, H, W = 8, 3, 436, 1024
    g = torch.Generator().manual_seed(3)
    flow = (torch.randn(B, 2, H, W, generator=g) * 4).cuda()
    f1 = torch.rand(B, C, H, W, generator=g).cuda()
    f2 = torch.rand(B, C, H, W, generator=g).cuda()
    gt = flow + torch.randn(B, 2, H, W, generator=g).cuda()
    sums = torch.empty(4, device="cuda")
    ws = torch.empty(lib.fd_photo_epe_workspace_floats(B, H, W), device="cuda")
    gflow = torch.empty_like(flow)
    gf2 = torch.empty_like(f2)
    out = torch.empty_like(f2)
    mask = torch.empty_like(f2)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    st = _lib.stream()
    P = _lib.ptr
    px = B * H * W
    res = {}

    clean = torch.zeros(256 << 20, dtype=torch.uint8, device="cuda")
    legs = []

    def rec(name, t, nbytes):
        res[name] = {"us": round(t * 1e6, 2), "GBps": round(nbytes / t / 1e9, 1), "bytes": nbytes}

    def timeit(fn, **kw):          # noqa: F811  (records the call so that the clean-L2 pass below can repeat it)
        legs.append(fn)
        return _timeit(fn, **kw)

    t = timeit(lambda: _lib.check(lib.fd_backwarp_photo_epe_fwd(P(f1), P(f2), P(flow), P(gt), P(sums), P(ws), B, C, H, W, st)), flush=flush, iters=iters, warmup=warmup)
    rec("photo_epe_fwd", t, 40 * px)
    wsb = torch.empty(lib.fd_warp_bwd_workspace_floats(B, C, H, W), device="cuda")
    t = timeit(lambda: _lib.check(lib.fd_backwarp_photo_epe_bwd(P(f1), P(f2), P(flow), P(gt), P(sums), 1.0, 1.0, P(gflow), P(gf2), P(wsb), B, C, H, W, st)), flush=flush, iters=iters, warmup=warmup)
    rec("photo_epe_bwd", t, 60 * px)
    t = timeit(lambda: _lib.check(lib.fd_backwarp_fwd(P(f2), P(flow), P(out), P(mask), B, C, H, W, st)), flush=flush, iters=iters, warmup=warmup)
    rec("backwarp_fwd", t, (8 + 12 + 12 + 12) * px)
    t = timeit(lambda: _lib.check(lib.fd_backwarp_bwd(P(f2), P(flow), P(out), P(gf2), P(gflow), P(wsb), B, C, H, W, st)), flush=flush, iters=iters, warmup=warmup)
    rec("backwarp_bwd", t, (8 + 12 + 12 + 12 + 8) * px)
    # the flow gradient alone (frames without gradient, as in a training step that learns only the flow): no scatter
    t = timeit(lambda: _lib.check(lib.fd_backwarp_photo_epe_bwd(P(f1), P(f2), P(flow), P(gt), P(sums), 1.0, 1.0, P(gflow), None, None, B, C, H, W, st)), flush=flush, iters=iters, warmup=warmup)
    rec("photo_epe_bwd_flow_only", t, 48 * px)
    t = timeit(lambda: _lib.check(lib.fd_backwarp_bwd(P(f2), P(flow), P(out), None, P(gflow), None, B, C, H, W, st)), flush=flush, iters=iters, warmup=warmup)
    rec("backwarp_bwd_flow_only", t, (8 + 12 + 12 + 8) * px)
    so = torch.empty_like(f2)
    wss = torch.empty(lib.fd_splat_fwd_workspace_floats(B, C, H, W, 1), device="cuda")
    t = timeit(lambda: _lib.check(lib.fd_splat_fwd(P(f2), P(flow), P(so), P(wss), B, C, H, W, 1, 0, 0, st)), flush=flush, iters=iters, warmup=warmup)
    rec("splat_fwd", t, (8 + 12 + 12) * px)
    t = timeit(lambda: _lib.check(lib.fd_splat_flowgrad(P(f2), P(flow), P(out), P(gflow), B, C, H, W, 1, 0, 0, st)), flush=flush, iters=iters, warmup=warmup)
    rec("splat_flowgrad", t, (8 + 12 + 12 + 8) * px)
    # warp_forward_flow on a three-channel image (what UnetWithWarp / the pyramid loss call): generic prepare / splat / finish
    # vs the fused two-launch path; bytes: image 12 + flow 8 + output 12 per pixel
    ten_in = torch.empty(B, 4, H, W, device="cuda")
    ret = torch.empty(B, 4, H, W, device="cuda")
    acc = torch.empty(B, H, W, 4, device="cuda")

    def generic():
        _lib.check(lib.fd_splat_prepare(P(f2), P(ten_in), B, C, H * W, st))
        _lib.check(lib.fd_splat_fwd(P(ten_in), P(flow), P(ret), P(acc), B, C + 1, H, W, 1, 0, 0, st))
        _lib.check(lib.fd_splat_finish(P(ret), P(so), B, C, H * W, 1, st))
    t = timeit(generic, flush=flush, iters=iters, warmup=warmup)
    rec("forward_warp_sum_generic", t, (12 + 8 + 12) * px)
    t = timeit(lambda: _lib.check(lib.fd_forward_warp_sum3(P(f2), P(flow), None, P(acc), P(so), None, B, H, W, 1, 0, 0, 1, st)),
               flush=flush, iters=iters, warmup=warmup)
    rec("forward_warp_sum_fused", t, (12 + 8 + 12) * px)
    # CLEAN_L2=1: the same launches with a clean L2 (see _timeit).  Measured: within 5 % of the dirty-L2 numbers
    # (photo_epe_fwd 72.7 vs 76.8 us), i.e. the write-back of the flush buffer is not what bounds these kernels.
    for name, fn in zip(list(res), legs if os.environ.get("CLEAN_L2") else []):
        t = _timeit(fn, flush=flush, clean=clean, iters=iters, warmup=2)
        res[name]["us_clean_l2"] = round(t * 1e6, 2)
        res[name]["GBps_clean_l2"] = round(res[name]["bytes"] / t / 1e9, 1)
    return res


if __name__ == "__main__":
    print(json.dumps(measure()))
