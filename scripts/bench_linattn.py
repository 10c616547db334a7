"""Times fd_linattn_tc (tcgen05 LinearAttention, csrc/fd_linattn_tc.cu) per launch at the UNet's shapes: CUDA events around the
three launches separately is not possible through the C ABI, so the whole block is timed and FD_LA_DBG (diagnostic switches,
see CtxParams::dbg) isolates the parts.  FD_LA_DBG only acts in a diagnostic build of the library:
FD_DIAG=1 python -m opticalflowdiffusion_b200.build --force."""
import json
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from opticalflowdiffusion_b200 import _lib  # noqa: E402

BF = torch.bfloat16


def main():
    lib = _lib.load(check_device=True)
    P = _lib.ptr
    res = {}
    for name, N, HW, C in (("full 64", 8, 440 * 1024, 64), ("half 64", 8, 220 * 512, 64), ("half 128", 8, 220 * 512, 128),
                           ("quarter 128", 8, 110 * 256, 128)):
        g = torch.Generator(device="cuda").manual_seed(1)
        x = torch.randn(N, HW, C, device="cuda", generator=g).to(BF)
        wqkv = torch.randn(384, C, device="cuda", generator=g) / C ** 0.5
        g1 = torch.ones(C, device="cuda")
        wout = torch.randn(C, 128, device="cuda", generator=g) / 128 ** 0.5
        bout, g2 = torch.zeros(C, device="cuda"), torch.ones(C, device="cuda")
        wq, wk = torch.empty(128, C, device="cuda", dtype=BF), torch.empty(128, C, device="cuda", dtype=BF)
        sq, sk, mk = (torch.empty(128, device="cuda") for _ in range(3))
        wv = torch.empty(128, C, device="cuda")
        _lib.check(lib.fd_linattn_tc_prep(P(wqkv), P(g1), P(wq), P(sq), P(wk), P(sk), P(mk), P(wv), C, _lib.stream()))
        out = torch.empty_like(x)
        ws = torch.empty(lib.fd_linattn_tc_workspace_floats(N, HW, C), device="cuda")

        def fn():
            _lib.check(lib.fd_linattn_tc(P(x), P(wk), P(sk), P(mk), P(wq), P(sq), P(wv), P(wout), P(bout), P(g2), P(out), P(ws), N, HW,
                                         C, 1e-5, _lib.stream()))
        for _ in range(3):
            fn()
        torch.cuda.synchronize()
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        iters = 10
        s.record()
        for _ in range(iters):
            fn()
        e.record()
        torch.cuda.synchronize()
        t = s.elapsed_time(e) / iters
        res[name] = {"us": round(t * 1e3, 1), "GBps_algorithmic": round(3 * x.numel() * 2 / t / 1e6, 1)}
    print(os.environ.get("FD_LA_DBG", "0"), json.dumps(res))


if __name__ == "__main__":
    main()
