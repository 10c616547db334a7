"""Times the mid-block attention core (fd_attention, the tcgen05 kernel of csrc/fd_attention_tc.cu) at the UNet's token counts: 55x128 (436x1024 frames), 46x96 (368x768 crops), 128x256 (1024x2048 frames)."""
import json
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from opticalflowdiffusion_b200 import _lib  # noqa: E402


def main():
    lib = _lib.load(check_device=True)
    P = _lib.ptr
    res = {}
    for name, N, HW in (("b8 7040", 8, 7040), ("b8 4416", 8, 4416), ("b2 32768", 2, 32768)):
        g = torch.Generator(device="cuda").manual_seed(1)
        qkv = (torch.randn(N, HW, 384, device="cuda", generator=g) * 1.5).to(torch.bfloat16)
        out = torch.empty(N, HW, 128, device="cuda", dtype=torch.bfloat16)

        def fn():
            _lib.check(lib.fd_attention(P(qkv), P(out), N, HW, _lib.stream()))
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
        t = s.elapsed_time(e) / iters * 1e-3
        flops = 4.0 * N * 4 * HW * HW * 32           # QK^T and PV
        res[name] = {"us": round(t * 1e6, 1), "TFLOPs": round(flops / t / 1e12, 1), "Gexp_per_s": round(N * 4 * HW * HW / t / 1e9, 1)}
    print(json.dumps(res))


if __name__ == "__main__":
    main()
