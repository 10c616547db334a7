"""CUDA-event timing of fd_conv_wgrad on the training shapes (batch 8, 368x768 crops)."""
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from opticalflowdiffusion_b200 import _lib  # noqa: E402

lib = _lib.load(check_device=True)
B = 8
SHAPES = [  # C0, C1, Cout, H, W, k
    (64, 0, 64, 368, 768, 3), (64, 64, 64, 368, 768, 3), (128, 0, 64, 368, 768, 3), (64, 0, 64, 184, 384, 3),
    (128, 0, 128, 184, 384, 3), (128, 64, 128, 184, 384, 3), (256, 0, 256, 92, 192, 3), (256, 128, 256, 92, 192, 3),
    (512, 0, 512, 46, 96, 3), (512, 256, 512, 46, 96, 3), (64, 0, 384, 368, 768, 1), (128, 0, 64, 368, 768, 1),
]
for c0, c1, cout, h, w, k in SHAPES:
    s0 = torch.randn(B, h, w, c0, device="cuda").bfloat16()
    s1 = torch.randn(B, h, w, c1, device="cuda").bfloat16() if c1 else None
    dy = torch.randn(B, h, w, cout, device="cuda").bfloat16()
    dw = torch.zeros(cout, k * k * (c0 + c1), device="cuda")

    def run():
        _lib.check(lib.fd_conv_wgrad(_lib.ptr(s0), c0, _lib.ptr(s1), c1, _lib.ptr(dy), _lib.ptr(dw), B, h, w, cout, k, k, k // 2,
                                     k // 2, 0, _lib.stream()))
    for _ in range(3):
        run()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    torch.cuda.synchronize()
    ev[0].record()
    for _ in range(10):
        run()
    ev[1].record()
    torch.cuda.synchronize()
    ms = ev[0].elapsed_time(ev[1]) / 10
    fl = 2.0 * B * h * w * cout * k * k * (c0 + c1)
    print(f"wgrad {c0}+{c1}->{cout} {h}x{w} k{k}: {ms * 1e3:8.1f} us  {fl / ms / 1e9:7.1f} TFLOP/s")
