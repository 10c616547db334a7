"""One launch of each config-#4 kernel after a warm-up (for `ncu -k regex:...`): same tensors as scripts/bench_warp.py."""
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from opticalflowdiffusion_b200 import _lib  # noqa: E402

lib = _lib.load(check_device=True)
B, C, H, W = 8, 3, 436, 1024
g = torch.Generator().manual_seed(3)
flow = (torch.randn(B, 2, H, W, generator=g) * 4).cuda()
f1 = torch.rand(B, C, H, W, generator=g).cuda()
f2 = torch.rand(B, C, H, W, generator=g).cuda()
gt = flow + torch.randn(B, 2, H, W, generator=g).cuda()
sums = torch.empty(4, device="cuda")
ws = torch.empty(lib.fd_photo_epe_workspace_floats(B, H, W), device="cuda")
wsb = torch.empty(lib.fd_warp_bwd_workspace_floats(B, C, H, W), device="cuda")
wss = torch.empty(lib.fd_splat_fwd_workspace_floats(B, C, H, W, 1), device="cuda")
gflow, gf2, out, mask = torch.empty_like(flow), torch.empty_like(f2), torch.empty_like(f2), torch.empty_like(f2)
flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
st, P = _lib.stream(), _lib.ptr
for _ in range(int(os.environ.get("REPS", 3))):
    flush.zero_()
    _lib.check(lib.fd_backwarp_photo_epe_fwd(P(f1), P(f2), P(flow), P(gt), P(sums), P(ws), B, C, H, W, st))
    flush.zero_()
    _lib.check(lib.fd_backwarp_photo_epe_bwd(P(f1), P(f2), P(flow), P(gt), P(sums), 1.0, 1.0, P(gflow), P(gf2), P(wsb), B, C, H, W, st))
    flush.zero_()
    _lib.check(lib.fd_backwarp_fwd(P(f2), P(flow), P(out), P(mask), B, C, H, W, st))
    flush.zero_()
    _lib.check(lib.fd_splat_fwd(P(f2), P(flow), P(out), P(wss), B, C, H, W, 1, 0, 0, st))
torch.cuda.synchronize()
print("ok")
