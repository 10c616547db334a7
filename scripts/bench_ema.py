"""Cost of the weight EMA (algorithm.ema_decay) on one GPU.

  * the optimiser kernels at the flow_diffuser parameter count (target=flow UNet, flat buffers with FusedAdam's padding):
    fd_adam_step (28 B per parameter: read p, g, m, v; write p, m, v) against fd_adam_ema_step (36 B: + read and write
    the EMA), us per call and GB/s over those bytes, CUDA events around `--launches` back-to-back launches.  One call's
    working set (>= 5 x 143 MB) exceeds the 126 MB L2, so every call streams from HBM;
  * the training step at 368x768, batch 8 (preprocess with GPU augmentation -> loss -> backward -> clip 100 + Adam), with
    EMA off and with EMA on at ema_update_every=1 and ema_update_after_step=0 (every step is an update step: the worst case).
Both comparisons alternate the two configurations in the same process, `--rounds` times, and report each round.  The
card's name and power limit are read in the same run and written beside the numbers, into ONE JSON file under --out.

    python scripts/bench_ema.py --out DIR [--rounds 3] [--steps 20] [--launches 200]
"""
import argparse
import json
import os
import statistics
import sys

import torch

sys.dont_write_bytecode = True
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from bench_samplers import PEAK_HBM_BYTES_S, card_info  # noqa: E402  (same directory)

TRAIN_H, TRAIN_W = 368, 768


def kernel_rounds(n, rounds, launches):
    from opticalflowdiffusion_b200 import _lib
    lib = _lib.load(check_device=True)
    p, m, ema = torch.randn(n, device="cuda"), torch.zeros(n, device="cuda"), torch.randn(n, device="cuda")
    g, v = torch.randn(n, device="cuda"), torch.zeros(n, device="cuda")
    sumsq = torch.zeros(1, device="cuda")
    _lib.check(lib.fd_sumsq(_lib.ptr(g), n, _lib.ptr(sumsq), _lib.stream()))
    st = _lib.stream()

    def adam(k):
        _lib.check(lib.fd_adam_step(_lib.ptr(p), _lib.ptr(g), _lib.ptr(m), _lib.ptr(v), n, 1e-5, 0.9, 0.999, 1e-8, 1e-6,
                                    k + 1, _lib.ptr(sumsq), 100.0, 1.0, st))

    def adam_ema(k):
        _lib.check(lib.fd_adam_ema_step(_lib.ptr(p), _lib.ptr(g), _lib.ptr(m), _lib.ptr(v), _lib.ptr(ema), n, 1e-5, 0.9,
                                        0.999, 1e-8, 1e-6, k + 1, _lib.ptr(sumsq), 100.0, 1.0, 1e-4, st))

    def timed(fn):
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        for k in range(launches):
            fn(k)
        e.record()
        torch.cuda.synchronize()
        return s.elapsed_time(e) * 1e-3 / launches

    for k in range(20):
        adam(k)
        adam_ema(k)
    out = {"fd_adam_step": {"bytes_per_call": 28 * n, "us_per_call": []},
           "fd_adam_ema_step": {"bytes_per_call": 36 * n, "us_per_call": []}}
    for _ in range(rounds):
        for name, fn in (("fd_adam_step", adam), ("fd_adam_ema_step", adam_ema)):
            out[name]["us_per_call"].append(timed(fn) * 1e6)
    for row in out.values():
        us = statistics.median(row["us_per_call"])
        row["us_median"] = us
        row["GB_per_s"] = row["bytes_per_call"] / (us * 1e-6) / 1e9
        row["fraction_of_7.7TB_s"] = row["bytes_per_call"] / (us * 1e-6) / PEAK_HBM_BYTES_S
    out["ema_extra_us"] = out["fd_adam_ema_step"]["us_median"] - out["fd_adam_step"]["us_median"]
    return out


def build(ema: bool, batch: int):
    from opticalflowdiffusion_b200 import FlowDiffuser
    from opticalflowdiffusion_b200.config import compose
    from opticalflowdiffusion_b200.datasets import synthetic_frames
    over = ["algorithm.target=flow"]
    if ema:
        over += ["algorithm.ema_decay=0.9999", "algorithm.ema_update_after_step=0", "algorithm.ema_update_every=1"]
    torch.manual_seed(0)
    algo = FlowDiffuser(compose(over).algorithm).cuda()
    algo.train()
    opt = algo.configure_optimizers()
    opt.max_grad_norm = 100.0
    g = torch.Generator().manual_seed(7)
    batch_dev = (synthetic_frames(batch, TRAIN_H, TRAIN_W, seed=200).cuda(),
                 synthetic_frames(batch, TRAIN_H, TRAIN_W, seed=300).cuda(),
                 (torch.randn(batch, 2, TRAIN_H, TRAIN_W, generator=g) * 5.0).cuda())

    def step():
        first, cond, _ = algo.preprocess(batch_dev, aug=True)
        loss = algo.loss(first, cond, None)
        loss.backward()
        opt.step()
        opt.zero_grad(set_to_none=True)

    return algo, opt, step


def train_rounds(batch, rounds, steps):
    from opticalflowdiffusion_b200 import _lib
    lib = _lib.load()
    runs = {name: build(name == "ema_every_step", batch) for name in ("ema_off", "ema_every_step")}
    for _, _, step in runs.values():
        for _ in range(3):
            step()
    torch.cuda.synchronize()
    out = {name: {"ms_per_step": [], "launches_per_step": None, "ema_updates": 0} for name in runs}
    for _ in range(rounds):
        for name, (algo, opt, step) in runs.items():
            s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            n0, upd = lib.fd_launch_count(), 0
            s.record()
            for _ in range(steps):
                step()
                upd += int(opt.ema_updated)
            e.record()
            torch.cuda.synchronize()
            out[name]["ms_per_step"].append(s.elapsed_time(e) / steps)
            out[name]["launches_per_step"] = (lib.fd_launch_count() - n0) / steps
            out[name]["ema_updates"] += upd
    for row in out.values():
        row["ms_median"] = statistics.median(row["ms_per_step"])
    out["ema_extra_ms"] = out["ema_every_step"]["ms_median"] - out["ema_off"]["ms_median"]
    out["peak_mem_gib"] = torch.cuda.max_memory_allocated() / 2 ** 30
    return out


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--out", required=True, help="directory for the JSON result")
    ap.add_argument("--batch", type=int, default=8)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--steps", type=int, default=20, help="timed training steps per configuration and round")
    ap.add_argument("--launches", type=int, default=200, help="timed kernel launches per kernel and round")
    args = ap.parse_args()
    from opticalflowdiffusion_b200 import _lib
    from opticalflowdiffusion_b200.unet import Unet
    _lib.load(check_device=True)          # no GPU -> error: nothing here falls back to the CPU
    n = sum((p.numel() + 3) // 4 * 4 for p in Unet(64, channels=5, out_dim=2).parameters())
    res = {"card": card_info(), "parameters_padded": n}
    res["kernels"] = kernel_rounds(n, args.rounds, args.launches)
    print(json.dumps(res["kernels"]), flush=True)
    res["train_step"] = dict(train_rounds(args.batch, args.rounds, args.steps), shape=[args.batch, TRAIN_H, TRAIN_W],
                             config="target=flow, GPU augmentation on, clip 100, Adam lr 1e-5 wd 1e-6; "
                                    "ema_every_step: ema_decay 0.9999, ema_update_after_step 0, ema_update_every 1")
    print(json.dumps(res["train_step"]), flush=True)
    res["card_after"] = card_info()
    os.makedirs(args.out, exist_ok=True)
    path = os.path.join(args.out, "bench_ema.json")
    with open(path, "w") as f:
        json.dump(res, f, indent=1)
    print("wrote", path)


if __name__ == "__main__":
    main()
