"""Sampler speed and accuracy on one GPU: DDIM-50 against multistep DPM-Solver++ (2M / 3M) at several step counts.

At 436x1024, batch 8, target=flow, every loop captured as a CUDA graph (use_cuda_graph=True) and replayed:
  * flows/s of each sampler: batch * reps / wall time of `reps` replays ending in a device synchronise;
  * mean end-point error in px (x flow_max) of each sampler's final flow against a 3M-200 run from the same x_T and cond;
  * the fused step kernel (fd_dpmpp_step, order 3, in place as in the loop: x_next == x, d_out == d_hist2) in us per call and
    GB/s over its 24 B per element, against the 7.7 TB/s HBM3e figure of the B200 data sheet; four input sets are cycled
    (0.57 GB) so that the 126 MB L2 does not hold the working set between calls.
The card's name and power limit are read in the same run and written beside the numbers, into ONE JSON file under --out.

Without --ckpt the UNet is randomly initialised: the end-point errors then show how fast the solvers converge on this
network, not the flow quality on trained data.  --ckpt PATH loads a FlowDiffuser state dict (or a Lightning checkpoint's
"state_dict") and measures the same on real weights.

    python scripts/bench_samplers.py --out DIR [--ckpt PATH] [--batch 8] [--reps 3]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import torch

sys.dont_write_bytecode = True
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

FLOW_MAX = 20.0
PEAK_HBM_BYTES_S = 7.7e12


def card_info():
    info = {"torch_device_name": torch.cuda.get_device_name(0)}
    try:
        r = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm,driver_version",
                            "--format=csv,noheader"], capture_output=True, text=True, timeout=60)
        name, power, clock, driver = (v.strip() for v in r.stdout.strip().split(","))
        info.update({"name": name, "power_limit": power, "max_sm_clock": clock, "driver": driver})
    except Exception as e:  # noqa: BLE001
        info["nvidia_smi_error"] = repr(e)
    return info


def build_algo(S, sampler, order, ckpt):
    from opticalflowdiffusion_b200 import FlowDiffuser
    from opticalflowdiffusion_b200.config import compose
    over = ["algorithm.target=flow", f"algorithm.sampling_timesteps={S}", "algorithm.return_all_timesteps=false",
            "algorithm.use_cuda_graph=true"]
    if sampler == "dpmpp":
        over += ["algorithm.sampler=dpmpp", f"algorithm.solver_order={order}"]
    torch.manual_seed(0)
    algo = FlowDiffuser(compose(over).algorithm)
    if ckpt:
        sd = torch.load(ckpt, map_location="cpu", weights_only=False)
        sd = sd.get("state_dict", sd)
        algo.load_state_dict(sd, strict=False)
    return algo.cuda().eval()


def time_sampler(algo, cond, x_T, reps):
    """Capture (first call) + one warm replay, then `reps` timed replays."""
    B = cond.shape[0]
    out = algo.model.sample(B, external_cond=cond, x_T=x_T, use_cuda_graph=True)
    out = algo.model.sample(B, external_cond=cond, x_T=x_T, use_cuda_graph=True)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(reps):
        out = algo.model.sample(B, external_cond=cond, x_T=x_T, use_cuda_graph=True)
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    return out, B * reps / dt, dt / reps


def step_kernel(n, iters=200):
    from opticalflowdiffusion_b200 import _lib
    from opticalflowdiffusion_b200.diffusion import ddim_time_pairs, dpmpp_coeffs, ConditionalDiffusion
    lib = _lib.load(check_device=True)
    d = ConditionalDiffusion(torch.nn.Identity(), 64, sampling_timesteps=10)
    pairs = ddim_time_pairs(1000, 10)
    times = [p[0] for p in pairs] + [-1]
    cx, c0, c1, c2, last = dpmpp_coeffs(d._host["alphas_cumprod"].tolist(), times, 5, 3)
    sets = [[torch.randn(n, device="cuda") for _ in range(4)] for _ in range(4)]     # x, model_out, d_hist1, d_hist2
    st = _lib.stream()

    def launch(k):
        x, mo, h1, h2 = sets[k % 4]
        _lib.check(lib.fd_dpmpp_step(_lib.ptr(x), _lib.ptr(mo), _lib.ptr(h1), _lib.ptr(h2), _lib.ptr(x), _lib.ptr(h2), n,
                                     cx, c0, c1, c2, last, st))

    for k in range(20):
        launch(k)
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s.record()
    for k in range(iters):
        launch(k)
    e.record()
    torch.cuda.synchronize()
    sec = s.elapsed_time(e) * 1e-3 / iters
    nbytes = 24 * n
    return {"n": n, "bytes_per_call": nbytes, "us_per_call": sec * 1e6, "GB_per_s": nbytes / sec / 1e9,
            "fraction_of_7.7TB_s": nbytes / sec / PEAK_HBM_BYTES_S,
            "note": "order 3, in place (x_next == x, d_out == d_hist2); 4 input sets cycled, 0.57 GB > L2; "
                    "CUDA events around 200 back-to-back launches"}


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--out", required=True, help="directory for the JSON result")
    ap.add_argument("--ckpt", default=None)
    ap.add_argument("--batch", type=int, default=8)
    ap.add_argument("--height", type=int, default=436)
    ap.add_argument("--width", type=int, default=1024)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--steps", default="10,15,20,25,50")
    args = ap.parse_args()
    from opticalflowdiffusion_b200 import _lib
    from opticalflowdiffusion_b200.datasets import synthetic_frames
    _lib.load(check_device=True)          # no GPU -> error: nothing here falls back to the CPU
    B, H, W = args.batch, args.height, args.width
    steps = [int(s) for s in args.steps.split(",")]
    res = {"card": card_info(), "shape": [B, 2, H, W], "target": "flow", "cuda_graph": True, "reps": args.reps,
           "weights": args.ckpt or "random init (torch.manual_seed(0)): end-point errors show solver convergence on this "
                                   "network, not flow quality on trained data",
           "epe_reference": "3M-200 from the same x_T and cond", "runs": []}
    cond = (2 * synthetic_frames(B, H, W, seed=5) - 1).cuda()
    x_T = torch.randn(B, 2, H, W, generator=torch.Generator().manual_seed(6)).cuda()

    ref_algo = build_algo(200, "dpmpp", 3, args.ckpt)
    t0 = time.perf_counter()
    ref = ref_algo.model.sample(B, external_cond=cond, x_T=x_T)       # eager
    torch.cuda.synchronize()
    res["reference_seconds_eager"] = time.perf_counter() - t0
    del ref_algo
    torch.cuda.empty_cache()

    configs = [("ddim", 1, 50)] + [("dpmpp", o, S) for o in (2, 3) for S in steps]
    for sampler, order, S in configs:
        algo = build_algo(S, sampler, order, args.ckpt)
        out, fps, sec = time_sampler(algo, cond, x_T, args.reps)
        epe = torch.sqrt(((out - ref) * FLOW_MAX).pow(2).sum(1)).mean().item()
        name = "DDIM-50" if sampler == "ddim" else f"{order}M-{S}"
        row = {"sampler": name, "nfe": S, "flows_per_s": fps, "seconds_per_batch": sec, "epe_px_vs_3M200": epe}
        print(json.dumps(row), flush=True)
        res["runs"].append(row)
        del algo, out
        torch.cuda.empty_cache()
    ddim = res["runs"][0]["flows_per_s"]
    for row in res["runs"]:
        row["speed_vs_ddim50"] = row["flows_per_s"] / ddim
    res["step_kernel"] = step_kernel(B * 2 * H * W)
    print(json.dumps(res["step_kernel"]))
    os.makedirs(args.out, exist_ok=True)
    path = os.path.join(args.out, "bench_samplers.json")
    with open(path, "w") as f:
        json.dump(res, f, indent=1)
    print("wrote", path)


if __name__ == "__main__":
    main()
