"""Speed of the flow evaluation path on one GPU.

  (a) fd_flow_eval at B = 8, 436x1024, K in {1, 4, 8}: microseconds per launch (CUDA events around back-to-back launches,
      four input sets cycled so that the working set exceeds the 126 MB L2 for K >= 4) and the achieved GB/s over the bytes
      it must move -- samples 8K + ground truth 8 + mean 8 + spread 4 bytes per pixel -- against the 7.7 TB/s HBM3e figure
      of the B200 data sheet; plus its worst deviation from the fp64 oracle at K = 4.
  (b) the evaluate path -- FlowDiffuser.evaluate_step: preprocess, K = 4 seeded x_T per image, DDIM-50 through the CUDA
      graph, fd_flow_eval -- in flows/s at 436x1024, against FlowDiffuser.sample alone on the same inputs (K calls of
      batch 8 with pre-drawn x_T), so the overhead of the evaluation path shows.
The card's name and power limit are read in the same run and written beside the numbers, into ONE JSON file under --out.
Weights are randomly initialised (torch.manual_seed(0)): the speeds do not depend on them.

    python scripts/bench_flow_eval.py --out DIR [--reps 3]
"""
import argparse
import json
import os
import sys
import time

import torch

sys.dont_write_bytecode = True
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))
sys.path.insert(0, os.path.join(ROOT, "tests"))

from bench_samplers import PEAK_HBM_BYTES_S, card_info  # noqa: E402

FLOW_MAX = 20.0


def kernel_time(B, K, H, W, iters=200):
    from opticalflowdiffusion_b200 import _lib
    lib = _lib.load(check_device=True)
    g = torch.Generator(device="cuda").manual_seed(K)
    sets = []
    for _ in range(4):
        s = torch.randn(B, K, 2, H, W, device="cuda", generator=g) * 0.25
        gt = torch.randn(B, 2, H, W, device="cuda", generator=g) * 6
        sets.append((s, gt, torch.empty(B, 2, H, W, device="cuda"), torch.empty(B, H, W, device="cuda")))
    rows = torch.empty(B, 8 + K, device="cuda", dtype=torch.float64)
    ws = torch.empty(lib.fd_flow_eval_workspace_floats(B, K, H, W), device="cuda")
    st = _lib.stream()

    def launch(i):
        s, gt, mean, spread = sets[i % 4]
        _lib.check(lib.fd_flow_eval(_lib.ptr(s), FLOW_MAX, _lib.ptr(gt), FLOW_MAX, _lib.ptr(mean), _lib.ptr(spread),
                                    _lib.ptr(rows), _lib.ptr(ws), B, K, H, W, st))

    for i in range(20):
        launch(i)
    a, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for i in range(iters):
        launch(i)
    e.record()
    torch.cuda.synchronize()
    sec = a.elapsed_time(e) * 1e-3 / iters
    nbytes = B * H * W * (8 * K + 8 + 8 + 4)
    return {"B": B, "K": K, "H": H, "W": W, "bytes_per_call": nbytes, "us_per_call": sec * 1e6,
            "GB_per_s": nbytes / sec / 1e9, "fraction_of_7.7TB_s": nbytes / sec / PEAK_HBM_BYTES_S,
            "working_set_GB": 4 * nbytes / 1e9}


def accuracy(B, K, H, W):
    import flow_eval_oracle as OR
    from opticalflowdiffusion_b200.evaluation import score_flows
    g = torch.Generator().manual_seed(1)
    s = torch.randn(B, K, 2, H, W, generator=g) * 0.25
    gt = torch.randn(B, 2, H, W, generator=g) * 6
    mean, spread, rows = score_flows(s.cuda(), FLOW_MAX, gt.cuda())
    m, sp, r, _ = OR.flow_eval(s, FLOW_MAX, gt)
    sums = [1, 6] + list(range(8, 8 + K))
    rel = ((rows.cpu()[:, sums] - r[:, sums]).abs() / r[:, sums].abs()).max()
    return {"shape": [B, K, 2, H, W], "max_abs_mean_err_px": float((mean.cpu().double() - m).abs().max()),
            "max_abs_spread_err_px": float((spread.cpu().double() - sp).abs().max()),
            "max_rel_sum_err": float(rel), "count_diffs": float((rows.cpu()[:, [0, 2, 3, 4, 5, 7]] -
                                                                  r[:, [0, 2, 3, 4, 5, 7]]).abs().max())}


def evaluate_throughput(B, K, H, W, reps):
    from opticalflowdiffusion_b200 import FlowDiffuser
    from opticalflowdiffusion_b200.config import compose
    from opticalflowdiffusion_b200.datasets import SyntheticSintelDataset
    torch.manual_seed(0)
    algo = FlowDiffuser(compose(["algorithm.target=flow", "algorithm.sampling_timesteps=50",
                                 "algorithm.return_all_timesteps=false", "algorithm.use_cuda_graph=true"]).algorithm)
    algo = algo.cuda().eval()
    ds = SyntheticSintelDataset(compose([f"dataset.height={H}", f"dataset.width={W}"]).dataset, split="validation")
    batch = tuple(torch.stack(x).cuda() for x in zip(*(ds[i] for i in range(B))))
    ids = list(range(B))
    cond = 2 * batch[0] - 1
    x_T = torch.randn(K, B, 2, H, W, device="cuda")

    def run_eval():
        return algo.evaluate_step(batch, ids, K, seed=0)

    def run_sample():
        return [algo.sample(cond, cond, x_T=x_T[k])[1] for k in range(K)]

    out = {}
    for name, fn in (("evaluate_step", run_eval), ("sample_only", run_sample)):
        fn()
        fn()                                          # capture, then one warm replay
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(reps):
            fn()
        torch.cuda.synchronize()
        dt = (time.perf_counter() - t0) / reps
        out[name] = {"flows_per_s": B * K / dt, "seconds_per_call": dt}
    out["evaluate_overhead"] = out["sample_only"]["flows_per_s"] / out["evaluate_step"]["flows_per_s"] - 1
    out["setup"] = (f"B={B} images x K={K} samples = {B * K} flows per call, {H}x{W}, target=flow, DDIM-50, CUDA graph, "
                    f"sampled in {K} chunks of {B} (the default max_batch); sample_only: {K} FlowDiffuser.sample calls "
                    f"of batch {B} on the same cond with pre-drawn x_T")
    return out


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--out", required=True, help="directory for the JSON result")
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--batch", type=int, default=8)
    ap.add_argument("--height", type=int, default=436)
    ap.add_argument("--width", type=int, default=1024)
    args = ap.parse_args()
    from opticalflowdiffusion_b200 import _lib
    _lib.load(check_device=True)          # no GPU -> error: nothing here falls back to the CPU
    B, H, W = args.batch, args.height, args.width
    res = {"card": card_info(), "kernel": [], "note": "kernel: CUDA events around 200 back-to-back launches, 4 input sets "
                                                      "cycled; evaluate: host clock around reps calls ending in a synchronise"}
    for K in (1, 4, 8):
        row = kernel_time(B, K, H, W)
        print(json.dumps(row), flush=True)
        res["kernel"].append(row)
        torch.cuda.empty_cache()
    res["accuracy_vs_fp64_oracle"] = accuracy(B, 4, H, W)
    print(json.dumps(res["accuracy_vs_fp64_oracle"]), flush=True)
    res["evaluate"] = evaluate_throughput(B, 4, H, W, args.reps)
    print(json.dumps(res["evaluate"]), flush=True)
    os.makedirs(args.out, exist_ok=True)
    path = os.path.join(args.out, "bench_flow_eval.json")
    with open(path, "w") as f:
        json.dump(res, f, indent=1)
    print("wrote", path)


if __name__ == "__main__":
    main()
