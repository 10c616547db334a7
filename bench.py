#!/usr/bin/env python
"""Headline benchmark of the flow_diffuser hot path (BASELINE.json configs[1]):
DDIM-50 flow sampling, Sintel-shaped synthetic 436x1024 frames, batch 8 per GPU.

    python bench.py --gpus N --steps K --warmup W            # this implementation (CUDA, sm_100a)
    python bench.py --impl reference --gpus N ...            # the reference algorithm on the host CPU cores
    python bench.py ... --dump-outputs DIR                   # also write what the last timed step computed, as .npy

One "step" = one DDIM-50 sampling pass over one batch of 8 frame pairs = 8 flows.
Prints ONE JSON line (rank 0).  Multi-GPU: one process per GPU under torchrun, the batch is sharded
by rank with no data-path collective (sampling has no exchange step) -> weak scaling.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True         # the tree may be read-only; the benchmark leaves it as it found it

DDIM_STEPS, TIMESTEPS = 50, 1000
# --config selects the workload; the default is BASELINE.json configs[1] (the configuration `metric` is quoted on),
# "matrix_flow_1024x2048" is configs[4] (the matrix_flow experiment's resolution; the reference itself cannot run it: its
# N x N attention matrix is 17 GB per sample, denoising_diffusion.py:263-265)
WORKLOADS = {
    "ddim50_436x1024": dict(
        H=436, W=1024, batch=8, metric="flows/sec DDIM-50 @436x1024",
        conv_gf=1590.3,        # SURVEY.md appendix A: algorithmic conv GFLOP per UNet forward at 440x1024
        fwd_gf=1635.28,        # SURVEY.md section 8d: whole forward (conv + attention matmuls)
        attn_gf=25.4,          # mid attention, N = 7040 tokens
        workload="flow_diffuser DDIM-50 sampling, Sintel-shaped synthetic 436x1024 (UNet runs on 440x1024), "
                 "target=flow, batch 8 per GPU, random-init weights seed 0",
        l2="working set >> L2: every bf16 activation tensor is 461 MB at full resolution, no reuse between steps"),
    "matrix_flow_1024x2048": dict(
        H=1024, W=2048, batch=2, metric="flows/sec DDIM-50 @1024x2048",
        conv_gf=1590.3 * (1024 * 2048) / (440 * 1024),      # appendix A: M scales linearly with pixels (x4.655)
        fwd_gf=8043.13,        # SURVEY.md section 6 / 8d row #5
        attn_gf=549.8,         # mid attention, N = 32768 tokens
        workload="matrix_flow experiment resolution: flow_diffuser DDIM-50 sampling, synthetic 1024x2048 frame pairs, "
                 "target=flow, batch 2 per GPU, random-init weights seed 0",
        l2="working set >> L2: every bf16 activation tensor is 537 MB at full resolution, no reuse between steps"),
}
WL = WORKLOADS["ddim50_436x1024"]
H, W, BATCH = WL["H"], WL["W"], WL["batch"]
CONV_GF_PER_SAMPLE, FWD_GF_PER_SAMPLE = WL["conv_gf"], WL["fwd_gf"]
CONFIG = {}


def select_workload(name: str):
    global WL, H, W, BATCH, CONV_GF_PER_SAMPLE, FWD_GF_PER_SAMPLE, CONFIG
    WL = WORKLOADS[name]
    H, W, BATCH = WL["H"], WL["W"], WL["batch"]
    CONV_GF_PER_SAMPLE, FWD_GF_PER_SAMPLE = WL["conv_gf"], WL["fwd_gf"]
    CONFIG = {"workload": WL["workload"], "name": name, "batch_per_gpu": BATCH, "ddim_steps": DDIM_STEPS,
              "timesteps": TIMESTEPS, "parallelism": "batch-sharded replicas", "l2": WL["l2"]}


def conv_traffic():
    """DRAM bytes (ncu dram__bytes_read.sum + dram__bytes_write.sum) of the conv launches of ONE forward of the
    selected workload, from the committed capture of the shipped code (scripts/agg_traffic.py -> profiles/), or None."""
    path = os.path.join(ROOT, "profiles", "r2_forward_traffic.json")
    try:
        with open(path) as f:
            d = json.load(f)
        ent = d.get(CONFIG.get("name", ""))
        if ent:
            return float(ent["conv_dram_bytes"]), "profiles/r2_forward_traffic.json: " + ent.get("source", "")
    except Exception:  # noqa: BLE001
        pass
    return None, "no ncu capture of this workload committed"


def load_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            p = json.load(f)
        return {"hbm": p["hbm_gbs"], "tf_burst": p["bf16_tflops"], "tf_sustained": p["bf16_tflops_sustained"],
                "src": "MEASURED_PEAKS.json"}
    except Exception:  # noqa: BLE001
        return {"hbm": 6650.0, "tf_burst": 1590.0, "tf_sustained": 1400.0, "src": "fallback (B200_PROFILING.md)"}


def load_red_rate():
    """Measured rate of red.global.add.v4.f32 to white-noise addresses (reductions / s) from profiles/r2_red_rate.txt, or None."""
    try:
        with open(os.path.join(ROOT, "profiles", "r2_red_rate.txt")) as f:
            rates = [float(l.split("us")[1].split("G reductions/s")[0]) for l in f
                     if l.startswith("v4.f32, white-noise") and "G reductions/s" in l]
        return max(rates) * 1e9 if rates else None
    except Exception:  # noqa: BLE001
        return None


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""

    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:  # noqa: BLE001
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is not None:
            self.proc.terminate()
        sm = sorted(int(r[0]) for r in self.rows if r and r[0].isdigit())
        mx = [int(r[1]) for r in self.rows if len(r) > 1 and r[1].isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(len(r) > 2 + i and r[2 + i].lower().startswith("active") for r in self.rows)]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons,
                "samples": len(sm)}


# ------------------------------------------------------------------------------------------------
# CPU reference arm / cpu_baseline: the oracle's fp32 restatement of the reference algorithm
# (the reference tree itself cannot travel to the GPU box) on all host threads.
# ------------------------------------------------------------------------------------------------
CPU_SAMPLE_HW = {"ddim50_436x1024": (436, 1024), "matrix_flow_1024x2048": (256, 512)}


def cpu_reference_step_seconds(steps: int, warmup: int, keep_io: bool = False):
    """Each step = ONE of the 50 DDIM steps of ONE sample (UNet forward + update) -> flows/s = 1 / (50 t).
    At 1024x2048 the reference's N x N attention matrix is 17 GB per sample (it cannot run there, SURVEY.md 8d row #5), so
    the sample is a 256x512 crop and the time is scaled by the pixel ratio (x16; the attention term grows faster, so the
    scaled time is a LOWER bound of the reference's cost).  Returns (seconds per full-size step, pixel scale, io)."""
    from oracle import flowdiff_oracle as O
    from opticalflowdiffusion_b200.unet_params import UnetParams
    # all host cores this process may use (torchrun pins OMP_NUM_THREADS=1 by default)
    try:
        torch.set_num_threads(max(1, len(os.sched_getaffinity(0))))
    except Exception:  # noqa: BLE001
        torch.set_num_threads(max(1, os.cpu_count() or 1))
    torch.manual_seed(0)
    sd = UnetParams(64, channels=5, out_dim=2).state_dict()
    sched = O.make_schedule(TIMESTEPS)
    h, w = CPU_SAMPLE_HW[CONFIG["name"]]
    scale = (H * W) / float(h * w)
    cond = O.replicate_pad_to_multiple(O.synthetic_frames(1, h, w, seed=0) * 2 - 1)[0]
    x = torch.randn(1, 2, cond.shape[-2], cond.shape[-1], generator=torch.Generator().manual_seed(1234))
    times = O.ddim_times(TIMESTEPS, DDIM_STEPS)
    ts, out = [], None
    with torch.no_grad():
        for i in range(warmup + steps):
            t0 = time.perf_counter()
            tt = torch.full((1,), times[0], dtype=torch.long)
            out = O.unet_forward(sd, x, cond, tt)
            O.ddim_update(sched, x, out, times[0], times[1])
            if i >= warmup:
                ts.append(time.perf_counter() - t0)
    io = (sd, x, cond, times[0], out) if keep_io else None
    return ts, scale, io


def cpu_sample_text(scale: float) -> str:
    h, w = CPU_SAMPLE_HW[CONFIG["name"]]
    txt = f"one of the {DDIM_STEPS} DDIM steps of ONE {h}x{w} sample (UNet forward + update) on the host cores, x{DDIM_STEPS} extrapolated"
    if scale != 1.0:
        txt += f", x{scale:.0f} by pixel count to {H}x{W} (the reference cannot allocate its attention matrix at that size)"
    return txt


def run_reference(args, rank: int):
    if rank != 0:
        return
    warm = max(0, args.warmup)
    ts, scale, _ = cpu_reference_step_seconds(args.steps, warm)
    threads = torch.get_num_threads()
    t = sum(ts) / len(ts)
    value = 1.0 / (DDIM_STEPS * t * scale)
    sample = cpu_sample_text(scale)
    # ms_per_step is what one timed step of THIS run took (the bounded sample), so steps x ms_per_step fits the driver's
    # clock; the whole-workload figure (one batch of BATCH flows) is extrapolated and labelled as such
    line = {"impl": "reference", "metric": WL["metric"], "value": value, "unit": "flows/s",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": warm, "ms_per_step": t * 1e3,
            "extrapolated": True, "sample_seconds_per_forward": t,
            "ms_per_step_full_workload_extrapolated": t * scale * 1e3 * DDIM_STEPS * BATCH,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": CONFIG,
            "cpu_baseline": {"value": value, "unit": "flows/s", "cores": threads, "kind": "port", "sample": sample},
            "e2e": {"value": value, "unit": "flows/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    _emit(line)


# ------------------------------------------------------------------------------------------------
# The GPU LIBRARY bar (SURVEY.md 2.2, BASELINE.md 3.5): the reference algorithm as PyTorch eager ops -- cuDNN convolutions,
# cuBLAS / ATen attention, ATen norms -- on the SAME B200, TF32 on as main.py:79-80 sets it, and once under bf16 autocast
# (Lightning's "bf16-mixed", exp_base.py:204).  The oracle's functional restatement is the same op sequence as the
# reference's nn.Modules (denoising_diffusion.py:81-417); it runs here as the thing being *compared against*, never as a
# fallback of the product path.
# ------------------------------------------------------------------------------------------------
def gpu_library_baseline(dev, full_loops: int = 1):
    from oracle import flowdiff_oracle as O
    from opticalflowdiffusion_b200.unet_params import UnetParams
    torch.backends.cuda.matmul.allow_tf32 = True          # torch.set_float32_matmul_precision("high"), main.py:79-80
    torch.backends.cudnn.allow_tf32 = True
    torch.backends.cudnn.benchmark = True                 # give the library its best algorithm per shape
    torch.manual_seed(0)
    sd = {k: v.to(dev) for k, v in UnetParams(64, channels=5, out_dim=2).state_dict().items()}
    sched = {k: v.to(dev) for k, v in O.make_schedule(TIMESTEPS).items()}
    cond = O.replicate_pad_to_multiple(O.synthetic_frames(BATCH, H, W, seed=100) * 2 - 1)[0].to(dev)
    x_T = torch.randn(BATCH, 2, cond.shape[-2], cond.shape[-1], device=dev)
    pairs = list(zip(O.ddim_times(TIMESTEPS, DDIM_STEPS)[:-1], O.ddim_times(TIMESTEPS, DDIM_STEPS)[1:]))
    res = {"what": "reference algorithm as PyTorch %s eager ops (cuDNN %s / cuBLAS) on this GPU, batch %d, %dx%d, DDIM-%d, "
                   "cudnn.benchmark on" % (torch.__version__, torch.backends.cudnn.version(), BATCH, cond.shape[-2], cond.shape[-1],
                                           DDIM_STEPS),
           "unit": "flows/s"}

    def loop(autocast: bool, n_steps: int):
        x = x_T.clone()
        with torch.no_grad():
            for tm, tn in pairs[:n_steps]:
                t = torch.full((BATCH,), tm, device=dev, dtype=torch.long)
                with torch.autocast("cuda", dtype=torch.bfloat16, enabled=autocast):
                    out = O.unet_forward(sd, x, cond, t)
                x, _ = O.ddim_update(sched, x, out.float(), tm, tn)
        return x

    for name, autocast in (("tf32", False), ("bf16_autocast", True)):
        try:
            loop(autocast, 3)                 # warm-up: cuDNN algorithm search, allocator
            torch.cuda.synchronize()
            s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s.record()
            for _ in range(full_loops):
                loop(autocast, DDIM_STEPS)
            e.record()
            torch.cuda.synchronize()
            sec = s.elapsed_time(e) * 1e-3 / full_loops
            res[name] = {"value": BATCH / sec, "ms_per_step": sec * 1e3, "ms_per_forward": sec * 1e3 / DDIM_STEPS,
                         "tflops": FWD_GF_PER_SAMPLE * BATCH * DDIM_STEPS / sec / 1e3}
        except torch.OutOfMemoryError as ex:  # the N x N attention matrix (17 GB per sample at 1024x2048)
            res[name] = {"unavailable": "out of memory: " + str(ex).split("\n")[0][:160]}
        torch.cuda.empty_cache()
    res["peak_mem_gib"] = torch.cuda.max_memory_allocated(dev) / 2 ** 30
    torch.backends.cudnn.benchmark = False
    return res


def gpu_library_train_baseline(dev, batch: int):
    """The same bar for the training step (BASELINE configs[2]): loss + backward (autograd through the eager ops) + Adam at
    368x768, batch `batch`, TF32 and bf16 autocast."""
    from oracle import flowdiff_oracle as O
    from opticalflowdiffusion_b200.unet_params import UnetParams
    torch.backends.cuda.matmul.allow_tf32 = True
    torch.backends.cudnn.allow_tf32 = True
    torch.backends.cudnn.benchmark = True
    res = {"what": "p_losses (target=flow) + backward + torch.optim.Adam through PyTorch eager ops on this GPU, 368x768",
           "unit": "samples/s"}
    sched = {k: v.to(dev) for k, v in O.make_schedule(TIMESTEPS).items()}
    for name, autocast in (("tf32", False), ("bf16_autocast", True)):
        b = batch
        while b >= 1:
            try:
                torch.manual_seed(0)
                sd = {k: v.to(dev).requires_grad_(True) for k, v in UnetParams(64, channels=5, out_dim=2).state_dict().items()}
                opt = torch.optim.Adam(list(sd.values()), lr=1e-5, weight_decay=1e-6)
                cond = (O.synthetic_frames(b, TRAIN_H, TRAIN_W, seed=200) * 2 - 1).to(dev)
                x0 = torch.clamp(torch.randn(b, 2, TRAIN_H, TRAIN_W, device=dev) * 0.25, -1, 1)
                noise = torch.randn(b, 2, TRAIN_H, TRAIN_W, device=dev)
                t = torch.randint(0, TIMESTEPS, (b,), device=dev)

                def step():
                    with torch.autocast("cuda", dtype=torch.bfloat16, enabled=autocast):
                        loss = O.p_losses_flow(sd, sched, x0, cond, t, noise)
                    loss.backward()
                    torch.nn.utils.clip_grad_norm_(list(sd.values()), 100.0)
                    opt.step()
                    opt.zero_grad(set_to_none=True)

                for _ in range(2):
                    step()
                torch.cuda.synchronize()
                s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                s.record()
                for _ in range(3):
                    step()
                e.record()
                torch.cuda.synchronize()
                sec = s.elapsed_time(e) * 1e-3 / 3
                res[name] = {"value": b / sec, "ms_per_step": sec * 1e3, "batch": b,
                             "peak_mem_gib": torch.cuda.max_memory_allocated(dev) / 2 ** 30}
                break
            except torch.OutOfMemoryError:
                res.setdefault("notes", []).append(f"{name}: batch {b} does not fit in memory through autograd of the eager ops")
                b //= 2
            finally:
                sd = opt = None
                torch.cuda.empty_cache()
                torch.cuda.reset_peak_memory_stats(dev)
    torch.backends.cudnn.benchmark = False
    return res


def run_torch_gpu(args, rank: int, local_rank: int):
    """--impl torch-gpu: the GPU library bar as its own arm (rank 0 only)."""
    if rank != 0:
        return
    dev = torch.device("cuda", local_rank)
    torch.cuda.set_device(dev)
    clocks = ClockSampler(local_rank)
    clocks.start()
    res = gpu_library_baseline(dev, full_loops=max(1, args.steps))
    clk = clocks.stop()
    best = res.get("tf32", {})
    line = {"impl": "torch-gpu", "metric": WL["metric"], "value": best.get("value"), "unit": "flows/s", "n_gpus": 1,
            "steps": max(1, args.steps), "warmup": 1, "ms_per_step": best.get("ms_per_step"), "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "tf32", "data": "synthetic", "config": CONFIG, "clocks": clk,
            "gpu_library_baseline": res, "gpu_launches": 0}
    if CONFIG["name"] == "ddim50_436x1024" and not args.skip_train:
        line["gpu_library_train_baseline"] = gpu_library_train_baseline(dev, args.train_batch)
    _emit(line)


def tiny_config(dev):
    """BASELINE configs[0]: the reference's own CPU-runnable case -- batch 1, 64x128 frame pair, target=flow.  The reference
    algorithm (oracle port, all host threads) is timed on one full DDIM-50 sampling pass and on 20 of the 1000 DDPM steps
    it runs as shipped (flow_diffuser.py:118-127 never passes sampling_timesteps); this implementation on DDIM-50 and the
    full DDPM-1000 chain, CUDA-graph off (launch-bound at this size)."""
    from oracle import flowdiff_oracle as O
    from opticalflowdiffusion_b200 import FlowDiffuser
    from opticalflowdiffusion_b200.config import compose
    h, w = 64, 128
    res = {"shape": [1, 2, h, w]}
    for name, steps in (("ddim50", 50), ("ddpm1000", None)):
        ov = ["algorithm.target=flow", f"algorithm.image_size=[{h},{w}]", "algorithm.return_all_timesteps=false"]
        if steps:
            ov.append(f"algorithm.sampling_timesteps={steps}")
        torch.manual_seed(0)
        algo = FlowDiffuser(compose(ov).algorithm).to(dev)
        cond = (O.synthetic_frames(1, h, w, seed=0) * 2 - 1).to(dev)
        zero = torch.zeros(1, 2, h, w, device=dev)
        algo.sample(cond, zero)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        algo.sample(cond, zero)
        torch.cuda.synchronize()
        res[name + "_gpu_s"] = time.perf_counter() - t0
        if name == "ddim50":
            sd = {k: v.detach().cpu() for k, v in algo.unet.state_dict().items()}
    sched = O.make_schedule(TIMESTEPS)
    cond_c = O.synthetic_frames(1, h, w, seed=0) * 2 - 1
    x = torch.randn(1, 2, h, w, generator=torch.Generator().manual_seed(1))
    with torch.no_grad():
        O.unet_forward(sd, x, cond_c, torch.tensor([999]))            # warm-up
        t0 = time.perf_counter()
        O.ddim_sample(sd, sched, x, cond_c, TIMESTEPS, 50)
        res["ddim50_reference_cpu_s"] = time.perf_counter() - t0
        t0 = time.perf_counter()
        for tt in range(999, 979, -1):
            out = O.unet_forward(sd, x, cond_c, torch.tensor([tt]))
            x, _ = O.ddpm_update(sched, x, out, tt, torch.zeros_like(x))
        res["ddpm1000_reference_cpu_s_extrapolated"] = (time.perf_counter() - t0) * 50.0
    res["cores"] = torch.get_num_threads()
    res["ddim50_speedup"] = res["ddim50_reference_cpu_s"] / res["ddim50_gpu_s"]
    return res


# --dump-outputs: an output of at most DUMP_FULL_MAX elements is written whole, a larger one as DUMP_SAMPLE elements at
# fixed, seeded flat indices.  The sampling outputs (with the hole mask of the samples) come to at most 32 + 3 x 8 MiB of
# float32.
DUMP_FULL_MAX = 1 << 23
DUMP_SAMPLE = 1 << 21


def dump_outputs(out_dir: str, arrays: dict):
    """Write each tensor of `arrays` as <out_dir>/<name>.npy in float32: whole (same shape) when it is small enough, else
    the 1-D sample flat[idx] with idx = sorted torch.randint(numel, (DUMP_SAMPLE,)) of a CPU generator seeded 0, so two
    runs or two builds at the same shape sample the same elements.  Every value written is finite: where an output holds
    NaN or inf (the forward splat leaves NaN holes in the samples), <name>.npy has 0 and <name>_nonfinite.npy has 1."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    for name, t in arrays.items():
        t = t.detach().float()
        if t.numel() > DUMP_FULL_MAX:
            idx = torch.randint(t.numel(), (DUMP_SAMPLE,), generator=torch.Generator().manual_seed(0)).sort().values
            t = t.reshape(-1)[idx.to(t.device)]
        finite = torch.isfinite(t)
        if not bool(finite.all()):
            np.save(os.path.join(out_dir, name + "_nonfinite.npy"), (~finite).float().cpu().numpy())
            t = torch.where(finite, t, torch.zeros_like(t))
        np.save(os.path.join(out_dir, name + ".npy"), t.cpu().numpy())


# ------------------------------------------------------------------------------------------------
def run_ours(args, rank: int, world: int, local_rank: int):
    import torch.distributed as dist
    from opticalflowdiffusion_b200 import FlowDiffuser, _lib
    from opticalflowdiffusion_b200.config import compose
    from opticalflowdiffusion_b200.datasets import synthetic_frames
    from opticalflowdiffusion_b200.parallel import max_over_ranks

    dev = torch.device("cuda", local_rank)
    torch.cuda.set_device(dev)
    lib = _lib.load(check_device=True)
    if world > 1:
        # NCCL prints its version banner to stdout when NCCL_DEBUG is set on the box; stdout carries exactly one JSON line
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
        dist.init_process_group("nccl", device_id=dev)
    cfg = compose(["algorithm.target=flow", f"algorithm.sampling_timesteps={DDIM_STEPS}",
                   f"algorithm.image_size=[{H},{W}]", "algorithm.return_all_timesteps=true",
                   f"algorithm.use_cuda_graph={'true' if args.graph else 'false'}"])
    torch.manual_seed(0)
    if args.skip_sample:
        tr = run_train_leg(args, cfg.algorithm, rank, world, dev)
        if rank == 0:
            _emit({"train": tr, "n_gpus": world})
        return
    algo = FlowDiffuser(cfg.algorithm).to(dev)
    algo.unet.prepare()
    frames = synthetic_frames(BATCH, H, W, seed=100 + rank)
    cond_host = (2 * frames - 1).pin_memory()
    flow_host = torch.zeros(BATCH, 2, H, W).pin_memory()
    out_host = torch.empty(BATCH, 2, H, W).pin_memory()
    cond_dev = cond_host.to(dev)
    flow_dev = flow_host.to(dev)
    gen = torch.Generator(device=dev).manual_seed(1234 + rank)
    x_T = torch.randn(BATCH, 2, H, W, device=dev, generator=gen)

    def sync():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    def step_resident():
        return algo.sample(cond_dev, flow_dev, x_T=x_T)

    def step_e2e():
        c = cond_host.to(dev, non_blocking=True)
        f = flow_host.to(dev, non_blocking=True)
        _, flows = algo.sample(c, f, x_T=x_T)
        out_host.copy_(flows[:, -1], non_blocking=True)
        torch.cuda.synchronize()

    def timed(fn, steps):
        """Seconds of `steps` calls of fn (slowest rank) and what the last call returned."""
        sync()
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        for _ in range(steps):
            out = fn()
        e.record()
        sync()
        return max_over_ranks(s.elapsed_time(e) * 1e-3, device=dev), out

    for _ in range(max(args.warmup, 3) if args.warmup >= 0 else 3):
        step_resident()
    clocks = ClockSampler(local_rank)
    if rank == 0:
        clocks.start()
    l0 = lib.fd_launch_count() + algo.model.graph_replayed_launches
    t_res, (samples, flows) = timed(step_resident, args.steps)
    launches = int(lib.fd_launch_count() + algo.model.graph_replayed_launches - l0)
    if args.dump_outputs and rank == 0:
        # what a caller of algo.sample receives: samples (B, 3, H, W) and the flow trajectory (B, 51, 2, H, W), and the
        # final flow (B, 2, H, W), whole, as the trajectory is only sampled
        dump_outputs(args.dump_outputs, {"samples": samples, "flows": flows, "flows_last": flows[:, -1]})
    del samples, flows
    t_e2e, _ = timed(step_e2e, args.steps)
    clk = clocks.stop() if rank == 0 else None

    # roofline pass (not timed above): CUDA events around every tensor-core conv launch of one UNet forward
    # (averaged over RF_REPS forwards: a single forward under the power cap varies by +-3 %)
    RF_REPS = 3
    t = torch.full((BATCH,), 999, device=dev, dtype=torch.long)
    torch.set_grad_enabled(False)          # the inference forward (with autograd on, unet(...) is the training forward)
    algo.unet(x_T, cond_dev, t)            # warm: the eager path's allocations are cached before anything is timed
    algo.unet._conv_timing = []
    for _ in range(RF_REPS):
        algo.unet(x_T, cond_dev, t)
    torch.cuda.synchronize()
    conv_s = sum(ev[0].elapsed_time(ev[1]) for _, _, ev in algo.unet._conv_timing) * 1e-3 / RF_REPS
    n_up = sum(1 for name, _, _ in algo.unet._conv_timing if name.startswith("ups.") and name.endswith(".3")) // RF_REPS
    n_phase = 3 * (n_up - 1) if getattr(algo.unet, "UPCONV_PHASES", False) and n_up > 1 else 0      # an Upsample conv = 4 phase launches
    conv_launches = len(algo.unet._conv_timing) // RF_REPS + n_phase
    algo.unet._conv_timing = None
    algo.unet(x_T, cond_dev, t)
    torch.cuda.synchronize()
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s.record()
    for _ in range(RF_REPS):
        algo.unet(x_T, cond_dev, t)
    e.record()
    torch.cuda.synchronize()
    fwd_s = s.elapsed_time(e) * 1e-3 / RF_REPS
    torch.set_grad_enabled(True)

    # cpu_baseline (rank 0, N = 1): one DDIM step of one sample through the oracle on the host cores; its output doubles as
    # the checker of a teacher-forced GPU forward on the very same input -> "parity" (the oracle is the checker here, the
    # GPU forward compared with it is the product path)
    cpu_base = parity = None
    if world == 1 and rank == 0 and not args.no_cpu_baseline:
        ts, scale, (sd_o, x_o, cond_o, t_o, out_o) = cpu_reference_step_seconds(1, 1, keep_io=True)
        tcpu = sum(ts) / len(ts)
        cpu_base = {"value": 1.0 / (DDIM_STEPS * tcpu * scale), "unit": "flows/s", "cores": torch.get_num_threads(),
                    "kind": "port", "sample": cpu_sample_text(scale) + " after one warm-up"}
        with torch.no_grad():
            got = algo.unet(x_o.to(dev), cond_o.to(dev), torch.full((1,), t_o, device=dev, dtype=torch.long)).cpu()
        err = (got - out_o).abs()
        epe = torch.sqrt(((got.clamp(-1, 1) - out_o.clamp(-1, 1)) * 20.0).pow(2).sum(1)).mean().item()
        parity = {"kind": "teacher-forced x0 prediction of one DDIM step (t = %d) vs the fp32 CPU oracle on the same input" % t_o,
                  "shape": list(x_o.shape), "max_abs_err": err.max().item(), "mean_abs_err": err.mean().item(),
                  "epe_px": epe, "tolerance": "max |err| <= 3e-2 on [-1, 1] data (tests/test_gpu_headline_parity.py)",
                  "free_running": "DDIM-50 436x1024 EPE vs the oracle trajectory: tests/test_gpu_headline_parity.py, "
                                  "numbers in profiles/r2_parity_headline.json"}
        del sd_o, x_o, cond_o, out_o, got
    default_wl = CONFIG["name"] == "ddim50_436x1024"
    tiny = None
    if world == 1 and rank == 0 and default_wl and not args.no_cpu_baseline:
        tiny = tiny_config(dev)
    # this implementation's training leg runs BEFORE the library baseline (40 s of eager kernels at the power cap heat the
    # board: measured 140 vs 150 samples/s for the same code when it ran after)
    train = None
    del algo
    algo = None
    torch.cuda.empty_cache()
    if not args.skip_train and default_wl:
        torch.cuda.reset_peak_memory_stats(dev)
        train = run_train_leg(args, cfg.algorithm, rank, world, dev)
    lib_base = None
    if world == 1 and rank == 0 and not args.no_gpu_baseline:
        torch.cuda.empty_cache()
        lib_base = gpu_library_baseline(dev)
        if default_wl and not args.skip_train:
            lib_base["train"] = gpu_library_train_baseline(dev, args.train_batch)
    if rank != 0:
        return
    peaks = load_peaks()
    traffic, traffic_src = conv_traffic()
    flows = world * BATCH * args.steps
    value = flows / t_res
    conv_tf = CONV_GF_PER_SAMPLE * BATCH * 1e9 / conv_s / 1e12
    line = {
        "metric": WL["metric"], "value": value, "unit": "flows/s", "n_gpus": world, "steps": args.steps,
        "warmup": max(args.warmup, 3), "ms_per_step": t_res / args.steps * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "bf16", "data": "synthetic", "config": CONFIG,
        "e2e": {"value": flows / t_e2e, "unit": "flows/s", "h2d_bytes_per_step": cond_host.numel() * 4 + flow_host.numel() * 4,
                "d2h_bytes_per_step": out_host.numel() * 4},
        "gpu_launches": launches, "cuda_graph": bool(args.graph),
        "clocks": clk,
        "roofline": {"bound": "tensor", "kernel": "conv_igemm_kernel (tcgen05 implicit GEMM, all %d conv launches of one forward)" % conv_launches,
                     "achieved": conv_tf, "peak": peaks["tf_sustained"], "unit": "TFLOP/s", "frac": conv_tf / peaks["tf_sustained"],
                     "traffic": traffic, "traffic_source": traffic_src + " (ncu dram__bytes_read.sum + dram__bytes_write.sum summed over "
                     "the conv launches of ONE forward at this batch: the unit of `achieved`; algorithmic FLOPs, not bytes, bound these kernels)",
                     "peak_source": peaks["src"] + " (sustained: the kernel is timed inside a long step)",
                     "note": "launches that also apply the preceding GroupNorm + SiLU to their input (fused operand transform) "
                             "carry that work in their time; the activation FLOPs are not counted.  `achieved` uses the ALGORITHMIC "
                             "conv FLOPs of the reference's layers (SURVEY.md appendix A); the three Upsample convs (12.5 % of them) "
                             "execute 4/9 of their MACs here (sub-pixel phase decomposition, fd_conv_igemm_up): executed MACs are "
                             "7.0 % fewer than algorithmic",
                     "executed_over_algorithmic_flops": 1.0 - (199.2 / 1590.3) * (5.0 / 9.0),
                     "conv_share_of_forward": conv_s / fwd_s, "forward_ms": fwd_s * 1e3,
                     "whole_step_tflops": FWD_GF_PER_SAMPLE * DDIM_STEPS * 1e9 * value / 1e12},
    }
    if parity is not None:
        line["parity"] = parity
    if tiny is not None:
        line["config1_tiny"] = tiny
    if lib_base is not None:
        line["gpu_library_baseline"] = lib_base
    if train is not None:
        line["train"] = train
    if world == 1 and not args.skip_warp and default_wl:
        # BASELINE configs[3]: fused backward-warp + photometric / EPE microbench, 8x2x436x1024 flow over 3-channel frames,
        # L2 flushed between iterations; GB/s over the ALGORITHMIC bytes (SURVEY.md 8d: fwd 40 B/px, bwd 60 B/px)
        sys.path.insert(0, os.path.join(ROOT, "scripts"))
        import bench_warp
        wm = bench_warp.measure(iters=20, warmup=5)
        line["warp_microbench"] = {k: dict(v, frac_of_hbm_peak=round(v["GBps"] / peaks["hbm"], 3)) for k, v in wm.items()
                                   if k in ("photo_epe_fwd", "photo_epe_bwd", "backwarp_fwd", "backwarp_bwd", "splat_fwd",
                                            "splat_flowgrad")}
        line["warp_microbench"]["hbm_peak_GBps"] = peaks["hbm"]
        # The three scatter legs (forward splat, gradient of the sampled frame) are bound by the L2's reduction units, not by
        # DRAM: they issue 4 pixel-interleaved 128-bit red.global.add per pixel to white-noise addresses, and the chip executes
        # those at the rate scripts/micro/red_rate.cu measures for exactly this pattern (profiles/r2_red_rate.txt).
        red = load_red_rate()
        if red is not None:
            n_red = 4 * BATCH * H * W
            for k in ("splat_fwd", "photo_epe_bwd", "backwarp_bwd"):
                leg = line["warp_microbench"].get(k)
                if leg:
                    leg["l2_reductions"] = n_red
                    leg["l2_reduction_floor_us"] = round(n_red / red * 1e6, 1)
                    leg["frac_of_l2_reduction_rate"] = round(n_red / (leg["us"] * 1e-6) / red, 3)
            line["warp_microbench"]["l2_reductions_per_s"] = red
            line["warp_microbench"]["l2_reduction_source"] = "profiles/r2_red_rate.txt (scripts/micro/red_rate.cu on this pool's B200)"
    if cpu_base is not None:
        line["cpu_baseline"] = cpu_base
    _emit(line)


TRAIN_H, TRAIN_W = 368, 768
TRAIN_GF_PER_SAMPLE = 3.0 * 1019.83      # SURVEY.md section 8d: forward 1019.83 GF at 368x768, fwd + bwd ~ 3x


def cpu_train_baseline():
    """The reference algorithm's training step (p_losses + backward through the oracle's fp32 restatement, no optimiser)
    on the host cores at a 64x64 crop, batch 1 (SURVEY.md 8d config #3), extrapolated to 368x768 by pixel count."""
    from oracle import flowdiff_oracle as O
    from opticalflowdiffusion_b200.unet_params import UnetParams
    try:
        torch.set_num_threads(max(1, len(os.sched_getaffinity(0))))
    except Exception:  # noqa: BLE001
        pass
    torch.manual_seed(0)
    sd = {k: v.clone().requires_grad_(True) for k, v in UnetParams(64, channels=5, out_dim=2).state_dict().items()}
    sched = O.make_schedule(TIMESTEPS)
    g = torch.Generator().manual_seed(3)
    x0 = torch.rand(1, 2, 64, 64, generator=g) * 2 - 1
    cond = torch.rand(1, 3, 64, 64, generator=g) * 2 - 1
    noise = torch.randn(1, 2, 64, 64, generator=g)
    t = torch.tensor([500])
    ts = []
    for i in range(3):
        t0 = time.perf_counter()
        loss = O.p_losses_flow(sd, sched, x0, cond, t, noise)
        loss.backward()
        ts.append(time.perf_counter() - t0)
    sec = min(ts[1:])
    scale = (TRAIN_H * TRAIN_W) / (64.0 * 64.0)
    return {"value": 1.0 / (sec * scale), "unit": "samples/s", "cores": torch.get_num_threads(), "kind": "port",
            "sample": "forward + backward of ONE 64x64 crop (p_losses, target=flow) after a warm-up, extrapolated x%.0f by "
                      "pixel count to 368x768" % scale}


def run_train_leg(args, algo_cfg, rank: int, world: int, dev):
    """BASELINE configs[2]: one training step (preprocess -> q_sample -> UNet fwd -> loss -> UNet bwd -> gradient
    all-reduce -> fused clip + Adam) at 368x768 crops, batch-sharded data parallel.  Returns the "train" object."""
    import torch.distributed as dist
    from opticalflowdiffusion_b200 import FlowDiffuser, _lib
    from opticalflowdiffusion_b200.datasets import synthetic_frames
    from opticalflowdiffusion_b200.optim import GradSync, allreduce_gradients
    from opticalflowdiffusion_b200.parallel import max_over_ranks, sync_module_from_rank0
    lib = _lib.load()
    B = args.train_batch
    torch.manual_seed(0)
    algo = FlowDiffuser(algo_cfg).to(dev)
    algo.train()
    opt = algo.configure_optimizers()
    opt.max_grad_norm = 100.0                                   # experiment=matrix_flow: training.clipping = 100
    gsync = None
    if world > 1:
        sync_module_from_rank0(algo)
        if not args.no_overlap:
            # DDP's bucketed exchange, overlapped with the backward (optim.GradSync); --no-overlap = one all-reduce after it
            gsync = GradSync(opt, comm_dtype=torch.bfloat16 if args.grad_bf16 else None).attach(algo.unet)
    g = torch.Generator().manual_seed(7 + rank)
    img_h = synthetic_frames(B, TRAIN_H, TRAIN_W, seed=200 + rank).pin_memory()
    tgt_h = synthetic_frames(B, TRAIN_H, TRAIN_W, seed=300 + rank).pin_memory()
    flow_h = (torch.randn(B, 2, TRAIN_H, TRAIN_W, generator=g) * 5.0).pin_memory()
    batch_dev = tuple(t.to(dev) for t in (img_h, tgt_h, flow_h))

    def sync():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    def one_step(batch):
        first, cond, _ = algo.preprocess(batch, aug=True)          # fused GPU augmentation (augment.py)
        loss = algo.loss(first, cond, None)
        loss.backward()
        allreduce_gradients(opt)
        opt.step()
        opt.zero_grad(set_to_none=True)
        return loss

    def step_resident():
        return one_step(batch_dev)

    # e2e: every step uploads its own inputs from pinned host memory and reads the loss back; like a DataLoader with
    # pin_memory + prefetch, the upload of step i+1 runs on a copy stream while step i computes (all inside the timed region)
    copy_stream = torch.cuda.Stream(device=dev)
    pending = []

    def upload():
        copy_stream.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(copy_stream):
            b = tuple(t.to(dev, non_blocking=True) for t in (img_h, tgt_h, flow_h))
            ev = torch.cuda.Event()
            ev.record(copy_stream)
        return b, ev

    # The loss of step i is copied to pinned host memory by step i and READ by the host while step i + 1 is being enqueued
    # (a training loop logs the previous step's loss; a full device synchronisation per step would only add the host's
    # launch time of ~600 kernels to every step).  Every step's loss still reaches the host inside the timed region: the
    # last one is read after the closing synchronisation of timed().
    loss_ring = [torch.empty((), pin_memory=True) for _ in range(2)]
    loss_done = [None, None]
    e2e_state = {"i": 0, "host_losses": []}

    def step_e2e():
        if not pending:
            pending.append(upload())
        batch, ev = pending.pop()
        cur = torch.cuda.current_stream()
        cur.wait_event(ev)
        for t in batch:
            t.record_stream(cur)
        pending.append(upload())
        loss = one_step(batch)
        i = e2e_state["i"]
        slot = i & 1
        loss_ring[slot].copy_(loss.detach(), non_blocking=True)
        done = torch.cuda.Event()
        done.record(cur)
        loss_done[slot] = done
        prev = loss_done[slot ^ 1]
        if prev is not None:                       # the previous step's loss: wait for ITS copy only, then read it
            prev.synchronize()
            e2e_state["host_losses"].append(float(loss_ring[slot ^ 1]))
            loss_done[slot ^ 1] = None
        e2e_state["i"] = i + 1

    def drain_e2e():
        for slot in (0, 1):
            if loss_done[slot] is not None:
                loss_done[slot].synchronize()
                e2e_state["host_losses"].append(float(loss_ring[slot]))
                loss_done[slot] = None

    def timed(fn, steps, finish=None):
        sync()
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        for _ in range(steps):
            fn()
        if finish is not None:
            finish()                                # e2e: the last step's loss is on the host before the clock stops
        e.record()
        sync()
        return max_over_ranks(s.elapsed_time(e) * 1e-3, device=dev)

    for _ in range(3):
        first_loss = step_resident()
    steps = args.steps
    l0 = lib.fd_launch_count()
    t_res = timed(step_resident, steps)
    launches = int(lib.fd_launch_count() - l0)
    for _ in range(3):                             # warm-up of the e2e path itself: the copy stream's allocator pool, pinned rings
        step_e2e()
    drain_e2e()
    e2e_state["host_losses"].clear()
    t_e2e = timed(step_e2e, steps, finish=drain_e2e)
    assert len(e2e_state["host_losses"]) == steps, "every e2e step must deliver its loss to the host"
    # phase split of one step (events on the launching stream)
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
    ev_aug = torch.cuda.Event(enable_timing=True)
    ev_aug.record()
    first, cond, _ = algo.preprocess(batch_dev, aug=True)
    ev[0].record()
    loss = algo.loss(first, cond, None)
    ev[1].record()
    loss.backward()
    ev[2].record()
    allreduce_gradients(opt)
    opt.step()
    opt.zero_grad(set_to_none=True)
    ev[3].record()
    torch.cuda.synchronize()
    cpu = None
    if world == 1 and rank == 0 and not args.no_cpu_baseline:
        cpu = cpu_train_baseline()
    samples = world * B * steps
    value = samples / t_res
    peak_mem = torch.cuda.max_memory_allocated(dev) / 2 ** 30
    return {"metric": "train samples/sec @368x768", "value": value, "unit": "samples/s", "ms_per_step": t_res / steps * 1e3,
            "batch_per_gpu": B, "global_batch": B * world, "steps": steps, "warmup": 3, "dtype": "bf16 activations / fp32 master weights, grads, Adam",
            "e2e": {"value": samples / t_e2e, "unit": "samples/s", "h2d_bytes_per_step": 4 * (img_h.numel() + tgt_h.numel() + flow_h.numel()),
                    "d2h_bytes_per_step": 4},
            "gpu_launches": launches, "loss_first": float(first_loss.detach()), "loss_last": float(loss.detach()),
            "phases_ms": {"augment+preprocess": ev_aug.elapsed_time(ev[0]), "forward+loss": ev[0].elapsed_time(ev[1]), "backward": ev[1].elapsed_time(ev[2]),
                          "allreduce+clip+adam": ev[2].elapsed_time(ev[3])},
            "tensor_tflops": TRAIN_GF_PER_SAMPLE * value / 1e3 / world, "peak_mem_gib": peak_mem, "cpu_baseline": cpu,
            "grad_exchange": ({"kind": "bucketed all-reduce overlapped with the backward (optim.GradSync)",
                               "buckets": gsync.buckets_last_backward, "bytes": gsync.bytes_last_backward,
                               "wire_dtype": "bf16" if args.grad_bf16 else "f32"} if gsync is not None else
                              {"kind": "none (1 GPU)" if world == 1 else "one all-reduce after the backward"}),
            "config": "flow_diffuser training step, target=flow, synthetic 368x768 crops, augmentation ON (GpuAugmentor: "
                      "reference Augmentor semantics, decisions on the host, arithmetic in 4 launches), Adam lr 1e-5 wd 1e-6, clip 100, "
                      "gradient all-reduce over NCCL when n_gpus > 1"}


_REAL_STDOUT = None


def _emit(obj):
    """The one JSON line of this run, on the process's original stdout."""
    text = json.dumps(obj) + "\n"
    sys.stdout.flush()
    if _REAL_STDOUT is None:
        sys.stdout.write(text)
        sys.stdout.flush()
    else:
        os.write(_REAL_STDOUT, text.encode())


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference", "torch-gpu"])
    ap.add_argument("--config", default="ddim50_436x1024", choices=sorted(WORKLOADS),
                    help="workload: BASELINE configs[1] (default, the headline) or configs[4] (matrix_flow resolution)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-gpu-baseline", action="store_true", help="omit the PyTorch-eager (cuDNN / cuBLAS) bar on the same GPU")
    ap.add_argument("--no-overlap", action="store_true", help="training leg: one all-reduce after the backward instead of GradSync")
    ap.add_argument("--grad-bf16", action="store_true", help="training leg: exchange gradient buckets as bf16")
    ap.add_argument("--graph", type=int, default=1, help="replay the DDIM loop as one CUDA graph (1) or launch eagerly (0)")
    ap.add_argument("--train-batch", type=int, default=8, help="per-GPU batch of the training leg (368x768 crops)")
    ap.add_argument("--skip-warp", action="store_true", help="omit the warp + photometric/EPE microbench (BASELINE configs[3])")
    ap.add_argument("--skip-train", action="store_true", help="omit the training leg (BASELINE configs[2])")
    ap.add_argument("--skip-sample", action="store_true", help="training leg only (debug; prints a reduced line)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed sampling steps, write what the last one computed as DIR/<name>.npy (float32; "
                         "an output larger than 2^23 elements as a fixed, seeded sample of 2^21 of them)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "ours" or args.skip_sample):
        ap.error("--dump-outputs writes the outputs of this implementation's sampling steps (--impl ours, no --skip-sample)")
    # stdout carries exactly ONE JSON line: libraries that chat on file descriptor 1 (NCCL prints its version banner there)
    # are sent to stderr for the duration of the run; _emit() writes the result to the real stdout
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)
    rank = int(os.environ.get("RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    local_rank = int(os.environ.get("LOCAL_RANK", 0))
    select_workload(args.config)
    if args.impl == "reference":
        run_reference(args, rank)
        return
    if args.impl == "torch-gpu":
        run_torch_gpu(args, rank, local_rank)
        return
    run_ours(args, rank, world, local_rank)
    if world > 1:
        import torch.distributed as dist
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
