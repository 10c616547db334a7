"""Scoring sampled flows against the ground truth.

The model is a conditional generator: for one frame it samples one plausible motion per draw of x_T.  A single sample is a
noisy, pessimistic estimate of its quality, so an image is scored with K samples at once (``fd_flow_eval``, one pass over
them): the end-point error (EPE) of their mean, the EPE of every sample and their per-pixel spread, an uncertainty map.

``score_flows`` launches the kernel on one batch; ``FlowScores`` gathers its per-image rows over a dataset (and over ranks)
into metrics that are pixel-weighted like RAFT's Sintel evaluation: sums over all images divided by the total number of
valid pixels.  Metrics are taken against the raw ground truth, not the ``flow_max``-clamped training target.

Seeding (``sample_seed``): x_T of sample k of the image with dataset index i is drawn from a device generator seeded with
``((seed & 0xFFFF) << 48) | ((i & 0xFFFFFFFF) << 16) | k``, so an image's samples do not depend on the batch it is in, the
chunking of the sampler calls or the number of ranks.
"""
from __future__ import annotations

import math
from typing import Dict, Optional, Tuple

import torch
import torch.distributed as dist

from . import _lib

Tensor = torch.Tensor

FIXED_COLUMNS = 8          # per_image columns before the K per-sample EPE sums (include/flowdiff.h, fd_flow_eval)
MAX_SAMPLES = 1 << 16      # k takes the low 16 bits of the seed


def sample_seed(seed: int, index: int, k: int) -> int:
    """Generator seed of x_T for sample ``k`` (0 <= k < 65536) of the image with dataset index ``index``."""
    if not 0 <= k < MAX_SAMPLES:
        raise ValueError(f"sample index {k} outside [0, {MAX_SAMPLES})")
    return ((int(seed) & 0xFFFF) << 48) | ((int(index) & 0xFFFFFFFF) << 16) | int(k)


def score_flows(samples: Tensor, flow_max: float, gt: Optional[Tensor] = None) -> Tuple[Tensor, Tensor, Tensor]:
    """K sampled flows per image -> ``(mean_px (B, 2, H, W), spread_px (B, H, W), per_image fp64 (B, 8 + K))``.

    ``samples``: fp32 CUDA (B, K, 2, H, W) in the sampler's normalised units (pixels / ``flow_max``).  ``gt``: fp32 CUDA
    (B, 2, H, W) in pixels, or None (then every pixel is valid and only the pixel count and spread sum are non-zero).
    Column 7 counts the valid pixels whose ground truth exceeds ``flow_max`` in a component: training clamps its targets
    there, so the model cannot reach them.
    The per_image columns are documented at ``fd_flow_eval`` in include/flowdiff.h.  Nothing is synchronised."""
    _lib.require_cuda(samples, gt)
    if samples.dim() != 5 or samples.shape[2] != 2:
        raise ValueError(f"samples must be (B, K, 2, H, W), got {tuple(samples.shape)}")
    B, K, _, H, W = samples.shape
    if min(B, K, H, W) == 0:
        raise ValueError(f"samples has an empty dimension: {tuple(samples.shape)}")
    if samples.dtype != torch.float32 or (gt is not None and gt.dtype != torch.float32):
        raise TypeError("samples and gt must be float32")
    if gt is not None:
        if tuple(gt.shape) != (B, 2, H, W):
            raise ValueError(f"gt must be {(B, 2, H, W)}, got {tuple(gt.shape)}")
        if gt.device != samples.device:
            raise ValueError("samples and gt are on different devices")
        gt = gt.contiguous()
    samples = samples.contiguous()
    lib = _lib.load()
    dev = samples.device
    mean = torch.empty((B, 2, H, W), device=dev, dtype=torch.float32)
    spread = torch.empty((B, H, W), device=dev, dtype=torch.float32)
    per_image = torch.empty((B, FIXED_COLUMNS + K), device=dev, dtype=torch.float64)
    ws = torch.empty(lib.fd_flow_eval_workspace_floats(B, K, H, W), device=dev, dtype=torch.float32)
    with torch.cuda.device(dev):
        _lib.check(lib.fd_flow_eval(_lib.ptr(samples), float(flow_max), _lib.ptr(gt), float(flow_max), _lib.ptr(mean),
                                    _lib.ptr(spread), _lib.ptr(per_image), _lib.ptr(ws), B, K, H, W, _lib.stream()))
    return mean, spread, per_image


def metrics_from_totals(totals, num_samples: int) -> Dict[str, float]:
    """Dataset metrics from the reduced sums (``FlowScores.totals`` layout): index c < 8 is per_image column c summed over
    images, 8 the sum over k of column 8 + k, 9 the sum over images of the best sample's EPE sum, 10 the image count."""
    t = [float(v) for v in totals]
    n, K = t[0], int(num_samples)

    def rate(x):
        return x / n if n > 0 else math.nan

    return {"epe": rate(t[1]), "1px": rate(t[2]), "3px": rate(t[3]), "5px": rate(t[4]), "fl": rate(t[5]),
            "epe_sample": rate(t[8] / K), "epe_best_of_k": rate(t[9]), "spread": rate(t[6]),
            "gt_beyond_flow_max": rate(t[7]), "pixels": int(n), "images": int(t[10]), "num_samples": K}


class FlowScores:
    """Dataset-level flow metrics from ``score_flows``' per-image rows.

    ``update`` keeps the rows on the device (no host synchronisation per batch); ``metrics`` sums them, applies ONE
    SUM all-reduce in fp64 when a process group of more than one rank is active (every rank must call it, also with no
    rows), and returns the same dict on every rank:

    * ``epe``, ``1px``, ``3px``, ``5px``, ``fl``: of the mean flow of the K samples;
    * ``epe_sample``: the expected EPE of a single sample, sum over k of the per-sample EPE sums / (K * pixels);
    * ``epe_best_of_k``: per IMAGE, the sample with the lowest mean EPE (a per-pixel minimum would flatter the model);
    * ``spread``: the mean per-pixel spread of the samples, px;
    * ``gt_beyond_flow_max``: fraction of valid pixels whose ground truth exceeds ``flow_max`` in a component;
    * ``pixels`` (valid), ``images``, ``num_samples``.

    Rates are sums over all images divided by the total valid pixel count."""

    def __init__(self, num_samples: int, device=None):
        self.num_samples = int(num_samples)
        self.device = device
        self.rows = []

    def update(self, per_image: Tensor) -> None:
        if per_image.dim() != 2 or per_image.shape[1] != FIXED_COLUMNS + self.num_samples:
            raise ValueError(f"per_image must be (n, {FIXED_COLUMNS + self.num_samples}), got {tuple(per_image.shape)}")
        if per_image.dtype != torch.float64:
            raise TypeError("per_image must be float64")
        self.rows.append(per_image.detach())
        if self.device is None:
            self.device = per_image.device

    def totals(self) -> Tensor:
        """This rank's sums (layout of ``metrics_from_totals``), fp64 on ``self.device``."""
        K = self.num_samples
        rows = torch.cat(self.rows) if self.rows else \
            torch.zeros((0, FIXED_COLUMNS + K), dtype=torch.float64, device=self.device)
        per_sample = rows[:, FIXED_COLUMNS:]
        best = per_sample.amin(dim=1).sum() if rows.shape[0] else rows.new_zeros(())
        return torch.cat((rows[:, :FIXED_COLUMNS].sum(0), per_sample.sum().view(1), best.view(1),
                          rows.new_full((1,), float(rows.shape[0]))))

    def metrics(self) -> Dict[str, float]:
        t = self.totals()
        if dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1:
            dist.all_reduce(t, op=dist.ReduceOp.SUM)
        return metrics_from_totals(t.tolist(), self.num_samples)
