"""TEST INFRASTRUCTURE ONLY -- CPU restatement of the multistep DPM-Solver++ sampler (``sampler: dpmpp``).

Not in the reference: written from the formulas of Lu et al., "DPM-Solver++: Fast Solver for Guided Sampling of Diffusion
Probabilistic Models" (arXiv:2211.01095), data prediction, deterministic, multistep, on the reference's DDIM grid and fp32
schedule (``flowdiff_oracle.ddim_times`` / ``make_schedule``), independently of the package.  It is pinned by its order-1
identity with ``flowdiff_oracle.ddim_sample``, by the closed-form solution for a constant prediction and by its convergence
order (tests/test_dpmpp_oracle.py).  Like flowdiff_oracle, it is imported by tests only.
"""
from __future__ import annotations

import math
from typing import Optional, Sequence, Tuple

import torch

from .flowdiff_oracle import ddim_times, unet_forward

Tensor = torch.Tensor


def _dpmpp_formula(sched, times: Sequence[int], i: int, order: int, x, d0, d1, d2):
    """The multistep DPM-Solver++ update (Lu et al., arXiv:2211.01095, data prediction) written as in the paper, in float64
    on scalars: a step from s = times[i] to t = times[i+1], D1 / D2 the predictions at times[i-1] / times[i-2]."""
    def asl(tt):
        a = float(sched["alphas_cumprod"][tt])
        return math.sqrt(a), math.sqrt(1.0 - a), math.log(math.sqrt(a)) - math.log(math.sqrt(1.0 - a))

    s, t = times[i], times[i + 1]
    _, sg_s, lam_s = asl(s)
    al_t, sg_t, lam_t = asl(t)
    h = lam_t - lam_s
    phi1 = math.expm1(-h)
    out = (sg_t / sg_s) * x - al_t * phi1 * d0
    if order == 1:
        return out
    h0 = lam_s - asl(times[i - 1])[2]
    r0 = h0 / h
    if order == 2:
        return out - 0.5 * al_t * phi1 * (d0 - d1) / r0
    h1 = asl(times[i - 1])[2] - asl(times[i - 2])[2]
    r1 = h1 / h
    phi2 = phi1 / h + 1.0
    phi3 = phi2 / h - 0.5
    e0, e1 = (d0 - d1) / r0, (d1 - d2) / r1
    dd1 = e0 + r0 / (r0 + r1) * (e0 - e1)
    dd2 = (e0 - e1) / (r0 + r1)
    return out + al_t * phi2 * dd1 - al_t * phi3 * dd2


def dpmpp_coeffs(sched, times: Sequence[int], i: int, order: int) -> Tuple[float, float, float, float, int]:
    """(cx, c0, c1, c2, last) of step i (float64): the update read off as a linear map, one unit input at a time.
    Order min(order, i + 1); the final step (times[i+1] < 0) returns D0 and is (0, 1, 0, 0, 1)."""
    if times[i + 1] < 0:
        return 0.0, 1.0, 0.0, 0.0, 1
    k = min(order, i + 1)
    unit = ((1.0, 0.0, 0.0, 0.0), (0.0, 1.0, 0.0, 0.0), (0.0, 0.0, 1.0, 0.0), (0.0, 0.0, 0.0, 1.0))
    cx, c0, c1, c2 = (_dpmpp_formula(sched, times, i, k, *u) for u in unit)
    return cx, c0, c1, c2, 0


def dpmpp_update(x: Tensor, model_out: Tensor, d1: Optional[Tensor], d2: Optional[Tensor], coeffs) -> Tuple[Tensor, Tensor]:
    """One DPM-Solver++ step in the kernel's op order: D0 = clamp(model_out, -1, 1);
    x_next = ((cx*x + c0*D0) + c1*D1) + c2*D2 with coefficients rounded to x's dtype; a term with a zero coefficient is
    not evaluated (a NaN in unused history stays out); last -> D0.  Returns (next x, D0)."""
    cx, c0, c1, c2, last = coeffs
    d0 = torch.clamp(model_out, -1.0, 1.0)
    if last:
        return d0, d0
    c = [torch.tensor(v, dtype=x.dtype) for v in (cx, c0, c1, c2)]
    out = c[0] * x + c[1] * d0
    if c[2].item() != 0.0:
        out = out + c[2] * d1
    if c[3].item() != 0.0:
        out = out + c[3] * d2
    return out, d0


def dpmpp_sample(sd, sched, x_T: Tensor, cond: Tensor, total_timesteps: int, sampling_timesteps: int, order: int,
                 prefix: str = "", return_all: bool = False, model=None):
    """Multistep DPM-Solver++ of the given order on the DDIM grid from a supplied x_T; the loop of ``ddim_sample`` with
    ``dpmpp_update`` in place of ``ddim_update``.  return_all -> (trajectory with time at dim 1, list of the D0s)."""
    times = ddim_times(total_timesteps, sampling_timesteps)
    x = x_T
    traj, ds = [x], []
    model = model or (lambda xx, cc, tt: unet_forward(sd, xx, cc, tt, prefix))
    for i, time in enumerate(times[:-1]):
        t = torch.full((x.shape[0],), time, dtype=torch.long, device=x.device)
        out = model(x, cond, t)
        coeffs = dpmpp_coeffs(sched, times, i, order)
        x, d0 = dpmpp_update(x, out, ds[-1] if i >= 1 else None, ds[-2] if i >= 2 else None, coeffs)
        traj.append(x)
        ds.append(d0)
    if return_all:
        return torch.stack(traj, dim=1), ds
    return x
