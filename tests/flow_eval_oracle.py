"""fp64 restatement of ``fd_flow_eval`` (include/flowdiff.h) and of ``evaluation.FlowScores.metrics``, on CPU tensors."""
import math

import torch

UNKNOWN = 1e9


def flow_eval(samples, scale, gt=None, gt_limit=None):
    """-> (mean px (B,2,H,W), spread px (B,H,W), per_image (B, 8+K), EPE of the mean flow px (B,H,W) or None), all fp64."""
    s = samples.double().cpu() * float(scale)                     # (B, K, 2, H, W) px
    B, K, _, H, W = s.shape
    mean = s.sum(1) / K
    spread = ((s - mean[:, None]) ** 2).sum(2).mean(1).sqrt()
    limit = float(scale if gt_limit is None else gt_limit)
    rows = torch.zeros(B, 8 + K, dtype=torch.float64)
    zero = torch.zeros((), dtype=torch.float64)
    if gt is None:
        rows[:, 0] = H * W
        rows[:, 6] = spread.flatten(1).sum(1)
        return mean, spread, rows, None
    g = gt.double().cpu()
    valid = (g.abs() < UNKNOWN).all(1)                            # NaN and +-inf fail the comparison
    epe = (mean - g).pow(2).sum(1).sqrt()
    epe_k = (s - g[:, None]).pow(2).sum(2).sqrt()                  # (B, K, H, W)
    mag = g.pow(2).sum(1).sqrt()

    def total(x):
        return torch.where(valid, x, zero).flatten(1).sum(1)

    rows[:, 0] = valid.flatten(1).sum(1)
    rows[:, 1] = total(epe)
    rows[:, 2] = total((epe < 1).double())
    rows[:, 3] = total((epe < 3).double())
    rows[:, 4] = total((epe < 5).double())
    rows[:, 5] = total(((epe > 3) & (epe > 0.05 * mag)).double())
    rows[:, 6] = total(spread)
    rows[:, 7] = total((g.abs().amax(1) > limit).double())
    for k in range(K):
        rows[:, 8 + k] = total(epe_k[:, k])
    return mean, spread, rows, torch.where(valid, epe, torch.full_like(epe, math.nan))


def metrics(rows, num_samples):
    """Dataset metrics of per-image rows (n, 8 + K): pixel-weighted sums, best of K chosen per image."""
    rows = rows.double()
    K = int(num_samples)
    n = float(rows[:, 0].sum())
    tot = rows.sum(0)

    def rate(x):
        return float(x) / n if n > 0 else math.nan

    best = sum(float(r[8:].min()) for r in rows)
    return {"epe": rate(tot[1]), "1px": rate(tot[2]), "3px": rate(tot[3]), "5px": rate(tot[4]), "fl": rate(tot[5]),
            "epe_sample": rate(tot[8:].sum() / K), "epe_best_of_k": rate(best), "spread": rate(tot[6]),
            "gt_beyond_flow_max": rate(tot[7]), "pixels": int(n), "images": rows.shape[0], "num_samples": K}
