"""-m gpu: fd_flow_eval against the fp64 oracle (tests/flow_eval_oracle.py), and the evaluation path end to end.

Kernel tolerances (fp32 against fp64): mean flow and spread |got - ref| <= 1e-6 * K * flow_max * max|samples| (K fp32 adds
of values up to flow_max * max|samples|); EPE and spread sums relative 1e-5 (each warp partial adds at most 8 + 5 fp32
terms per lane, about 1e-6 relative, before the fp64 sums); valid-pixel count and the beyond-flow_max count exact;
threshold counts exact except for pixels whose fp64 EPE lies within 1e-5 px of a threshold.

End to end (64x128, seeded random weights, DDIM-4): for target=flow, sample_flows with max_batch=1 is bitwise what sample()
returns for one image and the documented x_T.  For target=joint the UNet input carries the frame forward-splatted along the
current flow, which accumulates with float atomics, so two identical calls already differ: it is compared within
BATCH_TOL.  Batched sampling is compared within BATCH_TOL (normalised flow units) and the metrics of runs that batch the
images differently within METRIC_RTOL / METRIC_ATOL: batch invariance of the UNet kernels is not established.  Measured on a
B200 (1000 W limit): batched vs one image at a time, max |diff| 1.7e-2 (target=flow) and 0.54 (target=joint); metrics,
evaluate vs the manual loop 2e-9 relative, batch 2 vs batch 3 1.8e-5, two ranks vs one 0."""
import math
import os
import socket

import pytest
import torch
import torch.multiprocessing as mp

import flow_eval_oracle as OR
from opticalflowdiffusion_b200 import _lib
from opticalflowdiffusion_b200.evaluation import sample_seed, score_flows

pytestmark = pytest.mark.gpu

FLOW_MAX = 20.0
BATCH_TOL = {"flow": 5e-2, "joint": 1.0}    # max |flow| difference, normalised units, batched vs one-image sampling
METRIC_RTOL = 2e-3        # relative, metrics of differently batched evaluations
METRIC_ATOL = 2e-3        # absolute, rates in [0, 1]


def _inputs(B, K, H, W, seed, offset=0, special=True):
    g = torch.Generator().manual_seed(seed)
    s = torch.randn(B, K, 2, H, W, generator=g) * 0.25
    gt = torch.randn(B, 2, H, W, generator=g) * 6.0
    gt[:, :, ::7, ::5] *= 5.0                                   # some pixels beyond flow_max and far from the mean
    if special:
        flat = gt.view(B, 2, -1)
        n = flat.shape[-1]
        for j, v in enumerate((math.nan, math.inf, -math.inf, 1e9, -1e9)):
            flat[:, j % 2, (3 + 11 * j) % n] = v
        flat[:, 0, (5 * n) // 7] = 1e9 - 64.0                    # finite, just below the marker: valid
    dev_s = torch.empty(s.numel() + offset, device="cuda")[offset:].view_as(s)
    dev_g = torch.empty(gt.numel() + offset, device="cuda")[offset:].view_as(gt)
    dev_s.copy_(s)
    dev_g.copy_(gt)
    return s, gt, dev_s, dev_g


def _near(epe, t, eps=1e-5):
    return ((epe - t).abs() < eps).flatten(1).sum(1).double()


def _check_against_oracle(s, gt, dev_s, dev_g):
    K = s.shape[1]
    mean, spread, rows = score_flows(dev_s, FLOW_MAX, dev_g)
    torch.cuda.synchronize()
    m_ref, sp_ref, r_ref, epe = OR.flow_eval(s, FLOW_MAX, gt)
    tol = 1e-6 * K * FLOW_MAX * float(s.abs().max())
    worst = {"mean": float((mean.cpu().double() - m_ref).abs().max()), "spread": float((spread.cpu().double() - sp_ref).abs().max())}
    assert worst["mean"] <= tol and worst["spread"] <= tol, (worst, tol)
    rows = rows.cpu()
    assert torch.equal(rows[:, 0], r_ref[:, 0]) and torch.equal(rows[:, 7], r_ref[:, 7])
    sums = [1, 6] + list(range(8, 8 + K))
    rel = ((rows[:, sums] - r_ref[:, sums]).abs() / r_ref[:, sums].abs().clamp_min(1e-30)).max()
    assert rel <= 1e-5, float(rel)
    mag = gt.double().pow(2).sum(1).sqrt()
    for col, t in ((2, 1.0), (3, 3.0), (4, 5.0)):
        assert ((rows[:, col] - r_ref[:, col]).abs() <= _near(epe, t)).all(), col
    fl_near = _near(epe, 3.0) + ((epe - 0.05 * mag).abs() < 1e-5).flatten(1).sum(1)
    assert ((rows[:, 5] - r_ref[:, 5]).abs() <= fl_near).all()
    print(f"flow_eval K={K} shape={tuple(s.shape)}: max|mean err| {worst['mean']:.3e} px, max|spread err| "
          f"{worst['spread']:.3e} px (tol {tol:.1e}), max rel sum err {float(rel):.3e}")
    return mean, spread, rows


@pytest.mark.parametrize("B,K,H,W,offset", [
    (2, 1, 7, 13, 0), (3, 2, 5, 31, 0), (1, 3, 33, 45, 0), (2, 8, 17, 64, 0),     # ragged, W % 4 != 0, and the 16-byte path
    (2, 3, 64, 100, 0), (2, 8, 40, 128, 0),                                       # several blocks per image
    (2, 3, 40, 128, 1),                                                           # W % 4 == 0 at an odd float offset: scalar
])
def test_kernel_matches_oracle(B, K, H, W, offset):
    s, gt, dev_s, dev_g = _inputs(B, K, H, W, seed=B * 1000 + K * 100 + W + offset, offset=offset)
    _check_against_oracle(s, gt, dev_s, dev_g)


def test_kernel_matches_oracle_at_benchmark_shape():
    s, gt, dev_s, dev_g = _inputs(8, 4, 436, 1024, seed=11)
    _check_against_oracle(s, gt, dev_s, dev_g)


def test_without_ground_truth():
    s, _, dev_s, _ = _inputs(2, 3, 19, 36, seed=5)
    mean, spread, rows = score_flows(dev_s, FLOW_MAX)
    m_ref, sp_ref, r_ref, _ = OR.flow_eval(s, FLOW_MAX, None)
    rows = rows.cpu()
    assert torch.equal(rows[:, 0], r_ref[:, 0])
    assert float(((rows[:, 6] - r_ref[:, 6]) / r_ref[:, 6]).abs().max()) <= 1e-5
    assert rows[:, 1:6].abs().sum() == 0 and rows[:, 7:].abs().sum() == 0
    tol = 1e-6 * 3 * FLOW_MAX * float(s.abs().max())
    assert (mean.cpu().double() - m_ref).abs().max() <= tol and (spread.cpu().double() - sp_ref).abs().max() <= tol


@pytest.mark.parametrize("W", [64, 63])
def test_deterministic_and_any_workspace(W):
    """Two launches give the same bits; the workspace may hold anything (NaN here); mean / spread outputs are optional."""
    _, _, dev_s, dev_g = _inputs(3, 4, 50, W, seed=9)
    a = score_flows(dev_s, FLOW_MAX, dev_g)
    b = score_flows(dev_s, FLOW_MAX, dev_g)
    for x, y in zip(a, b):
        assert torch.equal(x, y)
    lib = _lib.load()
    ws = torch.full((lib.fd_flow_eval_workspace_floats(3, 4, 50, W),), math.nan, device="cuda")
    rows = torch.full_like(a[2], math.nan)
    _lib.check(lib.fd_flow_eval(_lib.ptr(dev_s), FLOW_MAX, _lib.ptr(dev_g), FLOW_MAX, None, None, _lib.ptr(rows),
                                _lib.ptr(ws), 3, 4, 50, W, _lib.stream()))
    assert torch.equal(rows, a[2])


def test_samples_equal_to_ground_truth_score_zero():
    """flow_max a power of two and K = 2 keep scale * (gt / scale) and the mean of two equal samples exact in fp32."""
    fm = 16.0
    gt = (torch.randn(2, 2, 24, 40, generator=torch.Generator().manual_seed(4)) * 7).cuda()
    s = (gt / fm)[:, None].repeat(1, 2, 1, 1, 1).contiguous()
    mean, spread, rows = score_flows(s, fm, gt)
    assert torch.equal(mean, gt) and torch.equal(spread, torch.zeros_like(spread))
    rows = rows.cpu()
    assert (rows[:, [1, 5, 6, 8, 9]] == 0).all() and torch.equal(rows[:, 2], rows[:, 0])
    assert rows[:, 0].tolist() == [24.0 * 40] * 2


# ------------------------------------------------------------------ end to end
def _algo(target, extra=()):
    from opticalflowdiffusion_b200 import FlowDiffuser
    from opticalflowdiffusion_b200.config import compose
    torch.manual_seed(0)
    over = [f"algorithm.target={target}", "algorithm.sampling_timesteps=4", "algorithm.zero_init=false", *extra]
    return FlowDiffuser(compose(over).algorithm).cuda()


def _one_by_one(algo, cond, ids, K, seed):
    """sample() on one image and one documented x_T at a time."""
    out = []
    keep = algo.return_all_timesteps
    algo.return_all_timesteps = False
    try:
        for b, i in enumerate(ids):
            for k in range(K):
                g = torch.Generator(device="cuda").manual_seed(sample_seed(seed, i, k))
                x_T = torch.randn((algo.model.channels,) + tuple(cond.shape[-2:]), generator=g, device="cuda")[None]
                _, flow = algo.sample(cond[b:b + 1], cond.new_empty((1, 2, 1, 1)), x_T=x_T)
                out.append(flow[-1] if algo.target == "target" else flow)
    finally:
        algo.return_all_timesteps = keep
    return torch.cat(out).view(len(ids), K, 2, *cond.shape[-2:])


@pytest.mark.parametrize("target,extra", [("flow", ()), ("flow", ("algorithm.use_cuda_graph=true",)), ("joint", ())])
def test_sample_flows_matches_sample(target, extra):
    from opticalflowdiffusion_b200.datasets import synthetic_frames
    algo = _algo(target, extra)
    cond = (2 * synthetic_frames(3, 64, 128, seed=2) - 1).cuda()
    ids, K, seed = [4, 9, 2], 2, 3
    ref = _one_by_one(algo, cond, ids, K, seed)
    one = algo.sample_flows(cond, ids, K, seed, max_batch=1)
    assert one.shape == (3, K, 2, 64, 128) and torch.isfinite(one).all()
    if target == "flow":
        assert torch.equal(one, ref)
    else:           # the forward splat of the UNet input accumulates with float atomics: two identical calls differ
        diff = float((one - ref).abs().max())
        print(f"sample_flows {target}: max_batch=1 vs sample(): max|diff| {diff:.3e} (normalised)")
        assert diff <= BATCH_TOL[target]
    assert not torch.equal(one[:, 0], one[:, 1])
    batched = algo.sample_flows(cond, ids, K, seed)
    diff = float((batched - ref).abs().max())
    print(f"sample_flows {target} {extra}: default chunking vs one image at a time: max|diff| {diff:.3e} (normalised)")
    assert diff <= BATCH_TOL[target]


OV = ["algorithm.target=flow", "algorithm.sampling_timesteps=4", "algorithm.zero_init=false", "dataset.height=64",
      "dataset.width=128", "dataset.length=5", "experiment.evaluation.num_samples=2", "experiment.evaluation.seed=1",
      "experiment.evaluation.data.batch_size=2"]


def _experiment(extra=()):
    from opticalflowdiffusion_b200.config import compose
    from opticalflowdiffusion_b200.experiments import build_experiment
    torch.manual_seed(0)
    return build_experiment(compose(OV + list(extra)), None, None)


def _close(a, b):
    for k in b:
        if isinstance(b[k], int):
            assert a[k] == b[k], k
        elif k in ("1px", "3px", "5px", "fl", "gt_beyond_flow_max"):
            assert abs(a[k] - b[k]) <= METRIC_ATOL, (k, a[k], b[k])
        else:
            assert a[k] == pytest.approx(b[k], rel=METRIC_RTOL), k


def _worst(a, b):
    return max(abs(a[k] - b[k]) / max(abs(b[k]), 1e-30) for k in b if not isinstance(b[k], int))


def test_evaluate_equals_manual_loop_and_is_batch_size_free():
    exp = _experiment()
    got = exp.evaluate()
    algo, ds = exp.algo, exp._build_dataset("validation")
    rows = []
    for i in range(len(ds)):
        img, _, flow = ds[i]
        cond = (2 * img[None] - 1).cuda()
        flows = _one_by_one(algo, cond, [i], 2, 1)
        rows.append(OR.flow_eval(flows.cpu(), FLOW_MAX, flow[None])[2])
    want = OR.metrics(torch.cat(rows), 2)
    assert got["images"] == 5 and got["pixels"] == 5 * 64 * 128 and got["num_samples"] == 2
    assert all(math.isfinite(v) for v in got.values())
    print(f"evaluate vs manual loop: worst relative metric difference {_worst(got, want):.3e}")
    _close(got, want)
    got3 = _experiment(["experiment.evaluation.data.batch_size=3"]).evaluate()
    print(f"evaluate batch 2 vs batch 3: worst relative metric difference {_worst(got3, got):.3e}")
    _close(got3, got)


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _worker(rank, world, port, q):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world), LOCAL_RANK="0",
                      FD_DIST_BACKEND="gloo")
    import torch.distributed as dist
    torch.manual_seed(100 + rank)                # different init per rank: evaluate must broadcast rank 0's weights
    from opticalflowdiffusion_b200.config import compose
    from opticalflowdiffusion_b200.experiments import build_experiment
    if rank == 0:
        torch.manual_seed(0)
    exp = build_experiment(compose(OV), None, None)
    q.put((rank, exp.evaluate()))
    dist.barrier()
    dist.destroy_process_group()


def test_two_rank_evaluate_equals_one_rank():
    single = _experiment().evaluate()
    world = 2
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, world, port, q)) for r in range(world)]
    for p in procs:
        p.start()
    out = sorted((q.get(timeout=600) for _ in range(world)), key=lambda r: r[0])
    for p in procs:
        p.join(120)
        assert p.exitcode == 0
    (_, m0), (_, m1) = out
    assert m0 == m1 and m0["images"] == 5
    print(f"evaluate 2 ranks (3 / 2 images) vs 1 rank: worst relative metric difference {_worst(m0, single):.3e}")
    _close(m0, single)
