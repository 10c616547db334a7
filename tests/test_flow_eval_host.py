"""Host side of the flow evaluation (no GPU): the fp64 oracle on hand-built tables, FlowScores' reduction and its
world-size-2 all-reduce, the x_T seeding of FlowDiffuser.sample_flows, the rank shards and the evaluate task's config."""
import math
import os
import socket

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

import flow_eval_oracle as OR
from opticalflowdiffusion_b200 import _lib, evaluation, parallel


def _rows(table):
    return torch.tensor(table, dtype=torch.float64)


def test_metrics_are_pixel_weighted():
    # image 0: 1 valid pixel with EPE 10; image 1: 3 valid pixels with EPE 1 each -> 13 / 4, not mean(10, 1) = 5.5
    rows = _rows([[1, 10, 0, 0, 0, 1, 2, 0, 10],
                  [3, 3, 0, 3, 3, 0, 3, 1, 3]])
    m = OR.metrics(rows, 1)
    assert m["epe"] == 13 / 4 and m["3px"] == 3 / 4 and m["fl"] == 1 / 4 and m["spread"] == 5 / 4
    assert m["gt_beyond_flow_max"] == 1 / 4 and m["pixels"] == 4 and m["images"] == 2
    fs = evaluation.FlowScores(1)
    fs.update(rows[:1])
    fs.update(rows[1:])
    assert fs.metrics() == m


def test_best_of_k_is_chosen_per_image():
    """Two pixels, two samples: sample 0 is exact at pixel 0 and 4 px off at pixel 1, sample 1 the other way round
    with 3 px.  Per pixel the minimum would be 0; per image the best sample is sample 1 with mean EPE 1.5."""
    gt = torch.zeros(1, 2, 1, 2)
    s = torch.zeros(1, 2, 2, 1, 2)
    s[0, 0, 0, 0, 1] = 4.0
    s[0, 1, 0, 0, 0] = 3.0
    _, _, rows, _ = OR.flow_eval(s, 1.0, gt)
    assert rows[0, 8:].tolist() == [4.0, 3.0]
    m = OR.metrics(rows, 2)
    assert m["epe_best_of_k"] == 1.5 and m["epe_sample"] == 7 / 4 and m["epe"] == 3.5 / 2
    fs = evaluation.FlowScores(2)
    fs.update(rows)
    assert fs.metrics() == m


def test_single_sample_scores_agree():
    g = torch.Generator().manual_seed(0)
    s = torch.randn(3, 1, 2, 5, 7, generator=g)
    gt = torch.randn(3, 2, 5, 7, generator=g) * 20
    _, spread, rows, _ = OR.flow_eval(s, 20.0, gt)
    assert torch.equal(spread, torch.zeros_like(spread))
    m = OR.metrics(rows, 1)
    assert m["epe_sample"] == m["epe_best_of_k"] == m["epe"] and m["spread"] == 0.0


def test_oracle_masks_unknown_ground_truth():
    gt = torch.ones(1, 2, 2, 3)
    gt[0, 0, 0, 0] = math.nan
    gt[0, 1, 0, 1] = math.inf
    gt[0, 0, 0, 2] = -math.inf
    gt[0, 1, 1, 0] = 1e9
    gt[0, 0, 1, 1] = 25.0                     # valid, beyond flow_max = 20
    s = torch.zeros(1, 2, 2, 2, 3)
    s[0, 1, :, 0, 0] = math.nan               # a NaN sample at an invalid pixel is masked
    _, _, rows, _ = OR.flow_eval(s, 20.0, gt)
    assert rows[0, 0] == 2 and rows[0, 7] == 1 and not rows.isnan().any()
    s[0, 1, :, 1, 2] = math.nan               # ... at a valid pixel it is reported
    _, _, rows, _ = OR.flow_eval(s, 20.0, gt)
    assert rows[0, 9].isnan() and rows[0, 1].isnan() and not rows[0, 8].isnan()
    _, _, rows, _ = OR.flow_eval(torch.zeros(2, 3, 2, 4, 5), 20.0, None)
    assert rows[:, 0].tolist() == [20.0, 20.0] and rows[:, 1:6].abs().sum() == 0 and rows[:, 7:].abs().sum() == 0


def test_flow_scores_match_the_oracle_metrics():
    g = torch.Generator().manual_seed(1)
    rows = []
    for b in range(4):
        s = torch.randn(2 + b % 2, 3, 2, 6, 5, generator=g)
        gt = torch.randn(s.shape[0], 2, 6, 5, generator=g) * 30
        gt[:, :, 0, b] = math.nan
        rows.append(OR.flow_eval(s, 20.0, gt)[2])
    fs = evaluation.FlowScores(3)
    for r in rows:
        fs.update(r)
    got, want = fs.metrics(), OR.metrics(torch.cat(rows), 3)
    assert got.keys() == want.keys()
    for k in want:
        assert got[k] == pytest.approx(want[k], rel=1e-12), k
    with pytest.raises(ValueError):
        fs.update(torch.zeros(2, 10, dtype=torch.float64))
    empty = evaluation.FlowScores(2).metrics()
    assert empty["pixels"] == 0 and empty["images"] == 0 and math.isnan(empty["epe"])


def test_score_flows_refuses_cpu_tensors():
    with pytest.raises(_lib.FlowDiffError):
        evaluation.score_flows(torch.zeros(1, 1, 2, 4, 4), 20.0)


def test_sample_seed_is_distinct_and_position_free():
    seeds = {evaluation.sample_seed(7, i, k) for i in range(300) for k in range(40)}
    assert len(seeds) == 300 * 40
    assert evaluation.sample_seed(7, 5, 3) == (7 << 48) | (5 << 16) | 3
    assert evaluation.sample_seed(1, 0, 0) != evaluation.sample_seed(2, 0, 0)
    assert max(seeds) < 1 << 64
    with pytest.raises(ValueError):
        evaluation.sample_seed(0, 0, 1 << 16)


@pytest.mark.parametrize("target", ["flow", "joint"])
def test_sample_flows_draws_x_T_per_image_and_sample(target):
    """sample_flows gives sample k of image i the same x_T whatever the batch it is in and the chunking, and
    restores return_all_timesteps.  The sampler itself is replaced here (it needs the GPU): it records x_T."""
    from opticalflowdiffusion_b200 import FlowDiffuser
    from opticalflowdiffusion_b200.config import compose
    algo = FlowDiffuser(compose([f"algorithm.target={target}"]).algorithm)
    seen = []

    def fake_sample(cond, flow, use_ema=None, x_T=None):
        assert not algo.return_all_timesteps and cond.shape[0] == x_T.shape[0] == flow.shape[0]
        seen.append(x_T.clone())
        return None, x_T[:, -2:].clone()            # the 2-channel final flow, as FlowDiffuser.sample returns it

    algo.sample = fake_sample
    cond = torch.zeros(3, 3, 4, 6)
    a = algo.sample_flows(cond, [10, 11, 12], 2, seed=5)
    xa = torch.cat(seen)
    seen.clear()
    b = algo.sample_flows(cond[1:2], [11], 2, seed=5, max_batch=1)
    assert len(seen) == 2 and algo.return_all_timesteps
    assert torch.equal(b[0], a[1]) and torch.equal(torch.cat(seen), xa[2:4])
    ch = algo.model.channels
    want = torch.randn((ch, 4, 6), generator=torch.Generator().manual_seed(evaluation.sample_seed(5, 12, 1)))
    assert torch.equal(xa[5], want)
    assert a.shape == (3, 2, 2, 4, 6) and not torch.equal(a[:, 0], a[:, 1])


def test_shard_range_covers_ragged_datasets():
    for n in (0, 1, 2, 5, 7, 13, 100):
        for world in range(1, 6):
            parts = [list(parallel.shard_range(n, r, world)) for r in range(world)]
            assert sum(parts, []) == list(range(n))


def test_compose_evaluate_task():
    from opticalflowdiffusion_b200.config import compose
    c = compose(["experiment.tasks=[evaluate]", "experiment.evaluation.num_samples=2"])
    ev = c.experiment.evaluation
    assert c.experiment.tasks == ["evaluate"] and ev.num_samples == 2 and ev.split == "validation"
    assert ev.seed == 0 and ev.limit_batch is None and ev.max_sample_batch is None and ev.data.batch_size == 8


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _rank_rows(K):
    g = torch.Generator().manual_seed(3)
    return [OR.flow_eval(torch.randn(n, K, 2, 5, 6, generator=g), 20.0, torch.randn(n, 2, 5, 6, generator=g) * 25)[2]
            for n in (3, 2)]


def _worker(rank, world, port, q):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        fs = evaluation.FlowScores(3)
        fs.update(_rank_rows(3)[rank])
        q.put((rank, fs.metrics()))
    finally:
        dist.destroy_process_group()


def test_flow_scores_all_reduce_world_size_2_gloo():
    world = 2
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, world, port, q)) for r in range(world)]
    for p in procs:
        p.start()
    out = sorted((q.get(timeout=120) for _ in range(world)), key=lambda r: r[0])
    for p in procs:
        p.join(60)
        assert p.exitcode == 0
    (_, m0), (_, m1) = out
    single = evaluation.FlowScores(3)
    for r in _rank_rows(3):
        single.update(r)
    want = single.metrics()
    assert m0 == m1
    for k in want:
        assert m0[k] == pytest.approx(want[k], rel=1e-12), k
    assert m0["images"] == 5
