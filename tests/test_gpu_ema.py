"""-m gpu: the weight EMA (algorithm.ema_decay) -- the fused Adam + EMA kernel, the EMA recurrence over real training
steps, its cost in launches, sampling from the EMA network (eager, CUDA graph, DPM-Solver++), checkpoints and resume, and
two data-parallel ranks."""
import hashlib
import os
import socket

import numpy as np
import pytest
import torch
import torch.multiprocessing as mp

from oracle import flowdiff_oracle as O

pytestmark = pytest.mark.gpu


def _algo(overrides, seed=0):
    from opticalflowdiffusion_b200 import FlowDiffuser
    from opticalflowdiffusion_b200.config import compose
    torch.manual_seed(seed)
    return FlowDiffuser(compose(overrides).algorithm).cuda()


def _batch(algo, B, H, W, seed=1):
    g = torch.Generator().manual_seed(seed)
    img = O.synthetic_frames(B, H, W, seed=seed).cuda()
    tgt = O.synthetic_frames(B, H, W, seed=seed + 1).cuda()
    flow = (torch.randn(B, 2, H, W, generator=g) * 2).cuda()
    first, cond, fl = algo.preprocess((img, tgt, flow), aug=False)
    t = torch.randint(0, 1000, (B,), generator=g).cuda()
    noise = torch.randn(first.shape, generator=g).cuda()
    return first, cond, fl, t, noise


def _train_step(algo, opt, batch):
    first, cond, fl, t, noise = batch
    loss = algo.loss(first, cond, fl, t=t, noise=noise)
    loss.backward()
    opt.step()
    opt.zero_grad(set_to_none=True)


def _flat(module):
    return torch.cat([p.detach().reshape(-1) for p in module.parameters()]).double().cpu()


def _lerp64(e, p, w):
    """The documented update in float64: torch.lerp's two-branch form."""
    return p - (p - e) * (1.0 - w) if w >= 0.5 else e + w * (p - e)


def _rel(a, b):
    return ((a - b).norm() / b.norm()).item()


# ----------------------------------------------------------------------------------------------------------------- kernel
@pytest.mark.parametrize("clip", [False, True])
def test_adam_ema_kernel(clip):
    """fd_adam_ema_step writes param / exp_avg / exp_avg_sq bitwise like fd_adam_step, and ema within 2 ulp (of
    max(|param|, |ema|)) of the fp64 evaluation of the documented formula, and exactly param at w = 1."""
    from opticalflowdiffusion_b200 import _lib
    lib = _lib.load(check_device=True)
    n = 1_000_003                                          # not a multiple of 4
    g = torch.Generator().manual_seed(11 + int(clip))
    p0 = torch.randn(n, generator=g).cuda()
    gr = (torch.randn(n, generator=g) * 3).cuda()
    m0 = (torch.randn(n, generator=g) * 0.1).cuda()
    v0 = (torch.rand(n, generator=g) * 0.01).cuda()
    e0 = (p0.cpu() + torch.randn(n, generator=g) * 0.05).cuda()
    sumsq = torch.zeros(1, device="cuda")
    if clip:
        _lib.check(lib.fd_sumsq(_lib.ptr(gr), n, _lib.ptr(sumsq), _lib.stream()))
    args = (1e-3, 0.9, 0.999, 1e-8, 1e-2, 3, _lib.ptr(sumsq) if clip else None, 100.0 if clip else 0.0, 0.5)
    pa, ma, va = p0.clone(), m0.clone(), v0.clone()
    _lib.check(lib.fd_adam_step(_lib.ptr(pa), _lib.ptr(gr), _lib.ptr(ma), _lib.ptr(va), n, *args, _lib.stream()))
    if clip:                                               # the clip really engaged: 0.5 * |g| > 100
        assert 0.5 * float(sumsq.sqrt()) > 100.0
    for w in (1.0, 0.9, 0.5, 0.4999, 0.1, 1e-4, 0.0):
        pb, mb, vb, eb = p0.clone(), m0.clone(), v0.clone(), e0.clone()
        _lib.check(lib.fd_adam_ema_step(_lib.ptr(pb), _lib.ptr(gr), _lib.ptr(mb), _lib.ptr(vb), _lib.ptr(eb), n, *args[:-1],
                                        args[-1], w, _lib.stream()))
        assert torch.equal(pa, pb) and torch.equal(ma, mb) and torch.equal(va, vb), w
        if w == 1.0:
            assert torch.equal(eb, pb)
        w32 = float(np.float32(w))
        ref = _lerp64(e0.double(), pb.double(), w32)
        # ulp at the operands' scale: each of the kernel's fp32 roundings (p - e, then the product and sum) is at most half
        # an ulp of a value no larger than max(|p|, |e|); a result that cancels to near zero keeps that absolute error
        scale = torch.maximum(pb.abs(), e0.abs())
        ulp = (torch.nextafter(scale, torch.tensor(float("inf"), device="cuda")) - scale).double()
        err = ((eb.double() - ref).abs() / ulp).max().item()
        assert err <= 2.0, (w, err)
    # arguments the entry point refuses
    with pytest.raises(_lib.FlowDiffError):
        _lib.check(lib.fd_adam_ema_step(_lib.ptr(pb), _lib.ptr(gr), _lib.ptr(mb), _lib.ptr(vb), _lib.ptr(eb), n, *args, 1.5,
                                        _lib.stream()))
    with pytest.raises(_lib.FlowDiffError):
        _lib.check(lib.fd_adam_ema_step(_lib.ptr(pb), _lib.ptr(gr), _lib.ptr(mb), _lib.ptr(vb), None, n, *args, 0.5,
                                        _lib.stream()))


# ------------------------------------------------------------------------------------------------------ training recurrence
@pytest.mark.parametrize("target", ["flow", "joint"])
def test_training_follows_the_ema_recurrence(target):
    """40 optimiser steps at 32x48 with after=5, every=3: ema_unet equals the float64 EMA recurrence replayed over the
    online weights after each step; the EMA's packed weights are invalidated exactly on the steps that updated it."""
    from opticalflowdiffusion_b200.optim import ema_weight
    after, every, beta = 5, 3, 0.9
    algo = _algo([f"algorithm.target={target}", "algorithm.zero_init=false", "algorithm.lr=1e-3",
                  f"algorithm.ema_decay={beta}", f"algorithm.ema_update_after_step={after}",
                  f"algorithm.ema_update_every={every}"])
    opt = algo.configure_optimizers()
    opt.max_grad_norm = 100.0
    batch = _batch(algo, 2, 32, 48)
    ema = _flat(algo.ema_unet)
    assert torch.equal(ema, _flat(algo.unet))
    worst = 0.0
    for k in range(1, 41):
        epoch = algo.ema_unet.weights_epoch
        _train_step(algo, opt, batch)
        w = ema_weight(k, beta, after, every)
        assert opt.step_count == k and opt.ema_updated == (w is not None)
        assert algo.ema_unet.weights_epoch == epoch + int(w is not None)
        if w is not None:
            ema = _lerp64(ema, _flat(algo.unet), w)
        worst = max(worst, _rel(_flat(algo.ema_unet), ema))
    print(f"target={target}: worst rel-L2 of the EMA vs its float64 replay over 40 steps {worst:.2e}")
    assert worst <= 1e-6
    assert _rel(_flat(algo.ema_unet), _flat(algo.unet)) > 1e-5      # the average lags the online weights


def test_ema_adds_no_launch():
    """fd_launch_count per training step: EMA off == EMA update step == skipped step."""
    from opticalflowdiffusion_b200 import _lib
    lib = _lib.load()

    def counts(overrides, steps):
        algo = _algo(["algorithm.target=flow", "algorithm.lr=1e-3", *overrides])
        opt = algo.configure_optimizers()
        batch = _batch(algo, 2, 32, 48)
        out = []
        for _ in range(steps):
            n0 = lib.fd_launch_count()
            _train_step(algo, opt, batch)
            torch.cuda.synchronize()
            out.append((int(lib.fd_launch_count() - n0), opt.ema_updated))
        return out

    off = counts([], 4)
    on = counts(["algorithm.ema_decay=0.99", "algorithm.ema_update_after_step=1", "algorithm.ema_update_every=2"], 4)
    assert [u for _, u in on] == [True, False, True, False]          # copy, skip, update, skip
    assert [c for c, _ in on] == [c for c, _ in off], (off, on)
    assert len({c for c, _ in on[1:]}) == 1, on                      # skipped == updated after the first step


# ----------------------------------------------------------------------------------------------------------------- sampling
def test_sampling_uses_the_ema_network():
    """sample() with EMA on == a fresh FlowDiffuser whose UNet holds the EMA tensors, bitwise from the same x_T: eager
    DDIM, CUDA-graph DDIM and DPM-Solver++ 2M; use_ema=False == the online network; an EMA graph is re-captured when the
    EMA moves into the optimiser's flat buffer and its replays follow later EMA updates."""
    ov = ["algorithm.target=flow", "algorithm.sampling_timesteps=3", "algorithm.lr=1e-2"]
    m = _algo(ov + ["algorithm.ema_decay=0.9", "algorithm.ema_update_after_step=1", "algorithm.ema_update_every=1"], seed=5)
    fresh = _algo(ov, seed=6)
    B, H, W = 1, 32, 64
    cond = (O.synthetic_frames(B, H, W, seed=8) * 2 - 1).cuda()
    flow = torch.zeros(B, 2, H, W, device="cuda")
    x_T = torch.randn(B, 2, H, W, generator=torch.Generator().manual_seed(9)).cuda()

    def sample(algo, graph, **kw):
        algo.use_cuda_graph = graph
        return algo.sample(cond, flow, x_T=x_T, **kw)[1]

    g_before = sample(m, True)                                # captured while the EMA still has its own storages
    opt = m.configure_optimizers()
    batch = _batch(m, B, H, W)
    for _ in range(3):
        _train_step(m, opt, batch)
    fresh.unet.load_state_dict(m.ema_unet.state_dict())
    assert _rel(_flat(m.ema_unet), _flat(m.unet)) > 1e-6
    e_ema, e_ref = sample(m, False), sample(fresh, False)
    assert torch.equal(e_ema, e_ref)
    g_ema, g_ref = sample(m, True), sample(fresh, True)
    assert torch.equal(g_ema, g_ref)
    assert (g_ema - e_ema).abs().max().item() < 5e-3 and (g_ema - g_before).abs().max().item() > 1e-4
    for d in (m.ema_model, fresh.model):
        d.sampler, d.solver_order = "dpmpp", 2
    assert torch.equal(sample(m, False), sample(fresh, False))
    for d in (m.ema_model, fresh.model):
        d.sampler = None
    online = sample(m, False, use_ema=False)
    assert (online - e_ema).abs().max().item() > 1e-4
    fresh.unet.load_state_dict(m.unet.state_dict())
    assert torch.equal(online, sample(fresh, False))
    # further training: the EMA graph (same storages) replays the updated EMA through prepare()
    for _ in range(2):
        _train_step(m, opt, batch)
    g2, e2 = sample(m, True), sample(m, False)
    assert (g2 - e2).abs().max().item() < 5e-3 and (g2 - g_ema).abs().max().item() > 1e-4


# -------------------------------------------------------------------------------------------------------------- checkpoints
def test_checkpoint_rules(tmp_path):
    """Save and load into a fresh EMA model: EMA bitwise; a checkpoint without EMA initialises the EMA from its weights;
    an EMA checkpoint loads into a model without EMA with the EMA keys reported as ignored."""
    from opticalflowdiffusion_b200 import io_formats as IO
    ema_ov = ["algorithm.target=flow", "algorithm.lr=1e-3", "algorithm.ema_decay=0.9", "algorithm.ema_update_after_step=0",
              "algorithm.ema_update_every=1"]
    m = _algo(ema_ov)
    opt = m.configure_optimizers()
    batch = _batch(m, 2, 32, 48)
    for _ in range(2):
        _train_step(m, opt, batch)
    path = str(tmp_path / "ema.ckpt")
    IO.save_checkpoint(m, path, optimizer=opt, global_step=2)
    dst = _algo(ema_ov, seed=3)
    rep = IO.load_checkpoint(dst, path)
    assert rep == {"missing": [], "unexpected": [], "ema_initialised": False}
    for (k, a), b in zip(m.ema_unet.state_dict().items(), dst.ema_unet.state_dict().values()):
        assert torch.equal(a, b), k
    plain = _algo(["algorithm.target=flow"], seed=4)
    rep = IO.load_checkpoint(plain, path)
    assert rep["missing"] == [] and rep["unexpected"] == [] and len(rep["ignored"]) == 276
    assert torch.equal(plain.unet.init_conv.weight, m.unet.init_conv.weight)
    path2 = str(tmp_path / "plain.ckpt")
    IO.save_checkpoint(plain, path2)
    dst = _algo(ema_ov, seed=5)
    rep = IO.load_checkpoint(dst, path2)
    assert rep == {"missing": [], "unexpected": [], "ema_initialised": True}
    for (k, a), b in zip(dst.ema_unet.state_dict().items(), plain.unet.state_dict().values()):
        assert torch.equal(a, b), k


def test_resume_continues_the_ema(tmp_path):
    """A run resumed from the step-2 checkpoint restores parameters, moments and EMA bitwise, and reproduces steps 3-4
    of the uninterrupted run.  One batch per epoch and the t / noise draws of steps 1-2 replayed make the resumed steps
    see the same inputs.  The backward's fp32 atomics may reorder parameter-gradient sums between runs, so the resumed run
    is compared with the first uninterrupted run against the distance between two uninterrupted runs."""
    from opticalflowdiffusion_b200.config import compose
    from opticalflowdiffusion_b200.experiments import build_experiment

    def run(ckpt, steps, out):
        import random
        ov = ["algorithm.target=flow", "algorithm.gpu_augment=true", "dataset.height=32", "dataset.width=32",
              "dataset.length=2", "experiment.training.data.batch_size=2", "experiment.training.data.shuffle=false",
              "experiment.training.checkpointing.every_n_train_steps=2", f"+output_dir={tmp_path / out}",
              "algorithm.ema_decay=0.5", "algorithm.ema_update_after_step=1", "algorithm.ema_update_every=1"]
        random.seed(0)
        torch.manual_seed(0)
        exp = build_experiment(compose(ov), None, ckpt)
        exp.algo.preprocess = (lambda f: (lambda batch, aug=True: f(batch, aug=False)))(exp.algo.preprocess)
        torch.manual_seed(123)
        if ckpt is not None:                       # the t / noise draws of steps 1-2 (p_losses: randint, then randn_like)
            for _ in range(2):
                torch.randint(0, 1000, (2,), device="cuda")
                torch.randn(2, 2, 32, 32, device="cuda")
        res = exp.train(max_steps=steps)
        return exp, res

    exp_a, res_a = run(None, 4, "a")
    ck = tmp_path / "a" / "checkpoints" / "step_0000002.ckpt"
    state = torch.load(str(ck), map_location="cpu", weights_only=False)["state_dict"]
    assert sum(k.startswith("ema_unet.") for k in state) == 276
    exp_r, _ = run(str(ck), 0, "r")                # restore only
    opt_r = exp_r.algo.optimizers
    opt_r._flatten()                               # the restored moments and the EMA move into the flat buffers
    assert opt_r.step_count == 2
    for k, v in exp_r.algo.state_dict().items():
        assert torch.equal(v.cpu(), state[k]), k
    saved = torch.load(str(ck), map_location="cpu", weights_only=False)["optimizer_states"][0]["state"]
    for i, p in enumerate(opt_r._params()):
        assert torch.equal(opt_r.state[p]["exp_avg"].cpu(), saved[i]["exp_avg"])
        assert torch.equal(opt_r.state[p]["exp_avg_sq"].cpu(), saved[i]["exp_avg_sq"])
    exp_b, res_b = run(str(ck), 2, "b")
    exp_c, res_c = run(None, 4, "c")
    assert res_a["global_step"] == res_b["global_step"] == res_c["global_step"] == 4
    assert exp_b.algo.optimizers.step_count == 4 and exp_b.algo.optimizers.ema_updated

    def state_of(exp):
        opt = exp.algo.optimizers
        return {"p": _flat(exp.algo.unet), "ema": _flat(exp.algo.ema_unet), "m": opt._m.double().cpu(),
                "v": opt._v.double().cpu()}

    a, b, c = state_of(exp_a), state_of(exp_b), state_of(exp_c)
    for k in a:
        floor, got = _rel(c[k], a[k]), _rel(b[k], a[k])
        print(f"{k}: resumed vs uninterrupted rel-L2 {got:.2e}; two uninterrupted runs {floor:.2e}")
        assert got <= max(10 * floor, 1e-6), (k, got, floor)


# -------------------------------------------------------------------------------------------------------------- two ranks
OV = ["algorithm.target=flow", "algorithm.gpu_augment=true", "algorithm.lr=1e-3", "dataset.height=32", "dataset.width=32",
      "dataset.length=8", "experiment.training.data.batch_size=2", "experiment.training.data.shuffle=false",
      "algorithm.ema_decay=0.9", "algorithm.ema_update_after_step=1", "algorithm.ema_update_every=1"]


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _worker(rank, world, port, q):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world), LOCAL_RANK="0",
                      FD_DIST_BACKEND="gloo")
    import random
    import torch.distributed as dist
    from opticalflowdiffusion_b200.config import compose
    from opticalflowdiffusion_b200.experiments import build_experiment
    random.seed(0)
    torch.manual_seed(1000 + rank)                      # different init per rank: the runner broadcasts rank 0's
    exp = build_experiment(compose(OV), None, None)
    exp.algo.preprocess = (lambda f: (lambda batch, aug=True: f(batch, aug=False)))(exp.algo.preprocess)
    e0 = float(exp.algo.ema_unet.final_res_block.block1.proj.weight.double().sum())
    torch.manual_seed(7)
    out = exp.train(max_steps=3)
    # plain Python values only: tensors sent through a multiprocessing queue live in shared memory owned by the sender
    sd = {k: hashlib.sha1(v.detach().cpu().numpy().tobytes()).hexdigest() for k, v in exp.algo.ema_unet.state_dict().items()}
    lag = _rel(_flat(exp.algo.ema_unet), _flat(exp.algo.unet))
    q.put((rank, e0, sd, out["steps"], exp.algo.optimizers.ema_updated, lag))
    dist.barrier()
    dist.destroy_process_group()


def test_two_ranks_keep_identical_emas():
    """Two gloo ranks on one GPU from different initial weights, 3 steps with after=1, every=1 (the copy and the lerp
    branch both run): the ranks end with hash-identical ema_unet tensors, without any EMA collective."""
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
    (_, e0, sd0, steps0, upd0, lag0), (_, e1, sd1, steps1, upd1, lag1) = out
    assert e0 != e1                                     # the ranks' EMAs started from different weights
    assert steps0 == steps1 == 3 and upd0 and upd1 and lag0 > 0 and lag0 == lag1
    assert len(sd0) == 276
    for k in sd0:
        assert sd0[k] == sd1[k], k
