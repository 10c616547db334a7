"""-m gpu: the DPM-Solver++ sampler (sampler: dpmpp).  The fused step kernel bit-exact against the oracle's fp32 op
sequence, the free-running sampler against the oracle's (flow, joint and the 436x1024 headline shape), order 1 against
the DDIM sampler, and the CUDA-graph capture of the loop."""
import os

import pytest
import torch

from oracle import dpmpp_oracle as P
from oracle import flowdiff_oracle as O

pytestmark = pytest.mark.gpu

FLOW_MAX = 20.0


def make_algo(overrides, seed=0):
    from opticalflowdiffusion_b200 import FlowDiffuser
    from opticalflowdiffusion_b200.config import compose
    torch.manual_seed(seed)
    return FlowDiffuser(compose(overrides).algorithm).cuda()


def _epe(a, b):
    return torch.sqrt(((a - b) * FLOW_MAX).pow(2).sum(1)).mean().item()


def _same(a, b):
    """Bitwise equal, NaN positions included."""
    a, b = a.cpu(), b.cpu()
    na, nb = torch.isnan(a), torch.isnan(b)
    return torch.equal(na, nb) and torch.equal(a.masked_fill(na, 0).view(torch.int32), b.masked_fill(nb, 0).view(torch.int32))


@pytest.mark.parametrize("shape", [(3, 2, 7, 11), (2, 2, 9, 12)])
def test_step_kernel_bit_exact(shape):
    """fd_dpmpp_step == P.dpmpp_update bit for bit given the package's coefficients, for orders 1-3 and the last step;
    model outputs beyond [-1, 1], NaNs in x / model output / history, a NaN-filled history slot that the order does not
    use (must not leak), n % 4 != 0 (float4 body + scalar tail), a misaligned view (scalar kernel), and the two allowed
    aliasings d_out == d_hist2 and x_next == x."""
    from opticalflowdiffusion_b200 import _lib
    from opticalflowdiffusion_b200.diffusion import dpmpp_coeffs
    lib = _lib.load(check_device=True)
    sched = O.make_schedule(1000)
    ac = sched["alphas_cumprod"].tolist()
    times = O.ddim_times(1000, 10)
    g = torch.Generator().manual_seed(sum(shape))
    x, mo, d1, d2 = (torch.randn(*shape, generator=g) * s for s in (1.0, 1.6, 0.7, 0.7))
    d1, d2 = d1.clamp(-1, 1), d2.clamp(-1, 1)
    flat = [v.view(-1) for v in (x, mo, d1, d2)]
    for k, v in enumerate(flat):
        v[(k * 37 + 5) % v.numel()] = float("nan")
    nan_slot = torch.full(shape, float("nan"))
    cases = [(0, 1, d1, d2), (3, 1, nan_slot, nan_slot), (1, 2, d1, nan_slot), (4, 2, d1, d2), (2, 3, d1, d2),
             (6, 3, d1, d2), (9, 3, d1, d2), (9, 1, nan_slot, nan_slot)]
    n = x.numel()
    for i, order, h1, h2 in cases:
        coeffs = dpmpp_coeffs(ac, times, i, order)
        ref_x, ref_d = P.dpmpp_update(x, mo, h1, h2, coeffs)
        cx, c0, c1, c2, last = coeffs
        xc, mc, h1c, h2c = x.cuda(), mo.cuda(), h1.cuda(), h2.cuda()
        out, dout = torch.empty_like(xc), torch.empty_like(xc)
        _lib.check(lib.fd_dpmpp_step(_lib.ptr(xc), _lib.ptr(mc), _lib.ptr(h1c), _lib.ptr(h2c), _lib.ptr(out), _lib.ptr(dout),
                                     n, cx, c0, c1, c2, last, _lib.stream()))
        assert _same(out, ref_x) and _same(dout, ref_d), (i, order)
        # aliasing: d_out over d_hist2, x_next over x
        xa, ha = xc.clone(), h2c.clone()
        _lib.check(lib.fd_dpmpp_step(_lib.ptr(xa), _lib.ptr(mc), _lib.ptr(h1c), _lib.ptr(ha), _lib.ptr(xa), _lib.ptr(ha),
                                     n, cx, c0, c1, c2, last, _lib.stream()))
        assert _same(xa, ref_x) and _same(ha, ref_d), ("aliased", i, order)
        # misaligned views (offset by one float): the scalar kernel
        big = [torch.empty(n + 1, device="cuda") for _ in range(6)]
        views = [b[1:].view(shape) for b in big]
        for v, src in zip(views[:4], (xc, mc, h1c, h2c)):
            v.copy_(src)
        _lib.check(lib.fd_dpmpp_step(*(_lib.ptr(v) for v in views), n, cx, c0, c1, c2, last, _lib.stream()))
        assert _same(views[4], ref_x) and _same(views[5], ref_d), ("scalar", i, order)
    # the argument checks: a used history slot must be given; d_out may not alias d_hist1
    coeffs = dpmpp_coeffs(ac, times, 4, 3)
    xc, mc, h = x.cuda(), mo.cuda(), d1.cuda()
    out = torch.empty_like(xc)
    assert lib.fd_dpmpp_step(_lib.ptr(xc), _lib.ptr(mc), None, _lib.ptr(h), _lib.ptr(out), _lib.ptr(h), n,
                             *coeffs[:4], 0, _lib.stream()) != 0
    assert lib.fd_dpmpp_step(_lib.ptr(xc), _lib.ptr(mc), _lib.ptr(h), None, _lib.ptr(out), _lib.ptr(h), n,
                             coeffs[0], coeffs[1], coeffs[2], 0.0, 0, _lib.stream()) != 0


@pytest.mark.parametrize("S", [5, 10])
def test_free_running_2m_3m_vs_oracle(S):
    """2M and 3M at 64x128, target=flow, bf16 UNet in the loop against the fp32 oracle: final flow EPE <= 0.25 px (the
    tolerance of the DDIM test in tests/test_gpu_sampling.py); the trajectory shape follows ddim_sample's."""
    m = make_algo(["algorithm.target=flow", f"algorithm.sampling_timesteps={S}", "algorithm.sampler=dpmpp"], seed=3)
    sd = {k: v.detach().cpu().clone() for k, v in m.unet.state_dict().items()}
    B, H, W = 1, 64, 128
    cond = O.synthetic_frames(B, H, W, seed=6) * 2 - 1
    x_T = torch.randn(B, 2, H, W, generator=torch.Generator().manual_seed(7))
    for order in (2, 3):
        m.model.solver_order = order
        with torch.no_grad():
            ref = P.dpmpp_sample(sd, O.make_schedule(1000), x_T, cond, 1000, S, order)
        traj = m.model.sample(B, external_cond=cond.cuda(), x_T=x_T, return_all_timesteps=True)
        assert traj.shape == (B, S + 1, 2, H, W) and torch.equal(traj[:, 0].cpu(), x_T)
        epe = _epe(traj[:, -1].cpu(), ref)
        print(f"dpmpp {order}M S={S} 64x128: EPE vs oracle {epe:.4f} px")
        assert epe <= 0.25, (order, S, epe)


def test_order1_equals_ddim_sampler():
    """sampler=dpmpp with solver_order=1 is the DDIM sampler (eta = 0) up to fp32 rounding.

    (a) Step by step: every state of the DDIM-10 trajectory and the UNet output at it go through fd_ddim_step and through
        fd_dpmpp_step (order 1); the two fp32 op orders agree to 8 ulp of max(1, |x|) (measured <= 5 ulp on their CPU
        restatements, which the kernels equal bit for bit).
    (b) Free-running, 10 steps from the same x_T.  A few-ulp difference of the state flips bf16 roundings of the UNet's
        input and activations, so two free runs differ at the scale of the bf16 UNet's own error, not at the scale of a
        replay of identical inputs: the DDIM sampler against itself from x_T moved by one ulp is printed as that floor.
        Asserted with the bounds of the bf16-in-the-loop trajectory test (tests/test_gpu_sampling.py): order 1 vs DDIM
        max |diff| <= 5e-2, mean <= 1e-2, and each sampler's final flow within 0.25 px EPE of the fp32 oracle's DDIM-10."""
    from opticalflowdiffusion_b200 import _lib
    from opticalflowdiffusion_b200.diffusion import ddim_time_pairs, dpmpp_coeffs
    lib = _lib.load(check_device=True)
    B, H, W, S = 2, 32, 64, 10
    cond_c = O.synthetic_frames(B, H, W, seed=2) * 2 - 1
    x_T_c = torch.randn(B, 2, H, W, generator=torch.Generator().manual_seed(5))
    cond, x_T = cond_c.cuda(), x_T_c.cuda()
    d = make_algo(["algorithm.target=flow", f"algorithm.sampling_timesteps={S}"], seed=4)
    p = make_algo(["algorithm.target=flow", f"algorithm.sampling_timesteps={S}", "algorithm.sampler=dpmpp",
                   "algorithm.solver_order=1"], seed=4)
    a = d.model.sample(B, external_cond=cond, x_T=x_T, return_all_timesteps=True)
    b = p.model.sample(B, external_cond=cond, x_T=x_T, return_all_timesteps=True)
    assert a.shape == b.shape == (B, S + 1, 2, H, W)

    pairs = ddim_time_pairs(1000, S)
    times = [q[0] for q in pairs] + [-1]
    ac = d.model._host["alphas_cumprod"].tolist()
    worst_ulp = 0.0
    with torch.no_grad():
        for i, (tm, tn) in enumerate(pairs):
            x = a[:, i].contiguous()
            mo = d.model.model_with_condition(x, torch.full((B,), tm, device="cuda", dtype=torch.long), None, cond)
            o1, o2, dh = torch.empty_like(x), torch.empty_like(x), torch.empty_like(x)
            _lib.check(lib.fd_ddim_step(_lib.ptr(x), _lib.ptr(mo), None, _lib.ptr(o1), None, x.numel(),
                                        *d.model._ddim_scalars(tm, tn), _lib.stream()))
            _lib.check(lib.fd_dpmpp_step(_lib.ptr(x), _lib.ptr(mo), None, None, _lib.ptr(o2), _lib.ptr(dh), x.numel(),
                                         *dpmpp_coeffs(ac, times, i, 1), _lib.stream()))
            scale = torch.clamp(o1.abs(), min=1.0)
            worst_ulp = max(worst_ulp, ((o1 - o2).abs() / scale).max().item() / 2 ** -23)
    assert worst_ulp <= 8, worst_ulp

    x_T_ulp = torch.nextafter(x_T, torch.full_like(x_T, float("inf")))
    a_ulp = d.model.sample(B, external_cond=cond, x_T=x_T_ulp, return_all_timesteps=True)
    diff = (a - b).abs()
    floor = (a - a_ulp).abs()
    sd = {k: v.detach().cpu().clone() for k, v in d.unet.state_dict().items()}
    with torch.no_grad():
        ref = O.ddim_sample(sd, O.make_schedule(1000), x_T_c, cond_c, 1000, S)
    epe_d, epe_p = _epe(a[:, -1].cpu(), ref), _epe(b[:, -1].cpu(), ref)
    print(f"order 1 vs DDIM-{S}: step level worst {worst_ulp:.1f} ulp; free-running max |diff| {diff.max().item():.3e} "
          f"mean {diff.mean().item():.3e}; DDIM vs DDIM from x_T + 1 ulp: max {floor.max().item():.3e} "
          f"mean {floor.mean().item():.3e}; EPE vs fp32 oracle DDIM: ddim {epe_d:.4f} px, dpmpp-1 {epe_p:.4f} px")
    assert diff.max().item() <= 5e-2 and diff.mean().item() <= 1e-2, (diff.max().item(), diff.mean().item())
    assert epe_d <= 0.25 and epe_p <= 0.25, (epe_d, epe_p)


def test_cuda_graph_dpmpp_follows_weight_updates():
    """use_cuda_graph=True captures the DPM-Solver++ loop (history buffers inside the capture): replay == replay bitwise,
    graph == eager within 5e-3, and the replay follows an optimiser step and load_state_dict (re-capture on moved
    parameters, as for DDIM)."""
    m = make_algo(["algorithm.target=flow", "algorithm.sampling_timesteps=4", "algorithm.lr=1e-2",
                   "algorithm.sampler=dpmpp", "algorithm.solver_order=3"], seed=5)
    B, H, W = 1, 32, 64
    cond = (O.synthetic_frames(B, H, W, seed=8) * 2 - 1).cuda()
    x_T = torch.randn(B, 2, H, W, generator=torch.Generator().manual_seed(9)).cuda()

    def both():
        g = m.model.sample(B, external_cond=cond, x_T=x_T, use_cuda_graph=True)
        e = m.model.sample(B, external_cond=cond, x_T=x_T)
        return g, e

    g0, e0 = both()
    r0 = m.model.sample(B, external_cond=cond, x_T=x_T, use_cuda_graph=True)
    assert torch.equal(g0, r0)
    assert (g0 - e0).abs().max().item() < 5e-3
    m.model.solver_order = 2                                # a different order is a different graph
    g2o, e2o = both()
    assert (g2o - e2o).abs().max().item() < 5e-3 and (g2o - g0).abs().max().item() > 0
    m.model.solver_order = 3
    opt = m.configure_optimizers()
    img = O.synthetic_frames(B, H, W, seed=1).cuda()
    flow = (torch.randn(B, 2, H, W, generator=torch.Generator().manual_seed(3)) * 5).cuda()
    loss = m.training_step((img, img, flow), 0)
    loss.backward()
    opt.step()
    opt.zero_grad(set_to_none=True)
    g1, e1 = both()
    assert (g1 - e1).abs().max().item() < 5e-3
    assert (g1 - g0).abs().max().item() > 1e-4
    sd = {k: v.clone() * 0.9 for k, v in m.state_dict().items() if v.dtype.is_floating_point and k.startswith("unet.")}
    m.load_state_dict(sd, strict=False)
    g3, e3 = both()
    assert (g3 - e3).abs().max().item() < 5e-3
    assert (g3 - g1).abs().max().item() > 1e-4


def test_joint_target_vs_oracle():
    """target=joint (the reference's default; the state carries the forward splat's NaN holes) through FlowDiffuser.sample
    with sampler=dpmpp (3M, S = 4) against P.dpmpp_sample driven by O.unet_with_warp, with the tolerances of the joint
    sampler test of tests/test_gpu_sampling.py: teacher-forced (the oracle's state in, every step) clamped flow prediction
    <= 3e-2 and hole pattern >= 96 % identical; free-running flow channels finite, the first step's flow <= 3e-2, the final
    hole fraction within 0.1 of the oracle's; and the final sample's NaN holes are those of the last prediction."""
    S, B, H, W = 4, 2, 32, 48
    m = make_algo(["algorithm.target=joint", "algorithm.zero_init=false", f"algorithm.sampling_timesteps={S}",
                   "algorithm.sampler=dpmpp", "algorithm.solver_order=3"], seed=12)
    sd = {k: v.detach().cpu().clone() for k, v in m.unet.state_dict().items()}
    cond = O.synthetic_frames(B, H, W, seed=13) * 2 - 1
    x_T = torch.randn(B, 5, H, W, generator=torch.Generator().manual_seed(14))
    times = O.ddim_times(1000, S)
    with torch.no_grad():
        ref, ref_d = P.dpmpp_sample(sd, O.make_schedule(1000), x_T, cond, 1000, S, 3, return_all=True,
                                    model=lambda x, c, t: O.unet_with_warp(sd, x, c, t, FLOW_MAX, True, False))
    cond_d = cond.cuda()
    worst_flow, worst_mask = 0.0, 1.0
    with torch.no_grad():
        for i in range(S):
            x = ref[:, i].contiguous().cuda()
            out = m.model.model_with_condition(x, torch.full((B,), times[i], device="cuda", dtype=torch.long), None, cond_d)
            out = out.cpu()
            inside = ref_d[i][:, 3:].abs() < 0.999
            ef = ((out[:, 3:].clamp(-1, 1) - ref_d[i][:, 3:]).abs() * inside).max().item()
            seen = ~torch.isnan(x[:, :3].cpu())
            agree = ((torch.isnan(out[:, :3]) == torch.isnan(ref_d[i][:, :3])) & seen).float().sum().item() / seen.float().sum().item()
            worst_flow, worst_mask = max(worst_flow, ef), min(worst_mask, agree)
        print("dpmpp joint, teacher-forced: worst flow err", worst_flow, "worst hole-mask agreement", worst_mask)
        assert worst_flow <= 3e-2 and worst_mask >= 0.96, (worst_flow, worst_mask)
        samples, flows = m.sample(cond_d, torch.zeros(B, 2, H, W, device="cuda"), x_T=x_T)
    assert samples.shape == (B, S + 1, 3, H, W) and flows.shape == (B, S + 1, 2, H, W)
    assert torch.isfinite(flows).all()
    assert torch.equal(samples[:, 0].cpu(), x_T[:, :3])
    assert (flows[:, 1].cpu() - ref[:, 1, 3:]).abs().max().item() <= 3e-2
    hole, hole_ref = torch.isnan(samples[:, -1]).float().mean().item(), torch.isnan(ref[:, -1, :3]).float().mean().item()
    print("final hole fraction", hole, "oracle", hole_ref)
    assert abs(hole - hole_ref) <= 0.1, (hole, hole_ref)
    with torch.no_grad():
        state = torch.cat((samples[:, S - 1], flows[:, S - 1]), dim=1).contiguous()
        last = m.model.model_with_condition(state, torch.full((B,), times[S - 1], device="cuda", dtype=torch.long), None,
                                            cond_d)
    assert torch.equal(torch.isnan(samples[:, -1]), torch.isnan(last[:, :3]))
    assert (samples[:, -1] - last[:, :3].clamp(-1, 1)).nan_to_num().abs().max().item() <= 1e-5


def test_2m10_436x1024_vs_oracle():
    """The headline shape: 2M with S = 10 at 436x1024, B = 1, against the fp32 oracle (10 CPU UNet forwards on the
    replicate-padded 440x1024 frames, cropped back as the CUDA path does inside Unet.forward): EPE <= 0.25 px."""
    try:
        torch.set_num_threads(max(1, len(os.sched_getaffinity(0))))
    except Exception:  # noqa: BLE001
        pass
    H, W, S = 436, 1024, 10
    m = make_algo(["algorithm.target=flow", f"algorithm.sampling_timesteps={S}", "algorithm.return_all_timesteps=false",
                   "algorithm.sampler=dpmpp", "algorithm.solver_order=2"], seed=0)
    sd = {k: v.detach().cpu().clone() for k, v in m.unet.state_dict().items()}
    cond = O.synthetic_frames(1, H, W, seed=100) * 2 - 1
    x_T = torch.randn(1, 2, H, W, generator=torch.Generator().manual_seed(1234))
    cond_p, pad = O.replicate_pad_to_multiple(cond)
    top, left = pad[2], pad[0]

    def model(x, c, t):
        xp, _ = O.replicate_pad_to_multiple(x)
        return O.unet_forward(sd, xp, cond_p, t)[..., top:top + H, left:left + W]

    with torch.no_grad():
        ref = P.dpmpp_sample(sd, O.make_schedule(1000), x_T, cond, 1000, S, 2, model=model)
    out = m.model.sample(1, external_cond=cond.cuda(), x_T=x_T)
    epe = _epe(out.cpu(), ref)
    print(f"dpmpp 2M-10 436x1024: EPE vs oracle {epe:.4f} px")
    assert epe <= 0.25, epe
