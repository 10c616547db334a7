"""CPU: the multistep DPM-Solver++ sampler (sampler: dpmpp) -- the oracle's restatement checked against DDIM, against the
closed-form solution for a constant prediction and for its convergence order, and the package's float64 step coefficients
against the oracle's."""
import math

import pytest
import torch

from oracle import dpmpp_oracle as P
from oracle import flowdiff_oracle as O

SCHED = O.make_schedule(1000)


def _flow_unet(seed):
    from opticalflowdiffusion_b200.unet_params import UnetParams
    torch.manual_seed(seed)
    return UnetParams(64, channels=5, out_dim=2).state_dict()


@pytest.mark.parametrize("S", [5, 50])
def test_order1_is_ddim(S):
    """DPM-Solver++(1) is DDIM with eta = 0 written as x_t = (sigma_t/sigma_s) x_s + (alpha_t - alpha_s sigma_t/sigma_s) D:
    the whole trajectory of a random-init flow UNet at 16x24 agrees to 1e-5 (fp32 rounding of the two op orders)."""
    sd = _flow_unet(11)
    cond = O.synthetic_frames(2, 16, 24, seed=3) * 2 - 1
    x_T = torch.randn(2, 2, 16, 24, generator=torch.Generator().manual_seed(4))
    with torch.no_grad():
        a, da = P.dpmpp_sample(sd, SCHED, x_T, cond, 1000, S, 1, return_all=True)
        b, db = O.ddim_sample(sd, SCHED, x_T, cond, 1000, S, return_all=True)
    assert a.shape == b.shape == (2, S + 1, 2, 16, 24)
    err = (a - b).abs().max().item()
    assert err <= 1e-5, err
    assert torch.equal(a[:, -1], da[-1])                   # the last step returns the last prediction, as DDIM does
    assert max((x - y).abs().max().item() for x, y in zip(da, db)) <= 1e-5


def _exact(x_T, times, k, c):
    """Closed-form solution of the probability-flow ODE for a constant data prediction c, at times[k] (float64)."""
    ac = SCHED["alphas_cumprod"].double()
    t = times[k]
    if t < 0:
        return torch.full_like(x_T, c, dtype=torch.float64)
    aT, sT = ac[times[0]].sqrt(), (1 - ac[times[0]]).sqrt()
    a, s = ac[t].sqrt(), (1 - ac[t]).sqrt()
    return (s / sT) * x_T.double() + (a - aT * s / sT) * c


@pytest.mark.parametrize("order", [1, 2, 3])
def test_constant_prediction_is_exact(order):
    """With D = c every difference term vanishes and each order integrates the ODE exactly: fp32 to 1e-6 at every grid
    point for S <= 20 (measured <= 6.3e-7; at S = 50 the rounding of 50 steps reaches 1.7e-6), float64 to 1e-12 at S = 50."""
    x_T = torch.randn(2, 2, 8, 8, generator=torch.Generator().manual_seed(0))
    for c in (-1.0, -0.3, 0.7, 1.0):
        model = lambda x, cc, t: torch.full_like(x, c)  # noqa: E731
        for S, dtype, tol in ((5, torch.float32, 1e-6), (10, torch.float32, 1e-6), (20, torch.float32, 1e-6),
                              (50, torch.float64, 1e-12)):
            x0 = x_T.to(dtype)
            traj, _ = P.dpmpp_sample(None, SCHED, x0, None, 1000, S, order, return_all=True, model=model)
            times = O.ddim_times(1000, S)
            err = max((traj[:, k].double() - _exact(x0, times, k, c)).abs().max().item() for k in range(1, S + 1))
            assert err <= tol, (c, S, dtype, err)


A, B_T = 1.0, 2.0


def _analytic(x, c, t):
    """A cheap smooth data prediction: D(x, t) = tanh(a x + b t / T)."""
    return torch.tanh(A * x + B_T * t.to(x.dtype).view(-1, 1, 1, 1) / 1000)


def test_convergence():
    """Errors against a 3M run with 1000 steps (max |err|, fp32, D(x, t) = tanh(x + 2 t / T), x_T ~ N(0, 1) 2x2x16x16).

    (a) The whole sampler on the DDIM grid, error of the last ODE state x(t_{S-1}) against the reference at the same t
        (the step to -1 returns D(x(t_{S-1}), t_{S-1}) for every solver alike).  Measured:
            S = 10: DDIM 7.46e-2, 2M 2.05e-2, 3M 2.10e-2 | S = 20: DDIM 4.42e-2, 2M 4.98e-3, 3M 4.16e-3
            S = 40: DDIM 2.58e-2, 2M 1.91e-3, 3M 1.12e-3 | S = 80: DDIM 1.50e-2
        2M with S steps beats DDIM with 2S at every S.  The observed orders on this grid are not the solvers' orders: the
        first step leaves t = 999 (alphas_cumprod = 3e-7) and spans h = 5.9, 5.5, 5.1, 4.8 in log-SNR at S = 10, 20, 40,
        80, so the order-1 warm-up step there does not shrink with S and bounds the endpoint's convergence.
    (b) The multistep formulas' own order: the oracle's step on the integer sub-grid t = 819 -> 19 with n = 10, 20, 40
        uniform steps, started from the reference state with the two earlier predictions taken on the reference trajectory
        (so every step runs at full order).  Measured: 1 -> 6.87e-2, 3.60e-2, 1.84e-2; 2M -> 1.84e-2, 5.79e-3, 1.77e-3;
        3M -> 1.71e-2, 3.90e-3, 6.44e-4; observed order n = 20 -> 40: 0.97, 1.71, 2.60 (asserted >= 0.8, 1.6, 2.4)."""
    x_T = torch.randn(2, 2, 16, 16, generator=torch.Generator().manual_seed(0))
    ref, _ = P.dpmpp_sample(None, SCHED, x_T, None, 1000, 1000, 3, return_all=True, model=_analytic)
    ref_times = O.ddim_times(1000, 1000)

    def at(t):
        return ref[:, ref_times.index(t)]

    err = {}
    for S in (10, 20, 40, 80):
        last = O.ddim_times(1000, S)[-2]
        d, _ = O.ddim_sample(None, SCHED, x_T, None, 1000, S, return_all=True, model=_analytic)
        err[("ddim", S)] = (d[:, -2] - at(last)).abs().max().item()
        if S < 80:
            for order in (2, 3):
                tr, _ = P.dpmpp_sample(None, SCHED, x_T, None, 1000, S, order, return_all=True, model=_analytic)
                err[(order, S)] = (tr[:, -2] - at(last)).abs().max().item()
    print("endpoint errors", {k: f"{v:.3e}" for k, v in err.items()})
    for S in (10, 20, 40):
        assert err[(2, S)] < err[("ddim", 2 * S)], (S, err)
        assert err[(3, S)] < err[("ddim", 2 * S)], (S, err)

    sub = {}
    for order in (1, 2, 3):
        for n in (10, 20, 40):
            dt = 800 // n
            times = [819 + 2 * dt, 819 + dt] + list(range(819, 18, -dt))
            ds = [torch.clamp(_analytic(at(t), None, torch.full((2,), t)), -1, 1) for t in times[:2]]
            x = at(819)
            for i in range(2, len(times) - 1):
                out = _analytic(x, None, torch.full((2,), times[i]))
                x, d0 = P.dpmpp_update(x, out, ds[-1], ds[-2], P.dpmpp_coeffs(SCHED, times, i, order))
                ds.append(d0)
            sub[(order, n)] = (x - at(19)).abs().max().item()
    rates = {order: math.log2(sub[(order, 20)] / sub[(order, 40)]) for order in (1, 2, 3)}
    print("sub-grid errors", {k: f"{v:.3e}" for k, v in sub.items()}, "orders 20 -> 40", rates)
    assert rates[1] >= 0.8 and rates[2] >= 1.6 and rates[3] >= 2.4, rates


def test_coefficients_package_vs_oracle():
    """diffusion.dpmpp_coeffs (expanded closed form) == the oracle's linear map read off the paper's update, float64."""
    from opticalflowdiffusion_b200.diffusion import dpmpp_coeffs
    ac = SCHED["alphas_cumprod"].tolist()
    worst = 0.0
    for S in (2, 3, 5, 10, 50, 200, 1000):
        times = O.ddim_times(1000, S)
        for order in (1, 2, 3):
            for i in range(S):
                got, ref = dpmpp_coeffs(ac, times, i, order), P.dpmpp_coeffs(SCHED, times, i, order)
                assert got[4] == ref[4] and (ref[4] == 1) == (i == S - 1)
                for g, r in zip(got[:4], ref[:4]):
                    if r == 0.0:
                        assert g == 0.0, (S, order, i, got, ref)
                    else:
                        worst = max(worst, abs(g - r) / abs(r))
                k = min(order, i + 1) if not ref[4] else 1
                assert (got[2] != 0.0) == (k >= 2) and (got[3] != 0.0) == (k >= 3), (S, order, i, got)
    assert worst <= 1e-12, worst


def test_config_and_constructor():
    """sampler defaults to null (today's DDIM / DDPM dispatch); dpmpp and solver_order reach ConditionalDiffusion;
    eta > 0 (the SDE variants) and unknown samplers / orders are refused."""
    from opticalflowdiffusion_b200 import FlowDiffuser
    from opticalflowdiffusion_b200.config import compose
    from opticalflowdiffusion_b200.diffusion import ConditionalDiffusion
    a = compose().algorithm
    assert a.sampler is None and a.solver_order == 2
    m = FlowDiffuser(compose(["algorithm.target=flow", "algorithm.sampling_timesteps=10"]).algorithm)
    assert m.model.sampler is None
    m = FlowDiffuser(compose(["algorithm.target=flow", "algorithm.sampling_timesteps=10", "algorithm.sampler=dpmpp",
                              "algorithm.solver_order=3"]).algorithm)
    assert m.model.sampler == "dpmpp" and m.model.solver_order == 3
    net = torch.nn.Identity()
    with pytest.raises(NotImplementedError):
        ConditionalDiffusion(net, 16, sampling_timesteps=10, ddim_sampling_eta=0.5, sampler="dpmpp")
    with pytest.raises(ValueError):
        ConditionalDiffusion(net, 16, sampler="unipc")
    with pytest.raises(ValueError):
        ConditionalDiffusion(net, 16, sampler="dpmpp", solver_order=4)
