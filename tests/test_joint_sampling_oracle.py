"""CPU: the oracle's sampler with ``target: joint`` (``O.ddpm_sample`` around ``O.unet_with_warp``; reference
denoising_diffusion.py:700-729 + flow_diffuser.py:20-63) against the trajectory of the UNMODIFIED reference
(oracle/make_goldens_joint_sampling.py: p_sample_loop over T = 5 steps, NaN holes of the forward splat carried in the state).

Tolerance: fp32 on both sides.  The hole pattern (NaN mask) must agree (<= 0.05 % of the entries may differ: splat weights at
the rounding level; measured 0).  The map state -> next state is ill-conditioned (a last-bit change of the predicted flow
moves splat weight between neighbouring cells), so rounding differences grow ~8x per step: measured max |err| 2e-7, 2e-5,
7e-5, 5e-4, 6e-3 over the five steps -- asserted: first step 2e-6, whole trajectory 2e-2 max and 1e-4 mean."""
import numpy as np
import pytest
import torch

from oracle import flowdiff_oracle as O

pytestmark = pytest.mark.usefixtures("golden_threads")


def T(a):
    return torch.from_numpy(np.asarray(a))


def joint_state(g):
    from opticalflowdiffusion_b200.unet_params import UnetParams
    torch.manual_seed(int(g["seed"]))
    sd = UnetParams(64, channels=9, out_dim=2).state_dict()
    sd["final_conv.weight"] = sd["final_conv.weight"] * float(g["head_scale"])
    sums = np.array([float(v.double().sum()) for v in sd.values()])
    np.testing.assert_allclose(sums, g["w_sums"], rtol=1e-12, atol=1e-12)
    return sd


def compare(traj, ref, max_mask_mismatch, atol, mean_tol=None):
    traj, ref = np.asarray(traj), np.asarray(ref)
    assert traj.shape == ref.shape
    mism = float((np.isnan(traj) != np.isnan(ref)).mean())
    both = ~np.isnan(traj) & ~np.isnan(ref)
    err = np.abs(np.where(both, traj - ref, 0.0))
    assert mism <= max_mask_mismatch, mism
    assert err.max() <= atol, err.max()
    if mean_tol is not None:
        assert err.sum() / both.sum() <= mean_tol, err.sum() / both.sum()
    return mism, float(err.max()), float(err.sum() / both.sum())


def test_joint_ddpm_trajectory(golden):
    g = golden("joint_ddpm5_32x48")
    sd = joint_state(g)
    sched = O.make_schedule(5)
    with torch.no_grad():
        traj = O.ddpm_sample(sd, sched, T(g["x_T"]), T(g["cond"]), 5, list(T(g["noises"])), return_all=True,
                             model=lambda x, c, t: O.unet_with_warp(sd, x, c, t, 20.0, True, False))
    ref = g["traj"]
    assert np.isnan(ref[:, -1, :3]).mean() > 0.2 and not np.isnan(ref[:, :, 3:]).any()      # holes in the image, none in the flow
    compare(traj.numpy()[:, :2], ref[:, :2], 0.0, 2e-6)
    compare(traj.numpy(), ref, 5e-4, 2e-2, mean_tol=1e-4)
