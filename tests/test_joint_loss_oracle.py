"""CPU: the oracle's restatement of the joint / target pyramid loss (``O.p_losses_joint`` / ``O.p_losses_target`` /
``O.pyramid_loss``; reference denoising_diffusion.py:823-983 + flow_diffuser.py:20-63) against goldens produced by the
UNMODIFIED reference classes (oracle/make_goldens_joint.py; the reference's own splat kernels compiled for the host).

Tolerances: loss value 1e-4 relative end to end through the fp32 UNet (the level^4-weighted pyramid amplifies last-bit
differences of the flow prediction), 2e-6 relative given the reference's own flow prediction; gradient w.r.t. the flow
prediction 1e-4 of its max."""
import numpy as np
import pytest
import torch

from oracle import flowdiff_oracle as O

pytestmark = pytest.mark.usefixtures("golden_threads")


def T(a):
    return torch.from_numpy(np.asarray(a))


def _sd(g, channels):
    from opticalflowdiffusion_b200.unet_params import UnetParams
    torch.manual_seed(int(g["seed"]))
    sd = UnetParams(64, channels=channels, out_dim=2).state_dict()
    sums = np.array([float(v.double().sum()) for v in sd.values()])
    np.testing.assert_allclose(sums, g["w_sums"], rtol=1e-12, atol=1e-12)
    return sd


def _model_out(g, target, fp):
    warped = O.warp_forward_flow(T(g["cond"])[:, :3], fp * 20.0)
    return torch.cat((warped, fp), 1)      # joint: full_output; target: additional_out (flow_diffuser.py:57-63)


@pytest.mark.parametrize("target,channels", [("joint", 9), ("target", 7)])
def test_pyramid_loss_given_reference_prediction(golden, target, channels):
    g = golden(f"p_losses_{target}_32x48")
    fp = T(g["flow_pred"]).clone().requires_grad_(True)
    first, cond, flow_n = T(g["first"]), T(g["cond"]), T(g["flow_n"])
    out = _model_out(g, target, fp)
    if target == "joint":
        loss = O.p_losses_joint(None, None, first, cond, None, None, model_out=out)
    else:
        loss = O.p_losses_target(None, None, first, cond, flow_n, None, None, model_out=out)
    np.testing.assert_allclose(float(loss.detach()), float(g["loss"]), rtol=2e-6)
    loss.backward()
    ref = g["grad_flow_pred"]
    assert np.abs(fp.grad.numpy() - ref).max() <= 1e-4 * np.abs(ref).max()
    # "val/ideal_loss": the model output overridden by the ground truth
    with torch.no_grad():
        warped = O.warp_forward_flow(cond[:, :3], flow_n * 20.0)
        ideal = O.pyramid_loss(warped, first[:, :3], flow_n, cond)
    assert abs(float(ideal) - float(g["ideal_loss"])) <= 1e-9


@pytest.mark.parametrize("target,channels", [("joint", 9), ("target", 7)])
def test_p_losses_end_to_end(golden, target, channels):
    g = golden(f"p_losses_{target}_32x48")
    sd = {k: v.clone().requires_grad_(True) for k, v in _sd(g, channels).items()}
    sched = O.make_schedule(1000)
    first, cond, flow_n, t, noise = T(g["first"]), T(g["cond"]), T(g["flow_n"]), T(g["t"]), T(g["noise"])
    if target == "joint":
        loss = O.p_losses_joint(sd, sched, first, cond, t, noise)
    else:
        loss = O.p_losses_target(sd, sched, first, cond, flow_n, t, noise)
    np.testing.assert_allclose(float(loss.detach()), float(g["loss"]), rtol=1e-4)
    loss.backward()
    gw, rw = sd["final_conv.weight"].grad.numpy(), g["grad_final_conv_w"]
    assert np.abs(gw - rw).max() <= 2e-3 * np.abs(rw).max()
    gb, rb = sd["init_conv.bias"].grad.numpy(), g["grad_init_conv_b"]
    assert np.abs(gb - rb).max() <= 2e-3 * np.abs(rb).max()
    s = float(sd["mid_attn.fn.fn.to_qkv.weight"].grad.double().abs().sum())
    assert abs(s - float(g["grad_mid_qkv_w_sum"])) <= 2e-3 * float(g["grad_mid_qkv_w_sum"])
