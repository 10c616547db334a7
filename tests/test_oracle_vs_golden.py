"""The CPU oracle (oracle/flowdiff_oracle.py) against golden vectors produced by the UNMODIFIED
reference (oracle/make_goldens.py).  This is what pins the oracle; everything on the GPU is then
compared with the oracle."""
import numpy as np
import pytest
import torch

from oracle import flowdiff_oracle as O

pytestmark = pytest.mark.usefixtures("golden_threads")
from opticalflowdiffusion_b200.unet_params import UnetParams


def T(a):
    return torch.from_numpy(np.asarray(a))


def _ref_weights(seed, channels, out_dim, gold):
    """Rebuild the reference's random init (same layer order + initialisers) and check the fingerprint."""
    torch.manual_seed(int(seed))
    p = UnetParams(64, channels=channels, out_dim=out_dim)
    sd = p.state_dict()
    sums = np.array([float(v.double().sum()) for v in sd.values()])
    asums = np.array([float(v.double().abs().sum()) for v in sd.values()])
    assert len(sums) == len(gold["w_sums"])
    np.testing.assert_allclose(sums, gold["w_sums"], rtol=1e-12, atol=1e-12)     # summation order differs per CPU
    np.testing.assert_allclose(asums, gold["w_asums"], rtol=1e-12, atol=1e-12)
    return sd


def test_schedule_bit_exact(golden):
    g = golden("schedule")
    s = O.make_schedule(1000)
    for k in O.SCHEDULE_BUFFERS:
        assert np.array_equal(s[k].numpy(), g[k]), k
    s6 = O.make_schedule(6)
    assert np.array_equal(s6["betas"].numpy(), g["betas_T6"])
    assert np.array_equal(s6["alphas_cumprod"].numpy(), g["alphas_cumprod_T6"])


@pytest.mark.parametrize("T_S", [(1000, 50), (1000, 7), (1000, 999), (50, 10), (6, 3)])
def test_ddim_grid_bit_exact(golden, T_S):
    g = golden("schedule")
    Tt, S = T_S
    assert O.ddim_times(Tt, S) == g[f"ddim_times_{Tt}_{S}"].tolist()


def test_nan_mse(golden):
    g = golden("misc")
    a, b = T(g["a"]), T(g["b"])
    assert np.array_equal(O.nan_mse(a, b).numpy(), g["nan_mse_mean"])
    assert np.array_equal(O.nan_mse(a, b, "none").numpy(), g["nan_mse_none"])


def test_backwarp_bit_exact(golden):
    g = golden("backwarp")
    out, mask = O.backwarp(T(g["img"]), T(g["flow"]))
    assert np.array_equal(mask.numpy(), g["mask"])
    assert np.array_equal(out.numpy(), g["out"])
    out2, mask2 = O.backwarp_torch(T(g["img"]), T(g["flow"]))
    assert np.array_equal(out2.numpy(), g["out"]) and np.array_equal(mask2.numpy(), g["mask"])
    np.testing.assert_allclose(O.charbonnier(T(g["img"]) - out).numpy(), g["charb"], rtol=1e-6, atol=0)


def test_backwarp_sintel_rows_bit_exact(golden):
    """The fp32 normalise/un-normalise round trip at W=1024, H=436 (SURVEY.md section 8a W1)."""
    g = golden("backwarp")
    full = torch.zeros(1, 2, 436, 1024)
    full[:, :, 200:204] = T(g["big_flow_rows"])
    img = T(g["big_img"].astype(np.float32))
    out, mask = O.backwarp(img, full)
    assert np.array_equal(mask[:, :, 200:204].numpy(), g["big_mask_rows"])
    assert np.array_equal(out[:, :, 200:204].numpy(), g["big_out_rows"])


def test_backwarp_grads(golden):
    g = golden("backwarp")
    img = T(g["img"]).requires_grad_(True)
    flow = T(g["flow"]).requires_grad_(True)
    out, _ = O.backwarp_torch(img, flow)
    (out * T(g["gout"])).sum().backward()
    np.testing.assert_allclose(img.grad.numpy(), g["grad_img"], rtol=1e-5, atol=1e-6)
    np.testing.assert_allclose(flow.grad.numpy(), g["grad_flow"], rtol=1e-5, atol=1e-5)


@pytest.mark.parametrize("cfg", [(1, 0, 0), (2, 0, 0), (2, 1, 1), (4, 1, 3), (8, 0, 0)])
def test_splat_vs_reference_kernels(golden, cfg):
    g = golden("splat")
    scale, ox, oy = cfg
    tag = f"s{scale}_{ox}_{oy}"
    x, flow = T(g["x"]), T(g["flow"])
    out = O.splat_forward(x, flow, scale, ox, oy)
    np.testing.assert_allclose(out.numpy(), g[f"out_{tag}"], rtol=1e-5, atol=1e-5)
    gout = T(g[f"gout_{tag}"])
    gin = O.splat_ingrad(x.shape, flow, gout, scale, ox, oy)
    np.testing.assert_allclose(gin.numpy(), g[f"gin_{tag}"], rtol=1e-5, atol=1e-5)
    gflow = O.splat_flowgrad(x, flow, gout, scale, ox, oy)
    np.testing.assert_allclose(gflow.numpy(), g[f"gflow_{tag}"], rtol=1e-4, atol=1e-4)


def test_unet_forward_and_taps(golden):
    g = golden("unet_flow_16x24")
    sd = _ref_weights(g["seed"], 5, 2, g)
    x, cond, t = T(g["x"]), T(g["cond"]), T(g["t"])
    with torch.no_grad():
        out, taps = O.unet_forward(sd, x, cond, t, return_taps=True)
        np.testing.assert_allclose(taps["temb"].numpy(), g["temb"], rtol=1e-5, atol=1e-6)
        for k in ("init_conv", "downs.0.0", "downs.0.2", "mid_block1", "mid_attn", "final_res_block"):
            np.testing.assert_allclose(taps[k].numpy(), g["tap_" + k], rtol=1e-4, atol=2e-5, err_msg=k)
        np.testing.assert_allclose(out.numpy(), g["unet_out"], rtol=1e-4, atol=2e-5)


def test_q_sample_loss_ddim_ddpm(golden):
    g = golden("unet_flow_16x24")
    sd = _ref_weights(g["seed"], 5, 2, g)
    sched = O.make_schedule(1000)
    x0, cond, t, noise = T(g["x0"]), T(g["cond"]), T(g["t"]), T(g["noise"])
    assert np.array_equal(O.q_sample(sched, x0, t, noise).numpy(), g["q_sample"])
    with torch.no_grad():
        loss = O.p_losses_flow(sd, sched, x0, cond, t, noise)
        np.testing.assert_allclose(loss.numpy(), g["p_losses"], rtol=1e-5)
        traj, _ = O.ddim_sample(sd, sched, T(g["ddim_xT"]), cond, 1000, 4, return_all=True)
        np.testing.assert_allclose(traj.numpy(), g["ddim4_traj"], rtol=1e-4, atol=1e-4)
        s6 = O.make_schedule(6)
        traj6 = O.ddpm_sample(sd, s6, T(g["ddpm_xT"]), cond, 6, list(T(g["ddpm_noises"])), return_all=True)
        np.testing.assert_allclose(traj6.numpy(), g["ddpm6_traj"], rtol=1e-4, atol=1e-4)


def test_loss_gradients(golden):
    g = golden("unet_flow_16x24")
    sd = _ref_weights(g["seed"], 5, 2, g)
    sd = {k: v.clone().requires_grad_(True) for k, v in sd.items()}
    sched = O.make_schedule(1000)
    loss = O.p_losses_flow(sd, sched, T(g["x0"]), T(g["cond"]), T(g["t"]), T(g["noise"]))
    loss.backward()
    np.testing.assert_allclose(sd["final_conv.weight"].grad.numpy(), g["grad_final_conv_w"], rtol=1e-3, atol=1e-6)
    np.testing.assert_allclose(sd["init_conv.bias"].grad.numpy(), g["grad_init_conv_b"], rtol=1e-3, atol=1e-6)
    np.testing.assert_allclose(float(sd["mid_attn.fn.fn.to_qkv.weight"].grad.double().abs().sum()),
                               float(g["grad_mid_qkv_w_sum"]), rtol=1e-3)


def test_joint_nan_mask_plumbing(golden):
    """UnetWithWarp's NaN -> 0 + mask channel (flow_diffuser.py:39-45) feeding the 9-channel UNet."""
    g = golden("unet_joint_16x16")
    sd = _ref_weights(g["seed"], 9, 2, g)
    x = T(g["x"]).clone()
    nans = torch.isnan(x)
    x[nans] = 0.0
    mask = torch.any(nans, dim=1)[:, None].float()
    with torch.no_grad():
        flow = O.unet_forward(sd, torch.cat((x, mask), 1), T(g["cond"]), T(g["t"]))
    np.testing.assert_allclose(flow.numpy(), g["flow"], rtol=1e-4, atol=2e-5)
