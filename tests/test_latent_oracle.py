"""CPU: the oracle's restatement of flow_diffuser's latent mode (``O.autoencoder_encode / _decode / _forward``,
``O.latent_preprocess``, ``O.p_losses_target(dim=16)``; reference flow_pred.py:17-58, flow_diffuser.py:81-95,143-168,
denoising_diffusion.py:823-983) against the golden produced by the UNMODIFIED reference classes
(oracle/make_goldens_latent.py).

The autoencoder / UNet weights are re-created from the recorded seeds with this package's parameter holders (same
construction order and initialisers as the reference; the per-tensor checksums in the golden prove it).
Tolerances: fp32 on both sides with different summation orders -> 2e-5 absolute on the [-1, 1] latents / [0, 1] images;
the level^4-weighted pyramid loss 2e-4 relative end to end, 2e-6 given the reference's own flow prediction."""
import numpy as np
import pytest
import torch

from oracle import flowdiff_oracle as O
from oracle import latent_golden

pytestmark = pytest.mark.usefixtures("golden_threads")


def T(a):
    return torch.from_numpy(np.asarray(a))


def ae_state(g):
    from opticalflowdiffusion_b200.unet_params import UnetParams
    torch.manual_seed(int(g["ae_seed"]))
    enc = UnetParams(64, channels=3, out_dim=16, dim_mults=(1, 2, 4), time_in=False)
    dec = UnetParams(64, channels=19, out_dim=3, dim_mults=(1, 2, 4), time_in=False)
    sd = {**{"model_enc." + k: v for k, v in enc.state_dict().items()}, **{"model_dec." + k: v for k, v in dec.state_dict().items()}}
    sums = np.array([float(v.double().sum()) for v in sd.values()])
    np.testing.assert_allclose(sums, g["ae_w_sums"], rtol=1e-12, atol=1e-12)
    return sd


def unet_state(g):
    """FlowDiffuser.__init__ builds the autoencoder first (consuming the generator), then the 33-channel UNet."""
    from opticalflowdiffusion_b200.unet_params import UnetParams
    torch.manual_seed(int(g["seed"]))
    UnetParams(64, channels=3, out_dim=16, dim_mults=(1, 2, 4), time_in=False)
    UnetParams(64, channels=19, out_dim=3, dim_mults=(1, 2, 4), time_in=False)
    sd = UnetParams(64, channels=33, out_dim=2).state_dict()
    sums = np.array([float(v.double().sum()) for v in sd.values()])
    np.testing.assert_allclose(sums, g["w_sums"], rtol=1e-12, atol=1e-12)
    return sd


def same_with_nans(a, b, atol):
    a, b = np.asarray(a), np.asarray(b)
    assert np.array_equal(np.isnan(a), np.isnan(b))
    if np.isnan(a).all():
        return
    assert np.nanmax(np.abs(a - b)) <= atol, np.nanmax(np.abs(a - b))


def test_autoencoder_and_preprocess(golden):
    g = latent_golden.load(golden("latent_32x48"))
    sd = ae_state(g)
    img, flow = T(g["img"]), T(g["flow"])
    with torch.no_grad():
        lat = O.autoencoder_encode(sd, img)
        assert np.abs(lat.numpy() - g["latent"]).max() <= 2e-5
        assert float(lat.abs().max()) == 1.0                      # the clamp is active on this input (4.5 % of the latent)
        dec = O.autoencoder_decode(sd, T(g["latent"]), img)
        assert np.abs(dec.numpy() - g["decoded"]).max() <= 2e-5
        same_with_nans(O.warp_forward_flow(T(g["latent"]), flow).numpy(), g["ae_forward_latent"], 1e-6)
        # (with holes in the splat the reference's decoder output is NaN everywhere -- GroupNorm / attention spread them --
        # which is what "dec_gt" logs there, flow_diffuser.py:308; kept)
        assert np.isnan(g["ae_forward"]).all() and np.isnan(g["ae_forward_latent"]).any()
        full = O.autoencoder_forward(sd, img, flow)
        same_with_nans(full.numpy(), g["ae_forward"], 5e-5)
        first, cond, flow_n = O.latent_preprocess(sd, img, flow, target="target")
    assert np.abs(cond.numpy() - g["cond"]).max() <= 2e-5
    assert np.array_equal(flow_n.numpy(), g["flow_n"])
    same_with_nans(first.numpy(), g["first"], 5e-5)


def test_latent_p_losses_target(golden):
    g = latent_golden.load(golden("latent_32x48"))
    first, cond, flow_n, t, noise = T(g["first"]), T(g["cond"]), T(g["flow_n"]), T(g["t"]), T(g["noise"])
    # given the reference's own flow prediction: value and gradient of the 16-channel pyramid loss
    fp = T(g["flow_pred"]).clone().requires_grad_(True)
    out = torch.cat((O.warp_forward_flow(cond[:, :16], fp * 20.0), fp), 1)
    loss = O.p_losses_target(None, None, first, cond, flow_n, None, None, model_out=out, dim=16)
    np.testing.assert_allclose(float(loss.detach()), float(g["loss"]), rtol=2e-6)
    loss.backward()
    ref = g["grad_flow_pred"]
    assert np.abs(fp.grad.numpy() - ref).max() <= 1e-4 * np.abs(ref).max()
    # end to end through the 33-channel UNet (wide init_conv)
    sd = {k: v.clone().requires_grad_(True) for k, v in unet_state(g).items()}
    sched = O.make_schedule(1000)
    loss = O.p_losses_target(sd, sched, first, cond, flow_n, t, noise, dim=16)
    np.testing.assert_allclose(float(loss.detach()), float(g["loss"]), rtol=2e-4)
    loss.backward()
    for k, ref in (("final_conv.weight", g["grad_final_conv_w"]), ("init_conv.weight", g["grad_init_conv_w"]),
                   ("init_conv.bias", g["grad_init_conv_b"])):
        got = sd[k].grad.numpy()
        assert np.abs(got - ref).max() <= 2e-3 * np.abs(ref).max(), k
