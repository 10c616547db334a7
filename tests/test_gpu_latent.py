"""-m gpu: flow_diffuser's latent mode (``latent: true``; SURVEY.md section 8f row N4) on the CUDA path against the golden
produced by the reference's own ``Autoencoder`` / ``FlowDiffuser`` (oracle/make_goldens_latent.py): the three-level,
time-free autoencoder UNets (flow_pred.py:17-58), the 33-channel flow UNet with the wide init_conv
(flow_diffuser.py:98-110), the frozen-autoencoder preprocess (:143-148) and the 16-channel pyramid loss.

Tolerances (bf16 activations / tensor-core operands vs the fp32 reference): latents and decoded images <= 3e-2 absolute
on [-1, 1] / [0, 1] data (same bound as the flow UNet's prediction, tests/test_gpu_unet.py); given the reference's flow
prediction the loss kernels agree to 1e-5 relative; end to end (bf16 UNet under the level^4-weighted pyramid) the loss agrees
to 3e-2 relative and the init_conv / final_conv gradients to 10 % relative L2 with cosine >= 0.99.
Measured on B200: latent max / mean error 0.017 / 0.0024, decoded 0.0070 / 0.0013, loss 0.84 %, gradients 1.5 % (final_conv),
4.4 % (init_conv.weight: the 49-tap wide path forward and its wgrad), 2.6 % (init_conv.bias), cosines >= 0.999."""
import os

import numpy as np
import pytest
import torch

from oracle import latent_golden

pytestmark = pytest.mark.gpu


def T(a):
    return torch.from_numpy(np.asarray(a))


def cfg_latent(**over):
    from opticalflowdiffusion_b200.config import compose
    cfg = compose(["algorithm.target=target", "algorithm.zero_init=false", "algorithm.latent=true"]).algorithm
    for k, v in over.items():
        cfg[k] = v
    return cfg


def make_autoencoder(g):
    from opticalflowdiffusion_b200.flow_pred import Autoencoder
    torch.manual_seed(int(g["ae_seed"]))
    ae = Autoencoder(cfg_latent())
    sums = np.array([float(v.double().sum()) for v in ae.state_dict().values()])
    np.testing.assert_allclose(sums, g["ae_w_sums"], rtol=1e-12, atol=1e-12)
    return ae


def make_algo(g, tmp_path):
    """The reference's own loading route: a FlowPred-style checkpoint ({'state_dict': {'ae.*': ...}}) read at construction."""
    from opticalflowdiffusion_b200 import FlowDiffuser
    ae = make_autoencoder(g)
    path = os.path.join(str(tmp_path), "model.ckpt")
    torch.save({"state_dict": {"ae." + k: v for k, v in ae.state_dict().items()}}, path)
    torch.manual_seed(int(g["seed"]))
    m = FlowDiffuser(cfg_latent(ae_checkpoint=path))
    assert m.ae_loaded and not any(p.requires_grad for p in m.ae.parameters())
    assert m.unet.channels == 33 and m.dim == 16
    sums = np.array([float(v.double().sum()) for v in m.unet.state_dict().values()])
    np.testing.assert_allclose(sums, g["w_sums"], rtol=1e-12, atol=1e-12)
    return m.cuda()


def test_autoencoder_encode_decode_vs_reference(golden):
    g = latent_golden.load(golden("latent_32x48"))
    ae = make_autoencoder(g).cuda()
    img, flow = T(g["img"]).cuda(), T(g["flow"]).cuda()
    lat = ae.encode(img)
    e_lat = (lat.cpu() - T(g["latent"])).abs()
    dec = ae.decode(T(g["latent"]).cuda(), img)
    e_dec = (dec.cpu() - T(g["decoded"])).abs()
    print("latent max/mean err", float(e_lat.max()), float(e_lat.mean()), "decoded", float(e_dec.max()), float(e_dec.mean()))
    assert lat.shape == (2, 16, 32, 48) and float(lat.abs().max()) <= 1.0
    assert float(e_lat.max()) <= 3e-2 and float(e_lat.mean()) <= 4e-3
    assert float(e_dec.max()) <= 3e-2 and float(e_dec.mean()) <= 4e-3
    # forward = encode, splat along the flow, decode: the splat's holes are NaN and the decoder spreads them everywhere
    # in the reference (GroupNorm / attention); same here
    wl = ae(img, flow, return_latent=True)
    assert torch.equal(torch.isnan(wl.cpu()), torch.isnan(T(g["ae_forward_latent"])))
    assert float((torch.nan_to_num(wl.cpu()) - torch.nan_to_num(T(g["ae_forward_latent"]))).abs().max()) <= 6e-2
    # shapes whose sides are multiples of 4 but not of 8 run unpadded, like the reference's three-level UNet
    assert ae.encode(torch.rand(1, 3, 20, 36, device="cuda")).shape == (1, 16, 20, 36)
    # the autoencoder is frozen: with autograd on it still runs the inference kernels; unfrozen it refuses
    ae.requires_grad_(False)                     # flow_diffuser.py:93-94
    with torch.enable_grad():
        assert not ae.model_enc(2 * img - 1).requires_grad
        for p in ae.model_enc.parameters():
            p.requires_grad_(True)
        with pytest.raises(NotImplementedError, match="three-level"):
            ae.model_enc(2 * img - 1)


def test_latent_preprocess_and_loss_vs_reference(golden, tmp_path):
    g = latent_golden.load(golden("latent_32x48"))
    m = make_algo(g, tmp_path)
    first, cond, flow_n = m.preprocess((T(g["img"]).cuda(), T(g["tgt"]).cuda(), T(g["flow"]).cuda()), aug=False)
    assert first.shape == (2, 16, 32, 48) and cond.shape == (2, 16, 32, 48)
    assert float((cond.cpu() - T(g["cond"])).abs().max()) <= 3e-2
    assert torch.equal(torch.isnan(first.cpu()), torch.isnan(T(g["first"])))          # the holes depend on the flow only
    np.testing.assert_allclose(flow_n.cpu().numpy(), g["flow_n"], rtol=0, atol=1e-7)
    # loss kernels over 16 channels given the reference's inputs and flow prediction: value and gradient
    first, cond, flow_n = T(g["first"]).cuda(), T(g["cond"]).cuda(), T(g["flow_n"]).cuda()
    t, noise = T(g["t"]).cuda(), T(g["noise"]).cuda()
    fp = T(g["flow_pred"]).cuda().requires_grad_(True)
    kw = dict(additional_tgt=flow_n, additional_weight=0.0)
    loss = m.model.p_losses(first, t, noise=noise, external_cond=cond, model_out_override=(m._model._warp(cond, fp), fp), **kw)
    np.testing.assert_allclose(float(loss.detach()), float(g["loss"]), rtol=1e-5)
    loss.backward()
    ref = g["grad_flow_pred"]
    assert np.abs(fp.grad.cpu().numpy() - ref).max() <= 1e-4 * np.abs(ref).max()
    # end to end through the 33-channel UNet (wide init_conv, forward and backward kernels)
    m.zero_grad()
    loss = m.model.p_losses(first, t, noise=noise, external_cond=cond, **kw)
    rel = abs(float(loss.detach()) - float(g["loss"])) / float(g["loss"])
    loss.backward()
    out = {}
    for name, p, ref in (("final_conv.weight", m.unet.final_conv.weight, g["grad_final_conv_w"]),
                         ("init_conv.weight", m.unet.init_conv.weight, g["grad_init_conv_w"]),
                         ("init_conv.bias", m.unet.init_conv.bias, g["grad_init_conv_b"])):
        got = p.grad.cpu().numpy()
        out[name] = (float(np.linalg.norm(got - ref) / np.linalg.norm(ref)),
                     float((got * ref).sum() / (np.linalg.norm(got) * np.linalg.norm(ref))))
    print("latent e2e loss", float(loss.detach()), "reference", float(g["loss"]), "rel", rel, "grads (rel L2, cosine)", out)
    assert rel <= 3e-2, rel
    for name, (r, c) in out.items():
        assert r <= 0.1 and c >= 0.99, (name, r, c)


def test_latent_training_step_sampling_and_validation(golden, tmp_path):
    g = latent_golden.load(golden("latent_32x48"))
    m = make_algo(g, tmp_path)
    m.model.sampling_timesteps, m.model.is_ddim_sampling = 3, True
    opt = m.configure_optimizers()
    batch = (T(g["img"]).cuda(), T(g["tgt"]).cuda(), T(g["flow"]).cuda())
    before = m.unet.init_conv.weight.detach().clone()
    ae_before = m.ae.model_enc.init_conv.weight.detach().clone()
    torch.manual_seed(1)
    tgt_, cond, flow_ = m.preprocess(batch, aug=False)
    loss = m.loss(tgt_, cond, flow_)
    loss.backward()
    opt.step()
    assert torch.isfinite(loss) and not torch.equal(before, m.unet.init_conv.weight)
    assert torch.equal(ae_before, m.ae.model_enc.init_conv.weight)                    # frozen
    samples, flows = m.sample(cond, flow_)
    last = samples[:, -1] if samples.dim() == 5 else samples
    assert last.shape == (2, 16, 32, 48)
    pf = flows[-1]
    assert pf.shape == (2, 2, 32, 48) and torch.isfinite(pf).all()
    m.logged = {}
    m.log_dict = lambda d, **k: m.logged.update({a: float(b) for a, b in d.items()})
    m.validation_step(batch, 0)
    assert {"val/loss", "val/mse", "val/ideal_loss"} <= set(m.logged) and np.isfinite(m.logged["val/loss"])
    dec = m.ae.decode(torch.nan_to_num(last) * m.latent_max, batch[0])
    assert dec.shape == (2, 3, 32, 48) and float(dec.min()) >= 0.0 and float(dec.max()) <= 1.0
