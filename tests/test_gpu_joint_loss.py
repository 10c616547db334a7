"""-m gpu: the joint / target pyramid loss (reference default ``target: joint``; denoising_diffusion.py:886-889,893-983,
flow_diffuser.py:38-63) on the CUDA path against goldens produced by the reference's own ``p_losses``
(oracle/make_goldens_joint.py).

Tolerances: given the reference's flow prediction the loss value agrees to 1e-5 relative and its gradient w.r.t. the
prediction to 1e-4 of its max (fp32 kernels, atomics reorder sums); end to end through the bf16 UNet the loss agrees to
5e-2 relative (the level^4-weighted splat terms amplify the bf16 error of the flow: a 1e-2 flow error is 0.2 px) and
the final_conv gradients to 30 % relative L2 with cosine >= 0.98 (see the comment at the assertion)."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu


def T(a):
    return torch.from_numpy(np.asarray(a))


def make_algo(g, target):
    from opticalflowdiffusion_b200 import FlowDiffuser
    from opticalflowdiffusion_b200.config import compose
    torch.manual_seed(int(g["seed"]))
    m = FlowDiffuser(compose([f"algorithm.target={target}", "algorithm.zero_init=false"]).algorithm)
    sums = np.array([float(v.double().sum()) for v in m.unet.state_dict().values()])
    np.testing.assert_allclose(sums, g["w_sums"], rtol=1e-12, atol=1e-12)
    return m.cuda()


def kwargs(g, target):
    return dict(additional_tgt=T(g["flow_n"]).cuda(), additional_weight=0.0) if target == "target" else {}


@pytest.mark.parametrize("target", ["joint", "target"])
def test_preprocess_matches_reference(golden, target):
    g = golden(f"p_losses_{target}_32x48")
    m = make_algo(g, target)
    first, cond, flow_n = m.preprocess((T(g["img"]).cuda(), T(g["tgt"]).cuda(), T(g["flow"]).cuda()), aug=False)
    ref = T(g["first"])
    assert first.shape == ref.shape, (first.shape, ref.shape)
    assert torch.equal(torch.isnan(first.cpu()), torch.isnan(ref)), (int(torch.isnan(first).sum()), int(torch.isnan(ref).sum()))
    np.testing.assert_allclose(torch.nan_to_num(first.cpu()).numpy(), torch.nan_to_num(ref).numpy(), rtol=1e-5, atol=2e-5)
    np.testing.assert_allclose(cond.cpu().numpy(), g["cond"], rtol=0, atol=1e-7)
    np.testing.assert_allclose(flow_n.cpu().numpy(), g["flow_n"], rtol=0, atol=1e-7)


@pytest.mark.parametrize("target", ["joint", "target"])
def test_pyramid_loss_value_and_gradient_given_reference_prediction(golden, target):
    g = golden(f"p_losses_{target}_32x48")
    m = make_algo(g, target)
    first, cond, flow_n = T(g["first"]).cuda(), T(g["cond"]).cuda(), T(g["flow_n"]).cuda()
    fp = T(g["flow_pred"]).cuda().requires_grad_(True)
    warped = m._model._warp(cond, fp)
    override = (warped, fp) if target == "target" else (torch.cat((warped, fp), dim=1), None)
    loss = m.model.p_losses(first, T(g["t"]).cuda(), noise=T(g["noise"]).cuda(), external_cond=cond,
                            model_out_override=override, **kwargs(g, target))
    np.testing.assert_allclose(float(loss.detach()), float(g["loss"]), rtol=1e-5)
    loss.backward()
    ref = g["grad_flow_pred"]
    err = np.abs(fp.grad.cpu().numpy() - ref).max() / np.abs(ref).max()
    assert err <= 1e-4, err
    # val/ideal_loss (flow_diffuser.py:256-259)
    with torch.no_grad():
        wi = m._model._warp(cond, flow_n)
        ov = (wi, flow_n) if target == "target" else (torch.cat((wi, flow_n), dim=1), None)
        ideal = m.model.p_losses(first, T(g["t"]).cuda(), noise=T(g["noise"]).cuda(), external_cond=cond,
                                 model_out_override=ov, **kwargs(g, target))
    assert abs(float(ideal) - float(g["ideal_loss"])) <= 1e-8


@pytest.mark.parametrize("target", ["joint", "target"])
def test_p_losses_end_to_end_through_the_unet(golden, target):
    g = golden(f"p_losses_{target}_32x48")
    m = make_algo(g, target)
    first, cond = T(g["first"]).cuda(), T(g["cond"]).cuda()
    loss = m.model.p_losses(first, T(g["t"]).cuda(), noise=T(g["noise"]).cuda(), external_cond=cond, **kwargs(g, target))
    rel = abs(float(loss.detach()) - float(g["loss"])) / float(g["loss"])
    print(target, "loss", float(loss.detach()), "reference", float(g["loss"]), "rel", rel)
    assert rel <= 5e-2, rel
    loss.backward()
    # gradient anchors of the reference's own backward (through splat_flowgrad and the whole UNet)
    # (relative L2 over the tensor: the level^4-weighted splat terms put a 0.2 px flow error of the bf16 UNet on a bilinear
    #  cell border here and there, which moves single entries by up to ~10 % of the largest one)
    gw, rw = m.unet.final_conv.weight.grad.cpu().numpy(), g["grad_final_conv_w"]
    rel_w = np.linalg.norm(gw - rw) / np.linalg.norm(rw)
    gb, rb = m.unet.final_conv.bias.grad.cpu().numpy(), g["grad_final_conv_b"]
    rel_b = np.linalg.norm(gb - rb) / np.linalg.norm(rb)
    cos_w = float((gw * rw).sum() / (np.linalg.norm(gw) * np.linalg.norm(rw)))
    print(target, "final_conv grad rel L2: weight", rel_w, "bias", rel_b, "cosine", cos_w)
    # measured on B200: joint 9-11 % / 6-11 %, target 6-9 % with the shipped kernels, and up to 17 % / 26 % (cosine 0.986) with
    # a two-pass variant of the training forward's residual GroupNorm (a different rounding path puts other pixels across a
    # splat cell border) while the loss itself agrees to 3e-4: this loss is ill-conditioned in the flow (a bilinear splat cell border is a
    # kink), so the end-to-end bound is loose -- the exact check of the loss kernels is the test above (1e-4)
    assert rel_w <= 0.3 and rel_b <= 0.3 and cos_w >= 0.98, (rel_w, rel_b, cos_w)
