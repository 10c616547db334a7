"""TEST INFRASTRUCTURE ONLY.  Golden vectors for flow_diffuser's latent mode (``latent: true``, SURVEY.md section 8f row N4)
from the UNMODIFIED reference classes: ``Autoencoder`` (flow_pred.py:17-58: encode / decode / forward on two three-level
UNets without time input) and ``FlowDiffuser`` with the frozen autoencoder (flow_diffuser.py:81-95 load, :143-148 preprocess,
``ConditionalDiffusion.p_losses`` with target='target' over latent_dim = 16 channels).

The reference fetches the autoencoder weights from wandb (flow_diffuser.py:84-92); here a checkpoint of a seeded,
reference-initialised ``Autoencoder`` is written to the local path the reference looks at first
(outputs/loaded_checkpoints/diffusion_control/<ae>/model.ckpt, relative to a temporary working directory), so the reference's
own loading code runs as shipped.  The forward splat is the reference's kernels compiled for the host (oracle/build_ref.py),
as in oracle/make_goldens_joint.py.

The file keeps only what needs the reference to recompute; oracle/latent_golden.py restores the rest (inputs from their
seed, ``cond``, the forward latent) bit for bit.

Run in the build container:  python oracle/make_goldens_latent.py  ->  tests/golden/latent_32x48.npz
"""
import os
import sys
import tempfile

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle import build_ref, latent_golden, ref_stubs  # noqa: E402
from oracle.make_goldens import quiet, weight_checksums  # noqa: E402
from oracle.make_goldens_flow_learner import HostSplat  # noqa: E402

GOLD = os.path.join(ROOT, "tests", "golden")
AE_SEED, MODEL_SEED, INPUT_SEED = 7, 0, 43


def main():
    ns = ref_stubs.import_reference()
    build_ref.build()
    ns.softsplat_new.softsplat_func = HostSplat
    B, H, W = 2, 32, 48
    cfg = ref_stubs.reference_cfg(target="target", image_size=64, zero_init=False, latent=True)
    torch.manual_seed(AE_SEED)
    ae0 = ns.flow_pred.Autoencoder(cfg)
    ae_sums, ae_asums = weight_checksums(ae0.state_dict())
    cwd = os.getcwd()
    with tempfile.TemporaryDirectory() as tmp:
        d = os.path.join(tmp, "outputs", "loaded_checkpoints", "diffusion_control", cfg.ae)
        os.makedirs(d)
        torch.save({"state_dict": {"ae." + k: v for k, v in ae0.state_dict().items()}}, os.path.join(d, "model.ckpt"))
        os.chdir(tmp)
        try:
            torch.manual_seed(MODEL_SEED)
            m = quiet(ns.flow_diffuser.FlowDiffuser, cfg)
        finally:
            os.chdir(cwd)
    assert all(torch.equal(a, b) for a, b in zip(m.ae.state_dict().values(), ae0.state_dict().values()))
    assert not any(p.requires_grad for p in m.ae.parameters())
    sums, asums = weight_checksums(m.unet.state_dict())
    inputs = latent_golden.draw_inputs(INPUT_SEED)
    img, tgt, flow = (torch.from_numpy(inputs[k]) for k in ("img", "tgt", "flow"))
    t = torch.tensor([710, 64], dtype=torch.long)
    with torch.no_grad():
        latent = m.ae.encode(img)
        decoded = m.ae.decode(latent, img)
        ae_fwd = quiet(m.ae, img, flow)
        ae_lat = quiet(m.ae, img, flow, return_latent=True)
    first, cond, flow_n = quiet(m.preprocess, (img, tgt, flow), aug=False)
    noise = torch.from_numpy(inputs["noise"])
    grabbed = {}

    def hook(_m, _i, out):
        out.retain_grad()
        grabbed["flow_pred"] = out
    h = m.unet.register_forward_hook(hook)
    m.zero_grad()
    loss = quiet(m.model.p_losses, first, t, noise=noise.clone(), external_cond=cond, additional_tgt=flow_n,
                 additional_weight=cfg.flow_weight)
    quiet(loss.backward)
    h.remove()
    torch.autograd.set_detect_anomaly(False)
    fp = grabbed["flow_pred"]
    assert torch.equal(cond, latent / float(latent_golden.LATENT_MAX))
    out = dict(ae_seed=AE_SEED, seed=MODEL_SEED, ae_w_sums=ae_sums, ae_w_asums=ae_asums, w_sums=sums, w_asums=asums,
               input_seed=INPUT_SEED, input_sums=latent_golden.input_sums(inputs), t=t.numpy(),
               latent=latent.numpy(), decoded=decoded.numpy(), ae_forward=ae_fwd.numpy(),
               ae_forward_latent_offset=latent_golden.forward_latent_offset(ae_lat.numpy(), first.detach().numpy()),
               first=first.detach().numpy(), flow_n=flow_n.numpy(), flow_pred=fp.detach().numpy(),
               grad_flow_pred=fp.grad.numpy(), loss=np.array(float(loss)),
               grad_final_conv_w=m.unet.final_conv.weight.grad.numpy(), grad_final_conv_b=m.unet.final_conv.bias.grad.numpy(),
               grad_init_conv_w=m.unet.init_conv.weight.grad.numpy(), grad_init_conv_b=m.unet.init_conv.bias.grad.numpy())
    np.savez_compressed(os.path.join(GOLD, "latent_32x48.npz"), **out)
    print("latent_32x48.npz loss", float(loss), "latent range", float(latent.min()), float(latent.max()),
          "clamped fraction", float((latent.abs() >= 1).float().mean()), "nan fraction of x0", float(torch.isnan(first).float().mean()),
          "unet channels", m.unet.channels)


if __name__ == "__main__":
    main()
