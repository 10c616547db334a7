"""CPU: the oracle's FlowLearner objective (SURVEY.md 8f row N1) against the golden produced by the reference's own
FlowLearner class (oracle/make_goldens_flow_learner.py: reference code + the reference's splat kernels compiled for the
host), and the host-side surface of the FlowLearner class here (parameter names, same random init)."""
import random

import numpy as np
import pytest
import torch

from oracle import flowdiff_oracle as O

pytestmark = pytest.mark.usefixtures("golden_threads")


def T(a):
    return torch.from_numpy(np.asarray(a))


class Cfg(dict):
    __getattr__ = dict.__getitem__


def make_cfg():
    return Cfg(flow_max=20, latent=False, zero_init=False, c2f=False, lr=8e-5, weight_decay=1e-6, sparsity_weight=0.0,
               occlusion_mask=True, train_aug=False, image_size=32)


def build_learner(seed):
    from opticalflowdiffusion_b200.flow_learner import FlowLearner
    random.seed(int(seed))
    torch.manual_seed(int(seed))
    return FlowLearner(make_cfg())


def test_same_init_and_keys_as_the_reference(golden):
    g = golden("flow_learner_32x32")
    m = build_learner(g["seed"])
    sd = m.unet.model.state_dict()
    assert not any(k.startswith("time_mlp") or ".mlp." in k for k in sd)          # Unet(time_in=False)
    sums = np.array([float(v.double().sum()) for v in sd.values()])
    np.testing.assert_allclose(sums, g["w_sums"], rtol=1e-12, atol=1e-12)
    assert len(m.state_dict()) == int(g["n_keys"])                               # unet.* and model.* aliases


def test_oracle_loss_and_gradients_match_the_reference(golden):
    g = golden("flow_learner_32x32")
    m = build_learner(g["seed"])
    sd = {k: v.clone().requires_grad_(True) for k, v in m.unet.model.state_dict().items()}
    img, tgt = T(g["img"]), T(g["tgt"])
    cond = torch.cat((2 * img - 1, 2 * tgt - 1), 1)
    with torch.no_grad():
        fw = O.unet_forward(sd, cond, None, None)
    np.testing.assert_allclose(fw.numpy(), g["model_out"][:, -3:], rtol=1e-4, atol=2e-5)
    loss = O.flow_learner_loss(sd, 2 * tgt - 1, cond)
    np.testing.assert_allclose(float(loss.detach()), float(g["loss"]), rtol=2e-5)
    loss.backward()
    np.testing.assert_allclose(sd["final_conv.weight"].grad.numpy(), g["grad_final_conv_w"], rtol=2e-3, atol=1e-6)
    np.testing.assert_allclose(sd["final_conv.bias"].grad.numpy(), g["grad_final_conv_b"], rtol=2e-3, atol=1e-7)
    np.testing.assert_allclose(sd["init_conv.bias"].grad.numpy(), g["grad_init_conv_b"], rtol=2e-3, atol=1e-7)
    np.testing.assert_allclose(float(sd["mid_attn.fn.fn.to_qkv.weight"].grad.double().abs().sum()),
                               float(g["grad_mid_qkv_w_sum"]), rtol=2e-3)
