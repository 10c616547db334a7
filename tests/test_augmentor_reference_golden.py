"""The augmentation (SURVEY.md 8f row N2) against goldens produced by the reference's OWN ``Augmentor``
(oracle/make_goldens_augment.py; augmentation.py:6-76): the per-item torchvision restatement ``flow_diffuser.Augmentor``
(CPU, bit-exact: same torchvision calls, same RNG consumption) and, on the GPU, ``augment.GpuAugmentor`` (<= 3e-5).

The golden holds the SHA-256 of every float32 output of the reference, not the outputs themselves: bit-exactness is
checked on the digest, and the GPU augmentor is compared with the host restatement's output once that output's digest
has matched the reference's."""
import hashlib
import random

import numpy as np
import pytest
import torch


def batch(seed, B, S):
    g = torch.Generator().manual_seed(1000 + seed)
    return (torch.rand(B, 3, S, S, generator=g), torch.rand(B, 3, S, S, generator=g), torch.randn(B, 2, S, S, generator=g) * 4)


def host_outputs(g, seed):
    """``flow_diffuser.Augmentor`` on the seeded batch of ``seed``, asserted bit for bit equal to the reference's output."""
    from opticalflowdiffusion_b200.flow_diffuser import Augmentor
    B, S = int(g["B"]), int(g["S"])
    random.seed(seed)
    torch.manual_seed(seed)
    aug = Augmentor()
    out = aug(tuple(t.clone() for t in batch(seed, B, S)))
    for name, o, c in zip(("img", "tgt", "flow"), out, (3, 3, 2)):
        a = np.ascontiguousarray(o.numpy())
        assert a.dtype == np.float32 and a.shape == (B, c, S, S), (name, seed, a.dtype, a.shape)
        assert hashlib.sha256(a.tobytes()).digest() == g[f"sha256_{name}_{seed}"].tobytes(), f"{name} seed {seed}"
    return out


def test_host_augmentor_equals_the_reference(golden):
    g = golden("augmentor_ref")
    for seed in g["seeds"]:
        host_outputs(g, int(seed))


@pytest.mark.gpu
def test_gpu_augmentor_equals_the_reference(golden):
    from opticalflowdiffusion_b200.augment import GpuAugmentor
    g = golden("augmentor_ref")
    B, S = int(g["B"]), int(g["S"])
    worst = 0.0
    for seed in g["seeds"]:
        seed = int(seed)
        ref = host_outputs(g, seed)
        random.seed(seed)
        torch.manual_seed(seed)
        aug = GpuAugmentor()
        out = aug(tuple(t.cuda() for t in batch(seed, B, S)))
        for name, o, r in zip(("img", "tgt", "flow"), out, ref):
            err = np.abs(o.cpu().numpy() - r.numpy()).max()
            worst = max(worst, float(err))
            assert err <= 3e-5, (name, seed, err)
    print("GpuAugmentor vs the reference Augmentor: worst |err|", worst)
