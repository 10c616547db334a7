"""TEST INFRASTRUCTURE ONLY.  Golden vectors for the training-time augmentation (SURVEY.md 8f row N2) from the reference's
OWN ``Augmentor`` (algorithms/diffusion_animation/augmentation.py:6-76, imported unmodified from /root/reference; it needs
only torch / torchvision / random).  For each seed: ``random.seed(s); torch.manual_seed(s)``, construct the Augmentor (its
jitter / blur parameters are drawn at construction), call it on a seeded square batch (the reference's resized crop assumes
square frames, :44-50).  Seeds are chosen so that every branch (jitter, grayscale, blur, h-flip, v-flip, resized crop)
fires for at least one item.  The golden stores the SHA-256 of each float32 output (the tests check bit-exactness on it),
which keeps the file small.

Run in the build container:  python oracle/make_goldens_augment.py  ->  tests/golden/augmentor_ref.npz
"""
import hashlib
import os
import random
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle import ref_stubs  # noqa: E402

GOLD = os.path.join(ROOT, "tests", "golden")
B, S = 4, 32


def batch(seed):
    g = torch.Generator().manual_seed(1000 + seed)
    return (torch.rand(B, 3, S, S, generator=g), torch.rand(B, 3, S, S, generator=g), torch.randn(B, 2, S, S, generator=g) * 4)


def main():
    ns = ref_stubs.import_reference()
    Augmentor = ns.augmentation.Augmentor
    d = {"B": np.array(B), "S": np.array(S)}
    seeds, changed = [], {"img": 0, "flip_or_crop": 0}
    for seed in range(40):
        random.seed(seed)
        torch.manual_seed(seed)
        aug = Augmentor()
        img, tgt, flow = batch(seed)
        o_img, o_tgt, o_flow = aug((img.clone(), tgt.clone(), flow.clone()))
        if len(seeds) < 12:
            seeds.append(seed)
            for name, o in (("img", o_img), ("tgt", o_tgt), ("flow", o_flow)):
                digest = hashlib.sha256(np.ascontiguousarray(o.numpy(), dtype=np.float32).tobytes()).digest()
                d[f"sha256_{name}_{seed}"] = np.frombuffer(digest, dtype=np.uint8)
            changed["img"] += int(not torch.equal(o_img, img))
            changed["flip_or_crop"] += int(not torch.equal(o_flow, flow))
    d["seeds"] = np.array(seeds)
    np.savez_compressed(os.path.join(GOLD, "augmentor_ref.npz"), **d)
    print("augmentor_ref.npz seeds", seeds, changed)


if __name__ == "__main__":
    main()
