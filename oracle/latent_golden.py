"""``tests/golden/latent_32x48.npz`` as oracle/make_goldens_latent.py computed it.

The file keeps only what needs the reference to recompute; ``load`` restores the rest exactly:
  * the inputs (img, tgt, flow, noise) are drawn again from the generator seed they were made with, and their stored
    sums prove it;
  * ``cond`` is the encoder latent over latent_max (the latent lies in [-1, 1], so the reference's clamp is the identity);
  * ``ae_forward_latent`` (the reference's ``ae(img, flow, return_latent=True)``) is stored as its float32 bit offset from
    latent_max * first: both splat the same latent along the same flow and differ in the last bits only."""
import numpy as np
import torch

LATENT_MAX = np.float32(2.0)           # configurations/algorithm/flow_diffuser.yaml
B, H, W = 2, 32, 48


def draw_inputs(seed: int):
    g = torch.Generator().manual_seed(seed)
    img = torch.rand(B, 3, H, W, generator=g)
    tgt = torch.rand(B, 3, H, W, generator=g)
    flow = torch.randn(B, 2, H, W, generator=g) * 3
    noise = torch.randn(B, 16, H, W, generator=g)
    return {"img": img.numpy(), "tgt": tgt.numpy(), "flow": flow.numpy(), "noise": noise.numpy()}


def input_sums(inputs) -> np.ndarray:
    return np.array([float(inputs[k].astype(np.float64).sum()) for k in ("img", "tgt", "flow", "noise")])


def forward_latent_offset(ae_forward_latent, first) -> np.ndarray:
    base = (LATENT_MAX * first).view(np.uint32)
    return (ae_forward_latent.view(np.uint32) - base).view(np.int32)          # modulo 2^32: exact both ways


def load(npz) -> dict:
    g = dict(npz)
    inputs = draw_inputs(int(g["input_seed"]))
    np.testing.assert_array_equal(input_sums(inputs), g["input_sums"],
                                  err_msg="the generator no longer draws the inputs the golden was made from")
    g.update(inputs)
    g["cond"] = g["latent"] / LATENT_MAX
    base = (LATENT_MAX * g["first"]).view(np.uint32)
    g["ae_forward_latent"] = (base + g.pop("ae_forward_latent_offset").view(np.uint32)).view(np.float32)
    return g
