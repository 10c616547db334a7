"""-m gpu: the full UNet forward through libflowdiff against the reference-generated golden (16x24)
and against the fp32 CPU oracle at 64x128 (BASELINE config #1 shape).

Tolerance (stated, bf16 activations + bf16 tensor-core operands with fp32 accumulation vs the fp32
reference): per-tensor max |err| <= 4 % of the tensor's max |value| and mean |err| <= 1.5 % of its
mean |value| for intermediates; the noise/x0 prediction itself <= 3e-2 absolute on [-1, 1] data."""
import numpy as np
import pytest
import torch

from oracle import flowdiff_oracle as O

pytestmark = pytest.mark.gpu


def T(a):
    return torch.from_numpy(np.asarray(a))


def build_unet(seed, channels, gold=None):
    from opticalflowdiffusion_b200.unet import Unet
    torch.manual_seed(int(seed))
    net = Unet(64, channels=channels, out_dim=2)
    if gold is not None:
        sums = np.array([float(v.double().sum()) for v in net.state_dict().values()])
        np.testing.assert_allclose(sums, gold["w_sums"], rtol=1e-12, atol=1e-12)   # summation order differs per CPU
    return net


def check(name, got, ref, max_frac=4e-2, mean_frac=1.5e-2):
    got, ref = got.float().cpu(), ref.float().cpu()
    err = (got - ref).abs()
    assert err.max().item() <= max_frac * ref.abs().max().item() + 1e-6, \
        f"{name}: max err {err.max().item():.4g} vs scale {ref.abs().max().item():.4g}"
    assert err.mean().item() <= mean_frac * ref.abs().mean().item() + 1e-6, \
        f"{name}: mean err {err.mean().item():.4g} vs mean {ref.abs().mean().item():.4g}"


def test_unet_golden_16x24(golden):
    g = golden("unet_flow_16x24")
    net = build_unet(g["seed"], 5, g)
    sd = {k: v.clone() for k, v in net.state_dict().items()}
    net = net.cuda()
    x, cond, t = T(g["x"]).cuda(), T(g["cond"]).cuda(), T(g["t"]).cuda()
    out, taps = net(x, cond, t, return_taps=True)
    assert torch.allclose(taps["temb"].cpu(), T(g["temb"]), rtol=1e-3, atol=2e-3)
    for k in ("init_conv", "downs.0.0", "downs.0.2", "mid_block1", "mid_attn", "final_res_block"):
        check(k, taps[k], T(g["tap_" + k]))
    ref = T(g["unet_out"])
    assert (out.cpu() - ref).abs().max().item() < 3e-2, (out.cpu() - ref).abs().max().item()
    # and the oracle on the same weights agrees with the golden (sanity of the comparison itself)
    with torch.no_grad():
        o2 = O.unet_forward(sd, T(g["x"]), T(g["cond"]), T(g["t"]))
    assert torch.allclose(o2, ref, rtol=1e-4, atol=2e-5)


def test_unet_joint_nan_mask_golden(golden):
    g = golden("unet_joint_16x16")
    net = build_unet(g["seed"], 9, g).cuda()
    out = net(T(g["x"]).cuda(), T(g["cond"]).cuda(), T(g["t"]).cuda(), nan_mask=True)
    assert (out.cpu() - T(g["flow"])).abs().max().item() < 3e-2


def test_unet_vs_oracle_64x128():
    net = build_unet(1, 5)
    sd = {k: v.clone() for k, v in net.state_dict().items()}
    net = net.cuda()
    g = torch.Generator().manual_seed(2)
    B, H, W = 1, 64, 128
    x = torch.randn(B, 2, H, W, generator=g)
    cond = O.synthetic_frames(B, H, W, seed=4) * 2 - 1
    t = torch.tensor([437])
    with torch.no_grad():
        ref, rt = O.unet_forward(sd, x, cond, t, return_taps=True)
    out, taps = net(x.cuda(), cond.cuda(), t.cuda(), return_taps=True)
    for k in ("init_conv", "downs.0.0", "downs.0.2", "mid_block1", "mid_attn", "final_res_block"):
        check(k, taps[k], rt[k])
    assert (out.cpu() - ref).abs().max().item() < 3e-2
    # determinism: per-tile GroupNorm partial sums are reduced in a fixed order and the cross-tile
    # accumulation is in double precision, so two runs agree to bf16 rounding flips at most
    with torch.no_grad():
        out2 = net(x.cuda(), cond.cuda(), t.cuda())
    assert (out2 - out).abs().max().item() < 5e-3
    # with autograd enabled the same call runs the training forward (unfused attention, activations kept for the
    # backward): same tolerance against the oracle
    out3 = net(x.cuda(), cond.cuda(), t.cuda())
    assert out3.requires_grad
    assert (out3.detach().cpu() - ref).abs().max().item() < 3e-2


def test_unet_fused_output_head_padded_shape():
    """Inference forward at a shape that needs replicate padding (44x140 -> 48x144): the fused tail (res_conv + GroupNorm
    residual + final_conv + crop in one launch) == the two-launch tail that return_taps=True takes == the oracle
    (InputPadder pad / unpad around the fp32 forward, utils.py:6-27 + denoising_diffusion.py:414-417)."""
    import torch.nn.functional as F
    net = build_unet(3, 5)
    sd = {k: v.clone() for k, v in net.state_dict().items()}
    net = net.cuda()
    g = torch.Generator().manual_seed(5)
    B, H, W = 2, 44, 140
    x = torch.randn(B, 2, H, W, generator=g)
    cond = O.synthetic_frames(B, H, W, seed=6) * 2 - 1
    t = torch.tensor([12, 903])
    ph, pw = (-H) % 8, (-W) % 8
    pad = [pw // 2, pw - pw // 2, ph // 2, ph - ph // 2]
    with torch.no_grad():
        ref = O.unet_forward(sd, F.pad(x, pad, mode="replicate"), F.pad(cond, pad, mode="replicate"), t)
        ref = ref[..., pad[2]:pad[2] + H, pad[0]:pad[0] + W]
        fused = net(x.cuda(), cond.cuda(), t.cuda())
        two = net(x.cuda(), cond.cuda(), t.cuda(), return_taps=True)[0]
    assert fused.shape == two.shape == (B, 2, H, W)
    assert (fused.cpu() - ref).abs().max().item() < 3e-2
    assert (two.cpu() - ref).abs().max().item() < 3e-2
    assert (fused - two).abs().max().item() < 1e-2
