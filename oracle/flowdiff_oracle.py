"""TEST INFRASTRUCTURE ONLY -- CPU restatement of the reference's flow_diffuser hot path.

This file is the parity oracle.  It is imported by ``tests/``, by
``__graft_entry__.smoke()`` and by ``bench.py``'s CPU-baseline / ``--impl reference``
legs, and by nothing else: the product package ``opticalflowdiffusion_b200`` never
imports it and has no CPU fallback.

It restates, with plain fp32 torch ops on the CPU and as pure functions over a
``state_dict`` (so it needs neither Lightning nor the reference tree at run time), the
arithmetic of:

  * ``Unet.forward``                     denoising_diffusion.py:272-417 (blocks :81-268)
  * the sigmoid beta schedule + buffers  denoising_diffusion.py:448-461, 511-583
  * ``q_sample`` / ``p_losses`` / ``_loss`` (target=flow, and the joint / target pyramid)   :806-812, :823-891, :893-983
  * ``UnetWithWarp.forward``             flow_diffuser.py:38-63
  * ``model_predictions`` / ``ddim_sample`` / ``p_sample`` loops  :634-664, :731-774, :677-729
  * ``warp_backward_flow``               warp.py:95-119
  * the three forward-splat kernels      softsplat_new.py:352-423, 489-565, 600-700
  * ``warp_forward_flow`` / ``softsplat`` wrappers  warp.py:121-156, softsplat_new.py:278-333
  * ``nan_mse`` / ``charbonnier``        warp.py:260-279, losses.py:3-6,46-47

PINNING: the reference ships no golden vectors or numeric tests for this path
(SURVEY.md section 4), so the oracle is pinned against the *reference code itself*:
``oracle/make_goldens.py`` imports the unmodified reference under ``oracle/ref_stubs.py``
in the build container, runs it on seeded inputs and commits the outputs under
``tests/golden/``; ``tests/test_oracle_vs_golden.py`` checks this file against them.
The forward splat is CUDA-only in the reference; its kernel source is compiled for the
host by ``oracle/build_ref.py`` into ``oracle/_ref/`` and the goldens come from that.
"""
from __future__ import annotations

import math
from typing import Dict, List, Optional, Sequence, Tuple

import torch
import torch.nn.functional as F

Tensor = torch.Tensor

# --------------------------------------------------------------------------------------
# UNet (denoising_diffusion.py:272-417)
# --------------------------------------------------------------------------------------


def _ws_conv3x3(x: Tensor, w: Tensor, b: Tensor) -> Tensor:
    """WeightStandardizedConv2d.forward, denoising_diffusion.py:106-114 (fp32 -> eps 1e-5)."""
    eps = 1e-5 if x.dtype == torch.float32 else 1e-3
    flat = w.reshape(w.shape[0], -1)
    mean = flat.mean(dim=1).reshape(-1, 1, 1, 1)
    var = flat.var(dim=1, unbiased=False).reshape(-1, 1, 1, 1)
    return F.conv2d(x, (w - mean) * (var + eps).rsqrt(), b, padding=1)


def _block(sd, p: str, x: Tensor, scale_shift=None, groups: int = 8) -> Tensor:
    """Block.forward, denoising_diffusion.py:179-188."""
    x = _ws_conv3x3(x, sd[p + "proj.weight"], sd[p + "proj.bias"])
    x = F.group_norm(x, groups, sd[p + "norm.weight"], sd[p + "norm.bias"], eps=1e-5)
    if scale_shift is not None:
        scale, shift = scale_shift
        x = x * (scale + 1) + shift
    return F.silu(x)


def _resnet_block(sd, p: str, x: Tensor, temb: Optional[Tensor]) -> Tensor:
    """ResnetBlock.forward, denoising_diffusion.py:202-214."""
    scale_shift = None
    if temb is not None and (p + "mlp.1.weight") in sd:
        e = F.linear(F.silu(temb), sd[p + "mlp.1.weight"], sd[p + "mlp.1.bias"])
        e = e[:, :, None, None]
        scale_shift = e.chunk(2, dim=1)
    h = _block(sd, p + "block1.", x, scale_shift)
    h = _block(sd, p + "block2.", h)
    if (p + "res_conv.weight") in sd:
        x = F.conv2d(x, sd[p + "res_conv.weight"], sd[p + "res_conv.bias"])
    return h + x


def _chan_layernorm(x: Tensor, g: Tensor, eps: Optional[float] = None) -> Tensor:
    """LayerNorm.forward, denoising_diffusion.py:121-125 (over channels, biased var, gain only).  ``eps`` defaults to the
    reference's choice by dtype (1e-5 for fp32, 1e-3 otherwise); a float64 restatement of the fp32 model passes 1e-5."""
    if eps is None:
        eps = 1e-5 if x.dtype == torch.float32 else 1e-3
    var = torch.var(x, dim=1, unbiased=False, keepdim=True)
    mean = torch.mean(x, dim=1, keepdim=True)
    return (x - mean) * (var + eps).rsqrt() * g


def _linear_attention(sd, p: str, x: Tensor, heads: int = 4, dim_head: int = 32, eps: Optional[float] = None) -> Tensor:
    """Residual(PreNorm(LinearAttention)), denoising_diffusion.py:81-87,127-135,229-244."""
    b, c, h, w = x.shape
    y = _chan_layernorm(x, sd[p + "norm.g"], eps)
    qkv = F.conv2d(y, sd[p + "fn.to_qkv.weight"])
    q, k, v = (t.reshape(b, heads, dim_head, h * w) for t in qkv.chunk(3, dim=1))
    q = q.softmax(dim=-2) * dim_head ** -0.5
    k = k.softmax(dim=-1)
    v = v / (h * w)
    ctx = torch.einsum("bhdn,bhen->bhde", k, v)
    out = torch.einsum("bhde,bhdn->bhen", ctx, q).reshape(b, heads * dim_head, h, w)
    out = F.conv2d(out, sd[p + "fn.to_out.0.weight"], sd[p + "fn.to_out.0.bias"])
    out = _chan_layernorm(out, sd[p + "fn.to_out.1.g"], eps)
    return out + x


def _full_attention(sd, p: str, x: Tensor, heads: int = 4, dim_head: int = 32) -> Tensor:
    """Residual(PreNorm(Attention)), denoising_diffusion.py:256-268."""
    b, c, h, w = x.shape
    y = _chan_layernorm(x, sd[p + "norm.g"])
    qkv = F.conv2d(y, sd[p + "fn.to_qkv.weight"])
    q, k, v = (t.reshape(b, heads, dim_head, h * w) for t in qkv.chunk(3, dim=1))
    q = q * dim_head ** -0.5
    sim = torch.einsum("bhdi,bhdj->bhij", q, k)
    attn = sim.softmax(dim=-1)
    out = torch.einsum("bhij,bhdj->bhid", attn, v)          # (b, heads, n, d)
    out = out.permute(0, 1, 3, 2).reshape(b, heads * dim_head, h, w)
    out = F.conv2d(out, sd[p + "fn.to_out.weight"], sd[p + "fn.to_out.bias"])
    return out + x


def time_embedding(sd, t: Tensor, dim: int = 64, prefix: str = "") -> Tensor:
    """SinusoidalPosEmb + time_mlp, denoising_diffusion.py:144-151, 319-324."""
    half = dim // 2
    freq = torch.exp(torch.arange(half, device=t.device) * -(math.log(10000) / (half - 1)))
    e = t[:, None] * freq[None, :]
    e = torch.cat((e.sin(), e.cos()), dim=-1)
    e = F.linear(e, sd[prefix + "time_mlp.1.weight"], sd[prefix + "time_mlp.1.bias"])
    e = F.gelu(e)
    return F.linear(e, sd[prefix + "time_mlp.3.weight"], sd[prefix + "time_mlp.3.bias"])


def _pixel_unshuffle2(x: Tensor) -> Tensor:
    """Rearrange('b c (h p1) (w p2) -> b (c p1 p2) h w'), denoising_diffusion.py:97."""
    b, c, H, W = x.shape
    x = x.reshape(b, c, H // 2, 2, W // 2, 2).permute(0, 1, 3, 5, 2, 4)
    return x.reshape(b, c * 4, H // 2, W // 2)


def unet_forward(sd: Dict[str, Tensor], x: Tensor, cond: Optional[Tensor], t: Tensor,
                 prefix: str = "", return_taps: bool = False):
    """Unet.forward, denoising_diffusion.py:363-417 (dim=64, no self-cond; the number of levels -- four for the flow UNet,
    three for the latent autoencoder's UNets, flow_pred.py:23-37 -- is read from the parameter names).

    ``sd`` holds the reference's parameter names (``init_conv.weight`` ...) under ``prefix``.
    ``return_taps`` additionally returns named intermediates for per-layer parity tests.
    """
    sd = {k[len(prefix):]: v for k, v in sd.items() if k.startswith(prefix)} if prefix else sd
    taps = {}
    if cond is not None:
        x = torch.cat((x, cond), dim=1)
    x = F.conv2d(x, sd["init_conv.weight"], sd["init_conv.bias"], padding=3)
    r = x.clone()
    taps["init_conv"] = x
    temb = None
    if "time_mlp.1.weight" in sd:            # Unet(time_in=False) has no time path at all (:306-318, 377-383)
        temb = time_embedding(sd, t)
        taps["temb"] = temb
    skips: List[Tensor] = []
    n_levels = sum(1 for i in range(8) if f"downs.{i}.0.block1.proj.weight" in sd)
    for i in range(n_levels):
        p = f"downs.{i}."
        x = _resnet_block(sd, p + "0.", x, temb)
        skips.append(x)
        if i == 0:
            taps["downs.0.0"] = x
        x = _resnet_block(sd, p + "1.", x, temb)
        x = _linear_attention(sd, p + "2.fn.", x)
        if i == 0:
            taps["downs.0.2"] = x
        skips.append(x)
        if i < n_levels - 1:
            x = F.conv2d(_pixel_unshuffle2(x), sd[p + "3.1.weight"], sd[p + "3.1.bias"])
        else:
            x = F.conv2d(x, sd[p + "3.weight"], sd[p + "3.bias"], padding=1)
        taps[f"downs.{i}"] = x
    x = _resnet_block(sd, "mid_block1.", x, temb)
    taps["mid_block1"] = x
    x = _full_attention(sd, "mid_attn.fn.", x)
    taps["mid_attn"] = x
    x = _resnet_block(sd, "mid_block2.", x, temb)
    taps["mid_block2"] = x
    for i in range(n_levels):
        p = f"ups.{i}."
        x = torch.cat((x, skips.pop()), dim=1)
        x = _resnet_block(sd, p + "0.", x, temb)
        x = torch.cat((x, skips.pop()), dim=1)
        x = _resnet_block(sd, p + "1.", x, temb)
        x = _linear_attention(sd, p + "2.fn.", x)
        if i < n_levels - 1:
            x = F.interpolate(x, scale_factor=2, mode="nearest")
            x = F.conv2d(x, sd[p + "3.1.weight"], sd[p + "3.1.bias"], padding=1)
        else:
            x = F.conv2d(x, sd[p + "3.weight"], sd[p + "3.bias"], padding=1)
        taps[f"ups.{i}"] = x
    x = torch.cat((x, r), dim=1)
    x = _resnet_block(sd, "final_res_block.", x, temb)
    taps["final_res_block"] = x
    out = F.conv2d(x, sd["final_conv.weight"], sd["final_conv.bias"])
    if return_taps:
        return out, taps
    return out


def autoencoder_encode(sd, x: Tensor, prefix: str = "") -> Tensor:
    """Autoencoder.encode, flow_pred.py:49-50: clamp(model_enc(2x - 1), -1, 1); ``sd`` holds ``model_enc.*`` / ``model_dec.*``."""
    return torch.clamp(unet_forward(sd, 2 * x - 1.0, None, None, prefix=prefix + "model_enc."), -1.0, 1.0)


def autoencoder_decode(sd, latent: Tensor, x: Tensor, prefix: str = "") -> Tensor:
    """Autoencoder.decode, flow_pred.py:53-57."""
    out = unet_forward(sd, torch.cat((latent, 2 * x - 1), dim=1), None, None, prefix=prefix + "model_dec.")
    return (torch.clamp(out, -1.0, 1.0) + 1.0) / 2.0


def autoencoder_forward(sd, x: Tensor, flow: Tensor, prefix: str = "") -> Tensor:
    """Autoencoder.forward, flow_pred.py:38-47: encode, forward-splat the latent along ``flow`` (pixels), decode."""
    lat = warp_forward_flow(autoencoder_encode(sd, x, prefix), flow)
    return autoencoder_decode(sd, lat, x, prefix)


def latent_preprocess(ae_sd, img: Tensor, flow: Tensor, flow_max: float = 20.0, latent_max: float = 2.0, target: str = "target"):
    """FlowDiffuser.preprocess with ``latent: true`` (flow_diffuser.py:136-168, aug off): the conditioning frame is the
    clamped, scaled latent; the diffusion target its forward splat along the ground-truth flow (+ the flow for 'joint')."""
    flow_n = torch.clamp(flow / flow_max, -1.0, 1.0)
    cond = torch.clamp(autoencoder_encode(ae_sd, img) / latent_max, -1.0, 1.0)
    first = warp_forward_flow(cond, flow_n * flow_max)
    if target == "joint":
        first = torch.cat((first, flow_n), dim=1)
    return first, cond, flow_n


# --------------------------------------------------------------------------------------
# Diffusion schedule + scheduler steps (denoising_diffusion.py:448-461, 511-583, 589-812)
# --------------------------------------------------------------------------------------


def sigmoid_beta_schedule(timesteps: int, start=-3, end=3, tau=1) -> Tensor:
    """denoising_diffusion.py:448-461 -- float64 throughout."""
    steps = timesteps + 1
    t = torch.linspace(0, timesteps, steps, dtype=torch.float64) / timesteps
    v_start = torch.tensor(start / tau).sigmoid()
    v_end = torch.tensor(end / tau).sigmoid()
    ac = (-((t * (end - start) + start) / tau).sigmoid() + v_end) / (v_end - v_start)
    ac = ac / ac[0]
    betas = 1 - (ac[1:] / ac[:-1])
    return torch.clip(betas, 0, 0.999)


SCHEDULE_BUFFERS = (
    "betas", "alphas_cumprod", "alphas_cumprod_prev", "sqrt_alphas_cumprod",
    "sqrt_one_minus_alphas_cumprod", "log_one_minus_alphas_cumprod", "sqrt_recip_alphas_cumprod",
    "sqrt_recipm1_alphas_cumprod", "posterior_variance", "posterior_log_variance_clipped",
    "posterior_mean_coef1", "posterior_mean_coef2", "loss_weight",
)


def make_schedule(timesteps: int = 1000, min_snr_gamma: float = 5.0) -> Dict[str, Tensor]:
    """The 13 fp32 buffers ConditionalDiffusion registers (denoising_diffusion.py:511-578).

    Computed in float64 and cast to float32 at the end, exactly like ``register_buffer`` at :530.
    ``loss_weight`` follows objective='pred_x0' with min_snr_loss_weight=True (flow_diffuser.py:121-126).
    """
    betas = sigmoid_beta_schedule(timesteps)
    alphas = 1.0 - betas
    ac = torch.cumprod(alphas, dim=0)
    ac_prev = F.pad(ac[:-1], (1, 0), value=1.0)
    post_var = betas * (1.0 - ac_prev) / (1.0 - ac)
    snr = ac / (1 - ac)
    out64 = {
        "betas": betas,
        "alphas_cumprod": ac,
        "alphas_cumprod_prev": ac_prev,
        "sqrt_alphas_cumprod": torch.sqrt(ac),
        "sqrt_one_minus_alphas_cumprod": torch.sqrt(1.0 - ac),
        "log_one_minus_alphas_cumprod": torch.log(1.0 - ac),
        "sqrt_recip_alphas_cumprod": torch.sqrt(1.0 / ac),
        "sqrt_recipm1_alphas_cumprod": torch.sqrt(1.0 / ac - 1),
        "posterior_variance": post_var,
        "posterior_log_variance_clipped": torch.log(post_var.clamp(min=1e-20)),
        "posterior_mean_coef1": betas * torch.sqrt(ac_prev) / (1.0 - ac),
        "posterior_mean_coef2": (1.0 - ac_prev) * torch.sqrt(alphas) / (1.0 - ac),
        "loss_weight": snr.clone().clamp_(max=min_snr_gamma),
    }
    return {k: v.to(torch.float32) for k, v in out64.items()}


def ddim_times(total_timesteps: int, sampling_timesteps: int) -> List[int]:
    """The DDIM grid, denoising_diffusion.py:737-738 (fp32 linspace -> .int() -> reversed)."""
    times = torch.linspace(-1, total_timesteps - 1, steps=sampling_timesteps + 1)
    return list(reversed(times.int().tolist()))


def _ext(a: Tensor, t: Tensor) -> Tensor:
    """extract(), denoising_diffusion.py:422-425, for 4-D x."""
    return a.gather(-1, t).reshape(-1, 1, 1, 1)


def q_sample(sched, x0: Tensor, t: Tensor, noise: Tensor) -> Tensor:
    """denoising_diffusion.py:806-812 (noise_space='image')."""
    return _ext(sched["sqrt_alphas_cumprod"], t) * x0 + _ext(sched["sqrt_one_minus_alphas_cumprod"], t) * noise


def predict_noise_from_start(sched, x_t: Tensor, t: Tensor, x0: Tensor) -> Tensor:
    """denoising_diffusion.py:595-599."""
    return (_ext(sched["sqrt_recip_alphas_cumprod"], t) * x_t - x0) / _ext(sched["sqrt_recipm1_alphas_cumprod"], t)


def ddim_update(sched, x: Tensor, x0_raw: Tensor, time: int, time_next: int, eta: float = 0.0,
                noise: Optional[Tensor] = None) -> Tuple[Tensor, Tensor]:
    """One DDIM step given the raw model output (objective pred_x0).

    model_predictions(clip_x_start=True) -> :653-656, then ddim_sample :752-767.
    Returns (next x, clipped x0)."""
    b = x.shape[0]
    t = torch.full((b,), time, dtype=torch.long, device=x.device)
    x0 = torch.clamp(x0_raw, min=-1.0, max=1.0)
    eps = predict_noise_from_start(sched, x, t, x0)
    if time_next < 0:
        return x0, x0
    alpha = sched["alphas_cumprod"][time]
    alpha_next = sched["alphas_cumprod"][time_next]
    sigma = eta * ((1 - alpha / alpha_next) * (1 - alpha_next) / (1 - alpha)).sqrt()
    c = (1 - alpha_next - sigma ** 2).sqrt()
    if noise is None:
        noise = torch.zeros_like(x)
    return x0 * alpha_next.sqrt() + c * eps + sigma * noise, x0


def ddpm_update(sched, x: Tensor, x0_raw: Tensor, time: int, noise: Optional[Tensor]) -> Tuple[Tensor, Tensor]:
    """One ancestral step: p_mean_variance + p_sample, denoising_diffusion.py:666-698, 613-623."""
    b = x.shape[0]
    t = torch.full((b,), time, dtype=torch.long, device=x.device)
    x0 = torch.clamp(x0_raw, -1.0, 1.0)
    mean = _ext(sched["posterior_mean_coef1"], t) * x0 + _ext(sched["posterior_mean_coef2"], t) * x
    logvar = _ext(sched["posterior_log_variance_clipped"], t)
    if time > 0:
        return mean + (0.5 * logvar).exp() * noise, x0
    return mean, x0


def ddim_sample(sd, sched, x_T: Tensor, cond: Tensor, total_timesteps: int, sampling_timesteps: int,
                prefix: str = "", return_all: bool = False, model=None):
    """ddim_sample, denoising_diffusion.py:731-774, eta = 0, starting from a supplied x_T."""
    times = ddim_times(total_timesteps, sampling_timesteps)
    x = x_T
    traj = [x]
    x0s = []
    model = model or (lambda xx, cc, tt: unet_forward(sd, xx, cc, tt, prefix))
    for time, time_next in zip(times[:-1], times[1:]):
        t = torch.full((x.shape[0],), time, dtype=torch.long, device=x.device)
        out = model(x, cond, t)
        x, x0 = ddim_update(sched, x, out, time, time_next)
        traj.append(x)
        x0s.append(x0)
    if return_all:
        return torch.stack(traj, dim=1), x0s
    return x


def ddpm_sample(sd, sched, x_T: Tensor, cond: Tensor, total_timesteps: int, noises: Sequence[Tensor],
                prefix: str = "", return_all: bool = False, model=None):
    """p_sample_loop, denoising_diffusion.py:700-729.  ``noises[i]`` is the draw used at step t = T-1-i."""
    x = x_T
    traj = [x]
    model = model or (lambda xx, cc, tt: unet_forward(sd, xx, cc, tt, prefix))
    for i, time in enumerate(reversed(range(total_timesteps))):
        t = torch.full((x.shape[0],), time, dtype=torch.long, device=x.device)
        out = model(x, cond, t)
        x, _ = ddpm_update(sched, x, out, time, noises[i] if time > 0 else None)
        traj.append(x)
    if return_all:
        return torch.stack(traj, dim=1)
    return x


def nan_mse(pred: Tensor, target: Tensor, reduction: str = "mean") -> Tensor:
    """warp.py:260-271."""
    pred, target = pred.flatten(), target.flatten()
    keep = ~(torch.isnan(target) | torch.isnan(pred))
    d = torch.square(pred[keep] - target[keep])
    return torch.nanmean(d) if reduction == "mean" else d


def p_losses_flow(sd, sched, x0: Tensor, cond: Tensor, t: Tensor, noise: Tensor, prefix: str = "") -> Tensor:
    """p_losses with target='flow' (objective pred_x0): denoising_diffusion.py:823-891 -> _loss level 1
    (:906-908, :973): nanmean of the NaN-filtered squared error of model_out[:, :3] vs x0[:, :3]."""
    x_t = q_sample(sched, x0, t, noise)
    out = unet_forward(sd, x_t, cond, t, prefix)
    return torch.nanmean(nan_mse(out[:, :3], x0[:, :3], reduction="none"))


def unet_with_warp(sd, x: Tensor, cond: Tensor, t: Tensor, flow_max: float = 20.0, full_output: bool = True,
                   additional_out: bool = False, prefix: str = "", dim: int = 3) -> Tensor:
    """UnetWithWarp.forward, flow_diffuser.py:38-63 (nan_safe=True): NaN -> 0 plus a 1-channel "any NaN" mask appended
    to x; flow = Unet(...); warped = forward splat of cond[:, :3] along flow * flow_max; cat(warped, flow) when
    ``full_output`` (target='joint'); the flow appended once more when ``additional_out`` (target='target').
    ``dim`` = 3, or latent_dim in latent mode (flow_diffuser.py:25)."""
    x = x.clone()
    nans = torch.isnan(x)
    x[nans] = 0.0
    mask = torch.any(nans, dim=1)[:, None]
    flow = unet_forward(sd, torch.cat((x, mask), dim=1), cond, t, prefix)
    out = warp_forward_flow(cond[:, :dim], flow[:, :2] * flow_max)
    if full_output:
        out = torch.cat((out, flow), dim=1)
    return torch.cat((out, flow), dim=1) if additional_out else out


def pyramid_loss(image_out: Tensor, target: Tensor, flow_out: Optional[Tensor] = None, cond: Optional[Tensor] = None,
                 flow_max: float = 20.0, levels=(2, 4, 8, 16), dim: int = 3) -> Tensor:
    """ConditionalDiffusion._loss, denoising_diffusion.py:893-983.  Level 1: NaN-filtered squared error of
    (image_out, target) (:906-908).  With a flow target (``flow_out`` given) every level L in 2,4,8,16 adds the
    NaN-filtered squared error between the splat of ``cond`` along the predicted flow at scale L and the splat of the
    TARGET image along zero flow at scale L (:947-953; the a = b = 0 shifted copies are identities), times L^4 (:965);
    all terms are concatenated and pooled by one nanmean (:973).  No SNR weight (:975-980), flow term disabled (:961-969)."""
    terms = [nan_mse(image_out, target, reduction="none")]
    if flow_out is not None:
        for level in levels:
            a = warp_forward_flow(cond[:, :dim], flow_out * flow_max, scale=level)       # UnetWithWarp._warp slices by dim
            b = warp_forward_flow(target[:, :dim], torch.zeros_like(flow_out) * flow_max, scale=level)
            terms.append(nan_mse(a, b, reduction="none") * level ** 4)
    return torch.nanmean(torch.cat(terms, dim=0))


def p_losses_joint(sd, sched, x0: Tensor, cond: Tensor, t: Tensor, noise: Tensor, flow_max: float = 20.0,
                   prefix: str = "", model_out: Optional[Tensor] = None) -> Tensor:
    """p_losses with target='joint' (x0 = cat(warped target image, normalised flow), 5 channels):
    denoising_diffusion.py:823-891 with the ``target.shape[1] == 5`` dispatch of :886-887."""
    if model_out is None:
        x_t = q_sample(sched, x0, t, noise)
        model_out = unet_with_warp(sd, x_t, cond, t, flow_max, True, False, prefix)
    return pyramid_loss(model_out[:, :3], x0[:, :3], model_out[:, 3:], cond, flow_max)


def p_losses_target(sd, sched, x0: Tensor, cond: Tensor, flow_tgt: Tensor, t: Tensor, noise: Tensor,
                    flow_max: float = 20.0, prefix: str = "", model_out: Optional[Tensor] = None, dim: int = 3) -> Tensor:
    """p_losses with target='target' (x0 = warped target image, ``additional_tgt`` = normalised flow): :868-885.
    The model is called with additional_out=True, its last 2 channels are the flow prediction."""
    if model_out is None:
        x_t = q_sample(sched, x0, t, noise)
        model_out = unet_with_warp(sd, x_t, cond, t, flow_max, False, True, prefix, dim)
    k = flow_tgt.shape[1]
    return pyramid_loss(model_out[:, :-k], x0, model_out[:, -k:], cond, flow_max, dim=dim)


# --------------------------------------------------------------------------------------
# Backward warp (warp.py:95-119; arithmetic of torch grid_sample, bilinear/zeros/align_corners)
# --------------------------------------------------------------------------------------


def _fma(a: Tensor, b: Tensor, c: Tensor) -> Tensor:
    """fp32 fused multiply-add emulated through float64 (the fp32 product is exact in float64)."""
    return (a.double() * b.double() + c.double()).float()


def backwarp_coords(flow: Tensor) -> Tuple[Tensor, Tensor]:
    """Un-normalised sampling coordinates (ix, iy) exactly as the reference op sequence produces
    them on the CPU: vgrid = grid + flow.flip(1); 2*v/max(S-1,1)-1 (warp.py:105-109, true fp32
    division); then grid_sample's align_corners un-normalisation as ATen's CPU kernel evaluates it,
    (g + 1) * ((S-1)/2).  The fp32 round trip is NOT the identity."""
    B, _, H, W = flow.shape
    xx = torch.arange(W, dtype=torch.float32).view(1, 1, W).expand(B, H, W)
    yy = torch.arange(H, dtype=torch.float32).view(1, H, 1).expand(B, H, W)
    vx = xx + flow[:, 1]
    vy = yy + flow[:, 0]
    gx = 2.0 * vx / max(W - 1, 1) - 1.0
    gy = 2.0 * vy / max(H - 1, 1) - 1.0
    ix = (gx + 1) * torch.tensor((W - 1) / 2, dtype=torch.float32)
    iy = (gy + 1) * torch.tensor((H - 1) / 2, dtype=torch.float32)
    return ix, iy


def backwarp(image: Tensor, flow: Tensor) -> Tuple[Tensor, Tensor]:
    """warp_backward_flow(first, second=image, flow) -> (output, mask), explicit 4-tap form.

    Follows ATen's CPU grid_sampler_2d (bilinear, padding zeros, align_corners=True) operation by
    operation -- w = ix - floor(ix), e = 1 - w, (nw, ne, sw, se) = (s*e, s*w, n*e, n*w); out-of-range
    taps read 0; the four taps are accumulated as nw_v*nw, then three fused multiply-adds in the
    order ne, sw, se -- which makes it BIT-EXACT against the reference's CPU output (checked by
    tests/test_oracle_vs_golden.py).  mask = grid_sample(ones) thresholded: <0.999 -> 0, >0 -> 1
    (warp.py:113-117)."""
    B, C, H, W = image.shape
    ix, iy = backwarp_coords(flow)
    x0 = torch.floor(ix)
    y0 = torch.floor(iy)
    x1 = x0 + 1
    y1 = y0 + 1
    w = ix - x0
    e = 1 - w
    n = iy - y0
    s = 1 - n
    out = None
    msk = None
    flat = image.reshape(B, C, H * W)
    for xs, ys, wt in ((x0, y0, s * e), (x1, y0, s * w), (x0, y1, n * e), (x1, y1, n * w)):
        ok = (xs >= 0) & (xs <= W - 1) & (ys >= 0) & (ys <= H - 1)
        xi = xs.clamp(0, W - 1).long()
        yi = ys.clamp(0, H - 1).long()
        idx = (yi * W + xi).reshape(B, 1, H * W).expand(B, C, H * W)
        val = flat.gather(2, idx).reshape(B, C, H, W) * ok[:, None]
        one = ok.float()
        if out is None:
            out = val * wt[:, None]
            msk = one * wt
        else:
            out = _fma(val, wt[:, None].expand_as(val), out)
            msk = _fma(one, wt, msk)
    mask = msk[:, None].expand(B, C, H, W).clone()
    mask[mask < 0.999] = 0
    mask[mask > 0] = 1
    return out, mask


def backwarp_torch(image: Tensor, flow: Tensor) -> Tuple[Tensor, Tensor]:
    """The same through torch.nn.functional.grid_sample, i.e. the op sequence of warp.py:95-119
    written without the reference's repeat/cat/flip plumbing (used to cross-check ``backwarp``)."""
    B, C, H, W = image.shape
    xx = torch.arange(W, dtype=torch.float32).view(1, 1, W).expand(B, H, W)
    yy = torch.arange(H, dtype=torch.float32).view(1, H, 1).expand(B, H, W)
    gx = 2.0 * (xx + flow[:, 1]) / max(W - 1, 1) - 1.0
    gy = 2.0 * (yy + flow[:, 0]) / max(H - 1, 1) - 1.0
    grid = torch.stack((gx, gy), dim=-1)
    out = F.grid_sample(image, grid, align_corners=True)
    mask = F.grid_sample(torch.ones_like(image), grid, align_corners=True)
    mask[mask < 0.999] = 0
    mask[mask > 0] = 1
    return out, mask


def charbonnier(x: Tensor, alpha: float = 0.5, eps: float = 1e-3) -> Tensor:
    """warp.py:278-279 / losses.py:46-47."""
    return torch.pow(torch.square(x) + eps ** 2, alpha)


def photometric_epe(frame1: Tensor, frame2: Tensor, flow: Tensor, flow_gt: Tensor):
    """The config-#4 microbench objective (SURVEY.md section 8d): W1 + P0 + EPE.

    warped, mask = warp_backward_flow(None, frame2, flow)
    L_photo = sum(mask * charbonnier(frame1 - warped)) / sum(mask)   (occlusion-weighted sum of
              losses.py:3-6 normalised by the weight mass)
    EPE     = mean sqrt(du^2 + dv^2)
    """
    warped, mask = backwarp_torch(frame2, flow)
    num = torch.sum(mask * charbonnier(frame1 - warped))
    den = torch.sum(mask)
    epe = torch.sqrt(torch.sum(torch.square(flow - flow_gt), dim=1)).mean()
    return num / den, epe, warped, mask


# --------------------------------------------------------------------------------------
# Forward splat (softsplat_new.py:352-423 / 489-565 / 600-700)
# --------------------------------------------------------------------------------------


def _splat_remap(f: Tensor, size: int, scale: int, offset: int, which: str, axis: str):
    """The scale/offset remap block shared (with per-kernel quirks) by the three kernels.

    which = 'out'      : softsplat_new.py:374-390  (upper branch only when scale > 1)
            'ingrad'   : :515-532  (upper branch always; X has the extra ``* offset_x`` line :517)
            'flowgrad' : :629-647  (upper branch always; Y uses ``* offset_y`` :640; returns dflt)
    The reference mixes float and double (the literal 1.0 / 0.0 are doubles): the upper-branch
    update is evaluated in double and rounded to float on assignment -- reproduced here.
    Returns (remapped coordinate fp32, dflt fp32)."""
    f64 = f.double()
    upper = f64 >= (float(size) - 1.0)
    if which == "out":
        upper = upper & (scale > 1)
    lower = (~upper) & ((f - offset).double() < 0.0)
    mid = ~(upper | lower)
    k = float(abs(offset - (size % scale)) % scale)
    if which == "flowgrad" and axis == "y":
        k = float(offset)
    fu = (f64 + ((f - float(size)).double() + 1.0) * k).float()
    if which == "ingrad" and axis == "x":
        fu = (fu.double() + ((fu - float(size)).double() + 1.0) * float(offset)).float()
    fu = (fu - offset) / scale
    fl = f - offset
    fm = (f - offset) / scale
    out = torch.where(upper, fu, torch.where(lower, fl, fm))
    dflt = torch.where(mid, torch.full_like(f, 1.0 / scale), torch.zeros_like(f))
    return out, dflt


def _splat_geometry(flow: Tensor, H: int, W: int, scale: int, off_x: int, off_y: int, which: str):
    B = flow.shape[0]
    xx = torch.arange(W, dtype=torch.float32).view(1, 1, W).expand(B, H, W)
    yy = torch.arange(H, dtype=torch.float32).view(1, H, 1).expand(B, H, W)
    fx = xx + flow[:, 0]            # channel 0 = dx here (opposite of the backward warp)
    fy = yy + flow[:, 1]
    finite = torch.isfinite(fx) & torch.isfinite(fy)
    fx = torch.where(finite, fx, torch.zeros_like(fx))
    fy = torch.where(finite, fy, torch.zeros_like(fy))
    fx, dxx = _splat_remap(fx, W, scale, off_x, which, "x")
    fy, dyy = _splat_remap(fy, H, scale, off_y, which, "y")
    x0 = torch.floor(fx)
    y0 = torch.floor(fy)
    return fx, fy, x0, y0, finite, dxx, dyy


def splat_forward(ten_in: Tensor, flow: Tensor, scale: int = 1, off_x: int = 0, off_y: int = 0) -> Tensor:
    """softsplat_out, softsplat_new.py:352-423, as an index_add scatter (fp32)."""
    B, C, H, W = ten_in.shape
    Ho, Wo = H // scale, W // scale
    fx, fy, x0, y0, finite, _, _ = _splat_geometry(flow, H, W, scale, off_x, off_y, "out")
    x1, y1 = x0 + 1, y0 + 1
    taps = ((x0, y0, (x1 - fx) * (y1 - fy)), (x1, y0, (fx - x0) * (y1 - fy)),
            (x0, y1, (x1 - fx) * (fy - y0)), (x1, y1, (fx - x0) * (fy - y0)))
    out = torch.zeros(B, C, Ho * Wo)
    src = ten_in.reshape(B, C, H * W)
    for xs, ys, wt in taps:
        ok = finite & (xs >= 0) & (xs < Wo) & (ys >= 0) & (ys < Ho)
        idx = (ys.clamp(0, Ho - 1) * Wo + xs.clamp(0, Wo - 1)).long().reshape(B, 1, H * W).expand(B, C, H * W)
        contrib = src * torch.where(ok, wt, torch.zeros_like(wt)).reshape(B, 1, H * W)
        out.scatter_add_(2, idx, contrib)
    return out.reshape(B, C, Ho, Wo)


def splat_ingrad(ten_in_shape, flow: Tensor, outgrad: Tensor, scale: int = 1, off_x: int = 0, off_y: int = 0):
    """softsplat_ingrad, softsplat_new.py:489-565 (4-tap gather of outgrad)."""
    B, C, H, W = ten_in_shape
    Ho, Wo = outgrad.shape[-2:]
    fx, fy, x0, y0, finite, _, _ = _splat_geometry(flow, H, W, scale, off_x, off_y, "ingrad")
    x1, y1 = x0 + 1, y0 + 1
    taps = ((x0, y0, (x1 - fx) * (y1 - fy)), (x1, y0, (fx - x0) * (y1 - fy)),
            (x0, y1, (x1 - fx) * (fy - y0)), (x1, y1, (fx - x0) * (fy - y0)))
    g = outgrad.reshape(B, C, Ho * Wo)
    acc = torch.zeros(B, C, H * W)
    for xs, ys, wt in taps:
        ok = finite & (xs >= 0) & (xs < Wo) & (ys >= 0) & (ys < Ho)
        idx = (ys.clamp(0, Ho - 1) * Wo + xs.clamp(0, Wo - 1)).long().reshape(B, 1, H * W).expand(B, C, H * W)
        acc = acc + g.gather(2, idx) * torch.where(ok, wt, torch.zeros_like(wt)).reshape(B, 1, H * W)
    return acc.reshape(B, C, H, W)


def splat_flowgrad(ten_in: Tensor, flow: Tensor, outgrad: Tensor, scale: int = 1, off_x: int = 0, off_y: int = 0):
    """softsplat_flowgrad, softsplat_new.py:600-700, including its quirks:
    channel 0 (d/dx) is scaled by dfltYY and channel 1 by dfltXX (:664-672); dflt is 0 outside
    the 'else' remap branch (:626-647, the "freeze gradient" comment)."""
    B, C, H, W = ten_in.shape
    Ho, Wo = outgrad.shape[-2:]
    fx, fy, x0, y0, finite, dxx, dyy = _splat_geometry(flow, H, W, scale, off_x, off_y, "flowgrad")
    x1, y1 = x0 + 1, y0 + 1
    corners = ((x0, y0), (x1, y0), (x0, y1), (x1, y1))
    w_dx = (-1.0 * (y1 - fy), +1.0 * (y1 - fy), -1.0 * (fy - y0), +1.0 * (fy - y0))
    w_dy = ((x1 - fx) * -1.0, (fx - x0) * -1.0, (x1 - fx) * +1.0, (fx - x0) * +1.0)
    g = outgrad.reshape(B, C, Ho * Wo)
    src = ten_in.reshape(B, C, H * W)
    res = []
    for wts, dflt in ((w_dx, dyy), (w_dy, dxx)):
        acc = torch.zeros(B, H * W)
        for ch in range(C):
            for (xs, ys), wt in zip(corners, wts):
                ok = finite & (xs >= 0) & (xs < Wo) & (ys >= 0) & (ys < Ho)
                idx = (ys.clamp(0, Ho - 1) * Wo + xs.clamp(0, Wo - 1)).long().reshape(B, H * W)
                term = g[:, ch].gather(1, idx) * src[:, ch] * wt.reshape(B, H * W) * dflt.reshape(B, H * W)
                acc = acc + torch.where(ok.reshape(B, H * W), term, torch.zeros_like(term))
        res.append(acc.reshape(B, H, W))
    return torch.stack(res, dim=1)


def warp_forward_flow(first: Tensor, flow: Tensor, scale: int = 1, set_nans: bool = True,
                      offset=(0, 0)) -> Tensor:
    """warp_forward_flow(..., warp_style='sum') -> softsplat(mode 'linear_unn'):
    warp.py:121-156 + softsplat_new.py:301-302, 329-330."""
    first = first.clone()
    weights = torch.ones_like(first[:, 0])
    nans = torch.isnan(first)
    first[nans] = 0.0
    weights[torch.any(nans, dim=1)] = 0.0
    offset = [o % scale for o in offset]
    ten_in = torch.cat([first * weights[:, None], weights[:, None]], 1)
    if torch.is_grad_enabled() and (ten_in.requires_grad or flow.requires_grad):
        ret = _SplatFn.apply(ten_in, flow, scale, offset[0], offset[1])      # softsplat_func under autograd (:339-733)
    else:
        ret = splat_forward(ten_in, flow, scale, offset[0], offset[1])
    img = ret[:, :-1]
    wsum = ret[:, -1:].expand_as(img)
    if set_nans:
        img = torch.where(wsum > 0, img, torch.full_like(img, float("nan")))
    return img


# --------------------------------------------------------------------------------------
# FlowLearner objective (flow_learner.py:133-222, warp.py:273-303, softsplat_new.py:278-333)
# --------------------------------------------------------------------------------------


class _SplatFn(torch.autograd.Function):
    """softsplat_func (softsplat_new.py:339-733) over the three restated kernels."""

    @staticmethod
    def forward(ctx, ten_in, flow, scale, off_x, off_y):
        ctx.save_for_backward(ten_in, flow)
        ctx.geom = (scale, off_x, off_y)
        return splat_forward(ten_in, flow, scale, off_x, off_y)

    @staticmethod
    def backward(ctx, gout):
        ten_in, flow = ctx.saved_tensors
        scale, ox, oy = ctx.geom
        gin = splat_ingrad(ten_in.shape, flow, gout, scale, ox, oy) if ctx.needs_input_grad[0] else None
        gflow = splat_flowgrad(ten_in, flow, gout, scale, ox, oy) if ctx.needs_input_grad[1] else None
        return gin, gflow, None, None, None


def softsplat_soft(ten_in: Tensor, flow: Tensor, metric: Tensor, scale: int, offset) -> Tensor:
    """softsplat(..., strMode='soft', scale, offset): softsplat_new.py:306-331."""
    x = torch.cat([ten_in * metric.exp(), metric.exp()], 1)
    out = _SplatFn.apply(x, flow, scale, offset[0], offset[1])
    norm = out[:, -1:] + 0.0000001
    return torch.cat((out[:, :-1] / norm, out[:, -1:]), dim=1)


def fill_holes_nan(img: Tensor, weights: Tensor) -> Tensor:
    """warp.py:273-276."""
    weights = weights.repeat((1, img.shape[1], 1, 1))
    return torch.where(weights > 0, img, torch.full_like(img, float("nan")))


def nan_charbonnier(pred: Tensor, target: Tensor) -> Tensor:
    """warp.py:281-287."""
    pred, target = pred.flatten(), target.flatten()
    keep = torch.logical_not(torch.logical_or(torch.isnan(target), torch.isnan(pred)))
    return torch.mean(charbonnier(pred[keep] - target[keep]))


def edgeaware_smoothness1(image: Tensor, flow: Tensor, edge_weight: float = 30) -> Tensor:
    """warp.py:289-303."""
    igy = image[:, :, 1:, :] - image[:, :, :-1, :]
    igx = image[:, :, :, 1:] - image[:, :, :, :-1]
    fgy = flow[:, :, 1:, :] - flow[:, :, :-1, :]
    fgx = flow[:, :, :, 1:] - flow[:, :, :, :-1]
    yw = torch.exp(-edge_weight * torch.mean(igy ** 2, dim=1, keepdim=True))
    xw = torch.exp(-edge_weight * torch.mean(igx ** 2, dim=1, keepdim=True))
    return (torch.mean(xw * charbonnier(fgx)) + torch.mean(yw * charbonnier(fgy))) / 2


FLOW_LEARNER_LEVELS = (1, 2, 4, 5, 7, 8, 10, 11, 14, 16)


def flow_learner_objective(img: Tensor, tgt: Tensor, flow_pred: Tensor, weights: Tensor,
                           levels=FLOW_LEARNER_LEVELS) -> Tensor:
    """The loop of FlowLearner.loss (flow_learner.py:160-205) given the prediction (flow in pixels, splat weights)."""
    photo = []
    for level in levels:
        terms = []
        for a in range(level):
            for b in range(level):
                ww = softsplat_soft(img, flow_pred, weights, level, (a, b))
                filled = fill_holes_nan(ww[:, :-1], ww[:, -1:])
                tt = softsplat_soft(tgt, torch.zeros_like(flow_pred), torch.ones_like(weights), level, (a, b))
                terms.append(nan_charbonnier(tt[:, :-1], filled))
        photo.append(sum(terms) / len(terms))
    loss = sum(photo) / len(photo)
    return loss + edgeaware_smoothness1(img, flow_pred) * 0.01


def flow_learner_loss(sd, tgt: Tensor, cond: Tensor, flow_max: float = 20.0, levels=FLOW_LEARNER_LEVELS,
                      prefix: str = "") -> Tensor:
    """FlowLearner.loss (flow_learner.py:133-222) for the flow representation: UnetWithWarp's inner Unet
    (channels 6, out_dim 3, time_in False) -> flow * flow_max + weights -> multi-scale soft-splat Charbonnier."""
    fw = unet_forward(sd, cond, None, None, prefix)
    return flow_learner_objective(cond[:, :3], tgt, fw[:, :2] * flow_max, fw[:, 2:], levels)


# --------------------------------------------------------------------------------------
# Synthetic Sintel-shaped inputs (SURVEY.md section 8d) shared by tests and bench
# --------------------------------------------------------------------------------------


def synthetic_frames(batch: int, height: int, width: int, seed: int = 0) -> Tensor:
    """Smooth random RGB frames in [0,1]: 4 low-frequency sinusoids + U[0,0.05] noise."""
    g = torch.Generator().manual_seed(seed)
    yy = torch.linspace(0, 1, height).view(1, 1, height, 1)
    xx = torch.linspace(0, 1, width).view(1, 1, 1, width)
    img = torch.zeros(batch, 3, height, width)
    for _ in range(4):
        fx = torch.rand(batch, 3, 1, 1, generator=g) * 6.0
        fy = torch.rand(batch, 3, 1, 1, generator=g) * 6.0
        ph = torch.rand(batch, 3, 1, 1, generator=g) * 6.2831853
        img = img + 0.125 * torch.sin(6.2831853 * (fx * xx + fy * yy) + ph)
    img = img + 0.5 + torch.rand(batch, 3, height, width, generator=g) * 0.05
    return img.clamp(0.0, 1.0)


def replicate_pad_to_multiple(x: Tensor, multiple: int = 8) -> Tuple[Tensor, Tuple[int, int, int, int]]:
    """InputPadder(mode='sintel') semantics, future/raft_utils.py:7-25."""
    ht, wd = x.shape[-2:]
    pad_ht = (((ht // multiple) + 1) * multiple - ht) % multiple
    pad_wd = (((wd // multiple) + 1) * multiple - wd) % multiple
    pad = (pad_wd // 2, pad_wd - pad_wd // 2, pad_ht // 2, pad_ht - pad_ht // 2)
    return F.pad(x, pad, mode="replicate"), pad
