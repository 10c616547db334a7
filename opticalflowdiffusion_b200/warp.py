"""Warp operators of the flow_diffuser path, same names and argument meaning as the reference's
``algorithms/diffusion_animation/warp.py`` (dispatcher :83-93, ``warp_backward_flow`` :95-119,
``warp_forward_flow`` :121-156, ``nan_mse`` :260-271, ``charbonnier`` :278-279) and
``softsplat_new.softsplat`` (:278-333), executed by the sm_100a kernels of ``libflowdiff.so``.

Only ``rep='flow'`` is implemented (the filter representation is never used by flow_diffuser,
SURVEY.md section 2).  All tensors must be CUDA fp32; there is no CPU path.
"""
from __future__ import annotations

from typing import Optional, Sequence, Tuple

import torch

from . import _lib

Tensor = torch.Tensor


def _f32c(t: Tensor) -> Tensor:
    _lib.require_cuda(t)
    if t.dtype != torch.float32:
        t = t.float()
    return t.contiguous()


# --------------------------------------------------------------------------------------
# backward warp
# --------------------------------------------------------------------------------------


def _workspace(floats: int, device) -> Optional[Tensor]:
    """A kernel workspace of the size the library asked for (None -> NULL when it needs none)."""
    return torch.empty(floats, device=device, dtype=torch.float32) if floats else None


def _bwd_workspace(lib, image: Tensor, need_image_grad: bool) -> Optional[Tensor]:
    """Workspace of the warp backward kernels (pixel-interleaved frame gradient): only a requested frame gradient uses it."""
    return _workspace(lib.fd_warp_bwd_workspace_floats(*image.shape), image.device) if need_image_grad else None


class _BackwarpFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, image: Tensor, flow: Tensor):
        image, flow = _f32c(image), _f32c(flow)
        B, C, H, W = image.shape
        assert flow.shape == (B, 2, H, W), (flow.shape, image.shape)
        out = torch.empty_like(image)
        mask = torch.empty_like(image)
        lib = _lib.load()
        _lib.check(lib.fd_backwarp_fwd(_lib.ptr(image), _lib.ptr(flow), _lib.ptr(out), _lib.ptr(mask),
                                       B, C, H, W, _lib.stream()))
        ctx.save_for_backward(image, flow)
        ctx.mark_non_differentiable(mask)
        return out, mask

    @staticmethod
    def backward(ctx, gout: Tensor, _gmask):
        image, flow = ctx.saved_tensors
        B, C, H, W = image.shape
        gout = _f32c(gout)
        gimage = torch.empty_like(image) if ctx.needs_input_grad[0] else None
        gflow = torch.empty_like(flow) if ctx.needs_input_grad[1] else None
        lib = _lib.load()
        ws = _bwd_workspace(lib, image, gimage is not None)
        _lib.check(lib.fd_backwarp_bwd(_lib.ptr(image), _lib.ptr(flow), _lib.ptr(gout), _lib.ptr(gimage),
                                       _lib.ptr(gflow), _lib.ptr(ws), B, C, H, W, _lib.stream()))
        return gimage, gflow


def warp_backward_flow(first: Optional[Tensor], second: Tensor, flow: Tensor) -> Tuple[Tensor, Tensor]:
    """``(output, mask)``: bilinear backward warp of ``second`` by ``flow`` (channel 0 = dy, channel 1 = dx;
    the reference flips, warp.py:105); ``mask`` is 1 where all four taps are inside (warp.py:113-117)."""
    return _BackwarpFn.apply(second, flow)


class _PhotoEpeFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, frame1: Tensor, frame2: Tensor, flow: Tensor, flow_gt: Tensor):
        frame1, frame2, flow, flow_gt = (_f32c(t) for t in (frame1, frame2, flow, flow_gt))
        B, C, H, W = frame2.shape
        lib = _lib.load()
        sums = torch.empty(4, device=flow.device, dtype=torch.float32)
        ws = torch.empty(lib.fd_photo_epe_workspace_floats(B, H, W), device=flow.device, dtype=torch.float32)
        _lib.check(lib.fd_backwarp_photo_epe_fwd(_lib.ptr(frame1), _lib.ptr(frame2), _lib.ptr(flow),
                                                 _lib.ptr(flow_gt), _lib.ptr(sums), _lib.ptr(ws),
                                                 B, C, H, W, _lib.stream()))
        ctx.save_for_backward(frame1, frame2, flow, flow_gt, sums)
        photo = sums[0] / sums[1]
        epe = sums[2] / sums[3]
        return photo, epe

    @staticmethod
    def backward(ctx, g_photo: Tensor, g_epe: Tensor):
        frame1, frame2, flow, flow_gt, sums = ctx.saved_tensors
        B, C, H, W = frame2.shape
        gflow = torch.empty_like(flow) if ctx.needs_input_grad[2] else None
        gframe2 = torch.empty_like(frame2) if ctx.needs_input_grad[1] else None
        lib = _lib.load()
        # the kernel scales by g_photo / sums[1] and g_epe / sums[3]: the upstream gradients stay on the device, folded into
        # a copy of the sums (no device-to-host read in the backward pass)
        sg = sums.clone()
        sg[1] = sums[1] / g_photo.detach().float()
        sg[3] = sums[3] / g_epe.detach().float()
        ws = _bwd_workspace(lib, frame2, gframe2 is not None)
        _lib.check(lib.fd_backwarp_photo_epe_bwd(_lib.ptr(frame1), _lib.ptr(frame2), _lib.ptr(flow),
                                                 _lib.ptr(flow_gt), _lib.ptr(sg), 1.0, 1.0,
                                                 _lib.ptr(gflow), _lib.ptr(gframe2), _lib.ptr(ws), B, C, H, W, _lib.stream()))
        return None, gframe2, gflow, None


def photometric_epe(frame1: Tensor, frame2: Tensor, flow: Tensor, flow_gt: Tensor) -> Tuple[Tensor, Tensor]:
    """Fused ``warp_backward_flow`` + occlusion-weighted Charbonnier (losses.py:3-6,46-47, normalised by the
    mask mass) + end-point error; one pass over the inputs, nothing materialised.  Differentiable in
    ``flow`` and ``frame2``."""
    return _PhotoEpeFn.apply(frame1, frame2, flow, flow_gt)


# --------------------------------------------------------------------------------------
# forward splat
# --------------------------------------------------------------------------------------


class softsplat_func(torch.autograd.Function):
    """softsplat_new.softsplat_func (:339-733): fp32 even under autocast."""

    @staticmethod
    def forward(ctx, tenIn: Tensor, tenFlow: Tensor, scale: int, offset_x: int, offset_y: int):
        tenIn, tenFlow = _f32c(tenIn), _f32c(tenFlow)
        B, C, H, W = tenIn.shape
        out = torch.empty(B, C, H // scale, W // scale, device=tenIn.device, dtype=torch.float32)
        lib = _lib.load()
        ws = _workspace(lib.fd_splat_fwd_workspace_floats(B, C, H, W, int(scale)), tenIn.device)
        _lib.check(lib.fd_splat_fwd(_lib.ptr(tenIn), _lib.ptr(tenFlow), _lib.ptr(out), _lib.ptr(ws), B, C, H, W,
                                    int(scale), int(offset_x), int(offset_y), _lib.stream()))
        ctx.save_for_backward(tenIn, tenFlow)
        ctx.geom = (int(scale), int(offset_x), int(offset_y))
        return out

    @staticmethod
    def backward(ctx, tenOutgrad: Tensor):
        tenIn, tenFlow = ctx.saved_tensors
        scale, ox, oy = ctx.geom
        B, C, H, W = tenIn.shape
        tenOutgrad = _f32c(tenOutgrad)
        lib = _lib.load()
        gin = gflow = None
        if ctx.needs_input_grad[0]:
            gin = torch.empty_like(tenIn)
            _lib.check(lib.fd_splat_ingrad(_lib.ptr(tenFlow), _lib.ptr(tenOutgrad), _lib.ptr(gin), B, C, H, W,
                                           scale, ox, oy, _lib.stream()))
        if ctx.needs_input_grad[1]:
            gflow = torch.empty_like(tenFlow)
            _lib.check(lib.fd_splat_flowgrad(_lib.ptr(tenIn), _lib.ptr(tenFlow), _lib.ptr(tenOutgrad),
                                             _lib.ptr(gflow), B, C, H, W, scale, ox, oy, _lib.stream()))
        return gin, gflow, None, None, None


def softsplat(tenIn: Tensor, tenFlow: Tensor, tenMetric: Optional[Tensor], strMode: str, scale: int = 1,
              offset: Sequence[int] = (0, 0)) -> Tensor:
    """softsplat_new.softsplat (:278-333) for the modes the flow_diffuser path uses."""
    mode = strMode.split("-")[0]
    assert mode in ("sum", "avg", "linear", "soft", "linear_unn")
    if mode in ("sum", "avg"):
        assert tenMetric is None
    else:
        assert tenMetric is not None
    if mode == "avg":
        tenIn = torch.cat([tenIn, tenIn.new_ones(tenIn.shape[0], 1, tenIn.shape[2], tenIn.shape[3])], 1)
    elif mode in ("linear", "linear_unn"):
        tenIn = torch.cat([tenIn * tenMetric, tenMetric], 1)
    elif mode == "soft":
        tenIn = torch.cat([tenIn * tenMetric.exp(), tenMetric.exp()], 1)
    tenOut = softsplat_func.apply(tenIn, tenFlow, scale, offset[0], offset[1])
    if mode in ("avg", "linear", "soft"):
        norm = tenOut[:, -1:, :, :]
        parts = strMode.split("-")
        if len(parts) == 1 or parts[1] == "addeps":
            norm = norm + 0.0000001
        elif parts[1] == "zeroeps":
            norm = torch.where(norm == 0.0, torch.ones_like(norm), norm)
        elif parts[1] == "clipeps":
            norm = norm.clip(0.0000001, None)
        return torch.cat((tenOut[:, :-1] / norm, tenOut[:, -1:]), dim=1)
    return tenOut


class _ForwardWarpSumFn(torch.autograd.Function):
    """warp_forward_flow(warp_style='sum') as prepare (NaN -> weight 0, append the weight channel),
    splat, finish (holes -> NaN); for three-channel images fused into the two launches of
    fd_forward_warp_sum3.  Gradient flows to ``flow`` only (cond has no grad in training, SURVEY.md
    S2) and to ``first`` on request."""

    @staticmethod
    def forward(ctx, first: Tensor, flow: Tensor, scale: int, set_nans: bool, off_x: int, off_y: int):
        first, flow = _f32c(first), _f32c(flow)
        B, C, H, W = first.shape
        lib = _lib.load()
        st = _lib.stream()
        if C == 3:
            # two launches, pixel-interleaved accumulation (one 128-bit reduction per tap): fd_forward_warp_sum3
            Ho, Wo = H // scale, W // scale
            need_bwd = bool(ctx.needs_input_grad[0] or ctx.needs_input_grad[1])
            ten_in = torch.empty(B, 4, H, W, device=first.device, dtype=torch.float32) if need_bwd else None
            acc = torch.empty(B, Ho, Wo, 4, device=first.device, dtype=torch.float32)
            img = torch.empty(B, 3, Ho, Wo, device=first.device, dtype=torch.float32)
            wsum = torch.empty(B, 1, Ho, Wo, device=first.device, dtype=torch.float32) if need_bwd else None
            _lib.check(lib.fd_forward_warp_sum3(_lib.ptr(first), _lib.ptr(flow), _lib.ptr(ten_in), _lib.ptr(acc), _lib.ptr(img),
                                                _lib.ptr(wsum), B, H, W, scale, off_x, off_y, int(bool(set_nans)), st))
            if need_bwd:
                ctx.save_for_backward(ten_in, flow, wsum)
            ctx.geom = (scale, off_x, off_y, bool(set_nans))
            return img
        ten_in = torch.empty(B, C + 1, H, W, device=first.device, dtype=torch.float32)
        _lib.check(lib.fd_splat_prepare(_lib.ptr(first), _lib.ptr(ten_in), B, C, H * W, st))
        Ho, Wo = H // scale, W // scale
        ret = torch.empty(B, C + 1, Ho, Wo, device=first.device, dtype=torch.float32)
        ws = _workspace(lib.fd_splat_fwd_workspace_floats(B, C + 1, H, W, scale), first.device)
        _lib.check(lib.fd_splat_fwd(_lib.ptr(ten_in), _lib.ptr(flow), _lib.ptr(ret), _lib.ptr(ws), B, C + 1, H, W, scale,
                                    off_x, off_y, st))
        img = torch.empty(B, C, Ho, Wo, device=first.device, dtype=torch.float32)
        _lib.check(lib.fd_splat_finish(_lib.ptr(ret), _lib.ptr(img), B, C, Ho * Wo, int(bool(set_nans)), st))
        ctx.save_for_backward(ten_in, flow, ret)
        ctx.geom = (scale, off_x, off_y, bool(set_nans))
        return img

    @staticmethod
    def backward(ctx, gimg: Tensor):
        ten_in, flow, ret = ctx.saved_tensors
        scale, ox, oy, set_nans = ctx.geom
        B, C1, H, W = ten_in.shape
        gimg = _f32c(gimg)
        # d(img)/d(ret[:, :C]) = 1 where the hole mask keeps the value (torch.where, warp.py:155), else 0
        if set_nans:
            gimg = torch.where(ret[:, -1:] > 0, gimg, torch.zeros_like(gimg))
        gout = torch.cat([gimg, torch.zeros_like(gimg[:, :1])], 1).contiguous()
        lib = _lib.load()
        gfirst = gflow = None
        if ctx.needs_input_grad[0]:
            gin = torch.empty_like(ten_in)
            _lib.check(lib.fd_splat_ingrad(_lib.ptr(flow), _lib.ptr(gout), _lib.ptr(gin), B, C1, H, W, scale, ox, oy,
                                           _lib.stream()))
            gfirst = gin[:, :-1] * ten_in[:, -1:]
        if ctx.needs_input_grad[1]:
            gflow = torch.empty_like(flow)
            _lib.check(lib.fd_splat_flowgrad(_lib.ptr(ten_in), _lib.ptr(flow), _lib.ptr(gout), _lib.ptr(gflow),
                                             B, C1, H, W, scale, ox, oy, _lib.stream()))
        return gfirst, gflow, None, None, None, None


def warp_forward_flow(first: Tensor, second: Optional[Tensor], flow: Tensor, scale: int = 1, set_nans: bool = True,
                      get_variance: bool = False, offset: Sequence[int] = (0, 0), warp_style: str = "sum") -> Tensor:
    """Forward splat of ``first`` along ``flow`` (channel 0 = dx, 1 = dy): warp.py:121-156."""
    if get_variance or warp_style != "sum":
        # the general path: the reference's python wrapper around the splat kernel
        first = first.clone()
        weights = torch.ones_like(first[:, 0])
        nans = torch.isnan(first)
        first[nans] = 0.0
        weights[torch.any(nans, dim=1)] = 0.0
        off = [o % scale for o in offset]
        mode = "linear_unn" if warp_style == "sum" else "linear"
        ret = softsplat(first, flow, weights[:, None], mode, scale, off)
        img = ret[:, :-1]
        wsum = ret[:, -1, None].repeat(1, img.shape[1], 1, 1)
        if get_variance:
            var = softsplat(torch.square(first), flow, weights[:, None].clone(), "linear_unn", scale, off)
            img = var[:, :-1] - torch.square(img)
        if set_nans:
            img = torch.where(wsum > 0, img, torch.full_like(img, float("nan")))
        return img
    off = [int(o) % int(scale) for o in offset]
    return _ForwardWarpSumFn.apply(first, flow, int(scale), bool(set_nans), off[0], off[1])


def warp(first, second, flow, rep: str = "flow", mode: str = "backward", **kwargs):
    """Dispatcher, warp.py:83-93."""
    if rep != "flow":
        raise NotImplementedError("only rep='flow' is on the flow_diffuser path (SURVEY.md section 2)")
    if mode == "backward":
        return warp_backward_flow(first, second, flow, **kwargs)
    if mode == "forward":
        return warp_forward_flow(first, second, flow, **kwargs)
    raise ValueError(mode)


# --------------------------------------------------------------------------------------
# losses
# --------------------------------------------------------------------------------------


class _NanMseFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, pred: Tensor, target: Tensor):
        pred, target = _f32c(pred), _f32c(target)
        assert pred.shape == target.shape
        n = pred.numel()
        lib = _lib.load()
        sums = torch.empty(3, device=pred.device, dtype=torch.float32)
        ws = torch.empty(lib.fd_nan_mse_workspace_floats(1, 1, n), device=pred.device, dtype=torch.float32)
        _lib.check(lib.fd_nan_mse_fwd(_lib.ptr(pred), _lib.ptr(target), _lib.ptr(sums), _lib.ptr(ws), 1, 1, n, n, n,
                                      _lib.stream()))
        ctx.save_for_backward(pred, target, sums)
        return sums[2].clone()

    @staticmethod
    def backward(ctx, g: Tensor):
        pred, target, sums = ctx.saved_tensors
        n = pred.numel()
        gpred = torch.empty_like(pred)
        lib = _lib.load()
        sg = sums.clone()
        sg[1] = sums[1] / g.detach().float()          # upstream gradient folded in on the device (no host read)
        _lib.check(lib.fd_nan_mse_bwd(_lib.ptr(pred), _lib.ptr(target), _lib.ptr(sg), 1.0, _lib.ptr(gpred),
                                      1, 1, n, n, n, n, _lib.stream()))
        return gpred, None


def nan_mse(pred: Tensor, target: Tensor, reduction: str = "mean") -> Tensor:
    """warp.py:260-271.  ``reduction='mean'`` is one fused reduction; ``'none'`` needs the compacted
    vector and is only kept for API parity (it is not on the fast path)."""
    if reduction == "mean":
        return _NanMseFn.apply(pred, target)
    pred, target = pred.flatten(), target.flatten()
    keep = ~(torch.isnan(target) | torch.isnan(pred))
    return torch.square(pred[keep] - target[keep])


def charbonnier(x: Tensor, alpha: float = 0.5, eps: float = 1e-3) -> Tensor:
    """warp.py:278-279 / losses.py:46-47."""
    return torch.pow(torch.square(x) + eps ** 2, alpha)


# --------------------------------------------------------------------------------------
# FlowLearner objective (flow_learner.py:133-222): fused loss terms
# --------------------------------------------------------------------------------------


class _SoftCharbFn(torch.autograd.Function):
    """softsplat's normalisation (softsplat_new.py:316-331) + fill_holes_nan (warp.py:273-276) + nan_charbonnier
    (warp.py:281-287) of one (level, offset) term, from the RAW soft splats S (prediction) and T (target)."""

    @staticmethod
    def forward(ctx, S: Tensor, T: Tensor):
        S, T = _f32c(S), _f32c(T)
        assert S.shape == T.shape
        B, C1, H, W = S.shape
        lib = _lib.load()
        sums = torch.empty(3, device=S.device, dtype=torch.float32)
        ws = torch.empty(lib.fd_loss_workspace_floats(B * H * W), device=S.device, dtype=torch.float32)
        _lib.check(lib.fd_soft_charb_fwd(_lib.ptr(S), _lib.ptr(T), _lib.ptr(sums), _lib.ptr(ws), B, C1 - 1, H * W, _lib.stream()))
        ctx.save_for_backward(S, T, sums)
        return sums[2].clone()

    @staticmethod
    def backward(ctx, g: Tensor):
        S, T, sums = ctx.saved_tensors
        B, C1, H, W = S.shape
        gS = torch.empty_like(S)
        g = g.detach().float().reshape(1).contiguous()
        _lib.check(_lib.load().fd_soft_charb_bwd(_lib.ptr(S), _lib.ptr(T), _lib.ptr(sums), _lib.ptr(g), _lib.ptr(gS), B, C1 - 1,
                                                 H * W, _lib.stream()))
        return gS, None


def soft_splat_charbonnier(S: Tensor, T: Tensor) -> Tensor:
    return _SoftCharbFn.apply(S, T)


def soft_splat_raw(tenIn: Tensor, tenFlow: Tensor, tenMetric: Tensor, scale: int, offset: Sequence[int]) -> Tensor:
    """The un-normalised 'soft' splat: softsplat_func(cat(in * exp(metric), exp(metric))) (softsplat_new.py:306-309)."""
    e = tenMetric.exp()
    return softsplat_func.apply(torch.cat([tenIn * e, e], 1), tenFlow, scale, offset[0], offset[1])


class _EdgeSmoothFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, image: Tensor, flow: Tensor):
        image, flow = _f32c(image), _f32c(flow)
        B, Ci, H, W = image.shape
        Cf = flow.shape[1]
        lib = _lib.load()
        out = torch.empty(1, device=flow.device, dtype=torch.float32)
        ws = torch.empty(lib.fd_loss_workspace_floats(B * H * W), device=flow.device, dtype=torch.float32)
        _lib.check(lib.fd_edge_smooth_fwd(_lib.ptr(image), _lib.ptr(flow), _lib.ptr(out), _lib.ptr(ws), B, Ci, Cf, H, W,
                                          _lib.stream()))
        ctx.save_for_backward(image, flow)
        return out[0].clone()

    @staticmethod
    def backward(ctx, g: Tensor):
        image, flow = ctx.saved_tensors
        B, Ci, H, W = image.shape
        gflow = torch.empty_like(flow)
        g = g.detach().float().reshape(1).contiguous()
        _lib.check(_lib.load().fd_edge_smooth_bwd(_lib.ptr(image), _lib.ptr(flow), _lib.ptr(g), _lib.ptr(gflow), B, Ci,
                                                  flow.shape[1], H, W, _lib.stream()))
        return None, gflow


def edgeaware_smoothness1(image: Tensor, flow: Tensor, edge_weight: float = 30) -> Tensor:
    """warp.py:289-303 (edge_weight is fixed at the reference's default of 30 in the kernel)."""
    assert edge_weight == 30
    return _EdgeSmoothFn.apply(image, flow)


def fill_holes_nan(img: Tensor, weights: Tensor) -> Tensor:
    """warp.py:273-276."""
    return torch.where(weights.expand_as(img) > 0, img, torch.full_like(img, float("nan")))


class _SoftLevelLossFn(torch.autograd.Function):
    """One pyramid level of FlowLearner's photometric loss (flow_learner.py:184-202) with all level^2 offsets batched:
    mean over (a, b) of nan_charbonnier(softsplat(tgt, 0), fill_holes(softsplat(img, flow))).  Seven launches per level
    (splat, target splat, loss, and their three backward kernels) instead of ~8 per offset."""

    @staticmethod
    def forward(ctx, ten_in: Tensor, flow: Tensor, tgt_in: Tensor, level: int):
        ten_in, flow, tgt_in = _f32c(ten_in), _f32c(flow), _f32c(tgt_in)
        B, C1, H, W = ten_in.shape
        lib, st = _lib.load(), _lib.stream()
        K, Ho, Wo = level * level, H // level, W // level
        assert C1 == 4, C1
        S = torch.empty(K, B, Ho, Wo, C1, device=ten_in.device, dtype=torch.float32)      # pixel-interleaved (r, g, b, weight)
        T = torch.empty_like(S)
        _lib.check(lib.fd_splat_fwd_multi(_lib.ptr(ten_in), _lib.ptr(flow), _lib.ptr(S), B, C1, H, W, level, st))
        zero = torch.zeros_like(flow)
        _lib.check(lib.fd_splat_fwd_multi(_lib.ptr(tgt_in), _lib.ptr(zero), _lib.ptr(T), B, C1, H, W, level, st))
        sums = torch.empty(K, 3, device=S.device, dtype=torch.float32)
        out = torch.empty(1, device=S.device, dtype=torch.float32)
        ws = torch.empty(lib.fd_soft_charb_multi_workspace_floats(B, Ho * Wo, K), device=S.device, dtype=torch.float32)
        _lib.check(lib.fd_soft_charb_multi_fwd(_lib.ptr(S), _lib.ptr(T), _lib.ptr(sums), _lib.ptr(out), _lib.ptr(ws), B, C1 - 1,
                                               Ho * Wo, K, st))
        ctx.save_for_backward(ten_in, flow, S, T, sums)
        ctx.level = level
        return out[0].clone()

    @staticmethod
    def backward(ctx, g: Tensor):
        ten_in, flow, S, T, sums = ctx.saved_tensors
        level = ctx.level
        K, B, Ho, Wo, C1 = S.shape
        H, W = ten_in.shape[-2:]
        lib, st = _lib.load(), _lib.stream()
        g = g.detach().float().reshape(1).contiguous()
        gS = torch.empty_like(S)
        _lib.check(lib.fd_soft_charb_multi_bwd(_lib.ptr(S), _lib.ptr(T), _lib.ptr(sums), _lib.ptr(g), _lib.ptr(gS), B, C1 - 1,
                                               Ho * Wo, K, st))
        gin = gflow = None
        if ctx.needs_input_grad[0]:
            gin = torch.empty_like(ten_in)
            _lib.check(lib.fd_splat_ingrad_multi(_lib.ptr(flow), _lib.ptr(gS), _lib.ptr(gin), B, C1, H, W, level, st))
        if ctx.needs_input_grad[1]:
            gflow = torch.empty_like(flow)
            _lib.check(lib.fd_splat_flowgrad_multi(_lib.ptr(ten_in), _lib.ptr(flow), _lib.ptr(gS), _lib.ptr(gflow), B, C1, H, W,
                                                   level, st))
        return gin, gflow, None, None


def soft_level_loss(ten_in: Tensor, flow: Tensor, tgt_in: Tensor, level: int) -> Tensor:
    return _SoftLevelLossFn.apply(ten_in, flow, tgt_in, int(level))
