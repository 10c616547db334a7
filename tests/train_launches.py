"""The distinct kernel launches of the UNet training step at the benchmark's shapes (bench.py: batch 8, 368 x 768 crops):
one training forward of ``Unet(64, 5, 2)`` with autograd on and its backward, and the error bounds their GPU checks
(tests/test_gpu_train_launches.py) hold each launch to.

``record_train(B, H, W)`` records both passes on the CPU with the fake library of tests/test_unet_host.py, as
``bench_launches.record`` does for the inference forward; ``TRAIN`` is that record at 8 x 368 x 768, committed, and
tests/test_train_launch_table.py re-records it.

Two legs check every linear kernel.  The exact leg feeds integer operands in {-1, 0, 1}: see ``exact_terms``.  The real leg
feeds Gaussian operands and holds the kernel to a rounding bound (the helpers below, next to those of bench_launches)."""
import math

import torch

import bench_launches as BL


def record_train(B, H, W):
    """{(name, scalars, nulls): count} of one training forward + backward of Unet(64, 5, 2) on a B x H x W batch."""
    return BL.record(B, H, W, train=True)


# ------------------------------------------------------------------------------------------------------------ exact leg
# Exact leg.  Operands are integers in {-1, 0, 1}; an output documented as += starts at FILL.  Then every partial sum a
# kernel forms is a multiple of FILL whose magnitude is at most the sum of |terms| of the whole reduction (plus |FILL|).
# When that is below 2^22, it is exact in fp32 under the accumulation model of ``bench_launches.gamma_mma``: an fp32
# addition (or a tensor-core step) loses at most one unit in the last place of a running sum of magnitude < 2^22 -- and
# the last place of such a sum is at most 2^-2 = FILL, below which none of these numbers has a bit.  So, whatever the
# summation order, split or atomics: fp32 outputs equal the fp64 reference exactly, bf16 outputs equal it rounded once
# (RNE, as fd_pack_bf16 does), and a second launch gives the same bits.
EXACT_LIMIT = 2.0 ** 22
FILL = 0.25


def exact_terms(name, scalars):
    """The largest sum of |terms| plus |FILL| any output element of ``name`` accumulates on the exact leg, or None for
    a kernel without an exact leg (nonlinear kernels, and those checked against other references)."""
    if name == "fd_conv_igemm":
        C0, C1, N, H, W, Cout, KH, KW, ph, pw, mode = scalars
        return (4 * C0 if mode else KH * KW * (C0 + C1)) + 2                   # + bias + residual
    if name == "fd_conv_igemm_ex":
        C0, C1, N, H, W, Cout, KH, KW, ph, pw, mode, out_mode = scalars
        return KH * KW * (C0 + C1) + 1                                        # + residual
    if name == "fd_conv_wgrad":
        return scalars[2] * scalars[3] * scalars[4] + FILL                    # N H W pixels per tap
    if name == "fd_bias_grad":
        return scalars[0] + FILL
    if name == "fd_final_conv_bwd":
        N, HW, Cin, Cout = scalars
        return max(Cout, N * HW + FILL)                                      # dx: Cout terms; dw, db: N HW
    if name == "fd_final_conv_crop":
        return scalars[3] + 1                                                # Cin + bias
    if name == "fd_linear_bwd_w":
        return scalars[2] + FILL                                             # B
    if name == "fd_linear_bwd_x":
        return scalars[4]                                                    # J
    return {"fd_upsample2x": 1, "fd_upsample2x_bwd": 4, "fd_add_bf16": 2, "fd_prep_weight_dgrad_batch": 1}.get(name)


# 128 input channels -> 64 output channels of a 3x3 pad-1 conv at W >= 128 run on the rolling-strip kernel as two passes
# over 64-channel halves; the first stores its partial sum (+ residual) as bf16, exact for integers up to 2^8 only, so the
# exact leg gives TWO_PASS_CH of the first half's channels non-zero weights at a time (9 TWO_PASS_CH + 1 <= 2^8), one
# launch per window of channels.
TWO_PASS_CH = 28


def two_pass(Cin, Cout, KH, KW, ph, pw, mode, W):
    return mode == 0 and (KH, KW, ph, pw) == (3, 3, 1, 1) and Cin == 128 and Cout == 64 and W >= 128


# ---------------------------------------------------------------------------------------------------------------- wgrad
def _pick_tile64(H, W):
    """fd_conv_wgrad.cu:210-222 (pick_tile64): rows x width of the 64-pixel K-block."""
    best, cost = (1, 64), None
    for wt in (64, 32, 16, 8):
        r = 64 // wt
        c = -(-W // wt) * wt * (-(-H // r) * r)
        if cost is None or c < cost:
            best, cost = (r, wt), c
    return best


def wgrad_ranges(scalars, sms):
    """(L, S) of one fd_conv_wgrad launch: L the longest pixel range one CTA accumulates in TMEM, S the largest number of
    CTA ranges whose partial sums are added into one dW element by fp32 atomics.
    Rolling-strip path (fd_conv_wgrad.cu:262, fd_conv_wgrad_strip.cu:276-281, 310-311): units = (64 x 64 block pair, image,
    128-pixel column block, row), cut into ``grid = min(sms, units)`` contiguous ranges.
    Generic path (fd_conv_wgrad.cu:276-337): 64-pixel tiles split into ``splits`` ranges per job."""
    C0, C1, N, H, W, Cout, KH, KW, ph, pw, mode = scalars
    if mode == 0 and (KH, KW, ph, pw) == (3, 3, 1, 1) and W >= 64 and Cout <= 128:
        rows = N * -(-W // 128) * H
        total = rows * ((C0 + C1) // 64) * (Cout // 64)
        grid = min(sms, total)
        return 128 * -(-total // grid), -(-rows // (total // grid)) + 1
    if mode == 1:
        n, h, w, taps = 1, N * H, W, 4
    elif (KH, KW, ph, pw) == (1, 1, 0, 0):
        n, h, w, taps = 1, 1, N * H * W, 1
    else:
        n, h, w, taps = N, H, W, KH * KW
    R, Wt = _pick_tile64(h, w)
    total = n * -(-w // Wt) * -(-h // R)
    bn = 256 if Cout % 256 == 0 else (128 if Cout % 128 == 0 else 64)
    base = -(-((C0 + C1) // 64) // 2) * (Cout // bn) * taps
    splits = max(1, min(-(-2 * sms // base), total // 4))
    return 64 * -(-total // splits), splits


def wgrad_bound(A, L, S, fill=FILL):
    """|dW - ref| of fd_conv_wgrad with A = sum |x dy| over all pixels: each CTA range's TMEM sum of L_r <= L pixels is off
    by gamma_mma(L_r) of its own sum |x dy|, so all of them together by 2^-22 L A; the S range sums and the fill are then
    added by fp32 atomics, 2^-24 each of at most A + |fill|."""
    return BL.gamma_mma(L) * A + S * 2.0 ** -24 * (A + abs(fill))


# ------------------------------------------------------------------------------------------------- GroupNorm backward
def gn_bwd_depth(N, HW, C, sms):
    """The longest chain of fp32 additions behind one of fd_gn_silu_bwd's per-(sample, channel) sums (fd_unet_bwd.cu:768-781):
    a thread's pixels in the reduce kernel, the ppb rows of its block, then a finalize slice's share of the bx blocks in
    four accumulators and the S slices."""
    ppb = max(256 // (C // 8), 1)
    bx = min(-(-HW // (ppb * 4)), sms * 8 // N + 1)
    S = min(1024 // (C // 8), 32)
    return -(-HW // (bx * ppb)) + ppb + -(-bx // S) + 2 + S, bx, ppb


def gn_bwd_sample(h, da, stats, gamma, beta, eps, depth, sc=None, sh=None):
    """The fp64 reference of fd_gn_silu_bwd for one sample (h, da: (P, C) float64 of the bf16 operands) and the bound of the
    kernel's fp32 evaluation (fd_unet_bwd.cu:39-303), term by term:
      g = da silu'(z), silu' = sg + z sg (1 - sg) with sg = tanh.approx(z / 2) / 2 + 1/2: EPS_TANH |t| / 2 in sg, times
      |d silu' / d sg| <= 1 + |z|, plus |silu''| <= 1/2 times the error of z (gn_affine) and a few roundings;
      S0 = sum g, S1 = sum g h, S2 = sum h: the element errors plus depth 2^-24 of the sums of |terms|;
      Sx = rstd (S1 - mean S0), from the fp32 sums (the cancellation of S1 against mean S0 is in the bound, not hidden);
      Q = -rstd^2 m2, R = -rstd m1 - Q mean from the group sums m1 = sum sc gamma S0 / cnt, m2 = sum sc gamma Sx / cnt;
      dh = a g + Q h + R (a = the folded forward slope).  Returns a dict of (reference, bound) pairs; the per-channel entries
      (S0, Sx, dbias) are what the accumulated outputs add up over the samples."""
    u = 2.0 ** -24
    P, C = h.shape
    cpg = C // 8
    cnt = P * cpg
    mean_g = stats[:, 0] / cnt
    rstd_g = ((stats[:, 1] / cnt - mean_g * mean_g).clamp(min=0) + eps).rsqrt()
    mean, rstd = mean_g.repeat_interleave(cpg), rstd_g.repeat_interleave(cpg)
    s1 = 1 + sc if sc is not None else torch.ones_like(gamma)
    z, dz = BL.gn_affine(h, stats, gamma, beta, eps, sc, sh)
    t = torch.tanh(z / 2)
    sg = 0.5 * t + 0.5
    sp = sg + z * sg * (1 - sg)
    dsp = (1 + z.abs()) * (0.5 * BL.EPS_TANH * t.abs() + 4 * u) + 0.5 * dz
    g = da * sp
    dg = da.abs() * dsp + u * g.abs()
    S0, S1, S2 = g.sum(0), (g * h).sum(0), h.sum(0)
    e0 = dg.sum(0) + depth * u * g.abs().sum(0)
    e1 = (dg * h.abs()).sum(0) + (depth + 1) * u * (g * h).abs().sum(0)
    e2 = depth * u * h.abs().sum(0)
    Sx = rstd * (S1 - mean * S0)
    eSx = rstd * (e1 + mean.abs() * e0 + 3 * u * (S1.abs() + (mean * S0).abs())) + 3 * u * Sx.abs()
    w = (s1 * gamma).abs()
    m1 = (s1 * gamma * S0).view(8, cpg).sum(1) / cnt
    m2 = (s1 * gamma * Sx).view(8, cpg).sum(1) / cnt
    em1 = ((w * e0).view(8, cpg).sum(1) + (cpg + 3) * u * (w * S0.abs()).view(8, cpg).sum(1)) / cnt
    em2 = ((w * eSx).view(8, cpg).sum(1) + (cpg + 3) * u * (w * Sx.abs()).view(8, cpg).sum(1)) / cnt
    Q = -rstd_g * rstd_g * m2
    eQ = rstd_g * rstd_g * em2 + 4 * u * Q.abs()
    R = -rstd_g * m1 - Q * mean_g
    eR = rstd_g * em1 + mean_g.abs() * eQ + 4 * u * ((rstd_g * m1).abs() + (Q * mean_g).abs())
    Qc, Rc, eQc, eRc = (v.repeat_interleave(cpg) for v in (Q, R, eQ, eR))
    a = gamma * rstd * s1
    dh = a * g + Qc * h + Rc
    edh = a.abs() * dg + 4 * u * (a * g).abs() + h.abs() * eQc + eRc + 2 * u * ((Qc * h).abs() + Rc.abs())
    db_ref = dh.sum(0)
    edb = rstd * w * e0 + S2.abs() * eQc + Qc.abs() * e2 + P * eRc + 4 * u * ((rstd * w * S0).abs() + (Qc * S2).abs() + P * Rc.abs())
    return {"dh": (dh, BL.OUT_ROUND * dh.abs() + (1 + BL.OUT_ROUND) * edh), "S0": (S0, e0), "Sx": (Sx, eSx),
            "dbias": (db_ref, edb), "s1": s1}


def accumulated(terms, fill=FILL):
    """fill + sum_n x_n of per-sample fp64 (x_n, bound_n) pairs, as the kernels add them with fp32 atomics: the bound adds
    one rounding of each partial sum, 2^-24 (|fill| + sum |x_n|) per term."""
    ref = fill + sum(x for x, _ in terms)
    mag = abs(fill) + sum(x.abs() for x, _ in terms)
    return ref, sum(b for _, b in terms) + len(terms) * 2.0 ** -24 * mag


# ------------------------------------------------------------------------------------------------- LayerNorm backward
def ln_bwd_ref(x, g, dy, eps):
    """fd_chan_layernorm_bwd on float64 rows x, dy (P, C) of the bf16 operands: (dx without the add, its fp32 error bound,
    xh, the bound of xh).  The error of xh is the forward's (check_chan_layernorm): C 2^-21 rstd (mean|x| + |x - mean|),
    the relative error of rstd C 2^-21; m1, m2 are fp32 means of C terms (C 2^-24 of their sums of |terms|)."""
    u = 2.0 ** -24
    C = x.shape[1]
    d = x - x.mean(1, keepdim=True)
    rstd = ((d * d).mean(1, keepdim=True) + eps).rsqrt()
    xh = d * rstd
    exh = C * 2.0 ** -21 * rstd * (x.abs().mean(1, keepdim=True) + d.abs())
    dd = dy * g
    m1, m2 = dd.mean(1, keepdim=True), (dd * xh).mean(1, keepdim=True)
    em1 = (C + 1) * u * dd.abs().mean(1, keepdim=True)
    em2 = (dd.abs() * exh).mean(1, keepdim=True) + (C + 2) * u * (dd * xh).abs().mean(1, keepdim=True)
    core = dd - m1 - xh * m2
    dx = rstd * core
    edx = rstd * (em1 + xh.abs() * em2 + m2.abs() * exh + 4 * u * (dd.abs() + m1.abs() + (xh * m2).abs())) + \
        C * 2.0 ** -21 * dx.abs()
    return dx, edx, xh, exh


def ln_dg_depth(npix, C, sms):
    """fd_chan_layernorm_bwd's dg sum (fd_unet_bwd.cu:398-402, 806-810): a thread's pixels, the block's threads on its
    channel (shared atomics) and one global atomic per block."""
    lanes = {64: 8, 128: 16, 256: 32, 512: 32}[C]
    grid = min(-(-npix * lanes // 256), sms * 8)
    return -(-npix // (grid * 256 // lanes)) + 256 // lanes + grid + 1


# ------------------------------------------------------------------------------------------------------- the table
# bench.py train leg: batch 8, 368 x 768 crops (no padding), one forward + backward, in launch order
TRAIN = [
    ('fd_prep_weight_dgrad_batch', (73, 32728), 'PP0', 1),
    ('fd_time_embed_save', (8, 64, 256), 'PPPPPPPP0', 1),
    ('fd_time_proj', (8, 256, 8064), 'PPPP0', 1),
    ('fd_pack_input_pad', (8, 2, 3, 368, 768, 0, 0, 368, 768, 0), 'PPP0', 1),
    ('fd_conv_igemm', (64, 0, 8, 368, 768, 64, 7, 1, 3, 0, 0), 'P0PP0P00', 1),
    ('fd_conv_igemm', (64, 0, 8, 368, 768, 64, 3, 3, 1, 1, 0), 'P0PP0PP0', 7),
    ('fd_gn_silu', (8064, 8, 282624, 64, 1e-05), 'PPPPP0P0', 5),
    ('fd_gn_silu', (0, 8, 282624, 64, 1e-05), 'PPPP0PP0', 2),
    ('fd_chan_layernorm', (2260992, 64, 1e-05), 'PP0P0', 2),
    ('fd_conv_igemm', (64, 0, 8, 368, 768, 384, 1, 1, 0, 0, 0), 'P0P00P00', 2),
    ('fd_linattn_save', (8, 282624), 'PPPP0', 2),
    ('fd_conv_igemm', (128, 0, 8, 368, 768, 64, 1, 1, 0, 0, 0), 'P0PP0P00', 2),
    ('fd_chan_layernorm', (2260992, 64, 1e-05), 'PPPP0', 2),
    ('fd_conv_igemm', (64, 0, 8, 184, 384, 64, 1, 1, 0, 0, 1), 'P0PP0P00', 1),
    ('fd_conv_igemm', (64, 0, 8, 184, 384, 64, 3, 3, 1, 1, 0), 'P0PP0PP0', 4),
    ('fd_gn_silu', (8064, 8, 70656, 64, 1e-05), 'PPPPP0P0', 2),
    ('fd_gn_silu', (0, 8, 70656, 64, 1e-05), 'PPPP0PP0', 2),
    ('fd_chan_layernorm', (565248, 64, 1e-05), 'PP0P0', 1),
    ('fd_conv_igemm', (64, 0, 8, 184, 384, 384, 1, 1, 0, 0, 0), 'P0P00P00', 1),
    ('fd_linattn_save', (8, 70656), 'PPPP0', 2),
    ('fd_conv_igemm', (128, 0, 8, 184, 384, 64, 1, 1, 0, 0, 0), 'P0PP0P00', 1),
    ('fd_chan_layernorm', (565248, 64, 1e-05), 'PPPP0', 1),
    ('fd_conv_igemm', (64, 0, 8, 92, 192, 128, 1, 1, 0, 0, 1), 'P0PP0P00', 1),
    ('fd_conv_igemm', (128, 0, 8, 92, 192, 128, 3, 3, 1, 1, 0), 'P0PP0PP0', 4),
    ('fd_gn_silu', (8064, 8, 17664, 128, 1e-05), 'PPPPP0P0', 2),
    ('fd_gn_silu', (0, 8, 17664, 128, 1e-05), 'PPPP0PP0', 2),
    ('fd_chan_layernorm', (141312, 128, 1e-05), 'PP0P0', 1),
    ('fd_conv_igemm', (128, 0, 8, 92, 192, 384, 1, 1, 0, 0, 0), 'P0P00P00', 1),
    ('fd_linattn_save', (8, 17664), 'PPPP0', 2),
    ('fd_conv_igemm', (128, 0, 8, 92, 192, 128, 1, 1, 0, 0, 0), 'P0PP0P00', 1),
    ('fd_chan_layernorm', (141312, 128, 1e-05), 'PPPP0', 1),
    ('fd_conv_igemm', (128, 0, 8, 46, 96, 256, 1, 1, 0, 0, 1), 'P0PP0P00', 1),
    ('fd_conv_igemm', (256, 0, 8, 46, 96, 256, 3, 3, 1, 1, 0), 'P0PP0PP0', 4),
    ('fd_gn_silu', (8064, 8, 4416, 256, 1e-05), 'PPPPP0P0', 2),
    ('fd_gn_silu', (0, 8, 4416, 256, 1e-05), 'PPPP0PP0', 2),
    ('fd_chan_layernorm', (35328, 256, 1e-05), 'PP0P0', 1),
    ('fd_conv_igemm', (256, 0, 8, 46, 96, 384, 1, 1, 0, 0, 0), 'P0P00P00', 1),
    ('fd_linattn_save', (8, 4416), 'PPPP0', 2),
    ('fd_conv_igemm', (128, 0, 8, 46, 96, 256, 1, 1, 0, 0, 0), 'P0PP0P00', 1),
    ('fd_chan_layernorm', (35328, 256, 1e-05), 'PPPP0', 1),
    ('fd_conv_igemm', (256, 0, 8, 46, 96, 512, 3, 3, 1, 1, 0), 'P0PP0P00', 1),
    ('fd_conv_igemm', (512, 0, 8, 46, 96, 512, 3, 3, 1, 1, 0), 'P0PP0PP0', 6),
    ('fd_gn_silu', (8064, 8, 4416, 512, 1e-05), 'PPPPP0P0', 4),
    ('fd_gn_silu', (0, 8, 4416, 512, 1e-05), 'PPPP0PP0', 2),
    ('fd_chan_layernorm', (35328, 512, 1e-05), 'PP0P0', 2),
    ('fd_conv_igemm', (512, 0, 8, 46, 96, 384, 1, 1, 0, 0, 0), 'P0P00P00', 2),
    ('fd_attention_lse', (8, 4416), 'PPP0', 1),
    ('fd_conv_igemm', (128, 0, 8, 46, 96, 512, 1, 1, 0, 0, 0), 'P0PPPP00', 1),
    ('fd_conv_igemm', (512, 256, 8, 46, 96, 512, 3, 3, 1, 1, 0), 'PPPP0PP0', 2),
    ('fd_conv_igemm_rt', (512, 256, 1e-05, 8, 46, 96, 512, 1, 1, 0, 0), 'PPPPPPPPP0', 2),
    ('fd_conv_igemm', (128, 0, 8, 46, 96, 512, 1, 1, 0, 0, 0), 'P0PP0P00', 1),
    ('fd_chan_layernorm', (35328, 512, 1e-05), 'PPPP0', 1),
    ('fd_upsample2x', (8, 46, 96, 512), 'PP0', 1),
    ('fd_conv_igemm', (512, 0, 8, 92, 192, 256, 3, 3, 1, 1, 0), 'P0PP0P00', 1),
    ('fd_conv_igemm', (256, 128, 8, 92, 192, 256, 3, 3, 1, 1, 0), 'PPPP0PP0', 2),
    ('fd_gn_silu', (8064, 8, 17664, 256, 1e-05), 'PPPPP0P0', 2),
    ('fd_conv_igemm', (256, 0, 8, 92, 192, 256, 3, 3, 1, 1, 0), 'P0PP0PP0', 2),
    ('fd_conv_igemm_rt', (256, 128, 1e-05, 8, 92, 192, 256, 1, 1, 0, 0), 'PPPPPPPPP0', 2),
    ('fd_chan_layernorm', (141312, 256, 1e-05), 'PP0P0', 1),
    ('fd_conv_igemm', (256, 0, 8, 92, 192, 384, 1, 1, 0, 0, 0), 'P0P00P00', 1),
    ('fd_conv_igemm', (128, 0, 8, 92, 192, 256, 1, 1, 0, 0, 0), 'P0PP0P00', 1),
    ('fd_chan_layernorm', (141312, 256, 1e-05), 'PPPP0', 1),
    ('fd_upsample2x', (8, 92, 192, 256), 'PP0', 1),
    ('fd_conv_igemm', (256, 0, 8, 184, 384, 128, 3, 3, 1, 1, 0), 'P0PP0P00', 1),
    ('fd_conv_igemm', (128, 64, 8, 184, 384, 128, 3, 3, 1, 1, 0), 'PPPP0PP0', 2),
    ('fd_gn_silu', (8064, 8, 70656, 128, 1e-05), 'PPPPP0P0', 2),
    ('fd_conv_igemm', (128, 0, 8, 184, 384, 128, 3, 3, 1, 1, 0), 'P0PP0PP0', 2),
    ('fd_conv_igemm_rt', (128, 64, 1e-05, 8, 184, 384, 128, 1, 1, 0, 0), 'PPPPPPPPP0', 2),
    ('fd_chan_layernorm', (565248, 128, 1e-05), 'PP0P0', 1),
    ('fd_conv_igemm', (128, 0, 8, 184, 384, 384, 1, 1, 0, 0, 0), 'P0P00P00', 1),
    ('fd_conv_igemm', (128, 0, 8, 184, 384, 128, 1, 1, 0, 0, 0), 'P0PP0P00', 1),
    ('fd_chan_layernorm', (565248, 128, 1e-05), 'PPPP0', 1),
    ('fd_upsample2x', (8, 184, 384, 128), 'PP0', 1),
    ('fd_conv_igemm', (128, 0, 8, 368, 768, 64, 3, 3, 1, 1, 0), 'P0PP0P00', 1),
    ('fd_conv_igemm', (64, 64, 8, 368, 768, 64, 3, 3, 1, 1, 0), 'PPPP0PP0', 3),
    ('fd_conv_igemm_rt', (64, 64, 1e-05, 8, 368, 768, 64, 1, 1, 0, 0), 'PPPPPPPPP0', 3),
    ('fd_conv_igemm', (64, 0, 8, 368, 768, 64, 3, 3, 1, 1, 0), 'P0PP0P00', 1),
    ('fd_final_conv_crop', (8, 368, 768, 64, 2, 0, 0, 368, 768), 'PPPP0', 1),
    ('fd_final_conv_bwd', (8, 282624, 64, 2), 'PPPPPP0', 1),
    ('fd_gn_silu_bwd', (0, 8, 282624, 64, 1e-05), 'PPPPP0PPP0PP0', 5),
    ('fd_bias_grad', (2260992, 64), 'PP0', 8),
    ('fd_conv_wgrad', (64, 64, 8, 368, 768, 64, 1, 1, 0, 0, 0), 'PPPP0', 3),
    ('fd_conv_igemm_ex', (64, 0, 8, 368, 768, 64, 1, 1, 0, 0, 0, 0), 'P0P00P00', 6),
    ('fd_conv_wgrad', (64, 0, 8, 368, 768, 64, 3, 3, 1, 1, 0), 'P0PP0', 8),
    ('fd_conv_igemm_ex', (64, 0, 8, 368, 768, 64, 3, 3, 1, 1, 0, 0), 'P0P00P00', 6),
    ('fd_gn_silu_bwd', (8064, 8, 282624, 64, 1e-05), 'PPPPPPPPPPPP0', 5),
    ('fd_conv_wgrad', (64, 64, 8, 368, 768, 64, 3, 3, 1, 1, 0), 'PPPP0', 3),
    ('fd_conv_igemm_ex', (64, 0, 8, 368, 768, 64, 3, 3, 1, 1, 0, 0), 'P0P0PP00', 8),
    ('fd_linear_bwd_w', (8064, 256, 8, 128, 256, 1), 'PPPP0', 7),
    ('fd_prep_weight_bwd_batch', (3, 192, 1e-05), 'PP0', 1),
    ('fd_chan_layernorm_bwd', (2260992, 64, 1e-05), 'PPP0PP0', 2),
    ('fd_conv_wgrad', (128, 0, 8, 368, 768, 64, 1, 1, 0, 0, 0), 'P0PP0', 2),
    ('fd_conv_igemm_ex', (64, 0, 8, 368, 768, 128, 1, 1, 0, 0, 0, 0), 'P0P00P00', 2),
    ('fd_linattn_bwd', (8, 282624), 'PPPPP0', 2),
    ('fd_conv_wgrad', (64, 0, 8, 368, 768, 384, 1, 1, 0, 0, 0), 'P0PP0', 2),
    ('fd_conv_igemm_ex', (384, 0, 8, 368, 768, 64, 1, 1, 0, 0, 0, 0), 'P0P00P00', 2),
    ('fd_chan_layernorm_bwd', (2260992, 64, 1e-05), 'PPPPPP0', 2),
    ('fd_conv_wgrad', (128, 0, 8, 368, 768, 64, 3, 3, 1, 1, 0), 'P0PP0', 1),
    ('fd_conv_igemm_ex', (64, 0, 8, 368, 768, 128, 3, 3, 1, 1, 0, 0), 'P0P00P00', 1),
    ('fd_upsample2x_bwd', (8, 184, 384, 128), 'PP0', 1),
    ('fd_chan_layernorm_bwd', (565248, 128, 1e-05), 'PPP0PP0', 1),
    ('fd_bias_grad', (565248, 128), 'PP0', 4),
    ('fd_conv_wgrad', (128, 0, 8, 184, 384, 128, 1, 1, 0, 0, 0), 'P0PP0', 1),
    ('fd_conv_igemm_ex', (128, 0, 8, 184, 384, 128, 1, 1, 0, 0, 0, 0), 'P0P00P00', 3),
    ('fd_linattn_bwd', (8, 70656), 'PPPPP0', 2),
    ('fd_conv_wgrad', (128, 0, 8, 184, 384, 384, 1, 1, 0, 0, 0), 'P0PP0', 1),
    ('fd_conv_igemm_ex', (384, 0, 8, 184, 384, 128, 1, 1, 0, 0, 0, 0), 'P0P00P00', 1),
    ('fd_chan_layernorm_bwd', (565248, 128, 1e-05), 'PPPPPP0', 1),
    ('fd_gn_silu_bwd', (0, 8, 70656, 128, 1e-05), 'PPPPP0PPP0PP0', 2),
    ('fd_conv_wgrad', (128, 64, 8, 184, 384, 128, 1, 1, 0, 0, 0), 'PPPP0', 2),
    ('fd_conv_igemm_ex', (128, 0, 8, 184, 384, 64, 1, 1, 0, 0, 0, 0), 'P0P00P00', 2),
    ('fd_conv_wgrad', (128, 0, 8, 184, 384, 128, 3, 3, 1, 1, 0), 'P0PP0', 2),
    ('fd_conv_igemm_ex', (128, 0, 8, 184, 384, 128, 3, 3, 1, 1, 0, 0), 'P0P00P00', 2),
    ('fd_gn_silu_bwd', (8064, 8, 70656, 128, 1e-05), 'PPPPPPPPPPPP0', 2),
    ('fd_conv_wgrad', (128, 64, 8, 184, 384, 128, 3, 3, 1, 1, 0), 'PPPP0', 2),
    ('fd_conv_igemm_ex', (128, 0, 8, 184, 384, 128, 3, 3, 1, 1, 0, 0), 'P0P0PP00', 2),
    ('fd_conv_igemm_ex', (128, 0, 8, 184, 384, 64, 3, 3, 1, 1, 0, 0), 'P0P0PP00', 2),
    ('fd_linear_bwd_w', (8064, 256, 8, 256, 256, 1), 'PPPP0', 4),
    ('fd_prep_weight_bwd_batch', (18, 2240, 1e-05), 'PP0', 1),
    ('fd_conv_wgrad', (256, 0, 8, 184, 384, 128, 3, 3, 1, 1, 0), 'P0PP0', 1),
    ('fd_conv_igemm_ex', (128, 0, 8, 184, 384, 256, 3, 3, 1, 1, 0, 0), 'P0P00P00', 1),
    ('fd_upsample2x_bwd', (8, 92, 192, 256), 'PP0', 1),
    ('fd_chan_layernorm_bwd', (141312, 256, 1e-05), 'PPP0PP0', 1),
    ('fd_bias_grad', (141312, 256), 'PP0', 4),
    ('fd_conv_wgrad', (128, 0, 8, 92, 192, 256, 1, 1, 0, 0, 0), 'P0PP0', 1),
    ('fd_conv_igemm_ex', (256, 0, 8, 92, 192, 128, 1, 1, 0, 0, 0, 0), 'P0P00P00', 3),
    ('fd_linattn_bwd', (8, 17664), 'PPPPP0', 2),
    ('fd_conv_wgrad', (256, 0, 8, 92, 192, 384, 1, 1, 0, 0, 0), 'P0PP0', 1),
    ('fd_conv_igemm_ex', (384, 0, 8, 92, 192, 256, 1, 1, 0, 0, 0, 0), 'P0P00P00', 1),
    ('fd_chan_layernorm_bwd', (141312, 256, 1e-05), 'PPPPPP0', 1),
    ('fd_gn_silu_bwd', (0, 8, 17664, 256, 1e-05), 'PPPPP0PPP0PP0', 2),
    ('fd_conv_wgrad', (256, 128, 8, 92, 192, 256, 1, 1, 0, 0, 0), 'PPPP0', 2),
    ('fd_conv_igemm_ex', (256, 0, 8, 92, 192, 256, 1, 1, 0, 0, 0, 0), 'P0P00P00', 2),
    ('fd_conv_wgrad', (256, 0, 8, 92, 192, 256, 3, 3, 1, 1, 0), 'P0PP0', 2),
    ('fd_conv_igemm_ex', (256, 0, 8, 92, 192, 256, 3, 3, 1, 1, 0, 0), 'P0P00P00', 2),
    ('fd_gn_silu_bwd', (8064, 8, 17664, 256, 1e-05), 'PPPPPPPPPPPP0', 2),
    ('fd_conv_wgrad', (256, 128, 8, 92, 192, 256, 3, 3, 1, 1, 0), 'PPPP0', 2),
    ('fd_conv_igemm_ex', (256, 0, 8, 92, 192, 256, 3, 3, 1, 1, 0, 0), 'P0P0PP00', 2),
    ('fd_conv_igemm_ex', (256, 0, 8, 92, 192, 128, 3, 3, 1, 1, 0, 0), 'P0P0PP00', 2),
    ('fd_linear_bwd_w', (8064, 256, 8, 512, 256, 1), 'PPPP0', 4),
    ('fd_prep_weight_bwd_batch', (9, 2304, 1e-05), 'PP0', 1),
    ('fd_conv_wgrad', (512, 0, 8, 92, 192, 256, 3, 3, 1, 1, 0), 'P0PP0', 1),
    ('fd_conv_igemm_ex', (256, 0, 8, 92, 192, 512, 3, 3, 1, 1, 0, 0), 'P0P00P00', 1),
    ('fd_upsample2x_bwd', (8, 46, 96, 512), 'PP0', 1),
    ('fd_chan_layernorm_bwd', (35328, 512, 1e-05), 'PPP0PP0', 1),
    ('fd_bias_grad', (35328, 512), 'PP0', 5),
    ('fd_conv_wgrad', (128, 0, 8, 46, 96, 512, 1, 1, 0, 0, 0), 'P0PP0', 2),
    ('fd_conv_igemm_ex', (512, 0, 8, 46, 96, 128, 1, 1, 0, 0, 0, 0), 'P0P00P00', 2),
    ('fd_linattn_bwd', (8, 4416), 'PPPPP0', 2),
    ('fd_conv_wgrad', (512, 0, 8, 46, 96, 384, 1, 1, 0, 0, 0), 'P0PP0', 2),
    ('fd_conv_igemm_ex', (384, 0, 8, 46, 96, 512, 1, 1, 0, 0, 0, 0), 'P0P00P00', 2),
    ('fd_chan_layernorm_bwd', (35328, 512, 1e-05), 'PPPPPP0', 2),
    ('fd_gn_silu_bwd', (0, 8, 4416, 512, 1e-05), 'PPPPP0PPP0PP0', 4),
    ('fd_conv_wgrad', (512, 256, 8, 46, 96, 512, 1, 1, 0, 0, 0), 'PPPP0', 2),
    ('fd_conv_igemm_ex', (512, 0, 8, 46, 96, 512, 1, 1, 0, 0, 0, 0), 'P0P00P00', 2),
    ('fd_conv_igemm_ex', (512, 0, 8, 46, 96, 256, 1, 1, 0, 0, 0, 0), 'P0P00P00', 2),
    ('fd_conv_wgrad', (512, 0, 8, 46, 96, 512, 3, 3, 1, 1, 0), 'P0PP0', 6),
    ('fd_conv_igemm_ex', (512, 0, 8, 46, 96, 512, 3, 3, 1, 1, 0, 0), 'P0P00P00', 4),
    ('fd_gn_silu_bwd', (8064, 8, 4416, 512, 1e-05), 'PPPPPPPPPPPP0', 4),
    ('fd_conv_wgrad', (512, 256, 8, 46, 96, 512, 3, 3, 1, 1, 0), 'PPPP0', 2),
    ('fd_conv_igemm_ex', (512, 0, 8, 46, 96, 512, 3, 3, 1, 1, 0, 0), 'P0P0PP00', 4),
    ('fd_conv_igemm_ex', (512, 0, 8, 46, 96, 256, 3, 3, 1, 1, 0, 0), 'P0P0PP00', 3),
    ('fd_linear_bwd_w', (8064, 256, 8, 1024, 256, 1), 'PPPP0', 4),
    ('fd_prep_weight_bwd_batch', (9, 4224, 1e-05), 'PP0', 1),
    ('fd_attention_bwd', (8, 4416), 'PPPPPP0', 1),
    ('fd_prep_weight_bwd_batch', (6, 2944, 1e-05), 'PP0', 1),
    ('fd_conv_wgrad', (256, 0, 8, 46, 96, 512, 3, 3, 1, 1, 0), 'P0PP0', 1),
    ('fd_chan_layernorm_bwd', (35328, 256, 1e-05), 'PPP0PP0', 1),
    ('fd_bias_grad', (35328, 256), 'PP0', 2),
    ('fd_conv_wgrad', (128, 0, 8, 46, 96, 256, 1, 1, 0, 0, 0), 'P0PP0', 1),
    ('fd_conv_igemm_ex', (256, 0, 8, 46, 96, 128, 1, 1, 0, 0, 0, 0), 'P0P00P00', 1),
    ('fd_conv_wgrad', (256, 0, 8, 46, 96, 384, 1, 1, 0, 0, 0), 'P0PP0', 1),
    ('fd_conv_igemm_ex', (384, 0, 8, 46, 96, 256, 1, 1, 0, 0, 0, 0), 'P0P00P00', 1),
    ('fd_chan_layernorm_bwd', (35328, 256, 1e-05), 'PPPPPP0', 1),
    ('fd_add_bf16', (9043968,), 'PPP0', 1),
    ('fd_gn_silu_bwd', (0, 8, 4416, 256, 1e-05), 'PPPPP0PPP0PP0', 2),
    ('fd_conv_wgrad', (256, 0, 8, 46, 96, 256, 3, 3, 1, 1, 0), 'P0PP0', 4),
    ('fd_conv_igemm_ex', (256, 0, 8, 46, 96, 256, 3, 3, 1, 1, 0, 0), 'P0P00P00', 2),
    ('fd_gn_silu_bwd', (8064, 8, 4416, 256, 1e-05), 'PPPPPPPPPPPP0', 2),
    ('fd_conv_igemm_ex', (256, 0, 8, 46, 96, 256, 3, 3, 1, 1, 0, 0), 'P0P0PP00', 2),
    ('fd_prep_weight_bwd_batch', (7, 2176, 1e-05), 'PP0', 1),
    ('fd_conv_wgrad', (128, 0, 8, 46, 96, 256, 1, 1, 0, 0, 1), 'P0PP0', 1),
    ('fd_conv_igemm_ex', (256, 0, 8, 46, 96, 512, 1, 1, 0, 0, 0, 1), 'P0P00P00', 1),
    ('fd_add_bf16', (18087936,), 'PPP0', 2),
    ('fd_chan_layernorm_bwd', (141312, 128, 1e-05), 'PPP0PP0', 1),
    ('fd_bias_grad', (141312, 128), 'PP0', 2),
    ('fd_conv_wgrad', (128, 0, 8, 92, 192, 128, 1, 1, 0, 0, 0), 'P0PP0', 1),
    ('fd_conv_igemm_ex', (128, 0, 8, 92, 192, 128, 1, 1, 0, 0, 0, 0), 'P0P00P00', 1),
    ('fd_conv_wgrad', (128, 0, 8, 92, 192, 384, 1, 1, 0, 0, 0), 'P0PP0', 1),
    ('fd_conv_igemm_ex', (384, 0, 8, 92, 192, 128, 1, 1, 0, 0, 0, 0), 'P0P00P00', 1),
    ('fd_chan_layernorm_bwd', (141312, 128, 1e-05), 'PPPPPP0', 1),
    ('fd_gn_silu_bwd', (0, 8, 17664, 128, 1e-05), 'PPPPP0PPP0PP0', 2),
    ('fd_conv_wgrad', (128, 0, 8, 92, 192, 128, 3, 3, 1, 1, 0), 'P0PP0', 4),
    ('fd_conv_igemm_ex', (128, 0, 8, 92, 192, 128, 3, 3, 1, 1, 0, 0), 'P0P00P00', 2),
    ('fd_gn_silu_bwd', (8064, 8, 17664, 128, 1e-05), 'PPPPPPPPPPPP0', 2),
    ('fd_conv_igemm_ex', (128, 0, 8, 92, 192, 128, 3, 3, 1, 1, 0, 0), 'P0P0PP00', 2),
    ('fd_prep_weight_bwd_batch', (7, 1280, 1e-05), 'PP0', 1),
    ('fd_conv_wgrad', (64, 0, 8, 92, 192, 128, 1, 1, 0, 0, 1), 'P0PP0', 1),
    ('fd_conv_igemm_ex', (128, 0, 8, 92, 192, 256, 1, 1, 0, 0, 0, 1), 'P0P00P00', 1),
    ('fd_add_bf16', (36175872,), 'PPP0', 2),
    ('fd_chan_layernorm_bwd', (565248, 64, 1e-05), 'PPP0PP0', 1),
    ('fd_bias_grad', (565248, 64), 'PP0', 2),
    ('fd_conv_wgrad', (128, 0, 8, 184, 384, 64, 1, 1, 0, 0, 0), 'P0PP0', 1),
    ('fd_conv_igemm_ex', (64, 0, 8, 184, 384, 128, 1, 1, 0, 0, 0, 0), 'P0P00P00', 1),
    ('fd_conv_wgrad', (64, 0, 8, 184, 384, 384, 1, 1, 0, 0, 0), 'P0PP0', 1),
    ('fd_conv_igemm_ex', (384, 0, 8, 184, 384, 64, 1, 1, 0, 0, 0, 0), 'P0P00P00', 1),
    ('fd_chan_layernorm_bwd', (565248, 64, 1e-05), 'PPPPPP0', 1),
    ('fd_gn_silu_bwd', (0, 8, 70656, 64, 1e-05), 'PPPPP0PPP0PP0', 2),
    ('fd_conv_wgrad', (64, 0, 8, 184, 384, 64, 3, 3, 1, 1, 0), 'P0PP0', 4),
    ('fd_conv_igemm_ex', (64, 0, 8, 184, 384, 64, 3, 3, 1, 1, 0, 0), 'P0P00P00', 2),
    ('fd_gn_silu_bwd', (8064, 8, 70656, 64, 1e-05), 'PPPPPPPPPPPP0', 2),
    ('fd_conv_igemm_ex', (64, 0, 8, 184, 384, 64, 3, 3, 1, 1, 0, 0), 'P0P0PP00', 2),
    ('fd_conv_wgrad', (64, 0, 8, 184, 384, 64, 1, 1, 0, 0, 1), 'P0PP0', 1),
    ('fd_conv_igemm_ex', (64, 0, 8, 184, 384, 256, 1, 1, 0, 0, 0, 1), 'P0P00P00', 1),
    ('fd_add_bf16', (144703488,), 'PPP0', 3),
    ('fd_conv_wgrad', (64, 0, 8, 368, 768, 64, 7, 1, 3, 0, 0), 'P0PP0', 1),
    ('fd_linear_bwd_x', (8064, 256, 256, 8, 8064, 256, 1), 'PPPP0', 1),
    ('fd_linear_bwd_w', (256, 256, 8, 256, 256, 2), 'PPPP0', 1),
    ('fd_linear_bwd_x', (256, 256, 256, 8, 256, 256, 2), 'PPPP0', 1),
    ('fd_linear_bwd_w', (256, 64, 8, 256, 64, 0), 'PPPP0', 1),
    ('fd_prep_weight_bwd_batch', (15, 1664, 1e-05), 'PP0', 1),
]
