"""CPU: the launch table of the benchmark's training step (tests/train_launches.py) matches what the UNet launches, every
kernel in it has a GPU checker, every exact-leg entry stays inside the exact-fp32 range, and the bounds of the backward
checkers pass fp32 emulations of the kernels' arithmetic while rejecting small mutations of it."""
import torch
import torch.nn.functional as F

import bench_launches as BL
import test_gpu_train_launches as GPU
import train_launches as TL
from test_bench_launch_table import _samples, bf16

D = torch.float64


def test_train_table_is_exact():
    """bench.py train leg at 8 x 368 x 768: every distinct launch of the forward and backward, with its count, in order."""
    assert BL.as_table(TL.record_train(8, 368, 768)) == TL.TRAIN
    assert len(TL.TRAIN) == 221 and sum(e[3] for e in TL.TRAIN) == 436


def test_every_kernel_has_a_checker():
    names = {e[0] for e in TL.TRAIN}
    assert len(names) == 25 and names <= set(GPU.CHECKERS), names - set(GPU.CHECKERS)


def test_exact_leg_partial_sums_stay_below_2_22():
    """The widest reduction, wgrad over N H W = 2,260,992 pixels, included."""
    linear = {"fd_conv_igemm", "fd_conv_igemm_ex", "fd_conv_wgrad", "fd_bias_grad", "fd_upsample2x", "fd_upsample2x_bwd",
              "fd_add_bf16", "fd_final_conv_crop", "fd_final_conv_bwd", "fd_linear_bwd_w", "fd_linear_bwd_x",
              "fd_prep_weight_dgrad_batch"}
    for name, scalars, _, _ in TL.TRAIN:
        t = TL.exact_terms(name, scalars)
        assert (t is not None) == (name in linear), name
        if t is not None:
            assert t < TL.EXACT_LIMIT, (name, scalars, t)
    assert max(TL.exact_terms(*e[:2]) for e in TL.TRAIN if e[0] == "fd_conv_wgrad") == 2260992 + TL.FILL
    assert 9 * TL.TWO_PASS_CH + 2 <= 2 ** 8              # the two-pass bf16 partial sum (+ bias + residual), exact leg


# ------------------------------------------------------------------------------------------------------------- wgrad
def _wgrad(x, dy, pixels=None):
    """dW (Cout, Cin, 3, 3) of a 3x3 pad-1 conv over the pixels selected by ``pixels`` (a bool mask of dy's), fp32
    accumulation of exact bf16 products (the emulated kernel) when the inputs are fp32."""
    if pixels is not None:
        dy = dy * pixels
    return torch.nn.grad.conv2d_weight(x, (dy.shape[1], x.shape[1], 3, 3), dy, padding=1)


def test_wgrad_bound_accepts_fp32_and_rejects_mutations():
    g = torch.Generator().manual_seed(3)
    N, C, H, W = 2, 64, 4, 256                      # two 128-pixel column blocks: the strip path's geometry
    x = _samples(N, C, H, W, g)
    dy = bf16(torch.randn(N, C, H, W, generator=g, dtype=D))
    ref = _wgrad(x, dy)
    A = _wgrad(x.abs(), dy.abs())
    Lr, S = TL.wgrad_ranges((C, 0, N, H, W, C, 3, 3, 1, 1, 0), 148)
    bound = TL.wgrad_bound(A, Lr, S, fill=0.0)

    def ratio(got):
        return BL.ratio((got - ref).abs(), bound)

    assert ratio(_wgrad(x.float(), dy.float()).double()) <= 1
    rng = torch.zeros(N, 1, H, W, dtype=torch.bool)
    rng[1, :, 2] = True                             # one CTA range: one 128-pixel row of one column block
    rng[1, :, 2, 128:] = False
    assert ratio(_wgrad(x, dy, ~rng)) > 1
    last = torch.ones(N, 1, H, W, dtype=torch.bool)
    last[..., 128:] = False                         # the last 128-pixel column block
    assert ratio(_wgrad(x, dy, last)) > 1
    assert ratio(ref[:, :, :, [1, 0, 2]]) > 1       # taps kx = 0 / 1 swapped


# ------------------------------------------------------------------------------------------------ GroupNorm backward
def _gn_case(g, N=3, HW=600, C=64):
    x = _samples(N, C, HW, 1, g).reshape(N, C, HW).transpose(1, 2).contiguous()
    x[..., :8] += 12 * (0.5 + 0.25 * torch.arange(N, dtype=D)).view(N, 1, 1)           # |mean| / std >= 10
    x = bf16(x)
    da = bf16(torch.randn(N, HW, C, generator=g, dtype=D) + torch.where(torch.arange(C) < C // 2, 0.5, 0.0))
    r = x.reshape(N, HW, 8, C // 8)
    stats = torch.stack((r.sum((1, 3)), (r * r).sum((1, 3))), -1)
    gamma = 1 + 0.3 * torch.randn(C, generator=g, dtype=D)
    beta = 0.2 * torch.randn(C, generator=g, dtype=D)
    return x, da, stats, gamma, beta


def _gn_bwd_emulated(x, da, stats, gamma, beta, eps=1e-5, blocks=4, drop_block=None, swap_stats=False, swap_qr=False,
                     assign=False):
    """fd_gn_silu_bwd in fp32 (fd_unet_bwd.cu:39-303): folded slope / offset, tanh-form silu', the three sums per
    (sample, channel) over ``blocks`` pixel blocks, the finalize and apply formulas.  Returns dh, dgamma, dbeta, dbias
    (the last three accumulated onto FILL) with optional mutations."""
    N, HW, C = x.shape
    cpg = C // 8
    cnt = HW * cpg
    st = stats[[1, 0] + list(range(2, N))] if swap_stats else stats
    f = torch.float32
    dh = torch.empty(N, HW, C, dtype=f)
    dgamma, dbeta, dbias = (torch.full((C,), TL.FILL, dtype=f) for _ in range(3))
    if assign:
        dgamma.zero_()
    for n in range(N):
        mean_d = st[n, :, 0] / cnt
        rstd = ((st[n, :, 1] / cnt - mean_d ** 2).clamp(min=0) + eps).rsqrt().to(f).repeat_interleave(cpg)
        mean = mean_d.to(f).repeat_interleave(cpg)
        a = gamma.to(f) * rstd
        b = beta.to(f) - mean * a
        h, d = x[n].to(f), da[n].to(f)
        z = a * h + b
        sg = 0.5 * torch.tanh(0.5 * z) + 0.5
        gz = d * (z * sg * (1 - sg) + sg)
        parts = [slice(i * HW // blocks, (i + 1) * HW // blocks) for i in range(blocks) if i != drop_block]
        S0 = sum(gz[p].sum(0) for p in parts)
        S1 = sum((gz[p] * h[p]).sum(0) for p in parts)
        S2 = sum(h[p].sum(0) for p in parts)
        Sx = rstd * (S1 - mean * S0)
        if assign:
            dgamma = Sx.clone()
        else:
            dgamma += Sx
        dbeta += S0
        m1 = (gamma.to(f) * S0).view(8, cpg).sum(1) / cnt
        m2 = (gamma.to(f) * Sx).view(8, cpg).sum(1) / cnt
        rg = rstd.view(8, cpg)[:, 0]
        Q = -rg * rg * m2
        R = -rg * m1 - Q * mean.view(8, cpg)[:, 0]
        if swap_qr:
            Q, R = Q[[1, 0] + list(range(2, 8))], R[[1, 0] + list(range(2, 8))]
        Qc, Rc = Q.repeat_interleave(cpg), R.repeat_interleave(cpg)
        dh[n] = bf16((a * gz + Qc * h + Rc).double()).to(f)
        dbias += rstd * gamma.to(f) * S0 + Qc * S2 + Rc * HW
    return dh.double(), dgamma.double(), dbeta.double(), dbias.double()


def _gn_bwd_worst(x, da, stats, gamma, beta, got):
    N, HW, C = x.shape
    depth = HW // 4 + 8
    dh, dgamma, dbeta, dbias = got
    worst, tg, tb, tbias = 0.0, [], [], []
    for n in range(N):
        r = TL.gn_bwd_sample(x[n], da[n], stats[n], gamma, beta, 1e-5, depth)
        worst = max(worst, BL.ratio((dh[n] - r["dh"][0]).abs(), r["dh"][1]))
        tg.append(r["Sx"])
        tb.append(r["S0"])
        tbias.append(r["dbias"])
    for got_v, terms in ((dgamma, tg), (dbeta, tb), (dbias, tbias)):
        ref, bound = TL.accumulated(terms)
        worst = max(worst, BL.ratio((got_v - ref).abs(), bound))
    return worst


def test_gn_bwd_bound_accepts_fp32_and_rejects_mutations():
    g = torch.Generator().manual_seed(4)
    case = _gn_case(g)
    assert _gn_bwd_worst(*case, _gn_bwd_emulated(*case)) <= 1
    for mutation in (dict(drop_block=2), dict(swap_stats=True), dict(swap_qr=True), dict(assign=True)):
        assert _gn_bwd_worst(*case, _gn_bwd_emulated(*case, **mutation)) > 1, mutation


# ------------------------------------------------------------------------------------------------ LayerNorm backward
def test_ln_bwd_bound_rejects_an_ignored_add():
    g = torch.Generator().manual_seed(5)
    P, C = 200, 64
    x = bf16(torch.randn(P, C, generator=g, dtype=D) * 2 + 1)
    dy = bf16(torch.randn(P, C, generator=g, dtype=D))
    add = bf16(torch.randn(P, C, generator=g, dtype=D))
    gain = 1 + 0.3 * torch.randn(C, generator=g, dtype=D)
    xf, df, gf = x.float(), dy.float(), gain.float()
    d = xf - xf.mean(1, keepdim=True)
    xh = d * torch.rsqrt((d * d).mean(1, keepdim=True) + 1e-5)
    dd = df * gf
    core = torch.rsqrt((d * d).mean(1, keepdim=True) + 1e-5) * (dd - dd.mean(1, keepdim=True) - xh * (dd * xh).mean(1, keepdim=True))
    ref, bound, _, _ = TL.ln_bwd_ref(x, gain, dy, 1e-5)
    ref = ref + add
    bound = BL.OUT_ROUND * ref.abs() + (1 + BL.OUT_ROUND) * (bound + 2.0 ** -24 * ref.abs())
    assert BL.ratio((bf16((core + add.float()).double()) - ref).abs(), bound) <= 1
    assert BL.ratio((bf16(core.double()) - ref).abs(), bound) > 1


# ------------------------------------------------------------------------------------------------------------- dgrad
def test_dgrad_bound_rejects_an_ignored_residual():
    g = torch.Generator().manual_seed(6)
    x = _samples(2, 64, 8, 12, g)
    w = bf16(torch.randn(64, 64, 3, 3, generator=g, dtype=D) / 24)
    res = _samples(2, 64, 8, 12, g)
    ref = F.conv2d(x, w, padding=1) + res
    A = F.conv2d(x.abs(), w.abs(), padding=1) + res.abs()
    bound = BL.conv_bound(ref, A, 9 * 64)
    conv = F.conv2d(x.float(), w.float(), padding=1)
    assert BL.ratio((bf16((conv + res.float()).double()) - ref).abs(), bound) <= 1
    assert BL.ratio((bf16(conv.double()) - ref).abs(), bound) > 1
