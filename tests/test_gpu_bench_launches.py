"""-m gpu: every distinct kernel launch of the benchmark's UNet inference forward (tests/bench_launches.py: all of
ddim50_436x1024 at batch 8, the two top levels of matrix_flow_1024x2048), run in isolation at exactly its launch shape
and null pattern and compared with a float64 restatement of the op on the same bf16 operands.

Inputs: every sample has its own offset and scale and every (sample, GroupNorm group) its own mean, so a swapped sample,
group or statistics row is off by far more than the bound.  GroupNorm statistics given to a kernel are the exact fp64
sums of its bf16 input.  Scale / shift rows have the UNet's stride (8064 floats) with the block at the end of the row and
NaN everywhere else in it, so a read outside the block shows.

Structure: outputs are prefilled with NaN (an unwritten element fails) and followed by a sentinel guard that must stay
intact; a second launch must give the same bits (the GroupNorm statistics are fp64 atomics: compared to 1e-12).

Bounds (tests/bench_launches.py): convolutions |got - ref| <= 2^-8 |ref| + K 2^-22 sum|x w| (+ the error of a kernel's own
activated input); the fused GroupNorm-SiLU paths add the tanh.approx.f32 error; the attention cores keep the per-kernel
tests' relative tolerances, sample by sample.  Each case prints max(err / bound)."""
import math

import pytest
import torch
import torch.nn.functional as F

import bench_launches as BL
from oracle import flowdiff_oracle as O

pytestmark = pytest.mark.gpu
BF, F64 = torch.bfloat16, torch.float64
SENTINEL = -(2.0 ** 99)
GUARD = 4096
NAN = float("nan")


@pytest.fixture(scope="module")
def L():
    from opticalflowdiffusion_b200 import _lib
    _lib.load(check_device=True)
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.cuda.reset_peak_memory_stats()
    yield _lib
    print(f"\n{torch.cuda.get_device_name()}: peak device memory {torch.cuda.max_memory_allocated() / 2 ** 30:.2f} GiB")


# ------------------------------------------------------------------------------------------------------------ inputs
def guarded(shape, dtype, fill):
    """(buffer, view): ``shape`` prefilled with ``fill``, followed by GUARD sentinel elements."""
    n = math.prod(shape)
    buf = torch.empty(n + GUARD, device="cuda", dtype=dtype)
    buf[:n].fill_(fill)
    buf[n:].fill_(SENTINEL)
    return buf, buf[:n].view(shape)


def guard_intact(buf, view):
    assert bool((buf[view.numel():] == SENTINEL).all()), "write past the end of the output"


def act(shape, seed):
    """bf16 (N, ..., C): sample n scaled by 0.5 + 0.25 n and offset by 0.3 (n - 3.5), each (n, group) its own mean."""
    N, C = shape[0], shape[-1]
    g = torch.Generator(device="cuda").manual_seed(seed)
    x = torch.randn(shape, generator=g, device="cuda")
    n = torch.arange(N, device="cuda", dtype=torch.float32)
    bshape = (N,) + (1,) * (len(shape) - 1)
    x.mul_((0.5 + 0.25 * n).view(bshape)).add_((0.3 * (n - 3.5)).view(bshape))
    mu = torch.randn(N, 8, generator=g, device="cuda").repeat_interleave(C // 8, 1)
    x.add_(mu.view((N,) + (1,) * (len(shape) - 2) + (C,)))
    return x.to(BF)


def rnd(shape, seed, scale=1.0, shift=0.0):
    g = torch.Generator(device="cuda").manual_seed(seed)
    return torch.randn(shape, generator=g, device="cuda") * scale + shift


def stats64(x):
    """Exact fp64 (sum, sum of squares) per (sample, group) of bf16 NHWC x."""
    N, C = x.shape[0], x.shape[-1]
    out = torch.empty(N, 8, 2, device="cuda", dtype=F64)
    for n in range(N):
        r = x[n].double().reshape(-1, 8, C // 8)
        out[n, :, 0] = r.sum((0, 2))
        out[n, :, 1] = (r * r).sum((0, 2))
    return out


def weight(Cout, Cin, KH, KW, seed):
    """bf16-rounded fp32 conv weight at the scale of the UNet's standardised weights."""
    return rnd((Cout, Cin, KH, KW), seed, (Cin * KH * KW) ** -0.5).to(BF).float()


def pack_w(w):
    """[Cout][Cin][KH][KW] -> bf16 [Cout][(ky*KW+kx)*Cin + ci]"""
    return w.permute(0, 2, 3, 1).reshape(w.shape[0], -1).contiguous().to(BF)


def ss_rows(N, C, stride, seed):
    """(rows, offset, scale, shift): (N, stride) fp32 rows, NaN except the (scale | shift) block at offset stride - 2C."""
    off = stride - 2 * C
    rows = torch.full((N, stride), NAN, device="cuda")
    n = torch.arange(N, device="cuda", dtype=torch.float32).view(N, 1)
    sc = rnd((N, C), seed, 0.3) + 0.1 * n - 0.35
    sh = rnd((N, C), seed + 1, 0.5) + 0.2 * (n - 3.5)
    rows[:, off:off + C] = sc
    rows[:, off + C:off + 2 * C] = sh
    return rows, off, sc.double(), sh.double()


def norm_params(C, seed):
    return rnd((C,), seed, 0.3, 1.0), rnd((C,), seed + 1, 0.2)


def nchw(t):
    """(H, W, C) or (P, C) of one sample -> float64 (1, C, H, W) / (1, C, P, 1)."""
    t = t.double()
    if t.dim() == 2:
        return t.t().reshape(1, t.shape[1], t.shape[0], 1)
    return t.permute(2, 0, 1).unsqueeze(0)


def report(name, scalars, nulls, **r):
    print(f"{name}{scalars} {nulls}: " + ", ".join(f"{k} {v:.3f}" for k, v in r.items()))


def conv_parts(x, w, bias, pad, res=None):
    """float64 conv of one sample and A = conv(|x|, |w|) + |bias| (+ residual and |residual|)."""
    b = bias.double() if bias is not None else None
    ref = F.conv2d(x, w, b, padding=pad)
    A = F.conv2d(x.abs(), w.abs(), padding=pad)
    if b is not None:
        A += b.abs().view(1, -1, 1, 1)
    if res is not None:
        ref += res
        A += res.abs()
    return ref, A


def check_stats(st, st2, sums_bounds):
    worst = 0.0
    for n, (sums, bounds) in enumerate(sums_bounds):
        worst = max(worst, BL.ratio((st[n] - sums).abs(), bounds))
    assert torch.allclose(st, st2, rtol=1e-12, atol=1e-12 * st.abs().max().item())      # fp64 atomics: order only
    return worst


# ------------------------------------------------------------------------------------------------------------ checkers
def check_conv(L, scalars, nulls, seed):
    """fd_conv_igemm: strip, CTA-pair, 1x1 and pixel-unshuffle (mode 1) paths; +- bias, residual, second source, stats."""
    lib = L.load()
    C0, C1, N, H, W, Cout, KH, KW, ph, pw, mode = scalars
    has_bias, has_res, has_stats = nulls[3] == "P", nulls[4] == "P", nulls[6] == "P"
    Hin, Win = (2 * H, 2 * W) if mode else (H, W)
    s0 = act((N, Hin, Win, C0), seed)
    s1 = act((N, Hin, Win, C1), seed + 1) if C1 else None
    if mode:
        w = weight(Cout, 4 * C0, 1, 1, seed + 2)
        # torch channel c*4 + p1*2 + p2 -> K = (p1*2+p2)*C + c
        wp = w.reshape(Cout, C0, 4).permute(0, 2, 1).reshape(Cout, 4 * C0).contiguous().to(BF)
    else:
        w = weight(Cout, C0 + C1, KH, KW, seed + 2)
        wp = pack_w(w)
    bias = rnd((Cout,), seed + 3) if has_bias else None
    res = act((N, H, W, Cout), seed + 4) if has_res else None

    def launch(fill):
        buf, out = guarded((N, H, W, Cout), BF, fill)
        sbuf, st = guarded((N, 8, 2), F64, 0.0) if has_stats else (None, None)
        L.check(lib.fd_conv_igemm(L.ptr(s0), C0, L.ptr(s1), C1, L.ptr(wp), L.ptr(bias), L.ptr(res), L.ptr(out), L.ptr(st),
                                  N, H, W, Cout, KH, KW, ph, pw, mode, L.stream()))
        torch.cuda.synchronize()
        guard_intact(buf, out)
        if has_stats:
            guard_intact(sbuf, st)
        return out, st

    # 128 input channels -> 64 at W >= 128 run on the rolling-strip kernel as two passes over 64-channel halves: pass 1 stores
    # its partial sum (+ the residual) as bf16 and pass 2 adds it back, one more bf16 rounding of that partial sum
    two_pass = (mode == 0 and (KH, KW, ph, pw) == (3, 3, 1, 1) and C0 + C1 == 128 and C0 in (64, 128) and Cout == 64 and
                W >= 128)
    out, st = launch(NAN)
    w64 = w.double()
    worst, sb = 0.0, []
    for n in range(N):
        x = nchw(torch.cat((s0[n], s1[n]), -1) if C1 else s0[n])
        if mode:
            x = O._pixel_unshuffle2(x)
        ref, A = conv_parts(x, w64, bias, (ph, pw), nchw(res[n]) if has_res else None)
        partial = None
        if two_pass:
            p0, a0 = conv_parts(x[:, :64], w64[:, :64], None, 1, nchw(res[n]) if has_res else None)
            partial = BL.OUT_ROUND * p0.abs() + BL.gamma_mma(9 * 64) * a0
            del p0, a0
        bound = BL.conv_bound(ref, A, wp.shape[1], partial)
        worst = max(worst, BL.ratio((nchw(out[n]) - ref).abs(), bound))
        if has_stats:
            sb.append(BL.stats_ref(ref[0], bound[0]))
        del x, ref, A, bound
    out2, st2 = launch(0.0)
    worst_st = check_stats(st, st2, sb) if has_stats else 0.0
    report("fd_conv_igemm", scalars, nulls, err_over_bound=worst, stats_err_over_bound=worst_st)
    assert worst <= 1 and worst_st <= 1
    assert torch.equal(out, out2)


def _gn_silu_sample(x, st, gamma, beta, eps, sc=None, sh=None):
    """silu(GroupNorm(x) (scale + 1) + shift) of one sample (P, C) in float64 and the bound of the kernels' fp32 form."""
    z, dz = BL.gn_affine(x.double(), st, gamma.double(), beta.double(), eps, sc, sh)
    return BL.silu_tanh(z, dz)


def check_gn_silu_fast(L, scalars, nulls, seed):
    """fd_gn_silu_fast: GroupNorm apply + (scale + 1, shift) + tanh-form SiLU (+ residual); grid-stride at large HW."""
    check_gn_silu_form(L, "fd_gn_silu_fast", BL.silu_tanh, scalars, nulls, seed)


def check_gn_silu_form(L, name, silu, scalars, nulls, seed):
    """GroupNorm apply + (scale + 1, shift) + SiLU (+ residual) of the kernel ``name`` against ``silu(z, dz)``, which gives
    silu(z) and the bound of the kernel's SiLU form."""
    lib = L.load()
    stride, N, HW, C, eps = scalars
    use_ss, use_res = nulls[4] == "P", nulls[5] == "P"
    x = act((N, HW, C), seed)
    st = stats64(x)
    gamma, beta = norm_params(C, seed + 1)
    rows, off, sc, sh = ss_rows(N, C, stride, seed + 2) if use_ss else (None, 0, None, None)
    res = act((N, HW, C), seed + 3) if use_res else None

    def launch(fill):
        buf, out = guarded((N, HW, C), BF, fill)
        L.check(getattr(lib, name)(L.ptr(x), L.ptr(st), L.ptr(gamma), L.ptr(beta), rows.data_ptr() + 4 * off if use_ss else None,
                                   stride, L.ptr(res), L.ptr(out), N, HW, C, eps, L.stream()))
        torch.cuda.synchronize()
        guard_intact(buf, out)
        return out

    out = launch(NAN)
    worst = 0.0
    for n in range(N):
        z, dz = BL.gn_affine(x[n].double(), st[n], gamma.double(), beta.double(), eps, sc[n] if use_ss else None,
                             sh[n] if use_ss else None)
        s, ds = silu(z, dz)
        ref = s + res[n].double() if use_res else s
        bound = BL.OUT_ROUND * ref.abs() + (1 + BL.OUT_ROUND) * ds
        worst = max(worst, BL.ratio((out[n].double() - ref).abs(), bound))
        del z, dz, s, ds, ref, bound
    report(name, scalars, nulls, err_over_bound=worst)
    assert worst <= 1
    assert torch.equal(out, launch(0.0))


def check_conv3x3_gnsilu_in(L, scalars, nulls, seed):
    """fd_conv3x3_gnsilu_in: block1's GroupNorm + scale/shift + SiLU applied to the strips of the 64 -> 64 conv's input."""
    lib = L.load()
    stride, eps, N, H, W = scalars
    C = 64
    x = act((N, H, W, C), seed)
    in_st = stats64(x)
    gamma, beta = norm_params(C, seed + 1)
    rows, off, sc, sh = ss_rows(N, C, stride, seed + 2)
    w = weight(C, C, 3, 3, seed + 4)
    wp = pack_w(w)
    bias = rnd((C,), seed + 5)

    def launch(fill):
        buf, out = guarded((N, H, W, C), BF, fill)
        sbuf, st = guarded((N, 8, 2), F64, 0.0)
        L.check(lib.fd_conv3x3_gnsilu_in(L.ptr(x), L.ptr(in_st), L.ptr(gamma), L.ptr(beta), rows.data_ptr() + 4 * off, stride,
                                         eps, L.ptr(wp), L.ptr(bias), None, L.ptr(out), L.ptr(st), N, H, W, L.stream()))
        torch.cuda.synchronize()
        guard_intact(buf, out)
        guard_intact(sbuf, st)
        return out, st

    out, st = launch(NAN)
    w64 = w.double()
    worst, sb = 0.0, []
    for n in range(N):
        s, ds = _gn_silu_sample(x[n].reshape(-1, C), in_st[n], gamma, beta, eps, sc[n], sh[n])
        da = BL.bf16_act(s, ds)
        s, da = nchw(s.view(H, W, C)), nchw(da.view(H, W, C))
        del ds
        ref = F.conv2d(s, w64, bias.double(), padding=1)
        A = F.conv2d(s.abs() + da, w64.abs(), padding=1) + bias.double().abs().view(1, -1, 1, 1)
        bound = BL.conv_bound(ref, A, 9 * C, F.conv2d(da, w64.abs(), padding=1))
        worst = max(worst, BL.ratio((nchw(out[n]) - ref).abs(), bound))
        sb.append(BL.stats_ref(ref[0], bound[0]))
        del s, da, ref, A, bound
    out2, st2 = launch(0.0)
    worst_st = check_stats(st, st2, sb)
    report("fd_conv3x3_gnsilu_in", scalars, nulls, err_over_bound=worst, stats_err_over_bound=worst_st)
    assert worst <= 1 and worst_st <= 1
    assert torch.equal(out, out2)


def _rt_inputs(C0, C1, N, H, W, Cout, seed):
    s0 = act((N, H, W, C0), seed)
    s1 = act((N, H, W, C1), seed + 1) if C1 else None
    w = weight(Cout, C0 + C1, 1, 1, seed + 2)
    bias = rnd((Cout,), seed + 3)
    raw = act((N, H, W, Cout), seed + 4)
    gamma, beta = norm_params(Cout, seed + 5)
    return s0, s1, w, bias, raw, stats64(raw), gamma, beta


def _rt_sample(n, s0, s1, w, bias, raw, raw_st, gamma, beta, eps):
    """res_conv(x) + silu(GroupNorm(raw)) of sample n (float64, NCHW), sum|x w| + |bias| + |silu|, and the silu's bound."""
    H, W, Cout = raw.shape[1:]
    x = nchw(torch.cat((s0[n], s1[n]), -1) if s1 is not None else s0[n])
    conv, A = conv_parts(x, w.double(), bias, 0)
    s, ds = _gn_silu_sample(raw[n].reshape(-1, Cout), raw_st[n], gamma, beta, eps)
    s, ds = nchw(s.view(H, W, Cout)), nchw(ds.view(H, W, Cout))
    return conv + s, A + s.abs(), ds


def check_conv_igemm_rt(L, scalars, nulls, seed):
    """fd_conv_igemm_rt: the 1x1 res_conv of cat(x0, x1) + silu(GroupNorm(h2)) in the conv's epilogue."""
    lib = L.load()
    C0, C1, eps, N, H, W, Cout, KH, KW, ph, pw = scalars
    s0, s1, w, bias, raw, raw_st, gamma, beta = _rt_inputs(C0, C1, N, H, W, Cout, seed)
    wp = pack_w(w)

    def launch(fill):
        buf, out = guarded((N, H, W, Cout), BF, fill)
        L.check(lib.fd_conv_igemm_rt(L.ptr(s0), C0, L.ptr(s1), C1, L.ptr(wp), L.ptr(bias), L.ptr(raw), L.ptr(raw_st), L.ptr(gamma),
                                     L.ptr(beta), eps, L.ptr(out), N, H, W, Cout, KH, KW, ph, pw, L.stream()))
        torch.cuda.synchronize()
        guard_intact(buf, out)
        return out

    out = launch(NAN)
    worst = 0.0
    for n in range(N):
        ref, A, ds = _rt_sample(n, s0, s1, w, bias, raw, raw_st, gamma, beta, eps)
        bound = BL.conv_bound(ref, A, C0 + C1, (1 + BL.OUT_ROUND) * ds)
        worst = max(worst, BL.ratio((nchw(out[n]) - ref).abs(), bound))
        del ref, A, ds, bound
    report("fd_conv_igemm_rt", scalars, nulls, err_over_bound=worst)
    assert worst <= 1
    assert torch.equal(out, launch(0.0))


def check_conv_igemm_rt_head(L, scalars, nulls, seed):
    """fd_conv_igemm_rt_head: fd_conv_igemm_rt's fp32 tile through the final 1x1 conv (fp32 weights), cropped to the
    H0 x W0 window at (pt, pl), fp32 NCHW.  Bound: the tile's error (accumulation + SiLU, no bf16 rounding) through |hw|, and
    the fp32 dot product of 64 terms plus the bias."""
    lib = L.load()
    C0, C1, eps, nout, N, H, W, H0, W0, pt, pl = scalars
    s0, s1, w, bias, raw, raw_st, gamma, beta = _rt_inputs(C0, C1, N, H, W, 64, seed)
    wp = pack_w(w)
    hw, hb = rnd((nout, 64), seed + 6, 1 / 8), rnd((nout,), seed + 7)

    def launch(fill):
        buf, out = guarded((N, nout, H0, W0), torch.float32, fill)
        L.check(lib.fd_conv_igemm_rt_head(L.ptr(s0), C0, L.ptr(s1), C1, L.ptr(wp), L.ptr(bias), L.ptr(raw), L.ptr(raw_st),
                                          L.ptr(gamma), L.ptr(beta), eps, L.ptr(hw), L.ptr(hb), nout, L.ptr(out), N, H, W, H0, W0,
                                          pt, pl, L.stream()))
        torch.cuda.synchronize()
        guard_intact(buf, out)
        return out

    out = launch(NAN)
    hw64, hb64 = hw.double().view(nout, 64, 1, 1), hb.double()
    worst = 0.0
    for n in range(N):
        v, A, ds = _rt_sample(n, s0, s1, w, bias, raw, raw_st, gamma, beta, eps)
        ev = BL.gamma_mma(C0 + C1) * A + ds + 2.0 ** -23 * v.abs()
        win = (slice(None), slice(None), slice(pt, pt + H0), slice(pl, pl + W0))
        ref = F.conv2d(v, hw64, hb64)[win]
        bound = F.conv2d(ev, hw64.abs())[win] + 65 * 2.0 ** -23 * (F.conv2d(v.abs(), hw64.abs())[win] + hb64.abs().view(1, -1, 1, 1))
        worst = max(worst, BL.ratio((out[n:n + 1].double() - ref).abs(), bound))
        del v, A, ds, ev, ref, bound
    report("fd_conv_igemm_rt_head", scalars, nulls, err_over_bound=worst)
    assert worst <= 1
    assert torch.equal(out, launch(0.0))


def check_conv_igemm_up(L, scalars, nulls, seed):
    """fd_conv_igemm_up: nearest x2 + conv3x3 as four 2x2 phase convolutions.  The reference is the conv on the up-sampled
    tensor with the fp32 weights; each phase weight is a sum of up to four of them in fp32 rounded once to bf16, which adds
    (2^-9 + 3 2^-24) sum |x| |w| <= (2^-9 + 2^-21) A to the bound."""
    lib = L.load()
    Cin, N, H, W, Cout = scalars
    x = act((N, H, W, Cin), seed)
    w = rnd((Cout, Cin, 3, 3), seed + 1, (9 * Cin) ** -0.5)
    bias = rnd((Cout,), seed + 2)
    w4 = torch.empty(4, Cout, 4 * Cin, device="cuda", dtype=BF)
    L.check(lib.fd_prep_weight_upconv(L.ptr(w), L.ptr(w4), Cout, Cin, L.stream()))

    def launch(fill):
        buf, out = guarded((N, 2 * H, 2 * W, Cout), BF, fill)
        L.check(lib.fd_conv_igemm_up(L.ptr(x), Cin, L.ptr(w4), L.ptr(bias), L.ptr(out), N, H, W, Cout, L.stream()))
        torch.cuda.synchronize()
        guard_intact(buf, out)
        return out

    out = launch(NAN)
    worst = 0.0
    for n in range(N):
        up = F.interpolate(nchw(x[n]), scale_factor=2, mode="nearest")
        ref, A = conv_parts(up, w.double(), bias, 1)
        bound = BL.OUT_ROUND * ref.abs() + (BL.gamma_mma(4 * Cin) + 2.0 ** -9 + 2.0 ** -21) * A
        worst = max(worst, BL.ratio((nchw(out[n]) - ref).abs(), bound))
        del up, ref, A, bound
    report("fd_conv_igemm_up", scalars, nulls, err_over_bound=worst)
    assert worst <= 1
    assert torch.equal(out, launch(0.0))


def rel_err(a, b):
    return ((a - b).abs().max() / b.abs().max().clamp(min=1e-6)).item()


def check_linattn_tc(L, scalars, nulls, seed):
    """fd_linattn_tc == the oracle's Residual(PreNorm(LinearAttention)) in float64, each sample by itself, at the
    tolerances of test_gpu_unet_ops.test_linear_attention_block_tcgen05 (whole block 2e-2, attention branch 4e-2)."""
    lib = L.load()
    N, HW, C, eps = scalars
    x = act((N, HW, C), seed)
    sd = {"norm.g": rnd((1, C, 1, 1), seed + 1, 0.3, 1.0),
          "fn.to_qkv.weight": rnd((384, C, 1, 1), seed + 2, 2.0 / C ** 0.5),
          "fn.to_out.0.weight": rnd((C, 128, 1, 1), seed + 3, 30 / 128 ** 0.5),
          "fn.to_out.0.bias": rnd((C,), seed + 4, 0.1),
          "fn.to_out.1.g": rnd((1, C, 1, 1), seed + 5, 0.3, 1.0)}
    wqkv = sd["fn.to_qkv.weight"].reshape(384, C).contiguous()
    g1, g2 = sd["norm.g"].reshape(C).contiguous(), sd["fn.to_out.1.g"].reshape(C).contiguous()
    wout, bout = sd["fn.to_out.0.weight"].reshape(C, 128).contiguous(), sd["fn.to_out.0.bias"]
    wq, wk = torch.empty(128, C, device="cuda", dtype=BF), torch.empty(128, C, device="cuda", dtype=BF)
    sq, sk, mk = (torch.empty(128, device="cuda") for _ in range(3))
    wv = torch.empty(128, C, device="cuda")
    L.check(lib.fd_linattn_tc_prep(L.ptr(wqkv), L.ptr(g1), L.ptr(wq), L.ptr(sq), L.ptr(wk), L.ptr(sk), L.ptr(mk), L.ptr(wv), C,
                                   L.stream()))
    ws = torch.empty(lib.fd_linattn_tc_workspace_floats(N, HW, C), device="cuda")

    def launch(fill):
        buf, out = guarded((N, HW, C), BF, fill)
        L.check(lib.fd_linattn_tc(L.ptr(x), L.ptr(wk), L.ptr(sk), L.ptr(mk), L.ptr(wq), L.ptr(sq), L.ptr(wv), L.ptr(wout),
                                  L.ptr(bout), L.ptr(g2), L.ptr(out), L.ptr(ws), N, HW, C, eps, L.stream()))
        torch.cuda.synchronize()
        guard_intact(buf, out)
        return out

    out = launch(NAN)
    sd64 = {k: v.double() for k, v in sd.items()}
    errs, branch = [], []
    for n in range(N):
        xn = nchw(x[n])
        ref = O._linear_attention(sd64, "", xn, eps=eps)
        got = nchw(out[n])
        errs.append(rel_err(got, ref))
        branch.append(rel_err(got - xn, ref - xn))
        del xn, ref, got
    report("fd_linattn_tc", scalars, nulls, worst_sample_rel_err=max(errs), worst_sample_branch_rel_err=max(branch))
    assert max(errs) < 2e-2 and max(branch) < 4e-2, (errs, branch)
    assert torch.equal(out, launch(0.0))


def _attn_core(qkv, linear):
    """qkv (1, 384, P, 1) float64 -> (1, 128, P, 1): the LinearAttention / Attention core (to_qkv / to_out excluded)."""
    from test_gpu_unet_ops import _attn_ref
    return _attn_ref(qkv, linear)


def _check_attention_core(L, name, scalars, nulls, seed, linear, tol):
    lib = L.load()
    N, HW = scalars
    g = torch.Generator(device="cuda").manual_seed(seed)
    n = torch.arange(N, device="cuda", dtype=torch.float32).view(N, 1, 1)
    qkv = (torch.randn(N, HW, 384, generator=g, device="cuda") * (1.0 + 0.07 * n) + 0.2 * (n - 3.5)).to(BF)
    ws = torch.empty(lib.fd_linattn_workspace_floats(N, HW), device="cuda") if linear else None

    def launch(fill):
        buf, out = guarded((N, HW, 128), BF, fill)
        if linear:
            L.check(lib.fd_linattn(L.ptr(qkv), L.ptr(out), L.ptr(ws), N, HW, L.stream()))
        else:
            L.check(lib.fd_attention(L.ptr(qkv), L.ptr(out), N, HW, L.stream()))
        torch.cuda.synchronize()
        guard_intact(buf, out)
        return out

    out = launch(NAN)
    errs = []
    for i in range(N):
        ref = _attn_core(nchw(qkv[i]), linear)
        errs.append(rel_err(nchw(out[i]), ref))
        del ref
    report(name, scalars, nulls, worst_sample_rel_err=max(errs))
    assert max(errs) < tol, errs
    assert torch.equal(out, launch(0.0))


def check_linattn(L, scalars, nulls, seed):
    """fd_linattn (C = 256 LinearAttention core), per sample at test_linear_attention_core's 1.5e-2."""
    _check_attention_core(L, "fd_linattn", scalars, nulls, seed, True, 1.5e-2)


def check_attention(L, scalars, nulls, seed):
    """fd_attention (mid block, tcgen05), per sample at test_full_attention_core's 2e-2."""
    _check_attention_core(L, "fd_attention", scalars, nulls, seed, False, 2e-2)


def check_chan_layernorm(L, scalars, nulls, seed):
    """fd_chan_layernorm (+ residual).  Bound: one output rounding, plus the fp32 mean and variance of C terms (the mean
    off by <= C 2^-24 mean|x|, the variance by <= C 2^-23 relative; the mean's error enters it only squared), doubled for
    rsqrtf and the products: C 2^-21 |g| rstd (mean|x| + |x - mean|)."""
    lib = L.load()
    npix, C, eps = scalars
    use_res = nulls[2] == "P"
    x = act((8, npix // 8, C), seed).view(npix, C)
    gain = rnd((C,), seed + 1, 0.3, 1.0)
    res = act((8, npix // 8, C), seed + 2).view(npix, C) if use_res else None

    def launch(fill):
        buf, out = guarded((npix, C), BF, fill)
        L.check(lib.fd_chan_layernorm(L.ptr(x), L.ptr(gain), L.ptr(res), L.ptr(out), npix, C, eps, L.stream()))
        torch.cuda.synchronize()
        guard_intact(buf, out)
        return out

    out = launch(NAN)
    xd, g64 = x.double(), gain.double()
    ref = O._chan_layernorm(xd, g64, eps)
    d = xd - xd.mean(1, keepdim=True)
    rstd = ((d * d).mean(1, keepdim=True) + eps).rsqrt()
    bound = BL.OUT_ROUND * (ref + (res.double() if use_res else 0)).abs() + \
        C * 2.0 ** -21 * g64.abs() * rstd * (xd.abs().mean(1, keepdim=True) + d.abs())
    if use_res:
        ref = ref + res.double()
    worst = BL.ratio((out.double() - ref).abs(), bound)
    report("fd_chan_layernorm", scalars, nulls, err_over_bound=worst)
    assert worst <= 1
    assert torch.equal(out, launch(0.0))


def check_time_embed(L, scalars, nulls, seed):
    """fd_time_embed: distinct timesteps per sample including 0 and 999, against the oracle in float64.  Bound propagated
    through the layers: sinf / cosf of the fp32 argument t f to 2^-21 (1 + |t f|), fp32 dot products of K terms to
    (K + 1) 2^-23 of sum |w x| + |b|, |gelu'| <= 1.13 plus erff's few ulp."""
    lib = L.load()
    B, dim, tdim = scalars
    t = torch.tensor([0, 999, 1, 17, 250, 500, 750, 998][:B], device="cuda")
    sd = {"time_mlp.1.weight": rnd((tdim, dim), seed, 0.1), "time_mlp.1.bias": rnd((tdim,), seed + 1),
          "time_mlp.3.weight": rnd((tdim, tdim), seed + 2, 0.05), "time_mlp.3.bias": rnd((tdim,), seed + 3)}

    def launch(fill):
        buf, out = guarded((B, tdim), torch.float32, fill)
        L.check(lib.fd_time_embed(L.ptr(t), L.ptr(sd["time_mlp.1.weight"]), L.ptr(sd["time_mlp.1.bias"]),
                                  L.ptr(sd["time_mlp.3.weight"]), L.ptr(sd["time_mlp.3.bias"]), L.ptr(out), B, dim, tdim, L.stream()))
        torch.cuda.synchronize()
        guard_intact(buf, out)
        return out

    out = launch(NAN)
    ref, bound = time_embed_ref(sd, t, dim, tdim)[4:]
    worst = BL.ratio((out.double() - ref).abs(), bound)
    report("fd_time_embed", scalars, nulls, err_over_bound=worst)
    assert worst <= 1
    assert torch.equal(out, launch(0.0))


def time_embed_ref(sd, t, dim, tdim):
    """(pe, its bound, the pre-GELU activations, their bound, temb, its bound) of the time MLP in float64."""
    sd64 = {k: v.double() for k, v in sd.items()}
    ref = O.time_embedding(sd64, t.double(), dim)
    half = dim // 2
    arg = t.double()[:, None] * torch.exp(torch.arange(half, device="cuda", dtype=F64) * -(math.log(10000) / (half - 1)))
    pe = torch.cat((arg.sin(), arg.cos()), 1)
    dpe = 2.0 ** -21 * (1 + torch.cat((arg, arg), 1).abs())
    w1, b1, w2, b2 = (sd64[k] for k in ("time_mlp.1.weight", "time_mlp.1.bias", "time_mlp.3.weight", "time_mlp.3.bias"))
    h = pe @ w1.t() + b1
    dh = dpe @ w1.abs().t() + (dim + 1) * 2.0 ** -23 * (pe.abs() @ w1.abs().t() + b1.abs())
    gel = F.gelu(h)
    dg = 1.13 * dh + 2.0 ** -21 * h.abs()
    bound = dg @ w2.abs().t() + (tdim + 1) * 2.0 ** -23 * (gel.abs() @ w2.abs().t() + b2.abs())
    return pe, dpe, h, dh, ref, bound


def check_time_proj(L, scalars, nulls, seed):
    """fd_time_proj: every block's (scale | shift) rows, silu(temb) @ w^T + b.  Bound: the exp-form SiLU (__expf,
    __fdividef) to 2^-20 |temb|, and the fp32 dot product of K terms to (K + 1) 2^-23 of sum |w s| + |b|."""
    lib = L.load()
    B, K, J = scalars
    n = torch.arange(B, device="cuda", dtype=torch.float32).view(B, 1)
    temb = rnd((B, K), seed, 1.0) * (0.5 + 0.25 * n) + 0.3 * (n - 3.5)
    w, b = rnd((J, K), seed + 1, 0.05), rnd((J,), seed + 2)

    def launch(fill):
        buf, out = guarded((B, J), torch.float32, fill)
        L.check(lib.fd_time_proj(L.ptr(temb), L.ptr(w), L.ptr(b), L.ptr(out), B, K, J, L.stream()))
        torch.cuda.synchronize()
        guard_intact(buf, out)
        return out

    out = launch(NAN)
    z = temb.double()
    s = F.silu(z)
    w64, b64 = w.double(), b.double()
    ref = s @ w64.t() + b64
    bound = (2.0 ** -20 * z.abs()) @ w64.abs().t() + (K + 1) * 2.0 ** -23 * (s.abs() @ w64.abs().t() + b64.abs())
    worst = BL.ratio((out.double() - ref).abs(), bound)
    report("fd_time_proj", scalars, nulls, err_over_bound=worst)
    assert worst <= 1
    assert torch.equal(out, launch(0.0))


def packed_input_ref(x, cond, H, W, pt, pl, nan_mask, wide):
    """The packed init_conv input, restated with torch: NaN -> 0 and the mask channel (any NaN over the x channels),
    replicate padding of the H0 x W0 planes at (pt, pl) into the H x W frame, then either the 7 horizontal taps unrolled
    (packed[b, h, w, kx * Ctot + c] = in[b, c, h, w + kx - 3], zero outside the row) or plain NHWC, zero above the used
    channels, bf16."""
    parts = [x]
    if nan_mask:
        nans = torch.isnan(x)
        parts = [torch.where(nans, torch.zeros_like(x), x), nans.any(1, keepdim=True).float()]
    if cond is not None:
        parts.append(cond)
    inp = torch.cat(parts, 1)
    B, Ctot, H0, W0 = inp.shape
    inp = F.pad(inp, (pl, W - W0 - pl, pt, H - H0 - pt), mode="replicate")
    if wide:
        packed = inp.permute(0, 2, 3, 1)
    else:
        row = F.pad(inp, (3, 3))
        packed = torch.stack([row[..., kx:kx + W] for kx in range(7)], 1).permute(0, 3, 4, 1, 2).reshape(B, H, W, 7 * Ctot)
    return F.pad(packed, (0, 64 - packed.shape[-1])).to(BF)


def _check_pack(L, scalars, seed, wide):
    lib = L.load()
    B, Cx, Cc, H0, W0, pt, pl, H, W, nan_mask = scalars
    n = torch.arange(B, device="cuda", dtype=torch.float32).view(B, 1, 1, 1)
    x = rnd((B, Cx, H0, W0), seed) * (1 + 0.5 * n) + n
    if nan_mask:
        g = torch.Generator(device="cuda").manual_seed(seed + 1)
        x[torch.rand(x.shape, generator=g, device="cuda") < 1e-3] = NAN
        x[:, :, 0, 0] = NAN                    # a corner that the replicate padding spreads
    cond = rnd((B, Cc, H0, W0), seed + 2) - n if Cc else None
    fn = lib.fd_pack_input_wide if wide else lib.fd_pack_input_pad

    def launch(fill):
        buf, out = guarded((B, H, W, 64), BF, fill)
        L.check(fn(L.ptr(x), L.ptr(cond), L.ptr(out), B, Cx, Cc, H0, W0, pt, pl, H, W, nan_mask, L.stream()))
        torch.cuda.synchronize()
        guard_intact(buf, out)
        return out

    out = launch(NAN)
    ref = packed_input_ref(x, cond, H, W, pt, pl, nan_mask, wide)
    assert torch.equal(out, ref), (out.float() - ref.float()).abs().nan_to_num(float("inf")).max()
    assert torch.equal(out, launch(0.0))


def check_pack_input_pad(L, scalars, nulls, seed):
    """fd_pack_input_pad: bit-exact against packed_input_ref (replicate padding folded into the packing)."""
    _check_pack(L, scalars, seed, False)
    report("fd_pack_input_pad", scalars, nulls, bit_exact=1.0)


CHECKERS = {
    "fd_time_embed": check_time_embed,
    "fd_time_proj": check_time_proj,
    "fd_pack_input_pad": check_pack_input_pad,
    "fd_conv_igemm": check_conv,
    "fd_conv3x3_gnsilu_in": check_conv3x3_gnsilu_in,
    "fd_gn_silu_fast": check_gn_silu_fast,
    "fd_linattn_tc": check_linattn_tc,
    "fd_linattn": check_linattn,
    "fd_attention": check_attention,
    "fd_chan_layernorm": check_chan_layernorm,
    "fd_conv_igemm_rt": check_conv_igemm_rt,
    "fd_conv_igemm_rt_head": check_conv_igemm_rt_head,
    "fd_conv_igemm_up": check_conv_igemm_up,
}

CASES = [pytest.param(wl, i, e, id=f"{wl}-{i:02d}-{e[0]}") for wl, table in (("default", BL.DEFAULT), ("matrix", BL.MATRIX))
         for i, e in enumerate(table)]


@pytest.mark.parametrize("workload, index, entry", CASES)
def test_bench_launch(L, workload, index, entry):
    name, scalars, nulls, _ = entry
    CHECKERS[name](L, scalars, nulls, 1000 * (workload == "matrix") + 16 * index)


@pytest.mark.parametrize("wide", [False, True])
def test_pack_input_nan_mask_and_ragged_padding(L, wide):
    """fd_pack_input_pad (9 channels) and fd_pack_input_wide (latent mode, 36 channels) with the NaN-mask channel and
    replicate padding on all four sides (1021 -> 1024 columns: one on the left, two on the right), bit-exact."""
    Cx = 32 if wide else 5
    _check_pack(L, (2, Cx, 3, 436, 1021, 2, 1, 440, 1024, 1), 7 + wide, wide)


def test_prep_weight_batch_benchmark_network(L):
    """fd_prep_weight_batch over every layer of the seed-0 benchmark network (Unet(64, 5, 2)): weight standardisation in
    float64 and the kind 0 / 1 / 2 layouts, to one bf16 rounding plus the fp32 mean / variance over K terms."""
    from opticalflowdiffusion_b200.unet import Unet
    torch.manual_seed(0)
    net = Unet(64, 5, 2).cuda()
    net.prepare()
    convs = net._convs
    assert len(convs) == 74
    worst = 0.0
    for name, pc in convs.items():
        w = pc.src.weight.detach().double()
        cout, cin, kh, kw = w.shape
        K = cin * kh * kw
        slack = torch.zeros_like(w)
        if pc.ws:
            flat = w.reshape(cout, -1)
            mean = flat.mean(1).view(-1, 1, 1, 1)
            rstd = (flat.var(1, unbiased=False).view(-1, 1, 1, 1) + net.WS_EPS).rsqrt()
            slack = K * 2.0 ** -22 * (w.abs() + flat.abs().mean(1).view(-1, 1, 1, 1)) * rstd
            w = (w - mean) * rstd
        if pc.kind == 0:
            ref, slack = (t.permute(0, 2, 3, 1).reshape(cout, -1) for t in (w, slack))
        elif pc.kind == 1:
            C = cin // 4
            ref, slack = (t.reshape(cout, C, 4).permute(0, 2, 1).reshape(cout, cin) for t in (w, slack))
        else:
            assert pc.kind == 2 and kw * cin <= 64
            # [Cout][ky * 64 + kx * Cin + c], zero above 7 * Cin in every ky block
            ref = torch.zeros(cout, kh, 64, device="cuda", dtype=F64)
            ref[:, :, :kw * cin] = w.permute(0, 2, 3, 1).reshape(cout, kh, kw * cin)
            ref = ref.reshape(cout, kh * 64)
            slack = torch.zeros_like(ref)
        got = pc.w.double()
        assert got.shape == ref.shape, name
        worst = max(worst, BL.ratio((got - ref).abs(), 2.0 ** -8 * ref.abs() + slack))
    print(f"fd_prep_weight_batch, 74 layers: err_over_bound {worst:.3f}")
    assert worst <= 1


def test_ddim_step_benchmark_shape(L):
    """fd_ddim_step at 8 x 2 x 436 x 1024 (the benchmark's sampler state) == the oracle's fp32 op sequence bit for bit."""
    from test_gpu_sampling import make_algo
    lib = L.load()
    m = make_algo(["algorithm.target=flow", "algorithm.sampling_timesteps=50"])
    sched = O.make_schedule(1000)
    g = torch.Generator().manual_seed(3)
    shape = (8, 2, 436, 1024)
    x = torch.randn(shape, generator=g) * (1 + 0.1 * torch.arange(8).view(8, 1, 1, 1))
    mo = torch.randn(shape, generator=g) * 1.5
    xc, moc = x.cuda(), mo.cuda()
    for time, time_next in ((999, 979), (19, -1), (500, 480)):
        ref, x0 = O.ddim_update(sched, x, mo, time, time_next)
        out_buf, out = guarded(shape, torch.float32, NAN)
        x0_buf, x0o = guarded(shape, torch.float32, NAN)
        recip, recipm1, san, c, sigma, last = m.model._ddim_scalars(time, time_next)
        L.check(lib.fd_ddim_step(L.ptr(xc), L.ptr(moc), None, L.ptr(out), L.ptr(x0o), xc.numel(), recip, recipm1, san, c, sigma,
                                 last, L.stream()))
        torch.cuda.synchronize()
        guard_intact(out_buf, out)
        guard_intact(x0_buf, x0o)
        assert torch.equal(out.cpu(), ref) and torch.equal(x0o.cpu(), x0)
