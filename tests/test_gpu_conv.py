"""-m gpu: the tcgen05 implicit-GEMM convolution against torch fp32 conv2d on the same bf16-rounded
operands (tolerance: fp32 accumulation-order noise + one bf16 rounding of the output)."""
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def L():
    from opticalflowdiffusion_b200 import _lib
    _lib.load(check_device=True)
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    return _lib


def nhwc_bf16(x):
    return x.permute(0, 2, 3, 1).contiguous().to(torch.bfloat16)


def pack_w(w):
    """[Cout][Cin][KH][KW] -> bf16 [Cout][(ky*KW+kx)*Cin + ci]"""
    return w.permute(0, 2, 3, 1).reshape(w.shape[0], -1).contiguous().to(torch.bfloat16)


def run_conv(L, xs, w, bias, pad, residual=None, stats=False, mode=0):
    lib = L.load()
    N = xs[0].shape[0]
    srcs = [nhwc_bf16(x) for x in xs]
    Cout = w.shape[0]
    if mode == 0:
        H, W = xs[0].shape[2:]
        KH, KW = w.shape[2:]
        wp = pack_w(w)
    else:
        H, W = xs[0].shape[2] // 2, xs[0].shape[3] // 2
        KH = KW = 1
        C = xs[0].shape[1]
        # torch channel c*4 + p1*2 + p2 -> K = (p1*2+p2)*C + c
        wp = w.reshape(Cout, C, 4).permute(0, 2, 1).reshape(Cout, 4 * C).contiguous().to(torch.bfloat16)
    out = torch.empty(N, H, W, Cout, device="cuda", dtype=torch.bfloat16)
    res = nhwc_bf16(residual) if residual is not None else None
    gn = torch.zeros(N, 8, 2, device="cuda", dtype=torch.float64) if stats else None
    L.check(lib.fd_conv_igemm(L.ptr(srcs[0]), srcs[0].shape[-1], L.ptr(srcs[1]) if len(srcs) > 1 else None,
                              srcs[1].shape[-1] if len(srcs) > 1 else 0, L.ptr(wp), L.ptr(bias), L.ptr(res),
                              L.ptr(out), L.ptr(gn), N, H, W, Cout, KH, KW, pad[0], pad[1], mode, L.stream()))
    torch.cuda.synchronize()
    return out.permute(0, 3, 1, 2).float(), gn


def ref_conv(xs, w, bias, pad, residual=None, mode=0):
    x = torch.cat([t.to(torch.bfloat16).float() for t in xs], 1)
    wq = w.to(torch.bfloat16).float()
    if mode == 1:
        b, c, H, W = x.shape
        x = x.reshape(b, c, H // 2, 2, W // 2, 2).permute(0, 1, 3, 5, 2, 4).reshape(b, c * 4, H // 2, W // 2)
    y = F.conv2d(x, wq, bias, padding=pad)
    if residual is not None:
        y = y + residual.to(torch.bfloat16).float()
    return y


def close(out, ref):
    err = (out - ref).abs()
    tol = 2e-2 * ref.abs().clamp(min=1.0)   # bf16 output rounding is 2^-9 relative; K up to 7k
    assert bool((err <= tol).all()), f"max err {err.max().item()} at ref scale {ref.abs().max().item()}"
    # and much tighter on average
    assert err.mean().item() < 4e-3 * ref.abs().mean().clamp(min=0.1).item()


CASES = [
    # N, Cins, Cout, H, W, k, pad, bias, residual, stats
    (2, (64,), 64, 16, 128, (3, 3), (1, 1), True, False, True),
    (1, (64,), 64, 3, 128, (3, 3), (1, 1), True, False, False),
    (2, (64, 64), 128, 12, 24, (3, 3), (1, 1), True, False, True),
    (2, (128, 64), 128, 8, 16, (3, 3), (1, 1), True, False, True),
    (2, (64,), 384, 10, 12, (1, 1), (0, 0), False, False, False),
    (2, (128,), 64, 10, 12, (1, 1), (0, 0), True, True, False),
    (1, (64,), 64, 20, 40, (7, 1), (3, 0), True, False, False),
    (2, (512,), 256, 2, 3, (3, 3), (1, 1), True, False, False),
    (2, (512, 256), 512, 4, 6, (3, 3), (1, 1), True, False, True),
    (1, (256,), 256, 33, 70, (3, 3), (1, 1), True, False, True),
    (2, (64,), 64, 220, 512, (3, 3), (1, 1), True, False, True),
    (2, (64, 64), 64, 21, 256, (3, 3), (1, 1), True, False, True),      # rolling-strip kernel, two sources
    (1, (128,), 64, 70, 200, (3, 3), (1, 1), True, False, False),       # rolling-strip kernel, 128-channel source, ragged W
    (2, (64,), 64, 37, 130, (3, 3), (1, 1), True, False, True),         # ragged W: second column block is 2 pixels wide
    (2, (256,), 256, 24, 40, (3, 3), (1, 1), True, False, True),        # CTA-pair kernel (cta_group::2), statistics, one N-tile
    (4, (384,), 512, 12, 20, (3, 3), (1, 1), True, False, True),        # CTA-pair kernel, two N-tiles, ragged tiles
    (2, (512, 256), 512, 8, 16, (1, 1), (0, 0), True, True, False),     # CTA-pair kernel, 1x1 with 12 K-blocks + residual
    (2, (256,), 768, 10, 24, (3, 3), (1, 1), False, False, False),      # CTA-pair kernel, three N-tiles, no bias
    (2, (128, 64), 128, 20, 48, (3, 3), (1, 1), True, False, True),     # CTA-pair kernel with N = 128 tiles, two sources
    (2, (128,), 128, 9, 30, (3, 3), (1, 1), True, True, False),         # ... N = 128, residual
    (2, (64,), 64, 30, 256, (3, 3), (1, 1), True, True, True),          # rolling-strip kernel with a residual (dgrad accumulation)
    (1, (64, 64), 64, 9, 130, (3, 3), (1, 1), False, True, False),      # two passes: caller's residual, then the partial sum
    (2, (128,), 128, 32, 64, (3, 3), (1, 1), True, False, True),        # N = 128 CTA pairs, two M-tiles per CTA (32 M-tiles)
    (2, (64, 64), 128, 16, 128, (3, 3), (1, 1), True, True, True),      # ... two sources + residual
    (1, (128,), 128, 24, 64, (3, 3), (1, 1), True, False, True),        # 12 M-tiles: one M-tile per CTA (count % 4 != 0 is 0 here -> 2 per CTA), 3 super-tiles
    (1, (128,), 128, 20, 64, (3, 3), (1, 1), False, False, False),      # 10 M-tiles: % 4 != 0 -> one M-tile per CTA
    (2, (64,), 64, 37, 256, (3, 3), (1, 1), True, False, True),         # rolling-strip kernel (A operand in tensor memory)
    (1, (64, 64), 64, 21, 200, (3, 3), (1, 1), True, True, True),       # ... two passes, ragged last column block, residual
    (3, (128,), 64, 5, 130, (3, 3), (1, 1), True, False, False),        # ... fewer rows than CTAs: some ranges are one row
]


@pytest.mark.parametrize("case", CASES)
def test_conv_igemm(L, case):
    N, cins, Cout, H, W, k, pad, has_bias, has_res, stats = case
    g = torch.Generator().manual_seed(hash(case) % 1000)
    xs = [torch.randn(N, c, H, W, generator=g).cuda() for c in cins]
    cin = sum(cins)
    w = (torch.randn(Cout, cin, k[0], k[1], generator=g) / (cin * k[0] * k[1]) ** 0.5).cuda()
    bias = torch.randn(Cout, generator=g).cuda() if has_bias else None
    res = torch.randn(N, Cout, H, W, generator=g).cuda() if has_res else None
    out, gn = run_conv(L, xs, w, bias, pad, res, stats)
    ref = ref_conv(xs, w, bias, pad, res)
    close(out, ref)
    out2, gn2 = run_conv(L, xs, w, bias, pad, res, stats)
    assert torch.equal(out, out2)                      # run-to-run bit-stable
    if stats:
        assert torch.allclose(gn, gn2, rtol=1e-12, atol=1e-9)
        r = ref.double().reshape(N, 8, -1)
        s = torch.stack((r.sum(-1), (r * r).sum(-1)), -1)
        assert torch.allclose(gn, s, rtol=1e-3, atol=1e-2 * r.shape[-1] ** 0.5), (gn - s).abs().max()


@pytest.mark.parametrize("case", [(2, 64, 128, 8, 12), (1, 128, 256, 32, 64), (2, 256, 512, 3, 5)])
def test_conv_pixel_unshuffle(L, case):
    N, C, Cout, H, W = case
    g = torch.Generator().manual_seed(C + H)
    x = torch.randn(N, C, 2 * H, 2 * W, generator=g).cuda()
    w = (torch.randn(Cout, 4 * C, 1, 1, generator=g) / (4 * C) ** 0.5).cuda()
    bias = torch.randn(Cout, generator=g).cuda()
    out, _ = run_conv(L, [x], w, bias, (0, 0), mode=1)
    close(out, ref_conv([x], w, bias, (0, 0), mode=1))


@pytest.mark.parametrize("case", [(2, 37, 256, True), (1, 21, 200, False), (3, 5, 130, True), (1, 70, 64, True)])
def test_strip_conv_fused_groupnorm_input(L, case):
    """fd_conv3x3_gnsilu_in = fd_gn_silu (GroupNorm affine + scale/shift + SiLU, Block.forward :176-187) fused into the 64 -> 64
    strip convolution that consumes it, against the two-pass form (same folded coefficients on the strip in shared memory; rows /
    pixels outside the image stay zero = padding of the ACTIVATED tensor)."""
    lib = L.load()
    N, H, W, use_ss = case
    g = torch.Generator().manual_seed(H * W + N)
    x = (torch.randn(N, H, W, 64, generator=g) * 1.5 + 0.3).to(torch.bfloat16).cuda()
    w = (torch.randn(64, 64, 3, 3, generator=g) / 24.0).cuda()
    wp = pack_w(w)
    bias = torch.randn(64, generator=g).cuda()
    gamma, beta = torch.randn(64, generator=g).cuda(), torch.randn(64, generator=g).cuda()
    ss = (torch.randn(N, 192, generator=g) * 0.5).cuda() if use_ss else None
    ss_ptr = ss.data_ptr() + 4 * 32 if use_ss else None          # (scale | shift) rows start at an offset, as in the UNet
    r = x.float().permute(0, 3, 1, 2).double().reshape(N, 8, -1)
    in_stats = torch.stack((r.sum(-1), (r * r).sum(-1)), -1).contiguous()
    # two passes
    act = torch.empty_like(x)
    L.check(lib.fd_gn_silu(L.ptr(x), L.ptr(in_stats), L.ptr(gamma), L.ptr(beta), ss_ptr, 192 if use_ss else 0, None, L.ptr(act),
                           N, H * W, 64, 1e-5, L.stream()))
    ref = torch.empty(N, H, W, 64, device="cuda", dtype=torch.bfloat16)
    gn_ref = torch.zeros(N, 8, 2, device="cuda", dtype=torch.float64)
    L.check(lib.fd_conv_igemm(L.ptr(act), 64, None, 0, L.ptr(wp), L.ptr(bias), None, L.ptr(ref), L.ptr(gn_ref), N, H, W, 64, 3, 3,
                              1, 1, 0, L.stream()))
    # fused
    out = torch.empty_like(ref)
    gn = torch.zeros_like(gn_ref)
    L.check(lib.fd_conv3x3_gnsilu_in(L.ptr(x), L.ptr(in_stats), L.ptr(gamma), L.ptr(beta), ss_ptr, 192 if use_ss else 0, 1e-5,
                                     L.ptr(wp), L.ptr(bias), None, L.ptr(out), L.ptr(gn), N, H, W, L.stream()))
    torch.cuda.synchronize()
    # the in-kernel SiLU uses tanh.approx (one MUFU op) instead of ex2 + rcp: the activation differs from fd_gn_silu's by
    # < 2^-10 relative before its bf16 rounding, i.e. an occasional 1-ulp flip of a conv input -> compare at that level
    err = (out.float() - ref.float()).abs()
    assert err.max().item() <= 2.5e-2 * ref.float().abs().max().item() and err.mean().item() <= 1e-3 * ref.float().abs().mean().item(), \
        (err.max().item(), err.mean().item())
    assert torch.allclose(gn, gn_ref, rtol=2e-3, atol=0.5)
    # and against torch on the same bf16-rounded activation
    y = F.conv2d(act.float().permute(0, 3, 1, 2), w.to(torch.bfloat16).float(), bias, padding=1)
    close(out.permute(0, 3, 1, 2).float(), y)


@pytest.mark.parametrize("shape", [(2, 64, 64, 64, 37, 150), (1, 128, 64, 128, 22, 64), (2, 256, 128, 256, 11, 32),
                                   (1, 512, 256, 512, 7, 16), (8, 64, 64, 64, 16, 128)])
def test_conv_residual_groupnorm_epilogue(L, shape):
    """fd_conv_igemm_rt: out = conv1x1(cat(x0, x1)) + silu(GroupNorm(h2)) with block2's GroupNorm apply folded into the
    res_conv's epilogue (ResnetBlock.forward :212-214) == the two-pass form (fd_gn_silu, then the conv with a residual) and
    == fp32 torch.  Statistics of h2 come from a producing conv (its epilogue accumulates them), like in the UNet."""
    lib = L.load()
    N, C0, C1, Cout, H, W = shape
    g = torch.Generator().manual_seed(Cout + H)
    x0 = torch.randn(N, C0, H, W, generator=g).cuda()
    x1 = torch.randn(N, C1, H, W, generator=g).cuda()
    w = (torch.randn(Cout, C0 + C1, 1, 1, generator=g) / (C0 + C1) ** 0.5).cuda()
    bias = torch.randn(Cout, generator=g).cuda()
    gamma = (torch.randn(Cout, generator=g) * 0.3 + 1).cuda()
    beta = (torch.randn(Cout, generator=g) * 0.2).cuda()
    # h2 and its statistics from a producing 3x3 conv
    a1 = torch.randn(N, Cout, H, W, generator=g).cuda()
    w2 = (torch.randn(Cout, Cout, 3, 3, generator=g) / (9 * Cout) ** 0.5 * 1.5).cuda()
    b2 = torch.randn(Cout, generator=g).cuda() * 0.1
    h2, st2 = run_conv(L, [a1], w2, b2, (1, 1), stats=True)
    h2q = nhwc_bf16(h2)
    s0, s1 = nhwc_bf16(x0), nhwc_bf16(x1)
    wp = pack_w(w)
    out = torch.empty(N, H, W, Cout, device="cuda", dtype=torch.bfloat16)
    L.check(lib.fd_conv_igemm_rt(L.ptr(s0), C0, L.ptr(s1), C1, L.ptr(wp), L.ptr(bias), L.ptr(h2q), L.ptr(st2), L.ptr(gamma),
                                 L.ptr(beta), 1e-5, L.ptr(out), N, H, W, Cout, 1, 1, 0, 0, L.stream()))
    # two-pass form
    a2 = torch.empty_like(h2q)
    L.check(lib.fd_gn_silu(L.ptr(h2q), L.ptr(st2), L.ptr(gamma), L.ptr(beta), None, 0, None, L.ptr(a2), N, H * W, Cout, 1e-5,
                           L.stream()))
    two = torch.empty_like(out)
    L.check(lib.fd_conv_igemm(L.ptr(s0), C0, L.ptr(s1), C1, L.ptr(wp), L.ptr(bias), L.ptr(a2), L.ptr(two), None, N, H, W, Cout,
                              1, 1, 0, 0, 0, L.stream()))
    torch.cuda.synchronize()
    got, two = out.permute(0, 3, 1, 2).float(), two.permute(0, 3, 1, 2).float()
    ref = ref_conv([x0, x1], w, bias, (0, 0)) + F.silu(F.group_norm(h2q.permute(0, 3, 1, 2).float(), 8, gamma, beta, eps=1e-5))
    scale = ref.abs().max().item()
    assert (got - ref).abs().max().item() <= 1.2e-2 * scale, ((got - ref).abs().max().item(), scale)
    assert (got - two).abs().max().item() <= 1.6e-2 * scale          # the two-pass form rounds the activated tensor to bf16
    assert (got - ref).abs().mean().item() <= 2e-3 * ref.abs().mean().item() + 1e-6


@pytest.mark.parametrize("shape", [(2, 64, 64, 24, 40, 21, 37, 2, 1, 2), (1, 64, 64, 16, 136, 16, 136, 0, 0, 2),
                                   (3, 64, 64, 9, 20, 5, 20, 3, 0, 3), (1, 128, 0, 40, 72, 33, 70, 7, 2, 1)])
def test_conv_residual_groupnorm_output_head(L, shape):
    """fd_conv_igemm_rt_head: the UNet's tail (final ResnetBlock's res_conv + silu(GroupNorm(h2)), final_conv 1x1, un-pad crop;
    Unet.forward :414-417 + InputPadder.unpad) in one launch == fd_conv_igemm_rt followed by fd_final_conv_crop (which reads the
    bf16-rounded activation: the fused head uses the fp32 tile, so it is the closer of the two to fp32 torch) == fp32 torch."""
    lib = L.load()
    N, C0, C1, H, W, H0, W0, pt, pl, nout = shape
    g = torch.Generator().manual_seed(H * W + nout)
    x0 = torch.randn(N, C0, H, W, generator=g).cuda()
    x1 = torch.randn(N, C1, H, W, generator=g).cuda() if C1 else None
    w = (torch.randn(64, C0 + C1, 1, 1, generator=g) / (C0 + C1) ** 0.5).cuda()
    bias = torch.randn(64, generator=g).cuda()
    gamma = (torch.randn(64, generator=g) * 0.3 + 1).cuda()
    beta = (torch.randn(64, generator=g) * 0.2).cuda()
    hw_ = (torch.randn(nout, 64, 1, 1, generator=g) / 8).cuda()
    hb = torch.randn(nout, generator=g).cuda()
    a1 = torch.randn(N, 64, H, W, generator=g).cuda()
    w2 = (torch.randn(64, 64, 3, 3, generator=g) / (9 * 64) ** 0.5 * 1.5).cuda()
    b2 = torch.randn(64, generator=g).cuda() * 0.1
    h2, st2 = run_conv(L, [a1], w2, b2, (1, 1), stats=True)
    h2q = nhwc_bf16(h2)
    s0 = nhwc_bf16(x0)
    s1 = nhwc_bf16(x1) if C1 else None
    wp = pack_w(w)
    got = torch.full((N, nout, H0, W0), float("nan"), device="cuda")
    L.check(lib.fd_conv_igemm_rt_head(L.ptr(s0), C0, L.ptr(s1), C1, L.ptr(wp), L.ptr(bias), L.ptr(h2q), L.ptr(st2), L.ptr(gamma),
                                      L.ptr(beta), 1e-5, L.ptr(hw_), L.ptr(hb), nout, L.ptr(got), N, H, W, H0, W0, pt, pl, L.stream()))
    mid = torch.empty(N, H, W, 64, device="cuda", dtype=torch.bfloat16)
    L.check(lib.fd_conv_igemm_rt(L.ptr(s0), C0, L.ptr(s1), C1, L.ptr(wp), L.ptr(bias), L.ptr(h2q), L.ptr(st2), L.ptr(gamma),
                                 L.ptr(beta), 1e-5, L.ptr(mid), N, H, W, 64, 1, 1, 0, 0, L.stream()))
    two = torch.empty_like(got)
    L.check(lib.fd_final_conv_crop(L.ptr(mid), L.ptr(hw_), L.ptr(hb), L.ptr(two), N, H, W, 64, nout, pt, pl, H0, W0, L.stream()))
    torch.cuda.synchronize()
    assert torch.isfinite(got).all()                     # every pixel of the window was written
    full = ref_conv([x0] + ([x1] if C1 else []), w, bias, (0, 0)) + \
        F.silu(F.group_norm(h2q.permute(0, 3, 1, 2).float(), 8, gamma, beta, eps=1e-5))
    ref = F.conv2d(full, hw_, hb)[:, :, pt:pt + H0, pl:pl + W0]
    scale = ref.abs().max().item()
    e_got, e_two = (got - ref).abs().max().item(), (two - ref).abs().max().item()
    assert e_got <= 6e-3 * scale, (e_got, scale)         # bf16 inputs / weights of the 1x1 conv, tanh.approx SiLU; no output rounding
    assert (got - two).abs().max().item() <= 1.2e-2 * scale
    assert (got - ref).abs().mean().item() <= max(1.5 * (two - ref).abs().mean().item(), 1e-3 * scale), (e_got, e_two)
    again = torch.empty_like(got)
    L.check(lib.fd_conv_igemm_rt_head(L.ptr(s0), C0, L.ptr(s1), C1, L.ptr(wp), L.ptr(bias), L.ptr(h2q), L.ptr(st2), L.ptr(gamma),
                                      L.ptr(beta), 1e-5, L.ptr(hw_), L.ptr(hb), nout, L.ptr(again), N, H, W, H0, W0, pt, pl, L.stream()))
    torch.cuda.synchronize()
    assert torch.equal(got, again)                       # no atomics on this path: bit-stable


@pytest.mark.parametrize("shape", [(2, 64, 64, 9, 20), (1, 128, 64, 22, 64), (2, 256, 128, 11, 32), (1, 512, 256, 7, 16),
                                   (1, 64, 64, 6, 130), (3, 64, 128, 5, 13)])
def test_upsample_conv_phase_decomposition(L, shape):
    """fd_conv_igemm_up: Upsample = nearest x2 + conv3x3(pad 1) (denoising_diffusion.py:89-93) computed as four 2x2 phase
    convolutions on the low-resolution tensor == conv3x3 on the materialised up-sampled tensor (torch fp32, bf16-rounded
    input and weights).  The phase weights are sums of up to four fp32 weights rounded ONCE to bf16, so the tolerance is the
    bf16 weight rounding (2^-9 relative per product) on top of the output rounding: max |err| <= 1.5e-2 of the output scale."""
    lib = L.load()
    N, Cin, Cout, H, W = shape
    g = torch.Generator().manual_seed(Cin + H)
    x = torch.randn(N, Cin, H, W, generator=g).cuda()
    w = (torch.randn(Cout, Cin, 3, 3, generator=g) / (9 * Cin) ** 0.5).cuda()
    bias = torch.randn(Cout, generator=g).cuda()
    w4 = torch.empty(4, Cout, 4 * Cin, device="cuda", dtype=torch.bfloat16)
    L.check(lib.fd_prep_weight_upconv(L.ptr(w), L.ptr(w4), Cout, Cin, L.stream()))
    xs = nhwc_bf16(x)
    out = torch.full((N, 2 * H, 2 * W, Cout), float("nan"), device="cuda", dtype=torch.bfloat16)
    L.check(lib.fd_conv_igemm_up(L.ptr(xs), Cin, L.ptr(w4), L.ptr(bias), L.ptr(out), N, H, W, Cout, L.stream()))
    torch.cuda.synchronize()
    got = out.permute(0, 3, 1, 2).float()
    assert torch.isfinite(got).all()                     # every output pixel of every phase was written
    up = F.interpolate(x.to(torch.bfloat16).float(), scale_factor=2, mode="nearest")
    ref = F.conv2d(up, w, bias, padding=1)
    scale = ref.abs().max().item()
    err = (got - ref).abs().max().item()
    assert err <= 1.5e-2 * scale, (err, scale)
    assert (got - ref).abs().mean().item() <= 2.5e-3 * ref.abs().mean().item() + 1e-6
