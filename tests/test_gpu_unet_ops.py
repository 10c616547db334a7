"""-m gpu: the memory-bound UNet kernels and the two attention cores against fp32 torch
restatements of the reference ops (oracle/flowdiff_oracle.py) on bf16-rounded inputs."""
import math

import pytest
import torch
import torch.nn.functional as F

from oracle import flowdiff_oracle as O

pytestmark = pytest.mark.gpu
BF = torch.bfloat16


@pytest.fixture(scope="module")
def L():
    from opticalflowdiffusion_b200 import _lib
    _lib.load(check_device=True)
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    return _lib


def nhwc(x):
    return x.permute(0, 2, 3, 1).contiguous().to(BF)


def nchw(x):
    return x.permute(0, 3, 1, 2).float()


def rel_err(a, b):
    return ((a - b).abs().max() / b.abs().max().clamp(min=1e-6)).item()


@pytest.mark.parametrize("C", [64, 128, 256, 512])
def test_gn_silu(L, C):
    lib = L.load()
    g = torch.Generator().manual_seed(C)
    N, H, W = 2, 6, 10
    x = (torch.randn(N, C, H, W, generator=g) * 2 + 0.5).to(BF).float().cuda()
    gamma, beta = torch.randn(C, generator=g).cuda(), torch.randn(C, generator=g).cuda()
    ss = torch.randn(N, 3 * C, generator=g).cuda()      # row stride 3C, block at offset C//2
    off = C // 2
    res = torch.randn(N, C, H, W, generator=g).to(BF).float().cuda()
    r = x.double().reshape(N, 8, -1)
    stats = torch.stack((r.sum(-1), (r * r).sum(-1)), -1).contiguous()
    xh, rh = nhwc(x), nhwc(res)      # keep the NHWC copies alive while the kernels run
    for use_ss, use_res in ((True, False), (False, True), (False, False)):
        out = torch.empty(N, H, W, C, device="cuda", dtype=BF)
        L.check(lib.fd_gn_silu(L.ptr(xh), L.ptr(stats), L.ptr(gamma), L.ptr(beta),
                               ss.data_ptr() + 4 * off if use_ss else None, 3 * C, L.ptr(rh) if use_res else None,
                               L.ptr(out), N, H * W, C, 1e-5, L.stream()))
        y = F.group_norm(x, 8, gamma, beta, eps=1e-5)
        if use_ss:
            sc, sh = ss[:, off:off + C], ss[:, off + C:off + 2 * C]
            y = y * (sc[:, :, None, None] + 1) + sh[:, :, None, None]
        y = F.silu(y)
        if use_res:
            y = y + res
        assert rel_err(nchw(out), y) < 1e-2


@pytest.mark.parametrize("C", [64, 128, 256, 512])
def test_chan_layernorm(L, C):
    lib = L.load()
    g = torch.Generator().manual_seed(C + 1)
    N, H, W = 2, 5, 7
    x = (torch.randn(N, C, H, W, generator=g) * 3 + 1).to(BF).float().cuda()
    gain = torch.randn(1, C, 1, 1, generator=g).cuda()
    res = torch.randn(N, C, H, W, generator=g).to(BF).float().cuda()
    xh, rh = nhwc(x), nhwc(res)
    for use_res in (False, True):
        out = torch.empty(N, H, W, C, device="cuda", dtype=BF)
        L.check(lib.fd_chan_layernorm(L.ptr(xh), L.ptr(gain), L.ptr(rh) if use_res else None, L.ptr(out),
                                      N * H * W, C, 1e-5, L.stream()))
        y = O._chan_layernorm(x, gain) + (res if use_res else 0)
        assert rel_err(nchw(out), y) < 1e-2


def test_upsample_and_layouts(L):
    lib = L.load()
    x = torch.randn(2, 64, 3, 5).to(BF).float().cuda()
    out = torch.empty(2, 6, 10, 64, device="cuda", dtype=BF)
    xh = nhwc(x)
    L.check(lib.fd_upsample2x(L.ptr(xh), L.ptr(out), 2, 3, 5, 64, L.stream()))
    assert torch.equal(nchw(out), F.interpolate(x, scale_factor=2, mode="nearest"))
    a = torch.empty(2, 3, 5, 64, device="cuda", dtype=BF)
    L.check(lib.fd_nchw_to_nhwc_bf16(L.ptr(x), L.ptr(a), 2, 64, 15, L.stream()))
    assert torch.equal(a, nhwc(x))
    b = torch.empty(2, 64, 3, 5, device="cuda")
    L.check(lib.fd_nhwc_bf16_to_nchw(L.ptr(a), L.ptr(b), 2, 64, 15, L.stream()))
    assert torch.equal(b, x)


def test_time_embed_and_proj(L):
    lib = L.load()
    g = torch.Generator().manual_seed(4)
    sd = {"time_mlp.1.weight": torch.randn(256, 64, generator=g) * 0.1, "time_mlp.1.bias": torch.randn(256, generator=g),
          "time_mlp.3.weight": torch.randn(256, 256, generator=g) * 0.05, "time_mlp.3.bias": torch.randn(256, generator=g)}
    t = torch.tensor([0, 1, 17, 500, 999])
    ref = O.time_embedding(sd, t)
    c = {k: v.cuda() for k, v in sd.items()}
    temb = torch.empty(5, 256, device="cuda")
    tc = t.cuda()
    L.check(lib.fd_time_embed(L.ptr(tc), L.ptr(c["time_mlp.1.weight"]), L.ptr(c["time_mlp.1.bias"]),
                              L.ptr(c["time_mlp.3.weight"]), L.ptr(c["time_mlp.3.bias"]), L.ptr(temb), 5, 64, 256, L.stream()))
    assert torch.allclose(temb.cpu(), ref, rtol=1e-3, atol=2e-3), (temb.cpu() - ref).abs().max()
    w, b = (torch.randn(384, 256, generator=g) * 0.05).cuda(), torch.randn(384, generator=g).cuda()
    out = torch.empty(5, 384, device="cuda")
    L.check(lib.fd_time_proj(L.ptr(temb), L.ptr(w), L.ptr(b), L.ptr(out), 5, 256, 384, L.stream()))
    assert torch.allclose(out, F.linear(F.silu(temb), w, b), rtol=1e-4, atol=1e-4)


@pytest.mark.parametrize("nan_mask", [False, True])
def test_pack_input_and_init_conv_weights(L, nan_mask):
    """pack_input + kind-2 weight packing + 7x1 implicit GEMM == 7x7 conv (denoising_diffusion.py:297)."""
    lib = L.load()
    g = torch.Generator().manual_seed(9)
    B, Cx, Cc, H, W = 2, 5 if nan_mask else 2, 3, 16, 24
    x = torch.randn(B, Cx, H, W, generator=g)
    if nan_mask:
        x[0, 1, 2, 3] = float("nan")
        x[1, 4, 15, 23] = float("nan")
    cond = torch.rand(B, Cc, H, W, generator=g)
    Ctot = Cx + int(nan_mask) + Cc
    w = torch.randn(64, Ctot, 7, 7, generator=g) / (Ctot * 49) ** 0.5
    bias = torch.randn(64, generator=g)
    packed = torch.empty(B, H, W, 64, device="cuda", dtype=BF)
    xc, cc, wc, bc = x.cuda(), cond.cuda(), w.cuda(), bias.cuda()
    L.check(lib.fd_pack_input(L.ptr(xc), L.ptr(cc), L.ptr(packed), B, Cx, Cc, H, W, int(nan_mask), L.stream()))
    wp = torch.empty(64, 7 * 64, device="cuda", dtype=BF)
    L.check(lib.fd_prep_weight(L.ptr(wc), L.ptr(wp), 64, Ctot, 7, 7, 2, 0, 0.0, L.stream()))
    out = torch.empty(B, H, W, 64, device="cuda", dtype=BF)
    L.check(lib.fd_conv_igemm(L.ptr(packed), 64, None, 0, L.ptr(wp), L.ptr(bc), None, L.ptr(out), None, B, H, W,
                              64, 7, 1, 3, 0, 0, L.stream()))
    xin = x.clone()
    if nan_mask:
        nans = torch.isnan(xin)
        xin[nans] = 0
        xin = torch.cat((xin, torch.any(nans, 1, keepdim=True).float()), 1)
    full = torch.cat((xin, cond), 1).to(BF).float()
    ref = F.conv2d(full, w.to(BF).float(), bias, padding=3)
    assert rel_err(nchw(out).cpu(), ref) < 1.5e-2


@pytest.mark.parametrize("kind", [0, 1])
def test_prep_weight_standardize(L, kind):
    lib = L.load()
    g = torch.Generator().manual_seed(kind)
    if kind == 0:
        w = torch.randn(128, 192, 3, 3, generator=g) * 0.3 + 0.1
        flat = w.reshape(128, -1)
        ws = (w - flat.mean(1).view(-1, 1, 1, 1)) * (flat.var(1, unbiased=False).view(-1, 1, 1, 1) + 1e-5).rsqrt()
        ref = ws.permute(0, 2, 3, 1).reshape(128, -1)
        std = 1
    else:
        w = torch.randn(128, 256, 1, 1, generator=g)
        C = 64
        ref = w.reshape(128, C, 4).permute(0, 2, 1).reshape(128, 256)
        std = 0
    out = torch.empty(ref.shape, device="cuda", dtype=BF)
    co, ci, kh, kw = w.shape
    wc = w.cuda()
    L.check(lib.fd_prep_weight(L.ptr(wc), L.ptr(out), co, ci, kh, kw, kind, std, 1e-5, L.stream()))
    assert torch.allclose(out.float().cpu(), ref.to(BF).float(), rtol=1e-2, atol=1e-3)


def test_final_conv(L):
    lib = L.load()
    g = torch.Generator().manual_seed(2)
    x = torch.randn(2, 64, 6, 9, generator=g).to(BF).float().cuda()
    w, b = torch.randn(2, 64, 1, 1, generator=g).cuda(), torch.randn(2, generator=g).cuda()
    out = torch.empty(2, 2, 6, 9, device="cuda")
    xh = nhwc(x)
    L.check(lib.fd_final_conv(L.ptr(xh), L.ptr(w), L.ptr(b), L.ptr(out), 2, 54, 64, 2, L.stream()))
    assert torch.allclose(out, F.conv2d(x, w, b), rtol=1e-4, atol=1e-4)


def _attn_ref(qkv, linear):
    """qkv (N, 384, H, W) fp32 -> (N, 128, H, W): the core of LinearAttention / Attention (to_qkv/to_out excluded)."""
    b, _, h, w = qkv.shape
    q, k, v = (t.reshape(b, 4, 32, h * w) for t in qkv.chunk(3, dim=1))
    if linear:
        q = q.softmax(dim=-2) * 32 ** -0.5
        k = k.softmax(dim=-1)
        v = v / (h * w)
        ctx = torch.einsum("bhdn,bhen->bhde", k, v)
        out = torch.einsum("bhde,bhdn->bhen", ctx, q)
        return out.reshape(b, 128, h, w)
    q = q * 32 ** -0.5
    sim = torch.einsum("bhdi,bhdj->bhij", q, k)
    out = torch.einsum("bhij,bhdj->bhid", sim.softmax(dim=-1), v)
    return out.permute(0, 1, 3, 2).reshape(b, 128, h, w)


@pytest.mark.parametrize("hw", [(2, 3), (8, 8), (16, 24), (55, 128), (100, 130)])
def test_linear_attention_core(L, hw):
    lib = L.load()
    H, W = hw
    g = torch.Generator().manual_seed(H * W)
    N = 2
    qkv = (torch.randn(N, 384, H, W, generator=g) * 1.5).to(BF).float().cuda()
    out = torch.empty(N, H, W, 128, device="cuda", dtype=BF)
    ws = torch.empty(lib.fd_linattn_workspace_floats(N, H * W), device="cuda")
    qh = nhwc(qkv)
    L.check(lib.fd_linattn(L.ptr(qh), L.ptr(out), L.ptr(ws), N, H * W, L.stream()))
    ref = _attn_ref(qkv, True)
    assert rel_err(nchw(out), ref) < 1.5e-2


@pytest.mark.parametrize("hw", [(2, 3), (8, 8), (5, 13), (16, 24), (55, 128)])
def test_full_attention_core(L, hw):
    lib = L.load()
    H, W = hw
    g = torch.Generator().manual_seed(H * W + 1)
    N = 2
    qkv = (torch.randn(N, 384, H, W, generator=g) * 1.5).to(BF).float().cuda()
    out = torch.empty(N, H, W, 128, device="cuda", dtype=BF)
    qh = nhwc(qkv)
    L.check(lib.fd_attention(L.ptr(qh), L.ptr(out), N, H * W, L.stream()))
    ref = _attn_ref(qkv, False)
    assert rel_err(nchw(out), ref) < 2e-2


@pytest.mark.parametrize("C", [64, 128])
@pytest.mark.parametrize("nhw", [(2, 9, 14), (1, 40, 72), (3, 16, 128), (8, 24, 64)])
def test_linear_attention_block_tcgen05(L, C, nhw):
    """fd_linattn_tc (tcgen05 / TMEM / TMA, two passes over x, no intermediate tensor) == the oracle's
    Residual(PreNorm(LinearAttention)) block (denoising_diffusion.py:81-87,127-135,216-244).  Shapes: a single ragged tile,
    several tiles per CTA with a ragged last one, several samples, more samples than fit one CTA range each.
    Tolerance: relative L2 <= 2e-2 (bf16 operands: x, the scaled q / k weights, exp(k), softmax(q), the folded context)."""
    lib = L.load()
    N, H, W = nhw
    g = torch.Generator().manual_seed(C + H * W)
    x = (torch.randn(N, C, H, W, generator=g) * 1.5 + 0.3).to(BF).float()
    sd = {"norm.g": torch.randn(1, C, 1, 1, generator=g) * 0.3 + 1,
          "fn.to_qkv.weight": torch.randn(384, C, 1, 1, generator=g) / C ** 0.5 * 2.0,
          "fn.to_out.0.weight": torch.randn(C, 128, 1, 1, generator=g) / 128 ** 0.5 * 30,
          "fn.to_out.0.bias": torch.randn(C, generator=g) * 0.1,
          "fn.to_out.1.g": torch.randn(1, C, 1, 1, generator=g) * 0.3 + 1}
    ref = O._linear_attention(sd, "", x)
    xc = nhwc(x.cuda())
    wqkv = sd["fn.to_qkv.weight"].reshape(384, C).contiguous().cuda()
    g1, g2 = sd["norm.g"].reshape(C).contiguous().cuda(), sd["fn.to_out.1.g"].reshape(C).contiguous().cuda()
    wout, bout = sd["fn.to_out.0.weight"].reshape(C, 128).contiguous().cuda(), sd["fn.to_out.0.bias"].cuda()
    wq, wk = torch.empty(128, C, device="cuda", dtype=BF), torch.empty(128, C, device="cuda", dtype=BF)
    sq, sk, mk = (torch.empty(128, device="cuda") for _ in range(3))
    wv = torch.empty(128, C, device="cuda")
    L.check(lib.fd_linattn_tc_prep(L.ptr(wqkv), L.ptr(g1), L.ptr(wq), L.ptr(sq), L.ptr(wk), L.ptr(sk), L.ptr(mk), L.ptr(wv), C,
                                   L.stream()))
    # the softmax shift is an upper bound of every k logit (Cauchy-Schwarz on the LayerNorm output)
    y = O._chan_layernorm(x, sd["norm.g"])
    k = torch.einsum("jc,nchw->njhw", wqkv[128:256].cpu(), y) * 1.4426950408889634
    assert bool((k.amax(dim=(0, 2, 3)) <= mk.cpu() + 1e-3).all())
    out = torch.empty_like(xc)
    ws = torch.empty(lib.fd_linattn_tc_workspace_floats(N, H * W, C), device="cuda")
    L.check(lib.fd_linattn_tc(L.ptr(xc), L.ptr(wk), L.ptr(sk), L.ptr(mk), L.ptr(wq), L.ptr(sq), L.ptr(wv), L.ptr(wout), L.ptr(bout),
                              L.ptr(g2), L.ptr(out), L.ptr(ws), N, H * W, C, 1e-5, L.stream()))
    torch.cuda.synchronize()
    got = nchw(out).cpu()
    assert torch.isfinite(got).all()
    err = rel_err(got, ref)
    # the attention branch alone (the residual x dominates the norm of the block's output)
    err_branch = rel_err(got - x, ref - x)
    print(f"C={C} {nhw}: rel L2 {err:.3e}, attention branch {err_branch:.3e}")
    assert err < 2e-2 and err_branch < 4e-2
    out2 = torch.empty_like(xc)
    L.check(lib.fd_linattn_tc(L.ptr(xc), L.ptr(wk), L.ptr(sk), L.ptr(mk), L.ptr(wq), L.ptr(sq), L.ptr(wv), L.ptr(wout), L.ptr(bout),
                              L.ptr(g2), L.ptr(out2), L.ptr(ws), N, H * W, C, 1e-5, L.stream()))
    assert torch.equal(out, out2)          # fixed-order reductions: run-to-run bit-stable
