"""-m gpu: the CUDA warp / splat / loss kernels (through the C ABI) against the oracle and the
reference-generated golden vectors."""
import numpy as np
import pytest
import torch

from oracle import flowdiff_oracle as O

pytestmark = pytest.mark.gpu


def T(a):
    return torch.from_numpy(np.asarray(a))


@pytest.fixture(scope="module")
def W():
    from opticalflowdiffusion_b200 import _lib, warp
    _lib.load(check_device=True)
    return warp


def test_backwarp_golden_bit_exact(W, golden):
    g = golden("backwarp")
    out, mask = W.warp_backward_flow(None, T(g["img"]).cuda(), T(g["flow"]).cuda())
    assert np.array_equal(mask.cpu().numpy(), g["mask"])
    assert np.array_equal(out.cpu().numpy(), g["out"])


def test_backwarp_sintel_rows_bit_exact(W, golden):
    g = golden("backwarp")
    full = torch.zeros(1, 2, 436, 1024)
    full[:, :, 200:204] = T(g["big_flow_rows"])
    img = T(g["big_img"].astype(np.float32))
    out, mask = W.warp_backward_flow(None, img.cuda(), full.cuda())
    assert np.array_equal(mask[:, :, 200:204].cpu().numpy(), g["big_mask_rows"])
    assert np.array_equal(out[:, :, 200:204].cpu().numpy(), g["big_out_rows"])


@pytest.mark.parametrize("shape", [(2, 3, 20, 28), (1, 1, 7, 5), (2, 3, 33, 64), (1, 2, 1, 9)])
def test_backwarp_vs_oracle_bit_exact(W, shape):
    B, C, H, Wd = shape
    g = torch.Generator().manual_seed(100 + H)
    img = torch.rand(B, C, H, Wd, generator=g)
    flow = torch.randn(B, 2, H, Wd, generator=g) * 3.0
    flow[0, :, 0, 0] = torch.tensor([-100.0, 100.0])
    o_ref, m_ref = O.backwarp(img, flow)
    o, m = W.warp_backward_flow(None, img.cuda(), flow.cuda())
    assert torch.equal(m.cpu(), m_ref)
    assert torch.equal(o.cpu(), o_ref)


def test_backwarp_grads_golden(W, golden):
    g = golden("backwarp")
    img = T(g["img"]).cuda().requires_grad_(True)
    flow = T(g["flow"]).cuda().requires_grad_(True)
    out, _ = W.warp_backward_flow(None, img, flow)
    (out * T(g["gout"]).cuda()).sum().backward()
    np.testing.assert_allclose(img.grad.cpu().numpy(), g["grad_img"], rtol=1e-5, atol=1e-6)
    np.testing.assert_allclose(flow.grad.cpu().numpy(), g["grad_flow"], rtol=1e-5, atol=1e-5)


def test_backwarp_grads_smooth_flow_merging(W):
    """Smooth flow -> neighbouring pixels hit the same taps: exercises the in-thread / cross-lane merge."""
    B, C, H, Wd = 2, 3, 24, 64
    g = torch.Generator().manual_seed(5)
    img = torch.rand(B, C, H, Wd, generator=g)
    flow = torch.zeros(B, 2, H, Wd)
    flow[:, 0] = 1.25
    flow[:, 1] = -2.5
    flow[1, 1, :, 32:] = 0.75
    gout = torch.randn(B, C, H, Wd, generator=g)
    ir, fr = img.clone().requires_grad_(True), flow.clone().requires_grad_(True)
    o, _ = O.backwarp_torch(ir, fr)
    (o * gout).sum().backward()
    ic, fc = img.cuda().requires_grad_(True), flow.cuda().requires_grad_(True)
    o2, _ = W.warp_backward_flow(None, ic, fc)
    (o2 * gout.cuda()).sum().backward()
    np.testing.assert_allclose(ic.grad.cpu().numpy(), ir.grad.numpy(), rtol=1e-5, atol=1e-5)
    np.testing.assert_allclose(fc.grad.cpu().numpy(), fr.grad.numpy(), rtol=1e-5, atol=1e-5)


@pytest.mark.parametrize("shape", [(2, 3, 20, 28), (2, 3, 17, 23), (1, 3, 64, 128)])
def test_photo_epe_fwd_bwd(W, shape):
    B, C, H, Wd = shape
    g = torch.Generator().manual_seed(3)
    flow = torch.randn(B, 2, H, Wd, generator=g) * 4.0
    f1 = torch.rand(B, C, H, Wd, generator=g)
    f2 = torch.rand(B, C, H, Wd, generator=g)
    gt = flow + torch.randn(B, 2, H, Wd, generator=g)
    fr, f2r = flow.clone().requires_grad_(True), f2.clone().requires_grad_(True)
    photo, epe, _, _ = O.photometric_epe(f1, f2r, fr, gt)
    (photo * 0.7 + epe * 1.3).backward()
    fc, f2c = flow.cuda().requires_grad_(True), f2.cuda().requires_grad_(True)
    p2, e2 = W.photometric_epe(f1.cuda(), f2c, fc, gt.cuda())
    (p2 * 0.7 + e2 * 1.3).backward()
    np.testing.assert_allclose(p2.item(), photo.item(), rtol=1e-5)
    np.testing.assert_allclose(e2.item(), epe.item(), rtol=1e-5)
    np.testing.assert_allclose(fc.grad.cpu().numpy(), fr.grad.numpy(), rtol=2e-4, atol=1e-7)
    np.testing.assert_allclose(f2c.grad.cpu().numpy(), f2r.grad.numpy(), rtol=2e-4, atol=1e-8)


def test_photo_epe_deterministic(W):
    g = torch.Generator().manual_seed(8)
    B, C, H, Wd = 2, 3, 64, 96
    args = [torch.rand(B, C, H, Wd, generator=g).cuda(), torch.rand(B, C, H, Wd, generator=g).cuda(),
            (torch.randn(B, 2, H, Wd, generator=g) * 4).cuda(), (torch.randn(B, 2, H, Wd, generator=g) * 4).cuda()]
    a = W.photometric_epe(*args)
    b = W.photometric_epe(*args)
    assert a[0].item() == b[0].item() and a[1].item() == b[1].item()


@pytest.mark.parametrize("cfg", [(1, 0, 0), (2, 0, 0), (2, 1, 1), (4, 1, 3), (8, 0, 0)])
def test_splat_golden(W, golden, cfg):
    g = golden("splat")
    scale, ox, oy = cfg
    tag = f"s{scale}_{ox}_{oy}"
    x = T(g["x"]).cuda().requires_grad_(True)
    flow = T(g["flow"]).cuda().requires_grad_(True)
    out = W.softsplat_func.apply(x, flow, scale, ox, oy)
    np.testing.assert_allclose(out.detach().cpu().numpy(), g[f"out_{tag}"], rtol=1e-5, atol=1e-5)
    out.backward(T(g[f"gout_{tag}"]).cuda())
    np.testing.assert_allclose(x.grad.cpu().numpy(), g[f"gin_{tag}"], rtol=1e-5, atol=1e-5)
    np.testing.assert_allclose(flow.grad.cpu().numpy(), g[f"gflow_{tag}"], rtol=1e-4, atol=1e-4)


@pytest.mark.parametrize("shape_scale", [((2, 4, 16, 24), 1), ((1, 3, 19, 21), 1), ((2, 4, 32, 64), 2), ((1, 4, 48, 40), 4),
                                         ((1, 4, 64, 64), 16)])
def test_splat_vs_oracle(W, shape_scale):
    (B, C, H, Wd), scale = shape_scale
    g = torch.Generator().manual_seed(31 + scale)
    x = torch.randn(B, C, H, Wd, generator=g)
    flow = torch.randn(B, 2, H, Wd, generator=g) * 3.0
    flow[0, 0, 1, 1] = float("nan")
    flow[0, :, 2, 2] = torch.tensor([float(Wd), float(H)])     # the ">= size-1" remap branch
    flow[0, :, H - 1, Wd - 1] = torch.tensor([0.3, 0.6])
    for ox, oy in ((0, 0), (scale - 1, scale // 2)):
        ref = O.splat_forward(x, flow, scale, ox, oy)
        xc, fc = x.cuda().requires_grad_(True), flow.cuda().requires_grad_(True)
        out = W.softsplat_func.apply(xc, fc, scale, ox, oy)
        # each target cell sums ~scale^2 atomically-ordered contributions: tolerance grows with scale
        tol = 1e-5 * max(1, scale)
        np.testing.assert_allclose(out.detach().cpu().numpy(), ref.numpy(), rtol=tol, atol=tol)
        gout = torch.randn(ref.shape, generator=g)
        out.backward(gout.cuda())
        np.testing.assert_allclose(xc.grad.cpu().numpy(), O.splat_ingrad(x.shape, flow, gout, scale, ox, oy).numpy(),
                                   rtol=1e-5, atol=1e-5)
        np.testing.assert_allclose(fc.grad.cpu().numpy(), O.splat_flowgrad(x, flow, gout, scale, ox, oy).numpy(),
                                   rtol=1e-4, atol=1e-4)


def test_splat_scale_consistency_property(W):
    """The property the reference fuzzes in warp_test.py:59-75:
    splat(src, flow, scale=L, offset)/L^2 == splat(splat(src, flow), 0, scale=L, offset)/L^2."""
    g = torch.Generator().manual_seed(77)
    src = torch.rand(1, 1, 128, 128, generator=g).cuda()
    for L, off in ((2, (0, 0)), (2, (1, 1)), (4, (1, 2))):
        ints = torch.randint(-2, 3, (1, 2, 128, 128), generator=g).float()
        frac = torch.rand(1, 2, 128, 128, generator=g) * 4 - 2
        pick = torch.rand(1, 1, 128, 128, generator=g) < 0.5
        flow = torch.where(pick, ints, frac).cuda()
        a = W.warp_forward_flow(src, None, flow, scale=L, set_nans=False, offset=off) / L ** 2
        full = W.warp_forward_flow(src, None, flow, set_nans=False)
        b = W.warp_forward_flow(full, None, torch.zeros_like(flow), scale=L, set_nans=False, offset=off) / L ** 2
        inner = (slice(None), slice(None), slice(2, -2), slice(2, -2))
        np.testing.assert_allclose(a[inner].cpu().numpy(), b[inner].cpu().numpy(), atol=1e-4)


def test_warp_forward_flow_vs_oracle(W):
    g = torch.Generator().manual_seed(12)
    first = torch.rand(2, 3, 24, 32, generator=g)
    first[0, 1, 3, 3] = float("nan")
    flow = torch.randn(2, 2, 24, 32, generator=g) * 2
    for scale, off in ((1, (0, 0)), (2, (1, 0))):
        ref = O.warp_forward_flow(first, flow, scale, True, off)
        out = W.warp_forward_flow(first.cuda(), None, flow.cuda(), scale=scale, offset=off).cpu()
        assert torch.equal(torch.isnan(out), torch.isnan(ref))
        np.testing.assert_allclose(torch.nan_to_num(out).numpy(), torch.nan_to_num(ref).numpy(), rtol=1e-5, atol=1e-5)
        # the generic (python-wrapper) path agrees with the fused one
        gen = W.warp_forward_flow(first.cuda(), None, flow.cuda(), scale=scale, offset=off, warp_style="sum",
                                  get_variance=False)
        assert gen.shape == out.shape


def test_nan_mse(W, golden):
    g = golden("misc")
    a = T(g["a"]).cuda().requires_grad_(True)
    b = T(g["b"]).cuda()
    loss = W.nan_mse(a, b)
    np.testing.assert_allclose(loss.item(), float(g["nan_mse_mean"]), rtol=1e-6)
    loss.backward()
    ar = T(g["a"]).clone().requires_grad_(True)
    O.nan_mse(ar, T(g["b"])).backward()
    np.testing.assert_allclose(a.grad.cpu().numpy(), ar.grad.numpy(), rtol=1e-5, atol=1e-8)
    np.testing.assert_array_equal(W.nan_mse(a.detach(), b, "none").cpu().numpy(), g["nan_mse_none"])
    # empty after filtering -> NaN like torch.nanmean of an empty tensor
    z = torch.full((4,), float("nan")).cuda()
    assert torch.isnan(W.nan_mse(z, z))


def test_full_size_properties(W):
    """BASELINE config #4 size (8x436x1024): size-independent properties instead of an oracle run."""
    B, C, H, Wd = 8, 3, 436, 1024
    g = torch.Generator().manual_seed(3)
    img = torch.rand(B, C, H, Wd, generator=g).cuda()
    zero = torch.zeros(B, 2, H, Wd).cuda()
    out, mask = W.warp_backward_flow(None, img, zero)
    # zero flow: the reference's fp32 normalise/un-normalise round trip is not exactly the identity
    # (SURVEY.md section 8a W1), so the warp reproduces the image only to a few ulps of the coordinate
    assert torch.allclose(out, img, atol=2e-4) and bool((mask == 1).all())
    shift = zero.clone()
    shift[:, 1] = 3.0                                                  # dx = +3: columns move left
    out, mask = W.warp_backward_flow(None, img, shift)
    assert torch.allclose(out[..., :-3], img[..., 3:], atol=2e-4)
    assert bool((mask[..., -3:] == 0).all()) and bool((mask[..., :-3] == 1).all())
    # linearity in the image
    flow = (torch.randn(B, 2, H, Wd, generator=g) * 4).cuda()
    img2 = torch.rand(B, C, H, Wd, generator=g).cuda()
    a, _ = W.warp_backward_flow(None, img, flow)
    b, _ = W.warp_backward_flow(None, img2, flow)
    c, _ = W.warp_backward_flow(None, img + img2, flow)
    assert torch.allclose(a + b, c, atol=1e-5)
    # splat conserves mass for in-bounds integer flow; photo loss of identical frames with zero flow = sqrt(1e-6)
    ones = torch.ones(B, 1, H, Wd).cuda()
    s = W.softsplat_func.apply(ones, zero, 1, 0, 0)
    assert torch.equal(s, ones)
    p, e = W.photometric_epe(img, img, zero, zero)
    np.testing.assert_allclose(p.item(), 1e-3, rtol=1e-4)
    assert e.item() == 0.0


@pytest.mark.parametrize("divisor", [1023.0, 435.0, 1.0, 3.0, 767.0, 367.0, 2047.0, 47.0, 16777216.0, 0.5, 3e7])
def test_hoisted_reciprocal_division_is_exact(divisor):
    """bw_div_rn == __fdiv_rn for EVERY fp32 numerator (2^32 bit patterns; NaNs compared as a class): the warp kernels'
    coordinate normalisation (warp.py:107-108) stays bit-identical to the reference with the reciprocal computed once per
    thread.  Divisors outside 1 .. 2^24 (last two cases) take __fdiv_rn itself."""
    from opticalflowdiffusion_b200 import _lib
    lib = _lib.load()
    bad = torch.full((1,), -1, dtype=torch.int64, device="cuda")
    _lib.check(lib.fd_warp_div_selftest(divisor, _lib.ptr(bad), _lib.stream()))
    torch.cuda.synchronize()
    assert int(bad.item()) == 0, int(bad.item())


@pytest.mark.parametrize("C", [3, 4])
@pytest.mark.parametrize("geom", [(1, 0, 0), (2, 1, 0), (4, 1, 3)])
def test_splat_forward_interleaved_vs_oracle(C, geom):
    """fd_splat_fwd at C = 3 / 4 (pixel-interleaved accumulation, one 128-bit reduction per tap, planar copy-out) == the
    oracle's splat (softsplat_new.py:352-423) up to the order of the atomics, NaN / Inf / far flows included; and
    fd_forward_warp_sum3 == the oracle's warp_forward_flow (prepare + splat + finish)."""
    from opticalflowdiffusion_b200 import _lib
    lib = _lib.load()
    scale, ox, oy = geom
    B, H, W = 2, 24, 40
    g = torch.Generator().manual_seed(C * 10 + scale)
    x = torch.randn(B, C, H, W, generator=g)
    flow = torch.randn(B, 2, H, W, generator=g) * 3
    flow[0, 0, 3, 4] = float("nan")
    flow[1, 1, 5, 6] = float("inf")
    flow[0, :, 0, 0] = -50.0
    Ho, Wo = H // scale, W // scale
    P, st = _lib.ptr, _lib.stream()
    ref = O.splat_forward(x, flow, scale, ox, oy)
    xc, fc = x.cuda(), flow.cuda()
    got = torch.full((B, C, Ho, Wo), float("nan"), device="cuda")
    ws = torch.empty(lib.fd_splat_fwd_workspace_floats(B, C, H, W, scale), device="cuda")
    _lib.check(lib.fd_splat_fwd(P(xc), P(fc), P(got), P(ws), B, C, H, W, scale, ox, oy, st))
    got = got.cpu()
    assert torch.isfinite(got).all()
    assert (got - ref).abs().max().item() <= 1e-5 * max(1.0, ref.abs().max().item())
    if C == 3:
        first = x.clone()
        first[0, 1, 7, 8] = float("nan")                      # NaN source pixel: weight 0
        img_ref = O.warp_forward_flow(first, flow, scale, True, (ox, oy))
        wsum_ref = O.splat_forward((~torch.isnan(first).any(1, keepdim=True)).float(), flow, scale, ox, oy)
        first = first.cuda()
        ten_in = torch.empty(B, 4, H, W, device="cuda")
        _lib.check(lib.fd_splat_prepare(P(first), P(ten_in), B, 3, H * W, st))
        ten2, acc = torch.empty_like(ten_in), torch.empty(B, Ho, Wo, 4, device="cuda")
        img, wsum = torch.empty(B, 3, Ho, Wo, device="cuda"), torch.empty(B, 1, Ho, Wo, device="cuda")
        _lib.check(lib.fd_forward_warp_sum3(P(first), P(fc), P(ten2), P(acc), P(img), P(wsum), B, H, W, scale, ox, oy, 1, st))
        img, wsum = img.cpu(), wsum.cpu()
        assert torch.equal(ten2, ten_in)
        assert torch.equal(torch.isnan(img), torch.isnan(img_ref))
        assert (img.nan_to_num() - img_ref.nan_to_num()).abs().max().item() <= 1e-5 * max(1.0, ref.abs().max().item())
        assert (wsum - wsum_ref).abs().max().item() <= 1e-5


def _misaligned(t):
    """A copy of ``t`` whose data pointer is NOT 16-byte aligned: the warp entry points then take the gather kernels of
    fd_warp.cu instead of the TMA-window kernels (both must give the same results)."""
    buf = torch.empty(t.numel() + 1, device=t.device, dtype=t.dtype)
    v = buf[1:].view(t.shape)
    v.copy_(t)
    assert v.data_ptr() % 16 != 0
    return v


@pytest.mark.parametrize("shape", [(1, 50, 68), (2, 17, 132), (3, 16, 128), (1, 97, 260), (1, 1024, 2048)])
def test_window_kernels_equal_gather_kernels_and_flow_only(shape):
    """The shared-memory-window kernels (fd_warp_win.cu: tiles of 16 x 128, 16-pixel halo, TMA zero fill, border tiles,
    out-of-window fallback) against the one-thread-per-pixel gather kernels on ragged / small / large shapes with flows that
    leave the window and the image: forward output and mask bit-identical, sums and gradients to the order of the atomics,
    the flow gradient of the window backward bit-identical with and without the frame gradient."""
    from opticalflowdiffusion_b200 import _lib
    lib = _lib.load()
    B, H, Wd = shape
    g = torch.Generator().manual_seed(H + Wd)
    flow = torch.randn(B, 2, H, Wd, generator=g) * 5
    flow[0, :, H // 2, Wd // 3] = torch.tensor([40.0, -33.0])          # outside the 16-pixel window
    flow[0, :, 0, 0] = torch.tensor([-3.0 * H, 2.0 * Wd])              # far outside the image (clamped cell)
    flow = flow.cuda()
    f1, f2 = torch.rand(B, 3, H, Wd, generator=g).cuda(), torch.rand(B, 3, H, Wd, generator=g).cuda()
    gt = (flow.cpu() + torch.randn(B, 2, H, Wd, generator=g)).cuda()
    gout = torch.randn(B, 3, H, Wd, generator=g).cuda()
    P, st = _lib.ptr, _lib.stream()
    mf, m1, m2, mg, mo = (_misaligned(t) for t in (flow, f1, f2, gt, gout))

    def fwd(f2_, fl_):
        out, mask = torch.empty_like(f2), torch.empty_like(f2)
        _lib.check(lib.fd_backwarp_fwd(P(f2_), P(fl_), P(out), P(mask), B, 3, H, Wd, st))
        return out, mask
    (o_w, m_w), (o_g, m_g) = fwd(f2, flow), fwd(m2, mf)
    assert torch.equal(o_w, o_g) and torch.equal(m_w, m_g)

    def photo(a1, a2, fl_, gt_):
        sums = torch.empty(4, device="cuda")
        ws = torch.empty(lib.fd_photo_epe_workspace_floats(B, H, Wd), device="cuda")
        _lib.check(lib.fd_backwarp_photo_epe_fwd(P(a1), P(a2), P(fl_), P(gt_), P(sums), P(ws), B, 3, H, Wd, st))
        return sums
    s_w, s_g = photo(f1, f2, flow, gt), photo(m1, m2, mf, mg)
    assert torch.allclose(s_w, s_g, rtol=2e-5, atol=1e-3), (s_w, s_g)

    def close(a, b):
        return (a - b).abs().max().item() <= 2e-5 * max(b.abs().max().item(), 1e-12)
    wsb = torch.empty(lib.fd_warp_bwd_workspace_floats(B, 3, H, Wd), device="cuda")
    assert wsb.numel() == 4 * B * H * Wd
    # window kernels with and without the frame gradient (flow only: no accumulation buffer), gather kernels on the views
    res = []
    for (a1, a2, fl_, gt_, frame_grad) in ((f1, f2, flow, gt, True), (f1, f2, flow, gt, False), (m1, m2, mf, mg, True)):
        gfl = torch.empty_like(flow)
        gf2 = torch.full_like(f2, float("nan")) if frame_grad else None
        _lib.check(lib.fd_backwarp_photo_epe_bwd(P(a1), P(a2), P(fl_), P(gt_), P(s_g), 1.0, 0.5, P(gfl), P(gf2),
                                                 P(wsb if frame_grad else None), B, 3, H, Wd, st))
        res.append((gfl, gf2))
    (gfl_w, gf2_w), (gfl_fo, _), (gfl_g, gf2_g) = res
    assert close(gfl_w, gfl_g) and close(gf2_w, gf2_g) and close(gfl_fo, gfl_g)
    assert torch.equal(gfl_fo, gfl_w)          # the flow gradient is written per pixel without atomics
    res = []
    for (a2, fl_, go_, frame_grad) in ((f2, flow, gout, True), (f2, flow, gout, False), (m2, mf, mo, True)):
        gfl = torch.empty_like(flow)
        gim = torch.full_like(f2, float("nan")) if frame_grad else None
        _lib.check(lib.fd_backwarp_bwd(P(a2), P(fl_), P(go_), P(gim), P(gfl), P(wsb if frame_grad else None), B, 3, H, Wd, st))
        res.append((gim, gfl))
    torch.cuda.synchronize()
    (gim_w, gfl_w), (_, gfl_fo), (gim_g, gfl_g) = res
    assert close(gim_w, gim_g) and close(gfl_w, gfl_g) and close(gfl_fo, gfl_g)
    assert torch.equal(gfl_fo, gfl_w)


def test_frame_gradient_without_workspace_is_an_error():
    """Shapes whose query returns a workspace need it for the frame gradient (the window backward kernels, the interleaved
    splat): a NULL workspace is refused by the argument checks, before anything is launched, and the outputs stay untouched."""
    from opticalflowdiffusion_b200 import _lib
    lib = _lib.load()
    B, C, H, Wd = 1, 3, 32, 128
    P, st = _lib.ptr, _lib.stream()
    f1, f2, gout = (torch.rand(B, C, H, Wd, device="cuda") for _ in range(3))
    flow, gt = torch.randn(B, 2, H, Wd, device="cuda"), torch.randn(B, 2, H, Wd, device="cuda")
    sums = torch.ones(4, device="cuda")
    assert lib.fd_warp_bwd_workspace_floats(B, C, H, Wd) > 0
    gfl, gim = torch.full_like(flow, float("nan")), torch.full_like(f2, float("nan"))
    assert lib.fd_backwarp_bwd(P(f2), P(flow), P(gout), P(gim), P(gfl), None, B, C, H, Wd, st) != 0
    assert "workspace" in lib.fd_last_error().decode()
    assert lib.fd_backwarp_photo_epe_bwd(P(f1), P(f2), P(flow), P(gt), P(sums), 1.0, 1.0, P(gfl), P(gim), None,
                                         B, C, H, Wd, st) != 0
    assert "workspace" in lib.fd_last_error().decode()
    for c in (3, 4):
        assert lib.fd_splat_fwd_workspace_floats(B, c, H, Wd, 1) > 0
        x, out = torch.rand(B, c, H, Wd, device="cuda"), torch.full((B, c, H, Wd), float("nan"), device="cuda")
        assert lib.fd_splat_fwd(P(x), P(flow), P(out), None, B, c, H, Wd, 1, 0, 0, st) != 0
        assert "workspace" in lib.fd_last_error().decode()
        assert torch.isnan(out).all()
    torch.cuda.synchronize()
    assert torch.isnan(gfl).all() and torch.isnan(gim).all()


def test_photo_epe_ticket_needs_no_clean_workspace():
    """The window kernel finds its last block through a {launch tag, count} word in the caller's workspace (no memset in front
    of the kernel): whatever the workspace holds -- zeros, all ones, the word an ABORTED launch would leave behind -- and when the
    very same launch is replayed from a CUDA graph (same tag every time), the sums are those of a clean run, bit for bit (the
    partials are reduced in a fixed order)."""
    from opticalflowdiffusion_b200 import _lib
    lib = _lib.load()
    B, H, Wd = 2, 70, 256
    g = torch.Generator().manual_seed(11)
    flow = (torch.randn(B, 2, H, Wd, generator=g) * 4).cuda()
    f1, f2 = torch.rand(B, 3, H, Wd, generator=g).cuda(), torch.rand(B, 3, H, Wd, generator=g).cuda()
    gt = (flow.cpu() + torch.randn(B, 2, H, Wd, generator=g)).cuda()
    P = _lib.ptr
    n_ws = lib.fd_photo_epe_workspace_floats(B, H, Wd)

    def run(ws, stream=None):
        sums = torch.full((4,), float("nan"), device="cuda")
        _lib.check(lib.fd_backwarp_photo_epe_fwd(P(f1), P(f2), P(flow), P(gt), P(sums), P(ws), B, 3, H, Wd,
                                                 stream if stream is not None else _lib.stream()))
        return sums

    ref = run(torch.zeros(n_ws, device="cuda"))
    assert torch.isfinite(ref).all()
    for fill in (float("nan"), 1.0, -3.0e38):
        assert torch.equal(run(torch.full((n_ws,), fill, device="cuda")), ref), fill
    ints = torch.full((n_ws,), -1, device="cuda", dtype=torch.int32)              # tag 0xffffffff, count 0xffffffff
    assert torch.equal(run(ints.view(torch.float32)), ref)
    ws = torch.empty(n_ws, device="cuda")
    for _ in range(3):                                                          # one workspace, consecutive launches
        assert torch.equal(run(ws), ref)
    # graph replay: the tag is baked into the captured launch
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        run(ws, side.cuda_stream)                                               # warm-up on the capture stream
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph, stream=side):
            out = run(ws, torch.cuda.current_stream().cuda_stream)
    torch.cuda.current_stream().wait_stream(side)
    for _ in range(3):
        out.fill_(float("nan"))
        graph.replay()
        torch.cuda.synchronize()
        assert torch.equal(out, ref)
