"""-m gpu: every distinct kernel launch of the benchmark's UNet training step (tests/train_launches.py: one training
forward and its backward at batch 8, 368 x 768), run in isolation at exactly its launch shape and null pattern, plus the
loss, q_sample and optimiser kernels of the same step at their sizes.

The harness is tests/test_gpu_bench_launches.py's: NaN-prefilled outputs followed by sentinel guards, per-sample float64
references, act() inputs (every sample its own offset and scale, every (sample, group) its own mean) and scale / shift rows
of stride 8064 with NaN outside the block.  Outputs the kernels accumulate into (+=) start at train_launches.FILL.

Exact leg (linear kernels): integer operands in {-1, 0, 1}; every partial sum is exact in fp32 (train_launches.exact_terms),
so fp32 outputs equal the float64 reference, bf16 outputs equal it rounded once, and a second launch gives the same bits.
Real leg (every entry): Gaussian operands and the rounding bound of the kernel's fp32 arithmetic; parameter-gradient
reductions get a sign-coherent upstream gradient on half of the channels, so that a lost block of pixels exceeds the
bound.  Each case prints max(err / bound)."""
import math

import pytest
import torch

import bench_launches as BL
import test_gpu_bench_launches as GPU
import train_launches as TL
from oracle import flowdiff_oracle as O
from test_gpu_bench_launches import BF, F64, NAN, act, guard_intact, guarded, report, rnd

pytestmark = pytest.mark.gpu
F32 = torch.float32
FILL = TL.FILL


@pytest.fixture(scope="module")
def L():
    from opticalflowdiffusion_b200 import _lib
    _lib.load(check_device=True)
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.cuda.reset_peak_memory_stats()
    yield _lib
    print(f"\n{torch.cuda.get_device_name()}: peak device memory {torch.cuda.max_memory_allocated() / 2 ** 30:.2f} GiB")


def sms():
    return torch.cuda.get_device_properties(0).multi_processor_count


def ints(shape, seed, dtype=BF):
    """Integers in {-1, 0, 1}: the exact leg's operands."""
    g = torch.Generator(device="cuda").manual_seed(seed)
    return torch.randint(-1, 2, shape, generator=g, device="cuda").to(dtype)


def coherent(shape, seed, offset=0.5):
    """bf16 Gaussian upstream gradient with +offset on the first half of the channels (sign-coherent there)."""
    C = shape[-1]
    d = rnd(shape, seed)
    d[..., :C // 2] += offset
    return d.to(BF)


def exact(name, scalars, got, ref):
    """The exact leg's comparison: fp32 outputs equal the float64 reference, bf16 outputs equal it rounded once."""
    assert TL.exact_terms(name, scalars) < TL.EXACT_LIMIT
    want = ref.to(got.dtype)
    bad = (got != want).sum().item()
    assert bad == 0, f"{name}{scalars}: {bad} elements differ from the exact result"


def tap_views(x, KH, KW, ph, pw, mode):
    """One sample's conv source (Hin, Win, C) as the (H, W, C) planes its taps read, in packed K order: mode 0 shifts by
    (ky - ph, kx - pw) with zero fill, mode 1 (pixel unshuffle) tap p1*2+p2 reads x[p1::2, p2::2]."""
    if mode == 1:
        for p in range(4):
            yield x[p >> 1::2, p & 1::2]
        return
    H, W, _ = x.shape
    for ky in range(KH):
        for kx in range(KW):
            dy, dx = ky - ph, kx - pw
            if (dy, dx) == (0, 0):
                yield x
                continue
            out = torch.zeros_like(x)
            out[max(0, -dy):min(H, H - dy), max(0, -dx):min(W, W - dx)] = \
                x[max(0, dy):min(H, H + dy), max(0, dx):min(W, W + dx)]
            yield out


def conv_sample(x, wp, KH, KW, ph, pw, mode, H, W):
    """sum over taps of x_tap @ W_tap^T and the same on |x|, |w|: (H W, Cout) float64."""
    Cout = wp.shape[0]
    w = wp.double()
    ref = torch.zeros(H * W, Cout, device="cuda", dtype=F64)
    A = torch.zeros_like(ref)
    cin = x.shape[-1]
    for t, v in enumerate(tap_views(x, KH, KW, ph, pw, mode)):
        v = v.reshape(-1, cin)
        wt = w[:, t * cin:(t + 1) * cin]
        ref += v @ wt.t()
        A += v.abs() @ wt.abs().t()
    return ref, A


def exact_windows(scalars_conv):
    """The channel windows of the exact leg: one launch over all channels, except in the rolling-strip kernel's two-pass
    geometry (train_launches.two_pass), whose first pass stores a bf16 partial sum that holds integers exactly only up to
    2^8.  There one launch per window of TWO_PASS_CH of the first pass's 64 channels (9 * 28 + 1 <= 256 terms) gives
    those channels their weights, the rest of the first half zero: every channel is covered by one exact launch."""
    if not TL.two_pass(*scalars_conv):
        return [None]
    return [(lo, min(lo + TL.TWO_PASS_CH, 64)) for lo in range(0, 64, TL.TWO_PASS_CH)]


def sparse_two_pass(wp, window):
    """``wp`` with the first pass's channels outside ``window`` zeroed (None: unchanged)."""
    if window is not None:
        Cout = wp.shape[0]
        v = wp.view(Cout, 9, -1)
        v[:, :, :window[0]] = 0
        v[:, :, window[1]:64] = 0
    return wp


def two_pass_partial(x, wp, res, H, W):
    """The bound the first pass's bf16 rounding adds (as in test_gpu_bench_launches.check_conv): one output rounding of
    the partial sum over the first 64 input channels (+ the residual) and its accumulation error."""
    Cout = wp.shape[0]
    p0, a0 = conv_sample(x[..., :64], wp.view(Cout, 9, -1)[:, :, :64].reshape(Cout, -1), 3, 3, 1, 1, 0, H, W)
    if res is not None:
        p0 += res
        a0 += res.abs()
    return BL.OUT_ROUND * p0.abs() + BL.gamma_mma(9 * 64) * a0


def cat_sample(s0, s1, n):
    return (torch.cat((s0[n], s1[n]), -1) if s1 is not None else s0[n]).double()


# ------------------------------------------------------------------------------------------------------ convolutions
def check_conv_train(L, scalars, nulls, seed):
    """fd_conv_igemm: the forward file's real leg, then the exact leg on its outputs (the statistics are not checked)."""
    GPU.check_conv(L, scalars, nulls, seed)
    lib = L.load()
    C0, C1, N, H, W, Cout, KH, KW, ph, pw, mode = scalars
    has_bias, has_res, has_stats = nulls[3] == "P", nulls[4] == "P", nulls[6] == "P"
    Hin, Win = (2 * H, 2 * W) if mode else (H, W)
    s0 = ints((N, Hin, Win, C0), seed)
    s1 = ints((N, Hin, Win, C1), seed + 1) if C1 else None
    K = 4 * C0 if mode else KH * KW * (C0 + C1)
    bias = ints((Cout,), seed + 3, F32) if has_bias else None
    res = ints((N, H, W, Cout), seed + 4) if has_res else None

    def launch():
        buf, out = guarded((N, H, W, Cout), BF, NAN)
        st = torch.zeros(N, 8, 2, device="cuda", dtype=F64) if has_stats else None
        L.check(lib.fd_conv_igemm(L.ptr(s0), C0, L.ptr(s1), C1, L.ptr(wp), L.ptr(bias), L.ptr(res), L.ptr(out), L.ptr(st),
                                  N, H, W, Cout, KH, KW, ph, pw, mode, L.stream()))
        torch.cuda.synchronize()
        guard_intact(buf, out)
        return out

    for window in exact_windows((C0 + C1, Cout, KH, KW, ph, pw, mode, W)):
        wp = sparse_two_pass(ints((Cout, K), seed + 2), window)
        out = launch()
        for n in range(N):
            ref, _ = conv_sample(cat_sample(s0, s1, n), wp, KH, KW, ph, pw, mode, H, W)
            if has_bias:
                ref += bias.double()
            if has_res:
                ref += res[n].double().reshape(-1, Cout)
            exact("fd_conv_igemm", scalars, out[n].reshape(-1, Cout), ref)
            del ref
        assert torch.equal(out, launch())
    report("fd_conv_igemm", scalars, nulls, exact_leg_bit_exact=1.0)


def check_conv_ex(L, scalars, nulls, seed):
    """fd_conv_igemm_ex as the data gradient: dy (C0 channels) through the packed dgrad weights handed in directly, plain,
    accumulating into the gradient already there (residual), or (out_mode 1) stored pixel-shuffled on the 2H x 2W grid."""
    lib = L.load()
    C0, C1, N, H, W, Cout, KH, KW, ph, pw, mode, out_mode = scalars
    assert C1 == 0 and mode == 0
    has_res = nulls[4] == "P"
    K = KH * KW * C0
    oshape = (N, 2 * H, 2 * W, Cout // 4) if out_mode else (N, H, W, Cout)

    def launch(dy, wp, res):
        buf, out = guarded(oshape, BF, NAN)
        L.check(lib.fd_conv_igemm_ex(L.ptr(dy), C0, None, 0, L.ptr(wp), None, L.ptr(res), L.ptr(out), None, N, H, W, Cout, KH, KW,
                                     ph, pw, 0, out_mode, L.stream()))
        torch.cuda.synchronize()
        guard_intact(buf, out)
        return out

    def ref_sample(dy, wp, res, n):
        ref, A = conv_sample(dy[n].double(), wp, KH, KW, ph, pw, 0, H, W)
        if has_res:
            r = res[n].double().reshape(-1, Cout)
            ref += r
            A += r.abs()
        if out_mode:       # channel (p1*2+p2)*Cq + c of (h, w) -> pixel (2h+p1, 2w+p2)
            ref, A = (t.view(H, W, 2, 2, Cout // 4).permute(0, 2, 1, 3, 4).reshape(-1, Cout // 4) for t in (ref, A))
        return ref, A

    # exact leg
    dy = ints((N, H, W, C0), seed)
    res = ints((N, H, W, Cout), seed + 2) if has_res else None
    for window in exact_windows((C0, Cout, KH, KW, ph, pw, 0, W)):
        wp = sparse_two_pass(ints((Cout, K), seed + 1), window)
        out = launch(dy, wp, res)
        for n in range(N):
            ref, _ = ref_sample(dy, wp, res, n)
            exact("fd_conv_igemm_ex", scalars, out[n].reshape(ref.shape), ref)
        assert torch.equal(out, launch(dy, wp, res))
    # real leg
    dy = act((N, H, W, C0), seed + 3)
    wp = GPU.pack_w(GPU.weight(Cout, C0, KH, KW, seed + 4))
    res = act((N, H, W, Cout), seed + 5) if has_res else None
    out = launch(dy, wp, res)
    worst = 0.0
    for n in range(N):
        ref, A = ref_sample(dy, wp, res, n)
        partial = None
        if TL.two_pass(C0, Cout, KH, KW, ph, pw, 0, W):
            partial = two_pass_partial(dy[n].double(), wp, res[n].double().reshape(-1, Cout) if has_res else None, H, W)
        worst = max(worst, BL.ratio((out[n].reshape(ref.shape).double() - ref).abs(), BL.conv_bound(ref, A, K, partial)))
        del ref, A
    report("fd_conv_igemm_ex", scalars, nulls, err_over_bound=worst, exact_leg_bit_exact=1.0)
    assert worst <= 1
    assert torch.equal(out, launch(dy, wp, res))


def check_wgrad(L, scalars, nulls, seed):
    """fd_conv_wgrad, rolling-strip and generic paths, mode 0 and 1: dw[co][tap*Cin + ci] += sum over pixels of
    src_tap * dy.  Real-leg bound train_launches.wgrad_bound with (L, S) from the launcher's own formulas."""
    lib = L.load()
    C0, C1, N, H, W, Cout, KH, KW, ph, pw, mode = scalars
    Hin, Win = (2 * H, 2 * W) if mode else (H, W)
    Cin = C0 + C1
    taps = 4 if mode else KH * KW

    def launch(s0, s1, dy):
        buf, dw = guarded((Cout, taps * Cin), F32, FILL)
        L.check(lib.fd_conv_wgrad(L.ptr(s0), C0, L.ptr(s1), C1, L.ptr(dy), L.ptr(dw), N, H, W, Cout, KH, KW, ph, pw, mode,
                                  L.stream()))
        torch.cuda.synchronize()
        guard_intact(buf, dw)
        return dw

    def reference(s0, s1, dy):
        ref = torch.zeros(Cout, taps * Cin, device="cuda", dtype=F64)
        A = torch.zeros_like(ref)
        for n in range(N):
            d = dy[n].double().reshape(-1, Cout)
            for t, v in enumerate(tap_views(cat_sample(s0, s1, n), KH, KW, ph, pw, mode)):
                v = v.reshape(-1, Cin)
                ref[:, t * Cin:(t + 1) * Cin] += d.t() @ v
                A[:, t * Cin:(t + 1) * Cin] += d.abs().t() @ v.abs()
            del d
        return ref + FILL, A

    s0, dy = ints((N, Hin, Win, C0), seed), ints((N, H, W, Cout), seed + 1)
    s1 = ints((N, Hin, Win, C1), seed + 2) if C1 else None
    dw = launch(s0, s1, dy)
    ref, _ = reference(s0, s1, dy)
    exact("fd_conv_wgrad", scalars, dw, ref)
    assert torch.equal(dw, launch(s0, s1, dy))
    s0, dy = act((N, Hin, Win, C0), seed + 3), act((N, H, W, Cout), seed + 4)
    s1 = act((N, Hin, Win, C1), seed + 5) if C1 else None
    dw = launch(s0, s1, dy)
    ref, A = reference(s0, s1, dy)
    Lr, S = TL.wgrad_ranges(scalars, sms())
    worst = BL.ratio((dw.double() - ref).abs(), TL.wgrad_bound(A, Lr, S))
    report("fd_conv_wgrad", scalars, nulls, err_over_bound=worst, exact_leg_bit_exact=1.0, L=Lr, S=S)
    assert worst <= 1


# ------------------------------------------------------------------------------------------- small linear kernels
def check_bias_grad(L, scalars, nulls, seed):
    """fd_bias_grad: db[c] += sum over pixels of dy.  Bound: the fp32 sums of fd_unet_bwd.cu:446-468 (a thread's pixels,
    the block's rows through shared atomics, one global atomic per block) at 2^-24 of sum |dy| + |fill| per level."""
    lib = L.load()
    npix, C = scalars
    ppb = max(256 // (C // 8), 1)
    bx = min(-(-npix // (ppb * 8)), sms() * 8)
    depth = -(-npix // (bx * ppb)) + ppb + bx + 1

    def launch(dy):
        buf, db = guarded((C,), F32, FILL)
        L.check(lib.fd_bias_grad(L.ptr(dy), L.ptr(db), npix, C, L.stream()))
        torch.cuda.synchronize()
        guard_intact(buf, db)
        return db

    dy = ints((npix, C), seed)
    db = launch(dy)
    exact("fd_bias_grad", scalars, db, dy.double().sum(0) + FILL)
    assert torch.equal(db, launch(dy))
    dy = coherent((npix, C), seed + 1)
    db = launch(dy)
    d = dy.double()
    ref = d.sum(0) + FILL
    worst = BL.ratio((db.double() - ref).abs(), depth * 2.0 ** -24 * (d.abs().sum(0) + FILL))
    report("fd_bias_grad", scalars, nulls, err_over_bound=worst, exact_leg_bit_exact=1.0)
    assert worst <= 1


def check_upsample2x(L, scalars, nulls, seed):
    """fd_upsample2x: a copy, so bit-exact on any data."""
    lib = L.load()
    N, H, W, C = scalars
    x = act((N, H, W, C), seed)
    buf, out = guarded((N, 2 * H, 2 * W, C), BF, NAN)
    L.check(lib.fd_upsample2x(L.ptr(x), L.ptr(out), N, H, W, C, L.stream()))
    torch.cuda.synchronize()
    guard_intact(buf, out)
    assert torch.equal(out, x.repeat_interleave(2, 1).repeat_interleave(2, 2))
    report("fd_upsample2x", scalars, nulls, bit_exact=1.0)


def check_upsample2x_bwd(L, scalars, nulls, seed):
    """fd_upsample2x_bwd: dx = sum of each 2 x 2 block of dy.  Exact leg against float64; real leg bit-exact against the
    kernel's own order ((a + b) + c) + d in fp32, rounded once."""
    lib = L.load()
    N, H, W, C = scalars

    def launch(dy):
        buf, dx = guarded((N, H, W, C), BF, NAN)
        L.check(lib.fd_upsample2x_bwd(L.ptr(dy), L.ptr(dx), N, H, W, C, L.stream()))
        torch.cuda.synchronize()
        guard_intact(buf, dx)
        return dx

    dy = ints((N, 2 * H, 2 * W, C), seed)
    exact("fd_upsample2x_bwd", scalars, launch(dy), dy.double().view(N, H, 2, W, 2, C).sum((2, 4)))
    dy = act((N, 2 * H, 2 * W, C), seed + 1)
    q = dy.float().view(N, H, 2, W, 2, C)
    want = (((q[:, :, 0, :, 0] + q[:, :, 0, :, 1]) + q[:, :, 1, :, 0]) + q[:, :, 1, :, 1]).to(BF)
    assert torch.equal(launch(dy), want)
    report("fd_upsample2x_bwd", scalars, nulls, bit_exact=1.0, exact_leg_bit_exact=1.0)


def check_add_bf16(L, scalars, nulls, seed):
    """fd_add_bf16: out = bf16(a + b in fp32); exact leg against float64, real leg bit-exact."""
    lib = L.load()
    n, = scalars

    def launch(a, b):
        buf, out = guarded((n,), BF, NAN)
        L.check(lib.fd_add_bf16(L.ptr(a), L.ptr(b), L.ptr(out), n, L.stream()))
        torch.cuda.synchronize()
        guard_intact(buf, out)
        return out

    a, b = ints((n,), seed), ints((n,), seed + 1)
    exact("fd_add_bf16", scalars, launch(a, b), a.double() + b.double())
    a, b = rnd((n,), seed + 2).to(BF), rnd((n,), seed + 3, 0.01).to(BF)
    assert torch.equal(launch(a, b), (a.float() + b.float()).to(BF))
    report("fd_add_bf16", scalars, nulls, bit_exact=1.0, exact_leg_bit_exact=1.0)


def check_final_conv_crop(L, scalars, nulls, seed):
    """fd_final_conv_crop: the 1x1 conv 64 -> Cout with fp32 weights, the H0 x W0 window, fp32 NCHW.  Bound: an fp32 dot
    product of Cin terms plus the bias, (Cin + 2) 2^-24 of sum |x w| + |b|."""
    lib = L.load()
    N, H, W, Cin, Cout, pt, pl, H0, W0 = scalars

    def launch(x, w, b):
        buf, out = guarded((N, Cout, H0, W0), F32, NAN)
        L.check(lib.fd_final_conv_crop(L.ptr(x), L.ptr(w), L.ptr(b), L.ptr(out), N, H, W, Cin, Cout, pt, pl, H0, W0, L.stream()))
        torch.cuda.synchronize()
        guard_intact(buf, out)
        return out

    def ref_sample(x, w, b, n):
        xs = x[n, pt:pt + H0, pl:pl + W0].double().reshape(-1, Cin)
        ref = (xs @ w.double().t() + b.double()).t().reshape(Cout, H0, W0)
        A = (xs.abs() @ w.double().abs().t() + b.double().abs()).t().reshape(Cout, H0, W0)
        return ref, A

    x, w, b = ints((N, H, W, Cin), seed), ints((Cout, Cin), seed + 1, F32), ints((Cout,), seed + 2, F32)
    out = launch(x, w, b)
    for n in range(N):
        exact("fd_final_conv_crop", scalars, out[n], ref_sample(x, w, b, n)[0])
    x, w, b = act((N, H, W, Cin), seed + 3), rnd((Cout, Cin), seed + 4, 1 / 8), rnd((Cout,), seed + 5)
    out = launch(x, w, b)
    worst = 0.0
    for n in range(N):
        ref, A = ref_sample(x, w, b, n)
        worst = max(worst, BL.ratio((out[n].double() - ref).abs(), (Cin + 2) * 2.0 ** -24 * A))
    report("fd_final_conv_crop", scalars, nulls, err_over_bound=worst, exact_leg_bit_exact=1.0)
    assert worst <= 1
    assert torch.equal(out, launch(x, w, b))


def check_final_conv_bwd(L, scalars, nulls, seed):
    """fd_final_conv_bwd: dx = dout^T w (bf16), dw += dout x, db += dout summed over the N HW pixels.  Bounds: dx one
    rounding plus 4 fp32 additions; dw, db the fp32 sums of fd_unet_bwd.cu:472-521 (a thread's pixels, 32 threads per
    block on one element through shared atomics, one global atomic per block)."""
    lib = L.load()
    N, HW, Cin, Cout = scalars
    grid = min(-(-N * HW * 8 // 256), sms() * 8)
    depth = -(-N * HW // (grid * 32)) + 32 + grid + 1

    def launch(x, w, dout):
        xb, dx = guarded((N, HW, Cin), BF, NAN)
        wb, dw = guarded((Cout, Cin), F32, FILL)
        bb, db = guarded((Cout,), F32, FILL)
        L.check(lib.fd_final_conv_bwd(L.ptr(x), L.ptr(w), L.ptr(dout), L.ptr(dx), L.ptr(dw), L.ptr(db), N, HW, Cin, Cout,
                                      L.stream()))
        torch.cuda.synchronize()
        for b, v in ((xb, dx), (wb, dw), (bb, db)):
            guard_intact(b, v)
        return dx, dw, db

    def reference(x, w, dout):
        dw = torch.zeros(Cout, Cin, device="cuda", dtype=F64)
        Aw = torch.zeros_like(dw)
        dxs = []
        for n in range(N):
            d, xs = dout[n].double(), x[n].double()
            dw += d @ xs
            Aw += d.abs() @ xs.abs()
            dxs.append((d.t() @ w.double(), d.abs().t() @ w.double().abs()))
        d = dout.double()
        return dxs, dw + FILL, Aw, d.sum((0, 2)) + FILL, d.abs().sum((0, 2))

    x, w, dout = ints((N, HW, Cin), seed), ints((Cout, Cin), seed + 1, F32), ints((N, Cout, HW), seed + 2, F32)
    dx, dw, db = launch(x, w, dout)
    dxs, dw_ref, _, db_ref, _ = reference(x, w, dout)
    for n in range(N):
        exact("fd_final_conv_bwd", scalars, dx[n], dxs[n][0])
    exact("fd_final_conv_bwd", scalars, dw, dw_ref)
    exact("fd_final_conv_bwd", scalars, db, db_ref)
    assert all(torch.equal(a, b) for a, b in zip((dx, dw, db), launch(x, w, dout)))
    x, w = act((N, HW, Cin), seed + 3), rnd((Cout, Cin), seed + 4, 0.1)
    dout = rnd((N, Cout, HW), seed + 5)
    dout[:, 0] += 0.5
    dx, dw, db = launch(x, w, dout)
    dxs, dw_ref, Aw, db_ref, Ab = reference(x, w, dout)
    worst_dx = max(BL.ratio((dx[n].double() - r).abs(), BL.OUT_ROUND * r.abs() + 5 * 2.0 ** -24 * a)
                   for n, (r, a) in enumerate(dxs))
    worst_dw = BL.ratio((dw.double() - dw_ref).abs(), depth * 2.0 ** -24 * (Aw + FILL) + 2.0 ** -24 * Aw)
    worst_db = BL.ratio((db.double() - db_ref).abs(), depth * 2.0 ** -24 * (Ab + FILL))
    report("fd_final_conv_bwd", scalars, nulls, dx_err_over_bound=worst_dx, dw_err_over_bound=worst_dw,
           db_err_over_bound=worst_db, exact_leg_bit_exact=1.0)
    assert max(worst_dx, worst_dw, worst_db) <= 1


# ------------------------------------------------------------------------------------------------ time-path layers
def _act64(x, act):
    """act(x), act'(x) in float64 and the bounds of the kernel's fp32 forms (fd_unet_bwd.cu:656-669: expf / erff / division,
    each a few ulp): act 2^-20 |act| + 2^-21 |x| (the absolute error of 1 + erff), act' 2^-20 (1 + |x| + x^2)."""
    if act == 0:
        return x, torch.ones_like(x), torch.zeros_like(x), torch.zeros_like(x)
    if act == 1:
        s = torch.sigmoid(x)
        f, d = x * s, s * (1 + x * (1 - s))
    else:
        f = torch.nn.functional.gelu(x)
        d = 0.5 * (1 + torch.erf(x / math.sqrt(2))) + x * torch.exp(-0.5 * x * x) / math.sqrt(2 * math.pi)
    return f, d, 2.0 ** -20 * f.abs() + 2.0 ** -21 * x.abs(), 2.0 ** -20 * (1 + x.abs() + x * x)


def check_linear_bwd_w(L, scalars, nulls, seed):
    """fd_linear_bwd_w: dW[j][k] += sum_b dY[b][j] act(X[b][k]), db[j] += sum_b dY[b][j]; dY rows of stride dy_stride with
    the J-block at the end and NaN elsewhere.  Exact leg at act 0 (the entry's own activation on the real leg)."""
    lib = L.load()
    dys, xs, B, J, K, act_ = scalars
    off = dys - J

    def launch(dY, X, a):
        wb, dW = guarded((J, K), F32, FILL)
        bb, db = guarded((J,), F32, FILL)
        L.check(lib.fd_linear_bwd_w(dY.data_ptr() + 4 * off, dys, L.ptr(X), xs, L.ptr(dW), L.ptr(db), B, J, K, a, L.stream()))
        torch.cuda.synchronize()
        guard_intact(wb, dW)
        guard_intact(bb, db)
        return dW, db

    def rows(blk):
        r = torch.full((B, dys), NAN, device="cuda")
        r[:, off:] = blk
        return r

    dY, X = ints((B, J), seed, F32), ints((B, xs), seed + 1, F32)
    dW, db = launch(rows(dY), X, 0)
    exact("fd_linear_bwd_w", scalars, dW, dY.double().t() @ X.double()[:, :K] + FILL)
    exact("fd_linear_bwd_w", scalars, db, dY.double().sum(0) + FILL)
    dY, X = rnd((B, J), seed + 2), rnd((B, xs), seed + 3, 1.5)
    dY[:, :J // 2] += 0.5
    dW, db = launch(rows(dY), X, act_)
    d, x = dY.double(), X.double()[:, :K]
    f, _, df, _ = _act64(x, act_)
    ref = d.t() @ f + FILL
    bound = d.abs().t() @ df + (B + 2) * 2.0 ** -24 * (d.abs().t() @ f.abs() + FILL)
    worst_w = BL.ratio((dW.double() - ref).abs(), bound)
    worst_b = BL.ratio((db.double() - d.sum(0) - FILL).abs(), (B + 1) * 2.0 ** -24 * (d.abs().sum(0) + FILL))
    report("fd_linear_bwd_w", scalars, nulls, dw_err_over_bound=worst_w, db_err_over_bound=worst_b, exact_leg_bit_exact=1.0)
    assert max(worst_w, worst_b) <= 1


def check_linear_bwd_x(L, scalars, nulls, seed):
    """fd_linear_bwd_x: dX[b][k] = act'(A[b][k]) sum_j dY[b][j] W[j][k] (8 j-lanes of J / 8 terms, then 8 partials).
    Exact leg at act 0."""
    lib = L.load()
    dys, as_, dxs, B, J, K, act_ = scalars

    def launch(dY, W, A, a):
        buf, dX = guarded((B, dxs), F32, NAN)
        L.check(lib.fd_linear_bwd_x(L.ptr(dY), dys, L.ptr(W), L.ptr(A), as_, L.ptr(dX), dxs, B, J, K, a, L.stream()))
        torch.cuda.synchronize()
        guard_intact(buf, dX)
        return dX[:, :K]

    dY, W, A = ints((B, dys), seed, F32), ints((J, K), seed + 1, F32), rnd((B, as_), seed + 2)
    exact("fd_linear_bwd_x", scalars, launch(dY, W, A, 0), dY.double()[:, :J] @ W.double())
    dY, W, A = rnd((B, dys), seed + 3), rnd((J, K), seed + 4, J ** -0.5), rnd((B, as_), seed + 5, 1.5)
    dX = launch(dY, W, A, act_)
    s = dY.double()[:, :J] @ W.double()
    sa = dY.double()[:, :J].abs() @ W.double().abs()
    _, d, _, dd = _act64(A.double()[:, :K], act_)
    ref = s * d
    bound = (J // 8 + 10) * 2.0 ** -24 * sa * d.abs() + s.abs() * dd + 2.0 ** -24 * ref.abs()
    worst = BL.ratio((dX.double() - ref).abs(), bound)
    report("fd_linear_bwd_x", scalars, nulls, err_over_bound=worst, exact_leg_bit_exact=1.0)
    assert worst <= 1


def check_time_embed_save(L, scalars, nulls, seed):
    """fd_time_embed_save: temb, the sinusoidal embedding pe and the pre-GELU activations, each within the forward
    checker's propagated bound (test_gpu_bench_launches.time_embed_ref)."""
    lib = L.load()
    B, dim, tdim = scalars
    t = torch.tensor([0, 999, 1, 17, 250, 500, 750, 998][:B], device="cuda")
    sd = {"time_mlp.1.weight": rnd((tdim, dim), seed, 0.1), "time_mlp.1.bias": rnd((tdim,), seed + 1),
          "time_mlp.3.weight": rnd((tdim, tdim), seed + 2, 0.05), "time_mlp.3.bias": rnd((tdim,), seed + 3)}
    bufs = [guarded(s, F32, NAN) for s in ((B, tdim), (B, dim), (B, tdim))]
    temb, pe, pre = (v for _, v in bufs)
    L.check(lib.fd_time_embed_save(L.ptr(t), *(L.ptr(sd[k]) for k in ("time_mlp.1.weight", "time_mlp.1.bias",
                                                                      "time_mlp.3.weight", "time_mlp.3.bias")),
                                   L.ptr(temb), L.ptr(pe), L.ptr(pre), B, dim, tdim, L.stream()))
    torch.cuda.synchronize()
    for b, v in bufs:
        guard_intact(b, v)
    pe_r, dpe, h, dh, ref, bound = GPU.time_embed_ref(sd, t, dim, tdim)
    r = {k: BL.ratio((got.double() - want).abs(), b) for k, got, want, b in
         (("temb", temb, ref, bound), ("pe", pe, pe_r, dpe), ("pre", pre, h, dh))}
    report("fd_time_embed_save", scalars, nulls, **{f"{k}_err_over_bound": v for k, v in r.items()})
    assert max(r.values()) <= 1


# ------------------------------------------------------------------------------------------- GroupNorm / LayerNorm
def check_gn_silu(L, scalars, nulls, seed):
    """fd_gn_silu (the training forward's exp-form SiLU, __expf / __fdividef): silu(z) to (2^-20 + 2^-24 |z|) |silu| (the
    exponent's argument rounding grows with |z|, ex2.approx and the division a few ulp) plus silu's Lipschitz constant on
    the error of z."""
    def silu_exp(z, dz):
        s = z * torch.sigmoid(z)
        return s, (2.0 ** -20 + 2.0 ** -24 * z.abs()) * s.abs() + BL.LIP_SILU * dz
    GPU.check_gn_silu_form(L, "fd_gn_silu", silu_exp, scalars, nulls, seed)


def far_act(shape, seed):
    """act() with group 0 of every sample moved 12 of its standard deviations away from zero and group 5 by -15: the
    (sample, group) pairs where the GroupNorm backward's raw-moment formulas cancel most."""
    N, C = shape[0], shape[-1]
    x = act(shape, seed).float()
    n = torch.arange(N, device="cuda", dtype=F32).view((N,) + (1,) * (len(shape) - 1))
    cpg = C // 8
    x[..., :cpg] += 12 * (0.5 + 0.25 * n)
    x[..., 5 * cpg:6 * cpg] -= 15 * (0.5 + 0.25 * n)
    return x.to(BF)


def check_gn_silu_bwd(L, scalars, nulls, seed):
    """fd_gn_silu_bwd: dh, and dgamma / dbeta / dbias (+=) and the d(scale, shift) rows, against train_launches.gn_bwd_sample
    sample by sample.  Inputs include (sample, group) pairs with |mean| / std >= 10 (far_act)."""
    lib = L.load()
    stride, N, HW, C, eps = scalars
    use_ss = nulls[5] == "P"
    h = far_act((N, HW, C), seed)
    st = GPU.stats64(h)
    da = coherent((N, HW, C), seed + 1)
    gamma, beta = GPU.norm_params(C, seed + 2)
    rows, off, sc, sh = GPU.ss_rows(N, C, stride, seed + 3) if use_ss else (None, 0, None, None)
    ws = torch.empty(lib.fd_gn_silu_bwd_workspace_floats(N, C), device="cuda")
    depth = TL.gn_bwd_depth(N, HW, C, sms())[0]

    def launch():
        hb, dh = guarded((N, HW, C), BF, NAN)
        acc = [guarded((C,), F32, FILL) for _ in range(3)]
        dss = torch.full((N, stride), NAN, device="cuda") if use_ss else None
        L.check(lib.fd_gn_silu_bwd(L.ptr(h), L.ptr(da), L.ptr(st), L.ptr(gamma), L.ptr(beta),
                                   rows.data_ptr() + 4 * off if use_ss else None, stride, L.ptr(dh), L.ptr(acc[0][1]),
                                   L.ptr(acc[1][1]), dss.data_ptr() + 4 * off if use_ss else None, L.ptr(acc[2][1]), L.ptr(ws),
                                   N, HW, C, eps, L.stream()))
        torch.cuda.synchronize()
        guard_intact(hb, dh)
        for b, v in acc:
            guard_intact(b, v)
        if use_ss:
            assert bool(torch.isnan(dss[:, :off]).all()), "write outside the d(scale, shift) block"
        return dh, acc[0][1], acc[1][1], acc[2][1], dss

    dh, dgamma, dbeta, dbias, dss = launch()
    g64, b64 = gamma.double(), beta.double()
    worst = dict(dh=0.0, dss=0.0)
    tg, tb, tbias = [], [], []
    u = 2.0 ** -24
    for n in range(N):
        r = TL.gn_bwd_sample(h[n].double(), da[n].double(), st[n], g64, b64, eps, depth, sc[n] if use_ss else None,
                             sh[n] if use_ss else None)
        worst["dh"] = max(worst["dh"], BL.ratio((dh[n].double() - r["dh"][0]).abs(), r["dh"][1]))
        (S0, e0), (Sx, eSx), s1 = r["S0"], r["Sx"], r["s1"]
        tg.append((s1 * Sx, s1.abs() * eSx + 2 * u * (s1 * Sx).abs()))
        tb.append((s1 * S0, s1.abs() * e0 + 2 * u * (s1 * S0).abs()))
        tbias.append(r["dbias"])
        if use_ss:
            dsc = g64 * Sx + b64 * S0
            esc = g64.abs() * eSx + b64.abs() * e0 + 3 * u * ((g64 * Sx).abs() + (b64 * S0).abs())
            got = dss[n, off:].double()
            worst["dss"] = max(worst["dss"], BL.ratio((got[:C] - dsc).abs(), esc), BL.ratio((got[C:] - S0).abs(), e0))
        del r
    for k, got, terms in (("dgamma", dgamma, tg), ("dbeta", dbeta, tb), ("dbias", dbias, tbias)):
        ref, bound = TL.accumulated(terms)
        worst[k] = BL.ratio((got.double() - ref).abs(), bound)
    report("fd_gn_silu_bwd", scalars, nulls, **{f"{k}_err_over_bound": v for k, v in worst.items()})
    assert max(worst.values()) <= 1
    assert torch.equal(dh, launch()[0])


def check_chan_layernorm_bwd(L, scalars, nulls, seed):
    """fd_chan_layernorm_bwd: dx (+ add) and dg += sum dy xh against train_launches.ln_bwd_ref, sample by sample."""
    lib = L.load()
    npix, C, eps = scalars
    use_add = nulls[3] == "P"
    P = npix // 8
    x = act((8, P, C), seed).view(npix, C)
    dy = coherent((npix, C), seed + 1)
    gain = rnd((C,), seed + 2, 0.3, 1.0)
    add = act((8, P, C), seed + 3).view(npix, C) if use_add else None
    depth = TL.ln_dg_depth(npix, C, sms())

    def launch():
        xb, dx = guarded((npix, C), BF, NAN)
        gb, dg = guarded((C,), F32, FILL)
        L.check(lib.fd_chan_layernorm_bwd(L.ptr(x), L.ptr(gain), L.ptr(dy), L.ptr(add), L.ptr(dx), L.ptr(dg), npix, C, eps,
                                          L.stream()))
        torch.cuda.synchronize()
        guard_intact(xb, dx)
        guard_intact(gb, dg)
        return dx, dg

    dx, dg = launch()
    worst, terms = 0.0, []
    for n in range(8):
        sl = slice(n * P, (n + 1) * P)
        d = dy[sl].double()
        ref, bound, xh, exh = TL.ln_bwd_ref(x[sl].double(), gain.double(), d, eps)
        if use_add:
            ref = ref + add[sl].double()
            bound = bound + 2.0 ** -24 * ref.abs()
        worst = max(worst, BL.ratio((dx[sl].double() - ref).abs(), BL.OUT_ROUND * ref.abs() + (1 + BL.OUT_ROUND) * bound))
        terms.append(((d * xh).sum(0), (d.abs() * exh).sum(0) + depth * 2.0 ** -24 * (d * xh).abs().sum(0)))
        del d, ref, bound, xh, exh
    ref, bound = TL.accumulated(terms)
    worst_dg = BL.ratio((dg.double() - ref).abs(), bound)
    report("fd_chan_layernorm_bwd", scalars, nulls, dx_err_over_bound=worst, dg_err_over_bound=worst_dg)
    assert worst <= 1 and worst_dg <= 1
    assert torch.equal(dx, launch()[0])


# ----------------------------------------------------------------------------------------------- attention cores
def _qkv(N, HW, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    n = torch.arange(N, device="cuda", dtype=F32).view(N, 1, 1)
    return (torch.randn(N, HW, 384, generator=g, device="cuda") * (1.0 + 0.07 * n) + 0.2 * (n - 3.5)).to(BF)


def _core64(qkv_n, linear):
    """The LinearAttention / Attention core of one sample in float64 with autograd: qkv (HW, 384) -> out (HW, 128)."""
    x = qkv_n.double().t().reshape(1, 384, -1, 1).requires_grad_(True)
    return x, GPU._attn_core(x, linear)[0].reshape(128, -1).t()


def _slices_err(got, want):
    return max(GPU.rel_err(got[:, s], want[:, s]) for s in (slice(0, 128), slice(128, 256), slice(256, 384)))


def check_linattn_save(L, scalars, nulls, seed):
    """fd_linattn_save: the core per sample at fd_linattn's 1.5e-2; its statistics give fd_linattn_bwd the same dqkv as the
    stats = NULL path (to test_linattn_bwd's 1e-2)."""
    lib = L.load()
    N, HW = scalars
    qkv = _qkv(N, HW, seed)
    ws = torch.empty(lib.fd_linattn_workspace_floats(N, HW), device="cuda")
    ob, out = guarded((N, HW, 128), BF, NAN)
    sb, stats = guarded((N, lib.fd_linattn_stats_floats()), F32, NAN)
    L.check(lib.fd_linattn_save(L.ptr(qkv), L.ptr(out), L.ptr(stats), L.ptr(ws), N, HW, L.stream()))
    torch.cuda.synchronize()
    guard_intact(ob, out)
    guard_intact(sb, stats)
    errs = []
    for n in range(N):
        with torch.no_grad():
            errs.append(GPU.rel_err(out[n].double(), _core64(qkv[n], True)[1]))
    dout = rnd((N, HW, 128), seed + 1).to(BF)
    wsb = torch.empty(lib.fd_linattn_bwd_workspace_floats(N, HW), device="cuda")
    d = []
    for s in (stats, None):
        dq = torch.empty_like(qkv)
        L.check(lib.fd_linattn_bwd(L.ptr(qkv), L.ptr(dout), L.ptr(dq), L.ptr(s), L.ptr(wsb), N, HW, L.stream()))
        d.append(dq)
    torch.cuda.synchronize()
    e2 = max(GPU.rel_err(d[0][n].double(), d[1][n].double()) for n in range(N))
    report("fd_linattn_save", scalars, nulls, worst_sample_rel_err=max(errs), saved_vs_recomputed_stats_rel_err=e2)
    assert max(errs) < 1.5e-2 and e2 < 1e-2


def check_linattn_bwd(L, scalars, nulls, seed):
    """fd_linattn_bwd with the forward's saved statistics: dq, dk, dv per sample against float64 autograd at
    test_linattn_bwd's 2e-2."""
    lib = L.load()
    N, HW = scalars
    qkv = _qkv(N, HW, seed)
    ws = torch.empty(lib.fd_linattn_workspace_floats(N, HW), device="cuda")
    att = torch.empty(N, HW, 128, device="cuda", dtype=BF)
    stats = torch.empty(N, lib.fd_linattn_stats_floats(), device="cuda")
    L.check(lib.fd_linattn_save(L.ptr(qkv), L.ptr(att), L.ptr(stats), L.ptr(ws), N, HW, L.stream()))
    del ws, att
    dout = rnd((N, HW, 128), seed + 1).to(BF)
    wsb = torch.empty(lib.fd_linattn_bwd_workspace_floats(N, HW), device="cuda")
    db, dq = guarded((N, HW, 384), BF, NAN)
    L.check(lib.fd_linattn_bwd(L.ptr(qkv), L.ptr(dout), L.ptr(dq), L.ptr(stats), L.ptr(wsb), N, HW, L.stream()))
    torch.cuda.synchronize()
    guard_intact(db, dq)
    errs = []
    for n in range(N):
        x, out = _core64(qkv[n], True)
        out.backward(dout[n].double())
        errs.append(_slices_err(dq[n].double(), x.grad[0, :, :, 0].t()))
        del x, out
    report("fd_linattn_bwd", scalars, nulls, worst_sample_rel_err=max(errs))
    assert max(errs) < 2e-2, errs


def check_attention_lse(L, scalars, nulls, seed):
    """fd_attention_lse: the core per sample at fd_attention's 2e-2, and the log2-domain log-sum-exp to 2e-2."""
    lib = L.load()
    N, HW = scalars
    qkv = _qkv(N, HW, seed)
    ob, out = guarded((N, HW, 128), BF, NAN)
    lb, lse = guarded((N, 4, HW), F32, NAN)
    L.check(lib.fd_attention_lse(L.ptr(qkv), L.ptr(out), L.ptr(lse), N, HW, L.stream()))
    torch.cuda.synchronize()
    guard_intact(ob, out)
    guard_intact(lb, lse)
    errs, lerr = [], 0.0
    for n in range(N):
        with torch.no_grad():
            errs.append(GPU.rel_err(out[n].double(), _core64(qkv[n], False)[1]))
            q, k = qkv[n].double()[:, :128], qkv[n].double()[:, 128:256]
            for hd in range(4):
                sim = (q[:, 32 * hd:32 * hd + 32] * 32 ** -0.5) @ k[:, 32 * hd:32 * hd + 32].t()
                ref = torch.logsumexp(sim, 1) / math.log(2)
                lerr = max(lerr, (lse[n, hd].double() - ref).abs().max().item())
                del sim, ref
    report("fd_attention_lse", scalars, nulls, worst_sample_rel_err=max(errs), lse_abs_err=lerr)
    assert max(errs) < 2e-2 and lerr < 2e-2


def check_attention_bwd(L, scalars, nulls, seed):
    """fd_attention_bwd from fd_attention_lse's output and lse: dq, dk, dv per sample against float64 autograd at
    test_attention_bwd's 2.5e-2; atomic-free, so a second launch gives the same bits."""
    lib = L.load()
    N, HW = scalars
    qkv = _qkv(N, HW, seed)
    out = torch.empty(N, HW, 128, device="cuda", dtype=BF)
    lse = torch.empty(N, 4, HW, device="cuda")
    L.check(lib.fd_attention_lse(L.ptr(qkv), L.ptr(out), L.ptr(lse), N, HW, L.stream()))
    dout = rnd((N, HW, 128), seed + 1).to(BF)
    wsb = torch.empty(lib.fd_attention_bwd_workspace_floats(N, HW), device="cuda")

    def launch():
        db, dq = guarded((N, HW, 384), BF, NAN)
        L.check(lib.fd_attention_bwd(L.ptr(qkv), L.ptr(out), L.ptr(dout), L.ptr(lse), L.ptr(dq), L.ptr(wsb), N, HW, L.stream()))
        torch.cuda.synchronize()
        guard_intact(db, dq)
        return dq

    dq = launch()
    errs = []
    for n in range(N):
        x, o = _core64(qkv[n], False)
        o.backward(dout[n].double())
        errs.append(_slices_err(dq[n].double(), x.grad[0, :, :, 0].t()))
        del x, o
    report("fd_attention_bwd", scalars, nulls, worst_sample_rel_err=max(errs))
    assert max(errs) < 2.5e-2, errs
    assert torch.equal(dq, launch())


# --------------------------------------------------------------------------------------------- weight (un)packing
def _bench_net():
    from opticalflowdiffusion_b200.unet import Unet
    torch.manual_seed(0)
    net = Unet(64, 5, 2).cuda()
    net.prepare()
    from opticalflowdiffusion_b200 import _lib
    net._lib, net._st = _lib.load(), _lib.stream()        # what Unet._begin sets for a forward
    return net


def check_prep_weight_dgrad_batch(L, scalars, nulls, seed):
    """fd_prep_weight_dgrad_batch over the seed-0 benchmark network, NaN-prefilled: a pure permutation,
    wd[ci][(T-1-tap)*Cout + co] = w[co][tap*Cin + ci], bit-exact."""
    net = _bench_net()
    convs = [pc for pc in net._convs.values() if pc.kind < 2]
    blocks = 0
    for pc in convs:
        cout, k = pc.w.shape
        taps = 1 if pc.kind == 1 else pc.kh * pc.kw
        pc.wd = torch.full((k // taps, taps * cout), NAN, device="cuda", dtype=BF)
        blocks += -(-(k // taps) // 32) * -(-cout // 32) * taps
    assert (len(convs), blocks) == scalars
    net._prepare_dgrad()
    torch.cuda.synchronize()
    for pc in convs:
        cout, k = pc.w.shape
        taps = 1 if pc.kind == 1 else pc.kh * pc.kw
        want = pc.w.reshape(cout, taps, k // taps).flip(1).permute(2, 1, 0).reshape(k // taps, taps * cout)
        assert torch.equal(pc.wd, want)
    report("fd_prep_weight_dgrad_batch", scalars, nulls, layers=len(convs), bit_exact=1.0)


def _unpack(g, kind, Cout, Cin, KH, KW):
    """fd_conv_wgrad's packed [Cout][K] -> torch [Cout][Cin][KH][KW] (the kinds of fd_prep_weight)."""
    if kind == 0:
        return g.view(Cout, KH, KW, Cin).permute(0, 3, 1, 2)
    if kind == 1:
        return g.view(Cout, 4, Cin // 4).permute(0, 2, 1).reshape(Cout, Cin, 1, 1)
    if kind == 2:
        return g.view(Cout, KH, 64)[:, :, :KW * Cin].reshape(Cout, KH, KW, Cin).permute(0, 3, 1, 2)
    return g.view(Cout, KH, KW, 64)[..., :Cin].permute(0, 3, 1, 2)


def check_prep_weight_bwd_batch(L, scalars, nulls, seed):
    """fd_prep_weight_bwd_batch for one gradient bucket of the seed-0 benchmark network, its layer table rebuilt by the
    UNet's own grouping code: dw += r (g - mean g - wt mean(g wt)) (or the unpacked g), every layer against float64.
    Bound: fp32 block sums of n = Cin KH KW terms (mean, variance, the two means of g) at n 2^-23 of their sums of |terms|,
    carried through wt = (w - mean) r and the final expression."""
    lib = L.load()
    n_layers, total_blocks, eps = scalars
    net = _bench_net()
    gb = net._grad_buffer()
    ws = net._wgrad_workspace()
    names = {}
    for name, pc in net._convs.items():
        if id(getattr(pc.src, "weight", None)) in gb.by_id:
            names.setdefault(net._grad_group_of(name), []).append(name)
    group = [g for g, e in ws["groups"].items() if (e[2], e[3]) == (n_layers, total_blocks)]
    assert len(group) == 1, group
    table, blk, n, blocks = ws["groups"][group[0]]
    gen = torch.Generator(device="cuda").manual_seed(seed)
    ws["flat"].copy_(torch.randn(ws["flat"].shape, generator=gen, device="cuda"))
    gb.flat.fill_(FILL)
    L.check(lib.fd_prep_weight_bwd_batch(L.ptr(table), L.ptr(blk), n, blocks, eps, L.stream()))
    torch.cuda.synchronize()
    worst, u = 0.0, 2.0 ** -24
    for name in names[group[0]]:
        pc = net._convs[name]
        w = pc.src.weight.detach().double()
        Cout, Cin, KH, KW = w.shape
        g = _unpack(ws["views"][name].double(), pc.kind, Cout, Cin, KH, KW).reshape(Cout, -1)
        got = gb.of(pc.src.weight).double().reshape(Cout, -1)
        wf = w.reshape(Cout, -1)
        m = wf.shape[1]
        if pc.ws:
            mean = wf.mean(1, keepdim=True)
            r = (wf.var(1, unbiased=False, keepdim=True) + eps).rsqrt()
            wt = (wf - mean) * r
            mg, mgw = g.mean(1, keepdim=True), (g * wt).mean(1, keepdim=True)
            core = g - mg - wt * mgw
            ref = FILL + r * core
            ewt = r * m * u * wf.abs().mean(1, keepdim=True) + wt.abs() * m * 2 * u
            emg = m * u * g.abs().mean(1, keepdim=True)
            emgw = (g.abs() * ewt).mean(1, keepdim=True) + m * 2 * u * (g * wt).abs().mean(1, keepdim=True)
            bound = r * (emg + wt.abs() * emgw + mgw.abs() * ewt + 4 * u * (g.abs() + mg.abs() + (wt * mgw).abs())) + \
                m * 2 * u * (r * core).abs() + u * ref.abs()
        else:
            # one fp32 addition FILL + g: round-to-nearest is off by at most half an ulp, <= 2^-24 |FILL + g| with equality
            # only at a power of two, where the sum is exact -- so this term reaches a ratio just below 1 whenever a sum
            # lands just above a power of two, and never exceeds it
            ref, bound = FILL + g, u * (FILL + g).abs()
        worst = max(worst, BL.ratio((got - ref).abs(), bound))
    report(f"fd_prep_weight_bwd_batch[{group[0]}]", scalars, nulls, err_over_bound=worst)
    assert worst <= 1


CHECKERS = {
    "fd_conv_igemm": check_conv_train,
    "fd_conv_igemm_rt": GPU.check_conv_igemm_rt,
    "fd_chan_layernorm": GPU.check_chan_layernorm,
    "fd_pack_input_pad": GPU.check_pack_input_pad,
    "fd_time_proj": GPU.check_time_proj,
    "fd_gn_silu": check_gn_silu,
    "fd_linattn_save": check_linattn_save,
    "fd_attention_lse": check_attention_lse,
    "fd_upsample2x": check_upsample2x,
    "fd_final_conv_crop": check_final_conv_crop,
    "fd_time_embed_save": check_time_embed_save,
    "fd_prep_weight_dgrad_batch": check_prep_weight_dgrad_batch,
    "fd_conv_igemm_ex": check_conv_ex,
    "fd_conv_wgrad": check_wgrad,
    "fd_gn_silu_bwd": check_gn_silu_bwd,
    "fd_chan_layernorm_bwd": check_chan_layernorm_bwd,
    "fd_linattn_bwd": check_linattn_bwd,
    "fd_attention_bwd": check_attention_bwd,
    "fd_bias_grad": check_bias_grad,
    "fd_add_bf16": check_add_bf16,
    "fd_upsample2x_bwd": check_upsample2x_bwd,
    "fd_final_conv_bwd": check_final_conv_bwd,
    "fd_linear_bwd_w": check_linear_bwd_w,
    "fd_linear_bwd_x": check_linear_bwd_x,
    "fd_prep_weight_bwd_batch": check_prep_weight_bwd_batch,
}


@pytest.mark.parametrize("index, entry", [pytest.param(i, e, id=f"{i:03d}-{e[0]}") for i, e in enumerate(TL.TRAIN)])
def test_train_launch(L, index, entry):
    name, scalars, nulls, _ = entry
    CHECKERS[name](L, scalars, nulls, 5000 + 16 * index)


# ------------------------------------------------------------------------------------- the rest of the training step
def test_q_sample_train_shape(L):
    """fd_q_sample at the train step's 8 x 2 x 368 x 768, bit-exact against the oracle."""
    from test_gpu_sampling import make_algo
    m = make_algo(["algorithm.target=flow"])
    g = torch.Generator().manual_seed(21)
    x0, noise = torch.randn(8, 2, 368, 768, generator=g), torch.randn(8, 2, 368, 768, generator=g)
    t = torch.tensor([0, 999, 1, 17, 250, 500, 750, 998])
    out = m.model.q_sample(x0.cuda(), t.cuda(), noise.cuda())
    assert torch.equal(out.cpu(), O.q_sample(O.make_schedule(1000), x0, t, noise))


@pytest.mark.parametrize("holes", [False, True])
def test_nan_mse_train_shape(L, holes):
    """fd_nan_mse_fwd / _bwd over n = 4,521,984 (8 x 2 x 368 x 768), with and without NaN holes in the target, through
    diffusion._SqErrSums as the training step calls them, against float64: the count exactly, the sum of squares to
    2^-10 relative (fp32 partial sums of at most n terms are far inside), and the gradient of sum / count, 2 (p - t) /
    count, to 2^-21 relative and zero at the holes."""
    from opticalflowdiffusion_b200.diffusion import _SqErrSums
    g = torch.Generator(device="cuda").manual_seed(22 + holes)
    pred = torch.randn(8, 2, 368, 768, generator=g, device="cuda").requires_grad_(True)
    target = torch.randn(8, 2, 368, 768, generator=g, device="cuda") * 1.5 + 0.2
    if holes:
        target[torch.rand(target.shape, generator=g, device="cuda") < 0.05] = NAN
    num, den = _SqErrSums.apply(pred, target)
    (num / den).backward()
    keep = ~torch.isnan(target)
    count = keep.sum().item()
    assert den.item() == count and (count < pred.numel()) == holes
    d = (pred.detach().double() - target.double())[keep]
    ref = (d * d).sum()
    assert abs(num.item() - ref.item()) <= 2.0 ** -10 * ref.item()
    want = torch.zeros_like(pred, dtype=F64)
    want[keep] = 2 * d / count
    err = (pred.grad.double() - want).abs()
    assert bool((err <= 2.0 ** -21 * want.abs()).all())
    assert bool((pred.grad[~keep] == 0).all())


def test_sumsq_and_adam_parameter_count(L):
    """fd_sumsq and fd_adam_step over the benchmark network's 35,717,314 parameters (2 mod 4: the scalar tail runs) with
    a gradient whose norm engages the clip at max_grad_norm = 100.  fd_sumsq: fp32 atomics of per-thread fp32 sums,
    bounded by (4 iterations + block sum + one atomic per block) 2^-24 of the sum; fd_adam_step as test_adam_clip."""
    lib = L.load()
    n = 35717314
    assert n % 4 == 2
    g = torch.Generator(device="cuda").manual_seed(23)
    grad = torch.randn(n, generator=g, device="cuda") * 0.1
    grad[-2:] = 50.0                        # the tail carries weight in the sum
    ss = torch.zeros(1, device="cuda")
    L.check(lib.fd_sumsq(L.ptr(grad), n, L.ptr(ss), L.stream()))
    ref = grad.double().pow(2).sum().item()
    grid = min(-(-(n // 4) // 256), sms() * 8)
    depth = 4 * -(-(n // 4) // (grid * 256)) + 16 + grid + 1
    assert abs(ss.item() - ref) <= depth * 2.0 ** -24 * ref
    assert math.sqrt(ref) > 100
    # parameters of the gradient's sign: the decayed gradient g + wd p never nears 0, where Adam's first step (m / sqrt v
    # = g / (|g| + eps)) would turn the last-bit difference between two clip factors into a difference of order lr
    p0 = torch.randn(n, generator=g, device="cuda").abs() * grad.sign()
    p = p0.clone()
    m, v = torch.zeros(n, device="cuda"), torch.zeros(n, device="cuda")
    L.check(lib.fd_adam_step(L.ptr(p), L.ptr(grad), L.ptr(m), L.ptr(v), n, 1e-3, 0.9, 0.999, 1e-8, 1e-2, 1, L.ptr(ss), 100.0, 1.0,
                             L.stream()))
    refp = torch.nn.Parameter(p0.clone())
    refp.grad = grad.clone()
    torch.nn.utils.clip_grad_norm_([refp], 100.0)
    torch.optim.Adam([refp], lr=1e-3, weight_decay=1e-2).step()
    assert torch.allclose(p, refp.detach(), rtol=1e-5, atol=1e-6), (p - refp.detach()).abs().max()
