"""CPU: the launch table of the benchmark's UNet forward (tests/bench_launches.py) matches what the UNet launches, every
kernel in it has a GPU checker, and the error bounds those checkers apply pass an exact fp32 emulation of the kernels'
arithmetic while rejecting small mutations of it."""
import pytest
import torch
import torch.nn.functional as F

import bench_launches as BL
import test_gpu_bench_launches as GPU


def test_default_workload_table_is_exact():
    """bench.py ddim50_436x1024: every distinct launch of the forward, with its count, in launch order."""
    assert BL.as_table(BL.record(8, 436, 1024)) == BL.DEFAULT


def test_matrix_flow_entries_are_launched():
    """bench.py matrix_flow_1024x2048: the committed top-level entries are launched with these counts."""
    got = BL.as_table(BL.record(2, 1024, 2048))
    missing = [e for e in BL.MATRIX if e not in got]
    assert not missing, missing


def test_every_kernel_has_a_checker():
    names = {e[0] for e in BL.DEFAULT + BL.MATRIX}
    assert names <= set(GPU.CHECKERS), names - set(GPU.CHECKERS)


# --------------------------------------------------------------------------------------------- the bounds have teeth
def bf16(t):
    return t.to(torch.bfloat16).to(t.dtype)


def _samples(N, C, H, W, g):
    """Every sample its own offset and scale, every (sample, group) its own mean, as the GPU checkers build them."""
    x = torch.randn(N, C, H, W, generator=g, dtype=torch.float64)
    scale = 0.5 + 0.25 * torch.arange(N, dtype=torch.float64)
    mu = torch.randn(N, 8, generator=g, dtype=torch.float64).repeat_interleave(C // 8, 1)
    return bf16(x * scale.view(N, 1, 1, 1) + mu.view(N, C, 1, 1) + 0.3 * torch.arange(N).view(N, 1, 1, 1))


def _conv_case(g, N=3, Cin=16, Cout=16, H=16, W=12):
    x = _samples(N, Cin, H, W, g)
    w = bf16(torch.randn(Cout, Cin, 3, 3, generator=g, dtype=torch.float64) / (9 * Cin) ** 0.5)
    bias = torch.randn(Cout, generator=g, dtype=torch.float64)
    return x, w, bias


def _conv_emulated(x, w, bias):
    """The kernel's arithmetic: fp32 accumulation of exact bf16 products, fp32 bias add, one bf16 output rounding."""
    return bf16(F.conv2d(x.float(), w.float(), bias.float(), padding=1)).double()


def _conv_ratio(x, w, bias, got):
    ref = F.conv2d(x, w, bias, padding=1)
    A = F.conv2d(x.abs(), w.abs(), padding=1) + bias.abs().view(1, -1, 1, 1)
    return BL.ratio((got - ref).abs(), BL.conv_bound(ref, A, w[0].numel()))


def test_conv_bound_accepts_fp32_and_rejects_mutations():
    g = torch.Generator().manual_seed(0)
    x, w, bias = _conv_case(g)
    good = _conv_emulated(x, w, bias)
    assert _conv_ratio(x, w, bias, good) <= 1
    w_drop = w.clone()
    w_drop[:, :, 0, 2] = 0                                        # one tap dropped
    assert _conv_ratio(x, w, bias, _conv_emulated(x, w_drop, bias)) > 1
    assert _conv_ratio(x, w, bias, _conv_emulated(x, w, 0 * bias)) > 1      # bias omitted
    shifted = good.clone()
    shifted[:, :, 8:] = good[:, :, 7:-1]                          # rows of the second 8-row tile moved down by one
    assert _conv_ratio(x, w, bias, shifted) > 1


def _stats(x):
    r = x.reshape(x.shape[0], 8, -1)
    return torch.stack((r.sum(-1), (r * r).sum(-1)), -1)


def _gn_silu_emulated(x, stats, gamma, beta, ss, C, eps=1e-5):
    """gn_silu_kernel<true> in fp32: folded a, b from the fp64 statistics, h = fma(a / 2, x, b / 2), y = fma(h, t, h) with
    t = tanh(h) off by the largest relative error tanh.approx.f32 may have, with alternating sign; bf16 output."""
    N, _, H, W = x.shape
    cnt = H * W * C / 8
    mean = stats[..., 0] / cnt
    var = (stats[..., 1] / cnt - mean * mean).clamp(min=0)
    rstd = (1.0 / (var + eps).sqrt()).float().repeat_interleave(C // 8, 1)
    meanf = mean.float().repeat_interleave(C // 8, 1)
    ga = gamma.float() * rstd
    be = beta.float() - meanf * ga
    if ss is not None:
        sc, sh = ss[:, :C].float() + 1, ss[:, C:].float()
        ga, be = ga * sc, be * sc + sh
    h = (0.5 * ga).view(N, C, 1, 1) * x.float() + (0.5 * be).view(N, C, 1, 1)
    sign = 1 - 2 * (torch.arange(h.numel()).view(h.shape) % 2)
    t = torch.tanh(h) * (1 + sign * 2.0 ** -11)
    return h + h * t


def _gn_silu_ratio(x, stats, gamma, beta, ss, got, conv_w=None, conv_b=None):
    """The GPU checkers' bound for fd_gn_silu_fast (conv_w None) or fd_conv3x3_gnsilu_in, sample by sample."""
    N, C = x.shape[:2]
    worst = 0.0
    for n in range(N):
        xs = x[n].reshape(C, -1).t()
        sc, sh = (ss[n, :C], ss[n, C:]) if ss is not None else (None, None)
        z, dz = BL.gn_affine(xs, stats[n], gamma, beta, 1e-5, sc, sh)
        s, ds = BL.silu_tanh(z, dz)
        s, ds = (t.t().reshape(1, *x.shape[1:]) for t in (s, ds))
        if conv_w is None:
            ref, bound = s, BL.OUT_ROUND * s.abs() + (1 + BL.OUT_ROUND) * ds
        else:
            da = BL.bf16_act(s, ds)
            ref = F.conv2d(s, conv_w, conv_b, padding=1)
            A = F.conv2d(s.abs() + da, conv_w.abs(), padding=1) + conv_b.abs().view(1, -1, 1, 1)
            bound = BL.conv_bound(ref, A, conv_w[0].numel(), F.conv2d(da, conv_w.abs(), padding=1))
        worst = max(worst, BL.ratio((got[n:n + 1] - ref).abs(), bound))
    return worst


@pytest.mark.parametrize("fused_conv", [False, True])
def test_gn_silu_bounds_accept_fp32_and_reject_swapped_samples(fused_conv):
    g = torch.Generator().manual_seed(1)
    N, C = 3, 16
    x = _samples(N, C, 10, 12, g)
    stats = _stats(x)
    gamma = 1 + 0.3 * torch.randn(C, generator=g, dtype=torch.float64)
    beta = 0.2 * torch.randn(C, generator=g, dtype=torch.float64)
    ss = 0.3 * torch.randn(N, 2 * C, generator=g, dtype=torch.float64) + 0.2 * torch.arange(N).view(N, 1)
    w = bf16(torch.randn(C, C, 3, 3, generator=g, dtype=torch.float64) / (9 * C) ** 0.5)
    b = torch.randn(C, generator=g, dtype=torch.float64)

    def run(st, rows):
        act = _gn_silu_emulated(x, st, gamma, beta, rows, C)
        if fused_conv:
            return bf16(F.conv2d(bf16(act.double()).float(), w.float(), b.float(), padding=1)).double()
        return bf16(act.double())

    check = (lambda got: _gn_silu_ratio(x, stats, gamma, beta, ss, got, w, b)) if fused_conv else \
        (lambda got: _gn_silu_ratio(x, stats, gamma, beta, ss, got))
    assert check(run(stats, ss)) <= 1
    swap = torch.tensor([1, 0, 2])
    assert check(run(stats[swap], ss)) > 1                      # statistics of two samples swapped
    assert check(run(stats, ss[swap])) > 1                      # scale / shift rows of two samples swapped


def test_conv_statistics_bound_rejects_swapped_samples():
    g = torch.Generator().manual_seed(2)
    x, w, bias = _conv_case(g)
    got = _conv_emulated(x, w, bias)
    got_stats = _stats(got)

    def worst(st):
        r = 0.0
        for n in range(x.shape[0]):
            ref = F.conv2d(x[n:n + 1], w, bias, padding=1)[0]
            A = F.conv2d(x[n:n + 1].abs(), w.abs(), padding=1)[0] + bias.abs().view(-1, 1, 1)
            sums, bounds = BL.stats_ref(ref, BL.conv_bound(ref, A, w[0].numel()))
            r = max(r, BL.ratio((st[n] - sums).abs(), bounds))
        return r

    assert worst(got_stats) <= 1
    assert worst(got_stats[torch.tensor([1, 0, 2])]) > 1
