"""The distinct kernel launches of the UNet inference forward at the benchmark's shapes, and the error bounds their GPU
checks (tests/test_gpu_bench_launches.py) hold each launch to.

``record(B, H, W)`` runs ``Unet(64, 5, 2)`` under ``torch.no_grad()`` on the CPU with the library replaced by the
recording fake of tests/test_unet_host.py and returns every distinct ``(name, scalars, nulls)`` with its count.  Weight
preparation and size queries (``*_floats``) are left out: the checkers call them as set-up.  ``DEFAULT`` and ``MATRIX`` are
that record, committed, for the two bench.py workloads; tests/test_bench_launch_table.py re-records them on the CPU.

The bound functions take float64 tensors on any device; tests/test_bench_launch_table.py shows on the CPU that exact fp32
emulations pass them and that small mutations of the result do not."""
import collections

import torch

from opticalflowdiffusion_b200 import _lib

# launches the checkers run as set-up, not as cases of their own
SETUP = ("fd_prep_weight_batch", "fd_prep_weight_upconv", "fd_linattn_tc_prep")


def record(B, H, W, train=False):
    """{(name, scalars, nulls): count} of one inference forward of Unet(64, 5, 2) on a B x H x W batch, in launch order.
    ``nulls`` has one character per pointer argument: "P" for a pointer, "0" for NULL (the stream is always "0").
    ``train``: the training forward (autograd on) and its backward from ``out.backward(ones)`` instead."""
    from test_unet_host import _Event, _FakeLib
    from opticalflowdiffusion_b200.unet import Unet

    lib = _FakeLib()
    saved = (_lib.load, _lib.stream, _lib.require_cuda, torch.cuda.Event)
    _lib.load, _lib.stream, _lib.require_cuda = (lambda check_device=False: lib), (lambda: 0), (lambda *t: None)
    torch.cuda.Event = _Event
    try:
        torch.manual_seed(0)
        net = Unet(64, 5, 2)
        args = torch.zeros(B, 2, H, W), torch.zeros(B, 3, H, W), torch.full((B,), 17)
        if train:
            out = net(*args)
            out.backward(torch.ones_like(out))
        else:
            with torch.no_grad():
                net(*args)
    finally:
        _lib.load, _lib.stream, _lib.require_cuda, torch.cuda.Event = saved
    seen = collections.OrderedDict()
    for c in lib.calls:
        if c.name in SETUP or c.name.endswith("_floats"):
            continue
        key = (c.name, c.scalars, "".join("0" if z else "P" for z in c.nulls))
        seen[key] = seen.get(key, 0) + 1
    return seen


def as_table(seen):
    return [(name, scalars, nulls, count) for (name, scalars, nulls), count in seen.items()]


# ---------------------------------------------------------------------------------------------------------------- bounds
OUT_ROUND = 2.0 ** -8       # one bf16 rounding of the output (unit roundoff 2^-9), doubled for |got| vs |ref|
ACT_ROUND = 2.0 ** -9       # one bf16 rounding of an activation the kernel feeds to the MMA
EPS_TANH = 2.0 ** -10.987   # maximum relative error of tanh.approx.f32 (PTX ISA)
LIP_SILU = 1.1              # max |silu'(z)| = 1.0998


def gamma_mma(K):
    """fp32 accumulation error of a K-term tensor-core dot product of bf16 operands, relative to sum |x w|.  The products
    are exact.  The textbook K * 2^-24 assumes round-to-nearest additions; the tensor cores align the products of one MMA
    step to the largest exponent and truncate, so each term can lose one unit in the last place of the running sum
    (2^-23) in the alignment and another in the truncated addition: 2^-22 per term."""
    return K * 2.0 ** -22


def conv_bound(ref, A, K, act=None):
    """|got - ref| of a convolution whose fp64 reference ``ref`` works on the same bf16 operands: one output rounding, the
    accumulation error on ``A`` = sum |x w| (+ |bias| + |residual|), and ``act`` = sum |w| * (error of the kernel's
    activated input) where the kernel computes its conv input itself."""
    b = OUT_ROUND * ref.abs() + gamma_mma(K) * A
    return b if act is None else b + act


def gn_affine(x, stats, gamma, beta, eps, scale=None, shift=None):
    """GroupNorm(8) of one sample x (P pixels, C channels; float64) from the fp64 sums ``stats`` (8, 2) the kernel is given,
    then (scale + 1, shift): the pre-activation z and the bound of its fp32 evaluation (the kernels fold mean, rstd, gamma,
    beta, scale and shift into z = a x + b in a handful of fp32 operations: 2^-20 of the magnitudes that enter)."""
    P, C = x.shape
    cnt = P * C / 8
    mean = stats[:, 0] / cnt
    rstd = ((stats[:, 1] / cnt - mean * mean).clamp(min=0) + eps).rsqrt()
    mean, rstd = mean.repeat_interleave(C // 8), rstd.repeat_interleave(C // 8)
    s1 = 1 + scale if scale is not None else torch.ones_like(gamma)
    sh = shift if shift is not None else torch.zeros_like(gamma)
    a = gamma * rstd * s1
    c = mean * a
    z = a * x + (beta * s1 - c + sh)
    mag = (a * x).abs() + c.abs() + (beta * s1).abs() + sh.abs()
    return z, 2.0 ** -20 * mag


def silu_tanh(z, dz):
    """silu(z) and the bound of the kernels' fp32 form h + h tanh.approx(h), h = z / 2, given the bound dz of z:
    |h| EPS_TANH |tanh h| <= |z| EPS_TANH / 2, one fp32 rounding, and silu's Lipschitz constant on dz."""
    s = z * torch.sigmoid(z)
    return s, 0.5 * EPS_TANH * z.abs() + 2.0 ** -23 * s.abs() + LIP_SILU * dz


def bf16_act(s, ds):
    """Bound of bf16(s~) - s for |s~ - s| <= ds: the error of the activation a kernel feeds to the MMA."""
    return ACT_ROUND * (s.abs() + ds) + ds


def stats_ref(ref, bound):
    """GroupNorm statistics of one sample (ref / bound: (C, pixels...) float64): the fp64 (sum, sum of squares) of every group
    of ``ref`` and their bounds sum(bound) and sum(2 |ref| bound + bound^2).  Both contain 2^-8 of sum |ref| (resp. 2 sum
    ref^2), far above the rounding of the kernel's fp32 partial sums (2^-24 per term over far fewer than 2^16 terms)."""
    r, b = ref.reshape(8, -1), bound.reshape(8, -1)
    sums = torch.stack((r.sum(1), (r * r).sum(1)), 1)
    bounds = torch.stack((b.sum(1), (2 * r.abs() * b + b * b).sum(1)), 1)
    return sums, bounds


def ratio(err, bound):
    """max(err / bound); <= 1 passes.  NaN (an unwritten element) counts as infinitely wrong."""
    err = torch.where(torch.isnan(err), torch.full_like(err, float("inf")), err)
    return (err / bound.clamp(min=1e-300)).max().item()


# bench.py ddim50_436x1024: batch 8, run on the 440 x 1024 frame (replicate pad of 2 rows at the top and bottom)
DEFAULT = [
    ("fd_time_embed", (8, 64, 256), "PPPPPP0", 1),
    ("fd_time_proj", (8, 256, 8064), "PPPP0", 1),
    ("fd_pack_input_pad", (8, 2, 3, 436, 1024, 2, 0, 440, 1024, 0), "PPP0", 1),
    ("fd_conv_igemm", (64, 0, 8, 440, 1024, 64, 7, 1, 3, 0, 0), "P0PP0P00", 1),
    ("fd_conv_igemm", (64, 0, 8, 440, 1024, 64, 3, 3, 1, 1, 0), "P0PP0PP0", 2),
    ("fd_conv3x3_gnsilu_in", (8064, 1e-05, 8, 440, 1024), "PPPPPPP0PP0", 5),
    ("fd_gn_silu_fast", (0, 8, 450560, 64, 1e-05), "PPPP0PP0", 2),
    ("fd_linattn_tc", (8, 450560, 64, 1e-05), "PPPPPPPPPPPP0", 2),
    ("fd_conv_igemm", (64, 0, 8, 220, 512, 64, 1, 1, 0, 0, 1), "P0PP0P00", 1),
    ("fd_conv_igemm", (64, 0, 8, 220, 512, 64, 3, 3, 1, 1, 0), "P0PP0PP0", 2),
    ("fd_conv3x3_gnsilu_in", (8064, 1e-05, 8, 220, 512), "PPPPPPP0PP0", 2),
    ("fd_gn_silu_fast", (0, 8, 112640, 64, 1e-05), "PPPP0PP0", 2),
    ("fd_linattn_tc", (8, 112640, 64, 1e-05), "PPPPPPPPPPPP0", 1),
    ("fd_conv_igemm", (64, 0, 8, 110, 256, 128, 1, 1, 0, 0, 1), "P0PP0P00", 1),
    ("fd_conv_igemm", (128, 0, 8, 110, 256, 128, 3, 3, 1, 1, 0), "P0PP0PP0", 4),
    ("fd_gn_silu_fast", (8064, 8, 28160, 128, 1e-05), "PPPPP0P0", 2),
    ("fd_gn_silu_fast", (0, 8, 28160, 128, 1e-05), "PPPP0PP0", 2),
    ("fd_linattn_tc", (8, 28160, 128, 1e-05), "PPPPPPPPPPPP0", 1),
    ("fd_conv_igemm", (128, 0, 8, 55, 128, 256, 1, 1, 0, 0, 1), "P0PP0P00", 1),
    ("fd_conv_igemm", (256, 0, 8, 55, 128, 256, 3, 3, 1, 1, 0), "P0PP0PP0", 4),
    ("fd_gn_silu_fast", (8064, 8, 7040, 256, 1e-05), "PPPPP0P0", 2),
    ("fd_gn_silu_fast", (0, 8, 7040, 256, 1e-05), "PPPP0PP0", 2),
    ("fd_chan_layernorm", (56320, 256, 1e-05), "PP0P0", 1),
    ("fd_conv_igemm", (256, 0, 8, 55, 128, 384, 1, 1, 0, 0, 0), "P0P00P00", 1),
    ("fd_linattn", (8, 7040), "PPP0", 2),
    ("fd_conv_igemm", (128, 0, 8, 55, 128, 256, 1, 1, 0, 0, 0), "P0PP0P00", 1),
    ("fd_chan_layernorm", (56320, 256, 1e-05), "PPPP0", 1),
    ("fd_conv_igemm", (256, 0, 8, 55, 128, 512, 3, 3, 1, 1, 0), "P0PP0P00", 1),
    ("fd_conv_igemm", (512, 0, 8, 55, 128, 512, 3, 3, 1, 1, 0), "P0PP0PP0", 6),
    ("fd_gn_silu_fast", (8064, 8, 7040, 512, 1e-05), "PPPPP0P0", 4),
    ("fd_gn_silu_fast", (0, 8, 7040, 512, 1e-05), "PPPP0PP0", 2),
    ("fd_chan_layernorm", (56320, 512, 1e-05), "PP0P0", 2),
    ("fd_conv_igemm", (512, 0, 8, 55, 128, 384, 1, 1, 0, 0, 0), "P0P00P00", 2),
    ("fd_attention", (8, 7040), "PP0", 1),
    ("fd_conv_igemm", (128, 0, 8, 55, 128, 512, 1, 1, 0, 0, 0), "P0PPPP00", 1),
    ("fd_conv_igemm", (512, 256, 8, 55, 128, 512, 3, 3, 1, 1, 0), "PPPP0PP0", 2),
    ("fd_conv_igemm_rt", (512, 256, 1e-05, 8, 55, 128, 512, 1, 1, 0, 0), "PPPPPPPPP0", 2),
    ("fd_conv_igemm", (128, 0, 8, 55, 128, 512, 1, 1, 0, 0, 0), "P0PP0P00", 1),
    ("fd_chan_layernorm", (56320, 512, 1e-05), "PPPP0", 1),
    ("fd_conv_igemm_up", (512, 8, 55, 128, 256), "PPPP0", 1),
    ("fd_conv_igemm", (256, 128, 8, 110, 256, 256, 3, 3, 1, 1, 0), "PPPP0PP0", 2),
    ("fd_gn_silu_fast", (8064, 8, 28160, 256, 1e-05), "PPPPP0P0", 2),
    ("fd_conv_igemm", (256, 0, 8, 110, 256, 256, 3, 3, 1, 1, 0), "P0PP0PP0", 2),
    ("fd_conv_igemm_rt", (256, 128, 1e-05, 8, 110, 256, 256, 1, 1, 0, 0), "PPPPPPPPP0", 2),
    ("fd_chan_layernorm", (225280, 256, 1e-05), "PP0P0", 1),
    ("fd_conv_igemm", (256, 0, 8, 110, 256, 384, 1, 1, 0, 0, 0), "P0P00P00", 1),
    ("fd_linattn", (8, 28160), "PPP0", 1),
    ("fd_conv_igemm", (128, 0, 8, 110, 256, 256, 1, 1, 0, 0, 0), "P0PP0P00", 1),
    ("fd_chan_layernorm", (225280, 256, 1e-05), "PPPP0", 1),
    ("fd_conv_igemm_up", (256, 8, 110, 256, 128), "PPPP0", 1),
    ("fd_conv_igemm", (128, 64, 8, 220, 512, 128, 3, 3, 1, 1, 0), "PPPP0PP0", 2),
    ("fd_gn_silu_fast", (8064, 8, 112640, 128, 1e-05), "PPPPP0P0", 2),
    ("fd_conv_igemm", (128, 0, 8, 220, 512, 128, 3, 3, 1, 1, 0), "P0PP0PP0", 2),
    ("fd_conv_igemm_rt", (128, 64, 1e-05, 8, 220, 512, 128, 1, 1, 0, 0), "PPPPPPPPP0", 2),
    ("fd_linattn_tc", (8, 112640, 128, 1e-05), "PPPPPPPPPPPP0", 1),
    ("fd_conv_igemm_up", (128, 8, 220, 512, 64), "PPPP0", 1),
    ("fd_conv_igemm", (64, 64, 8, 440, 1024, 64, 3, 3, 1, 1, 0), "PPPP0PP0", 3),
    ("fd_conv_igemm_rt", (64, 64, 1e-05, 8, 440, 1024, 64, 1, 1, 0, 0), "PPPPPPPPP0", 2),
    ("fd_conv_igemm", (64, 0, 8, 440, 1024, 64, 3, 3, 1, 1, 0), "P0PP0P00", 1),
    ("fd_conv_igemm_rt_head", (64, 64, 1e-05, 2, 8, 440, 1024, 436, 1024, 2, 0), "PPPPPPPPPPP0", 1),
]

# bench.py matrix_flow_1024x2048 (batch 2): only its two top levels (1024 x 2048 and 512 x 1024) and the fd_linattn core at
# 128 x 256.  Its lower levels run the kernel paths of DEFAULT at sizes DEFAULT already exceeds.
MATRIX = [
    ("fd_pack_input_pad", (2, 2, 3, 1024, 2048, 0, 0, 1024, 2048, 0), "PPP0", 1),
    ("fd_conv_igemm", (64, 0, 2, 1024, 2048, 64, 7, 1, 3, 0, 0), "P0PP0P00", 1),
    ("fd_conv_igemm", (64, 0, 2, 1024, 2048, 64, 3, 3, 1, 1, 0), "P0PP0PP0", 2),
    ("fd_conv3x3_gnsilu_in", (8064, 1e-05, 2, 1024, 2048), "PPPPPPP0PP0", 5),
    ("fd_gn_silu_fast", (0, 2, 2097152, 64, 1e-05), "PPPP0PP0", 2),
    ("fd_linattn_tc", (2, 2097152, 64, 1e-05), "PPPPPPPPPPPP0", 2),
    ("fd_conv_igemm", (64, 0, 2, 512, 1024, 64, 1, 1, 0, 0, 1), "P0PP0P00", 1),
    ("fd_conv_igemm", (64, 0, 2, 512, 1024, 64, 3, 3, 1, 1, 0), "P0PP0PP0", 2),
    ("fd_conv3x3_gnsilu_in", (8064, 1e-05, 2, 512, 1024), "PPPPPPP0PP0", 2),
    ("fd_gn_silu_fast", (0, 2, 524288, 64, 1e-05), "PPPP0PP0", 2),
    ("fd_linattn_tc", (2, 524288, 64, 1e-05), "PPPPPPPPPPPP0", 1),
    ("fd_linattn", (2, 131072), "PPP0", 1),
    ("fd_conv_igemm", (128, 64, 2, 512, 1024, 128, 3, 3, 1, 1, 0), "PPPP0PP0", 2),
    ("fd_gn_silu_fast", (8064, 2, 524288, 128, 1e-05), "PPPPP0P0", 2),
    ("fd_conv_igemm", (128, 0, 2, 512, 1024, 128, 3, 3, 1, 1, 0), "P0PP0PP0", 2),
    ("fd_conv_igemm_rt", (128, 64, 1e-05, 2, 512, 1024, 128, 1, 1, 0, 0), "PPPPPPPPP0", 2),
    ("fd_linattn_tc", (2, 524288, 128, 1e-05), "PPPPPPPPPPPP0", 1),
    ("fd_conv_igemm_up", (128, 2, 512, 1024, 64), "PPPP0", 1),
    ("fd_conv_igemm", (64, 64, 2, 1024, 2048, 64, 3, 3, 1, 1, 0), "PPPP0PP0", 3),
    ("fd_conv_igemm_rt", (64, 64, 1e-05, 2, 1024, 2048, 64, 1, 1, 0, 0), "PPPPPPPPP0", 2),
    ("fd_conv_igemm", (64, 0, 2, 1024, 2048, 64, 3, 3, 1, 1, 0), "P0PP0P00", 1),
    ("fd_conv_igemm_rt_head", (64, 64, 1e-05, 2, 2, 1024, 2048, 1024, 2048, 0, 0), "PPPPPPPPPPP0", 1),
]
