"""Host-side logic of the UNet forwards and backward on the CPU: the library is replaced by a fake that records every
call, so these tests check which kernels are launched with which sizes, not what they compute."""
from collections import namedtuple

import pytest
import torch

from opticalflowdiffusion_b200 import _lib
from opticalflowdiffusion_b200.unet import Unet

Call = namedtuple("Call", "name scalars nulls")     # nulls: one bool per pointer argument, True where it is NULL

# Unet(64, 5, 2) at 1 x 36 x 60 (run on the 40 x 64 frame): the algorithmic FLOPs of every conv launch of one inference
# forward, as the roofline pass of bench.py records them
FLOPS_36x60 = 8552775680.0


class _FakeLib:
    def __init__(self):
        self.calls = []

    def __getattr__(self, name):
        if not name.startswith("fd_"):
            raise AttributeError(name)
        argtypes = _lib.SIGNATURES[name][1]

        def fn(*args):
            assert len(args) == len(argtypes), (name, args)
            ptr = [t is _lib.c_void_p for t in argtypes]
            self.calls.append(Call(name, tuple(a for a, p in zip(args, ptr) if not p),
                                   tuple(not a for a, p in zip(args, ptr) if p)))
            return 4096 if name.endswith("_floats") else 0
        return fn

    def named(self, name):
        return [c for c in self.calls if c.name == name]


class _Event:
    def __init__(self, *args, **kwargs):
        pass

    def record(self, *args):
        pass


@pytest.fixture
def fake(monkeypatch):
    lib = _FakeLib()
    monkeypatch.setattr(_lib, "load", lambda check_device=False: lib)
    monkeypatch.setattr(_lib, "stream", lambda: 0)
    monkeypatch.setattr(_lib, "require_cuda", lambda *tensors: None)
    monkeypatch.setattr(torch.cuda, "Event", _Event)
    return lib


def _net(channels=5):
    torch.manual_seed(0)
    return Unet(64, channels, 2)


def _inputs(net, H, W):
    g = torch.Generator().manual_seed(1)
    return torch.randn(1, 2, H, W, generator=g), torch.randn(1, net.channels - 2, H, W, generator=g), torch.tensor([17])


@pytest.mark.parametrize("channels", [5, 35])
def test_forwards_pad_in_the_packing_and_crop_in_the_head(fake, monkeypatch, channels):
    """36 x 60 runs on the 40 x 64 frame: both forwards replicate-pad inside the packing kernel (pads 2, 2) and crop in
    the output head, without an ATen pad or copy."""
    def no_pad(*args, **kwargs):
        raise AssertionError("torch.nn.functional.pad called in the forward")

    monkeypatch.setattr(torch.nn.functional, "pad", no_pad)
    net = _net(channels)
    pack = "fd_pack_input_wide" if channels > 9 else "fd_pack_input_pad"
    x, cond, t = _inputs(net, 36, 60)
    with torch.no_grad():
        out = net(x, cond, t)
    assert out.shape == (1, 2, 36, 60)
    calls = fake.named(pack)
    assert len(calls) == 1 and calls[0].scalars[3:9] == (36, 60, 2, 2, 40, 64), calls

    fake.calls.clear()
    out, _ = net.forward_train(x, cond, t)
    assert out.shape == (1, 2, 36, 60)
    calls = fake.named(pack)
    assert len(calls) == 1 and calls[0].scalars[3:9] == (36, 60, 2, 2, 40, 64), calls
    last = fake.calls[-1]
    assert last.name == "fd_final_conv_crop" and last.scalars == (1, 40, 64, 64, 2, 2, 2, 36, 60), last


def test_conv_timing_records_every_conv_launch_once(fake):
    net = _net()
    x, cond, t = _inputs(net, 36, 60)
    net._conv_timing = []
    with torch.no_grad():
        net(x, cond, t)
    names = [name for name, _, _ in net._conv_timing]
    # the tcgen05 LinearAttention blocks (C = 64, 128) run their 1x1 convs inside fd_linattn_tc
    fused = {f"{blk}.{conv}" for blk in net._la_tc for conv in ("to_qkv", "to_out")}
    assert sorted(names) == sorted(set(net._convs) - fused)
    assert sum(flops for _, flops, _ in net._conv_timing) == FLOPS_36x60


def test_backward_announces_every_gradient_bucket_in_order(fake):
    class Sync:
        def __init__(self):
            self.buckets, self.finished = [], 0

        def bucket_ready(self, flat, lo, hi):
            self.buckets.append((lo, hi))

        def finish(self, flat):
            self.finished += 1

    net = _net()
    net.grad_sync = sync = Sync()
    x, cond, t = _inputs(net, 36, 60)
    out = net(x, cond, t)
    out.backward(torch.ones_like(out))
    ranges = net._grad_group_ranges()
    assert sync.buckets == [ranges[g] for g in net.GRAD_GROUPS]
    spans = sorted(sync.buckets)
    assert spans[0][0] == 0 and spans[-1][1] == net.grad_buffer.flat.numel()
    assert all(a[1] == b[0] for a, b in zip(spans[:-1], spans[1:]))
    assert sync.finished == 1
