"""Training-mode execution of the UNet: the forward pass that keeps what the backward needs, and the
backward pass itself, both as launches of ``libflowdiff.so`` kernels.

The reference trains through ``loss.backward()`` on the autograd graph of ``Unet.forward``
(denoising_diffusion.py:363-417, driven by flow_diffuser.py:217-235 / exp_base.py:193-214).  Here the whole UNet
is ONE ``torch.autograd.Function`` (``UnetFunction``): its forward records a tape of the kernels it launched, its
backward replays the tape in reverse with the matching backward kernels:

* every convolution: ``fd_conv_wgrad`` (tcgen05, K = pixels) + ``fd_prep_weight_bwd`` (unpacking + weight-
  standardisation backward) for the parameters, and the data gradient as the SAME implicit-GEMM convolution run
  on dy with flipped / transposed weights (``fd_prep_weight_dgrad``); where a tensor feeds several consumers the
  second gradient is added in the dgrad epilogue (its ``residual`` input) instead of a separate pass;
* GroupNorm + scale/shift + SiLU: ``fd_gn_silu_bwd`` (also yields the producing conv's bias gradient and the
  time-MLP gradients); channel LayerNorm, the two attention cores, nearest upsample, the final 1x1 conv and the
  time-embedding MLPs each have their kernel in ``csrc/fd_unet_bwd.cu`` / ``fd_attention_bwd.cu``.

Parameter gradients are accumulated in fp32 into one flat buffer (``unet.grad_buffer``); the Function returns
views of it, so ``p.grad`` is filled exactly as autograd would and any ``torch.optim`` optimiser -- or
``optim.FusedAdam`` on the flat buffer -- can step.  There is no PyTorch fallback for any of this arithmetic.
"""
from __future__ import annotations

from typing import Callable, Dict, List, Optional

import torch

from . import _lib

Tensor = torch.Tensor
BF16 = torch.bfloat16


def _batch_table(owner, attr: str, recs, blocks, dev):
    """Device copies of a batched-prep table (8 x int64 per layer) and its block prefix sums, cached on `owner`."""
    key = tuple(tuple(r) for r in recs)
    cur = getattr(owner, attr, None)
    if cur is None or cur[0] != key or cur[1].device != dev:
        cur = (key, torch.tensor(recs, dtype=torch.int64).to(dev), torch.tensor(blocks, dtype=torch.int32).to(dev))
        setattr(owner, attr, cur)
    return cur[1], cur[2]


class GradBuffer:
    """One flat fp32 buffer with a view per parameter (in ``module.parameters()`` order)."""

    def __init__(self, module: torch.nn.Module):
        params = list(module.parameters())
        dev = params[0].device
        sizes = [p.numel() for p in params]
        # 4-element alignment keeps every view 16-byte aligned
        offs, off = [], 0
        for n in sizes:
            offs.append(off)
            off += (n + 3) // 4 * 4
        self.flat = torch.zeros(off, device=dev, dtype=torch.float32)
        self.views: List[Tensor] = [self.flat[o:o + n].view_as(p) for o, n, p in zip(offs, sizes, params)]
        self.by_id: Dict[int, Tensor] = {id(p): v for p, v in zip(params, self.views)}
        self.device = dev
        self.key = tuple(id(p) for p in params)

    def zero_(self):
        self.flat.zero_()

    def of(self, param) -> Tensor:
        return self.by_id[id(param)]


class Tape:
    """Reverse-mode tape over bf16 NHWC activations.  Gradients are keyed by tensor identity; the closures keep
    their tensors alive until they have run."""

    def __init__(self, unet):
        self.unet = unet
        self.lib = unet._lib
        self.st = unet._st
        self.steps: List[Callable[[], None]] = []
        self.g: Dict[int, Tensor] = {}

    def record(self, fn: Callable[[], None]):
        self.steps.append(fn)

    def add_grad(self, t: Tensor, g: Tensor):
        k = id(t)
        cur = self.g.get(k)
        if cur is None:
            self.g[k] = g
        else:
            out = torch.empty_like(cur)
            _lib.check(self.lib.fd_add_bf16(_lib.ptr(cur), _lib.ptr(g), _lib.ptr(out), cur.numel(), self.st))
            self.g[k] = out

    def pop(self, t: Tensor) -> Tensor:
        return self.g.pop(id(t))

    def peek(self, t: Tensor) -> Optional[Tensor]:
        return self.g.get(id(t))

    def run(self):
        while self.steps:
            self.steps.pop()()
        self.g.clear()


class TrainMixin:
    """Methods mixed into ``unet.Unet``: training forward (records the tape) and helpers for the backward."""

    # ------------------------------------------------------------------ buffers / weights
    def _grad_buffer(self) -> GradBuffer:
        gb = getattr(self, "_gb", None)
        key = tuple(id(p) for p in self.parameters())
        dev = next(self.parameters()).device
        if gb is None or gb.key != key or gb.device != dev:
            gb = GradBuffer(self)
            self._gb = gb
        return gb

    @property
    def grad_buffer(self) -> GradBuffer:
        return self._grad_buffer()

    def _prepare_dgrad(self):
        """Flipped / transposed bf16 weights for the data-gradient convolutions; cached with the forward packing."""
        if getattr(self, "_dgrad_versions", None) == self._prepared_versions:
            return
        lib, st = self._lib, _lib.stream()
        recs, blocks = [], [0]
        for name, pc in self._convs.items():
            if pc.kind >= 2:
                continue
            cout, k = pc.w.shape
            taps = 1 if pc.kind == 1 else pc.kh * pc.kw
            cin = k // taps
            wd = getattr(pc, "wd", None)
            if wd is None or wd.device != pc.w.device:
                wd = torch.empty(cin, taps * cout, device=pc.w.device, dtype=BF16)
                pc.wd = wd
            recs.append([pc.w.data_ptr(), wd.data_ptr(), 0, cout, cin, taps, 0, 0])
            blocks.append(blocks[-1] + ((cin + 31) // 32) * ((cout + 31) // 32) * taps)
        # one launch for all layers (fd_prep_weight_dgrad_batch); the table is rebuilt only when a buffer moved
        table, blk = _batch_table(self, "_dgrad_table", recs, blocks, next(iter(self._convs.values())).w.device)
        _lib.check(lib.fd_prep_weight_dgrad_batch(_lib.ptr(table), _lib.ptr(blk), len(recs), blocks[-1], st))
        self._dgrad_versions = self._prepared_versions

    def _wgrad_workspace(self):
        """Flat fp32 buffer holding the packed weight gradient of every convolution (``fd_conv_wgrad`` accumulates into
        it) and the table for the single ``fd_prep_weight_bwd_batch`` launch that unpacks all of them at the end of the
        backward (78 zero-fills + 74 unpack launches per step otherwise)."""
        gb = self._gb
        convs = [(n, pc) for n, pc in self._convs.items() if id(getattr(pc.src, "weight", None)) in gb.by_id]
        key = (gb.flat.data_ptr(),) + tuple(pc.src.weight.data_ptr() for _, pc in convs)
        ws = getattr(self, "_gw_ws", None)
        if ws is not None and ws["key"] == key:
            return ws
        offs, off = [], 0
        for _, pc in convs:
            offs.append(off)
            off += (pc.w.numel() + 3) // 4 * 4
        dev = gb.flat.device
        flat = torch.zeros(off, device=dev, dtype=torch.float32)
        views, recs, blocks = {}, [], [0]
        for (name, pc), o in zip(convs, offs):
            v = flat[o:o + pc.w.numel()].view(pc.w.shape)
            views[name] = v
            wt = pc.src.weight
            recs.append([v.data_ptr(), wt.data_ptr(), gb.of(wt).data_ptr(), wt.shape[0], wt.shape[1], wt.shape[2], wt.shape[3],
                         pc.kind | (int(pc.ws) << 8)])
            blocks.append(blocks[-1] + wt.shape[0])
        ws = {"key": key, "flat": flat, "views": views, "n": len(recs), "blocks": blocks[-1],
              "table": torch.tensor(recs, dtype=torch.int64).to(dev), "blk": torch.tensor(blocks, dtype=torch.int32).to(dev)}
        # one sub-table per gradient bucket (GRAD_GROUPS): a bucket's weight gradients are unpacked -- and handed to the
        # gradient exchange -- as soon as the backward has walked past its layers, not at the end of the backward
        per = {}
        for (name, _), rec in zip(convs, recs):
            per.setdefault(self._grad_group_of(name), []).append(rec)
        ws["groups"] = {}
        for gname, grecs in per.items():
            gblocks = [0]
            for r in grecs:
                gblocks.append(gblocks[-1] + r[3])
            ws["groups"][gname] = (torch.tensor(grecs, dtype=torch.int64).to(dev), torch.tensor(gblocks, dtype=torch.int32).to(dev),
                                   len(grecs), gblocks[-1])
        self._gw_ws = ws
        return ws

    # ------------------------------------------------------------------ gradient buckets
    # Buckets of the flat gradient in the order the backward completes them (reverse layer order).  Every bucket is a
    # CONTIGUOUS range of the flat buffer (parameters are laid out in module order: init_conv, time_mlp, downs, ups, mid,
    # final) -- the unit of DDP's bucketed all-reduce (exp_base.py:198), overlapped with the rest of the backward by
    # optim.GradSync.  The deep levels hold 90 % of the parameters and finish first; the full-resolution levels, whose
    # backward takes longest, hold almost none, so only the small "front" bucket is exchanged after the last kernel.
    GRAD_GROUPS = ("final", "ups.23", "ups.1", "ups.0", "mid", "downs.3", "downs.2", "front")

    @staticmethod
    def _grad_group_of(name: str) -> str:
        if name.startswith(("final_res_block", "final_conv")):
            return "final"
        if name.startswith(("ups.2", "ups.3")):
            return "ups.23"
        if name.startswith(("ups.1", "ups.0", "downs.3", "downs.2")):
            return name[:name.index(".", name.index(".") + 1)]
        if name.startswith("mid_"):
            return "mid"
        return "front"            # init_conv, time_mlp, downs.0, downs.1

    def _grad_group_ranges(self):
        """{group: (lo, hi)} element ranges of the flat gradient buffer."""
        gb = self._gb
        cached = getattr(self, "_gg_ranges", None)
        if cached is not None and cached[0] is gb:
            return cached[1]
        base = gb.flat.data_ptr()
        ranges = {}
        for pname, p in self.named_parameters():
            g = self._grad_group_of(pname)
            v = gb.of(p)
            lo = (v.data_ptr() - base) // 4
            hi = (lo + v.numel() + 3) // 4 * 4
            cur = ranges.get(g)
            ranges[g] = (lo, hi) if cur is None else (min(cur[0], lo), max(cur[1], hi))
        hi_all = gb.flat.numel()
        spans = sorted(ranges.values())
        assert spans[0][0] == 0 and all(a[1] == b[0] for a, b in zip(spans[:-1], spans[1:])) and spans[-1][1] <= hi_all, spans
        self._gg_ranges = (gb, ranges)
        return ranges

    def _t_group_boundary(self, tape: "Tape", group: str):
        """Recorded BEFORE a group's first forward op, hence run AFTER its last backward op: unpack the group's packed
        weight gradients (+ weight-standardisation backward) into the flat buffer and announce the bucket."""
        lib, st = self._lib, self._st

        def bwd():
            ws = self._gw_ws
            ent = ws["groups"].get(group)
            if ent is not None:
                _lib.check(lib.fd_prep_weight_bwd_batch(_lib.ptr(ent[0]), _lib.ptr(ent[1]), ent[2], ent[3], self.WS_EPS, st))
            sync = getattr(self, "grad_sync", None)
            if sync is not None:
                lo, hi = self._grad_group_ranges()[group]
                sync.bucket_ready(self._gb.flat, lo, hi)

        tape.record(bwd)

    # ------------------------------------------------------------------ recorded ops
    def _t_conv(self, tape: Tape, name: str, src0: Tensor, src1: Optional[Tensor] = None,
                residual: Optional[Tensor] = None, stats: Optional[Tensor] = None, need_dgrad: bool = True,
                res_gn=None) -> Tensor:
        """``res_gn = (h2, stats2, norm, producing conv's bias)``: the residual is silu(GroupNorm(h2)), applied inside the
        conv's epilogue (fd_conv_igemm_rt); its backward is the GroupNorm + SiLU backward with this conv's dy as upstream."""
        if res_gn is not None:
            out = self._conv_res_gn(name, src0, src1, res_gn[0], res_gn[1], res_gn[2])
        else:
            out = self._conv(name, src0, src1, residual, stats)
        pc = self._convs[name]
        lib, st, gb = self._lib, self._st, self._gb

        def bwd():
            dy = tape.pop(out)
            n, h, w, cout = out.shape
            c0 = src0.shape[-1]
            c1 = src1.shape[-1] if src1 is not None else 0
            if residual is not None:
                tape.add_grad(residual, dy)
            if res_gn is not None:
                h2, st2, norm, conv_bias = res_gn
                dh = torch.empty_like(h2)
                wsb = torch.empty(lib.fd_gn_silu_bwd_workspace_floats(n, cout), device=h2.device, dtype=torch.float32)
                _lib.check(lib.fd_gn_silu_bwd(_lib.ptr(h2), _lib.ptr(dy), _lib.ptr(st2), _lib.ptr(norm.weight), _lib.ptr(norm.bias),
                                              None, 0, _lib.ptr(dh), _lib.ptr(gb.of(norm.weight)), _lib.ptr(gb.of(norm.bias)), None,
                                              _lib.ptr(gb.of(conv_bias)), _lib.ptr(wsb), n, h * w, cout, self.GN_EPS, st))
                tape.add_grad(h2, dh)
            mod = pc.src
            if mod.bias is not None and stats is None:      # with statistics the GroupNorm backward delivers it
                _lib.check(lib.fd_bias_grad(_lib.ptr(dy), _lib.ptr(gb.of(mod.bias)), n * h * w, cout, st))
            # packed weight gradient into this conv's slice of the workspace (zeroed at the start of the backward); the
            # unpacking + weight-standardisation backward of ALL convs is one launch at the end (forward_train.backward)
            gw = self._gw_ws["views"][name]
            _lib.check(lib.fd_conv_wgrad(_lib.ptr(src0), c0, _lib.ptr(src1), c1, _lib.ptr(dy), _lib.ptr(gw), n, h, w, cout,
                                         pc.kh, pc.kw, pc.pad[0], pc.pad[1], pc.mode, st))
            if not need_dgrad:
                return
            if pc.mode == 1:
                dsrc = torch.empty_like(src0)
                _lib.check(lib.fd_conv_igemm_ex(_lib.ptr(dy), cout, None, 0, _lib.ptr(pc.wd), None, None, _lib.ptr(dsrc), None,
                                                n, h, w, 4 * c0, 1, 1, 0, 0, 0, 1, st))
                tape.add_grad(src0, dsrc)
                return
            row_bytes = pc.wd.shape[1] * 2
            lo = 0
            for src in (src0, src1):
                if src is None:
                    continue
                c = src.shape[-1]
                prev = tape.peek(src)
                dsrc = torch.empty_like(src)
                _lib.check(lib.fd_conv_igemm_ex(_lib.ptr(dy), cout, None, 0, pc.wd.data_ptr() + lo * row_bytes, None,
                                                _lib.ptr(prev), _lib.ptr(dsrc), None, n, h, w, c, pc.kh, pc.kw, pc.pad[0],
                                                pc.pad[1], 0, 0, st))
                tape.g[id(src)] = dsrc            # prev (if any) was added in the epilogue
                lo += c

        tape.record(bwd)
        return out

    def _t_gn_silu(self, tape: Tape, h: Tensor, stats: Tensor, norm, ss: Optional[Tensor], dss: Optional[Tensor], ss_off: int,
                   residual: Optional[Tensor], conv_bias) -> Tensor:
        out = self._gn_silu(h, stats, norm, ss, ss_off, residual, exact=True)
        lib, st, gb = self._lib, self._st, self._gb

        def bwd():
            da = tape.pop(out)
            n, hh, ww, c = h.shape
            if residual is not None:
                tape.add_grad(residual, da)
            dh = torch.empty_like(h)
            ws = torch.empty(lib.fd_gn_silu_bwd_workspace_floats(n, c), device=h.device, dtype=torch.float32)
            ss_ptr = ss.data_ptr() + 4 * ss_off if ss is not None else None
            dss_ptr = dss.data_ptr() + 4 * ss_off if ss is not None else None
            _lib.check(lib.fd_gn_silu_bwd(_lib.ptr(h), _lib.ptr(da), _lib.ptr(stats), _lib.ptr(norm.weight), _lib.ptr(norm.bias),
                                          ss_ptr, ss.shape[1] if ss is not None else 0, _lib.ptr(dh),
                                          _lib.ptr(gb.of(norm.weight)), _lib.ptr(gb.of(norm.bias)), dss_ptr,
                                          _lib.ptr(gb.of(conv_bias)), _lib.ptr(ws), n, hh * ww, c, self.GN_EPS, st))
            tape.add_grad(h, dh)

        tape.record(bwd)
        return out

    def _t_chan_ln(self, tape: Tape, x: Tensor, gain, residual: Optional[Tensor] = None) -> Tensor:
        out = self._chan_ln(x, gain, residual)
        lib, st, gb = self._lib, self._st, self._gb

        def bwd():
            dy = tape.pop(out)
            n, hh, ww, c = x.shape
            if residual is not None:
                tape.add_grad(residual, dy)
            prev = tape.peek(x)
            dx = torch.empty_like(x)
            _lib.check(lib.fd_chan_layernorm_bwd(_lib.ptr(x), _lib.ptr(gain), _lib.ptr(dy), _lib.ptr(prev), _lib.ptr(dx),
                                                 _lib.ptr(gb.of(gain)), n * hh * ww, c, self.LN_EPS, st))
            tape.g[id(x)] = dx

        tape.record(bwd)
        return out

    def _t_resnet(self, tape: Tape, name: str, rb, x0: Tensor, x1: Optional[Tensor], ss: Tensor, dss: Tensor,
                  need_dgrad: bool = True) -> Tensor:
        st1, st2 = self._next_stats(), self._next_stats()
        if rb.mlp is not None and ss is not None:
            lin, temb, gb, lib, st = rb.mlp[1], tape.temb, self._gb, self._lib, self._st

            def mlp_bwd(o=self._tproj_off[name]):     # runs after block1's GroupNorm backward wrote this block's d(scale, shift)
                _lib.check(lib.fd_linear_bwd_w(dss.data_ptr() + 4 * o, dss.shape[1], _lib.ptr(temb), self.time_dim,
                                               _lib.ptr(gb.of(lin.weight)), _lib.ptr(gb.of(lin.bias)), dss.shape[0],
                                               lin.weight.shape[0], self.time_dim, 1, st))

            tape.record(mlp_bwd)
        h1 = self._t_conv(tape, name + ".block1.proj", x0, x1, stats=st1, need_dgrad=need_dgrad)
        a1 = self._t_gn_silu(tape, h1, st1, rb.block1.norm, ss, dss, self._tproj_off[name], None, rb.block1.proj.bias)
        h2 = self._t_conv(tape, name + ".block2.proj", a1, stats=st2)
        if (name + ".res_conv") in self._convs:
            return self._t_conv(tape, name + ".res_conv", x0, x1, need_dgrad=need_dgrad,
                                res_gn=(h2, st2, rb.block2.norm, rb.block2.proj.bias))
        assert x1 is None
        return self._t_gn_silu(tape, h2, st2, rb.block2.norm, None, None, 0, x0, rb.block2.proj.bias)

    def _t_linear_attention(self, tape: Tape, name: str, res, x: Tensor) -> Tensor:
        n, h, w, c = x.shape
        lib, st = self._lib, self._st
        y = self._t_chan_ln(tape, x, res.fn.norm.g)
        qkv = self._t_conv(tape, name + ".to_qkv", y)
        att = torch.empty(n, h, w, 128, device=x.device, dtype=BF16)
        ws = torch.empty(lib.fd_linattn_workspace_floats(n, h * w), device=x.device, dtype=torch.float32)
        stats = torch.empty(n, lib.fd_linattn_stats_floats(), device=x.device, dtype=torch.float32)
        _lib.check(lib.fd_linattn_save(_lib.ptr(qkv), _lib.ptr(att), _lib.ptr(stats), _lib.ptr(ws), n, h * w, st))
        del ws

        def bwd():
            datt = tape.pop(att)
            dqkv = torch.empty_like(qkv)
            wsb = torch.empty(lib.fd_linattn_bwd_workspace_floats(n, h * w), device=x.device, dtype=torch.float32)
            _lib.check(lib.fd_linattn_bwd(_lib.ptr(qkv), _lib.ptr(datt), _lib.ptr(dqkv), _lib.ptr(stats), _lib.ptr(wsb), n, h * w,
                                          st))
            tape.add_grad(qkv, dqkv)

        tape.record(bwd)
        o = self._t_conv(tape, name + ".to_out", att)
        return self._t_chan_ln(tape, o, res.fn.fn.to_out[1].g, residual=x)

    def _t_attention(self, tape: Tape, name: str, res, x: Tensor) -> Tensor:
        n, h, w, c = x.shape
        lib, st = self._lib, self._st
        y = self._t_chan_ln(tape, x, res.fn.norm.g)
        qkv = self._t_conv(tape, name + ".to_qkv", y)
        att = torch.empty(n, h, w, 128, device=x.device, dtype=BF16)
        lse = torch.empty(n, 4, h * w, device=x.device, dtype=torch.float32)
        _lib.check(lib.fd_attention_lse(_lib.ptr(qkv), _lib.ptr(att), _lib.ptr(lse), n, h * w, st))

        def bwd():
            datt = tape.pop(att)
            dqkv = torch.empty_like(qkv)
            wsb = torch.empty(lib.fd_attention_bwd_workspace_floats(n, h * w), device=x.device, dtype=torch.float32)
            _lib.check(lib.fd_attention_bwd(_lib.ptr(qkv), _lib.ptr(att), _lib.ptr(datt), _lib.ptr(lse), _lib.ptr(dqkv),
                                            _lib.ptr(wsb), n, h * w, st))
            tape.add_grad(qkv, dqkv)

        tape.record(bwd)
        return self._t_conv(tape, name + ".to_out", att, residual=x)

    # ------------------------------------------------------------------ forward (training)
    def forward_train(self, x: Tensor, external_cond: Optional[Tensor], time: Tensor, nan_mask: bool = False):
        """``Unet.forward`` keeping the tape.  Returns ``(out, backward)`` where ``backward(dout)`` accumulates every
        parameter gradient into ``self.grad_buffer`` (caller zero-fills) and returns nothing: the network input
        (noised target + conditioning frames) carries no gradient in the reference's training step."""
        _lib.require_cuda(x, external_cond, time)
        if self.time_in and time is None:
            raise ValueError("when Unet takes time arg, time argument must be passed in")
        self.prepare()
        self._lib = _lib.load()
        self._st = _lib.stream()
        self._prepare_dgrad()
        self._grad_buffer()
        lib, st = self._lib, self._st
        B, Cx, H0, W0 = x.shape
        Cc = external_cond.shape[1] if external_cond is not None else 0
        assert Cx + int(nan_mask) + Cc == self.channels, (Cx, nan_mask, Cc, self.channels)
        dev = x.device
        x = x.detach().float()
        cond = external_cond.detach().float() if external_cond is not None else None
        ph, pw = (-H0) % 8, (-W0) % 8
        pad = (pw // 2, pw - pw // 2, ph // 2, ph - ph // 2)
        if ph or pw:
            x = torch.nn.functional.pad(x, pad, mode="replicate")
            if cond is not None:
                cond = torch.nn.functional.pad(cond, pad, mode="replicate")
        x = x.contiguous()
        cond = cond.contiguous() if cond is not None else None
        H, W = H0 + ph, W0 + pw
        tape = Tape(self)
        gb = self._gb
        ss = dss = None
        self._t_group_boundary(tape, "front")        # first record = last to run: after init_conv and the time MLP
        if self.time_in:
            time = time.to(torch.int64).contiguous()

            temb = torch.empty(B, self.time_dim, device=dev, dtype=torch.float32)
            pe = torch.empty(B, self.dim, device=dev, dtype=torch.float32)
            pre = torch.empty(B, self.time_dim, device=dev, dtype=torch.float32)
            tm = self.time_mlp
            _lib.check(lib.fd_time_embed_save(_lib.ptr(time), _lib.ptr(tm[1].weight), _lib.ptr(tm[1].bias), _lib.ptr(tm[3].weight),
                                              _lib.ptr(tm[3].bias), _lib.ptr(temb), _lib.ptr(pe), _lib.ptr(pre), B, self.dim,
                                              self.time_dim, st))
            J = self._tproj_w.shape[0]
            ss = torch.empty(B, J, device=dev, dtype=torch.float32)
            dss = torch.zeros(B, J, device=dev, dtype=torch.float32)
            _lib.check(lib.fd_time_proj(_lib.ptr(temb), _lib.ptr(self._tproj_w), _lib.ptr(self._tproj_b), _lib.ptr(ss), B,
                                        self.time_dim, J, st))

            tape.temb = temb

            def time_bwd():
                # (each ResnetBlock's mlp Linear gradient was taken inside its own block: _t_resnet.mlp_bwd)
                td = self.time_dim
                dtemb = torch.empty(B, td, device=dev, dtype=torch.float32)
                _lib.check(lib.fd_linear_bwd_x(_lib.ptr(dss), J, _lib.ptr(self._tproj_w), _lib.ptr(temb), td, _lib.ptr(dtemb), td,
                                               B, J, td, 1, st))
                _lib.check(lib.fd_linear_bwd_w(_lib.ptr(dtemb), td, _lib.ptr(pre), td, _lib.ptr(gb.of(tm[3].weight)),
                                               _lib.ptr(gb.of(tm[3].bias)), B, td, td, 2, st))
                dpre = torch.empty(B, td, device=dev, dtype=torch.float32)
                _lib.check(lib.fd_linear_bwd_x(_lib.ptr(dtemb), td, _lib.ptr(tm[3].weight), _lib.ptr(pre), td, _lib.ptr(dpre), td,
                                               B, td, td, 2, st))
                _lib.check(lib.fd_linear_bwd_w(_lib.ptr(dpre), td, _lib.ptr(pe), self.dim, _lib.ptr(gb.of(tm[1].weight)),
                                               _lib.ptr(gb.of(tm[1].bias)), B, td, self.dim, 0, st))

            tape.record(time_bwd)          # runs last: every block's d(scale, shift) is in dss by then

        self._stats = torch.zeros(2 * len(self._resblocks), B, 8, 2, device=dev, dtype=torch.float64)
        self._stats_i = 0
        packed = torch.empty(B, H, W, 64, device=dev, dtype=BF16)
        if self._wide_input:
            _lib.check(lib.fd_pack_input_wide(_lib.ptr(x), _lib.ptr(cond), _lib.ptr(packed), B, Cx, Cc, H, W, 0, 0, H, W,
                                              int(nan_mask), st))
        else:
            _lib.check(lib.fd_pack_input(_lib.ptr(x), _lib.ptr(cond), _lib.ptr(packed), B, Cx, Cc, H, W, int(nan_mask), st))
        h = self._t_conv(tape, "init_conv", packed, need_dgrad=False)
        r = h
        skips: List[Tensor] = []
        n_levels = len(self.downs)
        for i, (b1, b2, attn, down) in enumerate(self.downs):
            if i >= 2:
                self._t_group_boundary(tape, f"downs.{i}")
            h = self._t_resnet(tape, f"downs.{i}.0", b1, h, None, ss, dss)
            skips.append(h)
            h = self._t_resnet(tape, f"downs.{i}.1", b2, h, None, ss, dss)
            h = self._t_linear_attention(tape, f"downs.{i}.2", attn, h)
            skips.append(h)
            h = self._t_conv(tape, f"downs.{i}.3", h)
        self._t_group_boundary(tape, "mid")
        h = self._t_resnet(tape, "mid_block1", self.mid_block1, h, None, ss, dss)
        h = self._t_attention(tape, "mid_attn", self.mid_attn, h)
        h = self._t_resnet(tape, "mid_block2", self.mid_block2, h, None, ss, dss)
        for i, (b1, b2, attn, up) in enumerate(self.ups):
            if i <= 2:
                self._t_group_boundary(tape, ("ups.0", "ups.1", "ups.23")[i])
            h = self._t_resnet(tape, f"ups.{i}.0", b1, h, skips.pop(), ss, dss)
            h = self._t_resnet(tape, f"ups.{i}.1", b2, h, skips.pop(), ss, dss)
            h = self._t_linear_attention(tape, f"ups.{i}.2", attn, h)
            if i < n_levels - 1:
                n_, hh, ww, cc = h.shape
                up_t = torch.empty(n_, 2 * hh, 2 * ww, cc, device=dev, dtype=BF16)
                _lib.check(lib.fd_upsample2x(_lib.ptr(h), _lib.ptr(up_t), n_, hh, ww, cc, st))

                def up_bwd(h=h, up_t=up_t, n_=n_, hh=hh, ww=ww, cc=cc):
                    d = tape.pop(up_t)
                    dx = torch.empty_like(h)
                    _lib.check(lib.fd_upsample2x_bwd(_lib.ptr(d), _lib.ptr(dx), n_, hh, ww, cc, st))
                    tape.add_grad(h, dx)

                tape.record(up_bwd)
                h = self._t_conv(tape, f"ups.{i}.3", up_t)
                del up_t
            else:
                h = self._t_conv(tape, f"ups.{i}.3", h)
        self._t_group_boundary(tape, "final")
        h = self._t_resnet(tape, "final_res_block", self.final_res_block, h, r, ss, dss)
        out = torch.empty(B, self.out_dim, H, W, device=dev, dtype=torch.float32)
        fc = self.final_conv
        _lib.check(lib.fd_final_conv(_lib.ptr(h), _lib.ptr(fc.weight), _lib.ptr(fc.bias), _lib.ptr(out), B, H * W, self.dim,
                                     self.out_dim, st))
        h_last = h
        self._stats = None

        def backward(dout: Tensor):
            _lib.require_cuda(dout)
            dout = dout.float()
            if ph or pw:
                dout = torch.nn.functional.pad(dout, pad)        # the cropped border received no gradient
            dout = dout.contiguous()
            dh = torch.empty_like(h_last)
            _lib.check(lib.fd_final_conv_bwd(_lib.ptr(h_last), _lib.ptr(fc.weight), _lib.ptr(dout), _lib.ptr(dh),
                                             _lib.ptr(gb.of(fc.weight)), _lib.ptr(gb.of(fc.bias)), B, H * W, self.dim,
                                             self.out_dim, st))
            tape.g[id(h_last)] = dh
            ws = self._wgrad_workspace()
            ws["flat"].zero_()
            tape.run()          # the group boundaries unpack the packed weight gradients bucket by bucket (_t_group_boundary)

        if ph or pw:
            out = out[:, :, pad[2]:pad[2] + H0, pad[0]:pad[0] + W0].contiguous()
        return out, backward


class UnetFunction(torch.autograd.Function):
    """The UNet as one autograd node: ``out = UnetFunction.apply(unet, x, cond, time, nan_mask, *unet.parameters())``."""

    @staticmethod
    def forward(ctx, unet, x, cond, time, nan_mask, *params):
        with _lib.nvtx_range("unet.forward_train"):
            out, backward = unet.forward_train(x, cond, time, nan_mask)
        ctx.unet = unet
        ctx.run_backward = backward
        return out

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, dout):
        unet = ctx.unet
        if ctx.run_backward is None:
            raise RuntimeError("UnetFunction: the activations were released by the first backward pass "
                               "(retain_graph / double backward are not supported on this path)")
        gb = unet.grad_buffer
        gb.zero_()
        with _lib.nvtx_range("unet.backward"):
            ctx.run_backward(dout)
        ctx.run_backward = None
        sync = getattr(unet, "grad_sync", None)
        if sync is not None:
            sync.finish(gb.flat)          # the launching stream waits for the bucket all-reduces issued during the backward
        # hand autograd its own copy of the flat buffer's views: p.grad accumulation (+=) must not alias the
        # buffer the next backward zero-fills
        flat = gb.flat.clone()
        views = []
        off = 0
        for v in gb.views:
            o = v.storage_offset()
            views.append(flat[o:o + v.numel()].view(v.shape))
        unet.last_flat_grad = flat
        return (None, None, None, None, None) + tuple(views)
