"""The noise-prediction UNet of flow_diffuser (reference: ``Unet``, denoising_diffusion.py:272-417)
executed by the sm_100a kernels of ``libflowdiff.so``.

``Unet`` *is* the reference's parameter tree (same attribute names -> same ``state_dict`` keys, same
construction order -> same random init under a given ``torch.manual_seed``); its ``forward`` walks
that tree and launches kernels through the C ABI:

* activations are bf16 NHWC; every convolution is ``fd_conv_igemm`` (tcgen05 + TMA), which also
  accumulates the GroupNorm statistics of its output, so ``Block`` = conv + one ``fd_gn_silu`` pass;
* skip concats, the pixel-unshuffle of ``Downsample`` and the ``+ res_conv(x)`` of ``ResnetBlock`` are
  folded into the conv's operand maps / epilogue, never materialised;
* weight standardisation + bf16 packing is one tiny launch per conv (``prepare``), cached while
  the parameters are unchanged;
* all 18 ResnetBlock time-MLPs run as one ``fd_time_proj`` over their concatenated weights.

There is no PyTorch fallback: a missing library or a non-sm_100 device raises.
"""
from __future__ import annotations

from functools import partial
from typing import Dict, List, Optional, Tuple

import torch

from . import _lib
from .unet_params import UnetParams, _ResnetBlock
from .unet_train import TrainMixin, UnetFunction, _batch_table

Tensor = torch.Tensor
BF16 = torch.bfloat16


class _PackedConv:
    __slots__ = ("w", "wd", "bias", "cout", "kh", "kw", "pad", "mode", "src", "kind", "ws")

    def __init__(self, src, kind: int, ws: bool, kh: int, kw: int, pad: Tuple[int, int], mode: int):
        self.src, self.kind, self.ws = src, kind, ws
        self.kh, self.kw, self.pad, self.mode = kh, kw, pad, mode
        self.cout = src.weight.shape[0]
        self.w: Optional[Tensor] = None
        self.wd: Optional[Tensor] = None     # dgrad packing (unet_train.py)
        self.bias: Optional[Tensor] = None


class Unet(UnetParams, TrainMixin):
    """Unet(dim=64, channels=C_in, out_dim=2): same constructor meaning as the reference (:272-293)."""

    GN_EPS = 1e-5       # nn.GroupNorm default (:176)
    # Upsample (nearest x2 + 3x3 conv, :89-93) runs as four 2x2 phase convolutions on the low-resolution tensor
    # (fd_conv_igemm_up, inference path): 2.25x fewer MACs for 12.5 % of the forward's conv FLOPs, no up-sampled tensor.
    # bench.py reads this to count the forward's conv launches.
    UPCONV_PHASES = True
    WS_EPS = 1e-5       # WeightStandardizedConv2d with fp32 input (:107)
    LN_EPS = 1e-5       # LayerNorm with fp32 input (:122)

    def __init__(self, dim: int = 64, channels: int = 5, out_dim: int = 2, dim_mults=(1, 2, 4, 8), groups: int = 8,
                 time_in: bool = True):
        super().__init__(dim, channels, out_dim, tuple(dim_mults), groups, time_in)
        assert dim == 64 and tuple(dim_mults) in ((1, 2, 4, 8), (1, 2, 4)) and groups == 8, \
            "the sm_100a path is specialised to the flow_diffuser UNets (dim 64, mults 1-2-4-8 or 1-2-4, 8 groups)"
        assert channels <= 64, "init_conv takes at most 64 input channels"
        # <= 9 channels: 7 horizontal taps x 9 channels fit one 64-wide K chunk (init_conv as a 7x1 conv, kind 2); more
        # (latent mode, flow_diffuser.py:98-110 / flow_pred.py:23-37): channels zero-padded to 64, 49-tap implicit GEMM (kind 3)
        self._wide_input = channels > 9
        self._convs: Optional[Dict[str, _PackedConv]] = None
        self._resblocks: List[Tuple[str, _ResnetBlock]] = []
        self._tproj_w: Optional[Tensor] = None
        self._tproj_b: Optional[Tensor] = None
        self._tproj_off: Dict[str, int] = {}
        self._up_w: Dict[int, Tensor] = {}       # phase-decomposed Upsample weights (fd_prep_weight_upconv)
        self._la_tc: Dict[str, Dict[str, Tensor]] = {}       # tcgen05 LinearAttention operands (fd_linattn_tc_prep)
        self._prep_table = None
        self._prepared_versions = None
        self.weights_epoch = 0      # bumped by optimisers that update the parameters through raw pointers
        self._conv_timing: Optional[list] = None     # bench.py's roofline pass sets a list: see _launch_conv

    # ------------------------------------------------------------------ weight preparation
    def _build_conv_table(self):
        convs: Dict[str, _PackedConv] = {}

        def add(name, mod, kind=0, ws=False, mode=0):
            kh, kw = mod.weight.shape[2:]
            if kind == 2 and self._wide_input:
                convs[name] = _PackedConv(mod, 3, False, 7, 7, (3, 3), 0)
            elif kind == 2:
                convs[name] = _PackedConv(mod, 2, False, 7, 1, (3, 0), 0)
            else:
                convs[name] = _PackedConv(mod, kind, ws, kh, kw, (kh // 2, kw // 2), mode)

        def add_res(name, rb: _ResnetBlock):
            add(name + ".block1.proj", rb.block1.proj, ws=True)
            add(name + ".block2.proj", rb.block2.proj, ws=True)
            if not isinstance(rb.res_conv, torch.nn.Identity):
                add(name + ".res_conv", rb.res_conv)
            self._resblocks.append((name, rb))

        def add_attn(name, res):
            fn = res.fn.fn
            linear = isinstance(fn.to_out, torch.nn.Sequential)
            add(name + ".to_qkv", fn.to_qkv)
            add(name + ".to_out", fn.to_out[0] if linear else fn.to_out)

        self._resblocks = []
        add("init_conv", self.init_conv, kind=2)
        n = len(self.downs)
        for i, (b1, b2, attn, down) in enumerate(self.downs):
            add_res(f"downs.{i}.0", b1)
            add_res(f"downs.{i}.1", b2)
            add_attn(f"downs.{i}.2", attn)
            if i < n - 1:
                add(f"downs.{i}.3", down[1], kind=1, mode=1)
            else:
                add(f"downs.{i}.3", down)
        add_res("mid_block1", self.mid_block1)
        add_attn("mid_attn", self.mid_attn)
        add_res("mid_block2", self.mid_block2)
        for i, (b1, b2, attn, up) in enumerate(self.ups):
            add_res(f"ups.{i}.0", b1)
            add_res(f"ups.{i}.1", b2)
            add_attn(f"ups.{i}.2", attn)
            add(f"ups.{i}.3", up[1] if i < n - 1 else up)
        add_res("final_res_block", self.final_res_block)
        self._convs = convs

    def _linattn_blocks(self):
        for i, stage in enumerate(self.downs):
            yield f"downs.{i}.2", stage[2]
        for i, stage in enumerate(self.ups):
            yield f"ups.{i}.2", stage[2]

    def _versions(self):
        return (self.weights_epoch,) + tuple(p._version for p in self.parameters()) + \
            tuple(p.data_ptr() for p in self.parameters())

    @torch.no_grad()
    def prepare(self, force: bool = False):
        """Standardise + pack every conv weight to bf16 [Cout][K]; concatenate the time-MLP weights.
        Cached until a parameter is modified in place or replaced."""
        ver = self._versions()
        if not force and self._convs is not None and ver == self._prepared_versions:
            return
        lib = _lib.load(check_device=True)
        if self._convs is None:
            self._build_conv_table()
        st = _lib.stream()
        recs, blocks, dev = [], [0], None
        for pc in self._convs.values():
            w = pc.src.weight
            _lib.require_cuda(w)
            dev = w.device
            cout, cin, kh, kw = w.shape
            kp = 7 * 64 if pc.kind == 2 else (49 * 64 if pc.kind == 3 else cin * kh * kw)
            if pc.w is None or pc.w.device != w.device:
                pc.w = torch.empty(cout, kp, device=w.device, dtype=BF16)
            if w.dtype == torch.float32 and w.is_contiguous():
                # batched below: one launch standardises + packs every layer (a training step re-packs all ~80 of them)
                recs.append([w.data_ptr(), pc.w.data_ptr(), 0, cout, cin, kh, kw, pc.kind | (int(pc.ws) << 8)])
                blocks.append(blocks[-1] + cout)
            else:
                _lib.check(lib.fd_prep_weight(_lib.ptr(w.detach().float().contiguous()), _lib.ptr(pc.w), cout, cin, kh, kw,
                                              pc.kind, int(pc.ws), self.WS_EPS, st))
            pc.bias = pc.src.bias.detach().float().contiguous() if pc.src.bias is not None else None
        if recs:
            table, blk = _batch_table(self, "_prep_table", recs, blocks, dev)
            _lib.check(lib.fd_prep_weight_batch(_lib.ptr(table), _lib.ptr(blk), len(recs), blocks[-1], self.WS_EPS, st))
        ws, bs, off = [], [], 0
        self._tproj_off = {}
        for name, rb in self._resblocks:
            self._tproj_off[name] = off
            if rb.mlp is None:
                continue
            lin = rb.mlp[1]
            off += lin.weight.shape[0]
            ws.append(lin.weight.detach().float())
            bs.append(lin.bias.detach().float())
        # phase-decomposed weights of the Upsample convs (fd_prep_weight_upconv), rewritten in place
        up = self._up_w
        for i, stage in enumerate(self.ups):
            if i >= len(self.ups) - 1:
                continue
            conv = stage[3][1]
            wt = conv.weight
            cout, cin = wt.shape[:2]
            buf = up.get(i)
            if buf is None or buf.device != wt.device:
                buf = up[i] = torch.empty(4, cout, 4 * cin, device=wt.device, dtype=BF16)
            _lib.check(lib.fd_prep_weight_upconv(_lib.ptr(wt.detach().float().contiguous()), _lib.ptr(buf), cout, cin, st))
        # operands of the tcgen05 LinearAttention blocks (fd_linattn_tc_prep): buffers allocated once, rewritten in place
        la = self._la_tc
        for name, res in self._linattn_blocks():
            fn = res.fn.fn
            if fn.dim not in (64, 128):
                continue
            wqkv = fn.to_qkv.weight
            ent = la.get(name)
            if ent is None or ent["wq"].device != wqkv.device:
                dv, C = wqkv.device, fn.dim
                ent = la[name] = {"wq": torch.empty(128, C, device=dv, dtype=BF16), "wk": torch.empty(128, C, device=dv, dtype=BF16),
                                  "sq": torch.empty(128, device=dv), "sk": torch.empty(128, device=dv),
                                  "mk": torch.empty(128, device=dv), "wv": torch.empty(128, C, device=dv)}
            _lib.check(lib.fd_linattn_tc_prep(_lib.ptr(wqkv.detach().float().contiguous()), _lib.ptr(res.fn.norm.g), _lib.ptr(ent["wq"]),
                                              _lib.ptr(ent["sq"]), _lib.ptr(ent["wk"]), _lib.ptr(ent["sk"]), _lib.ptr(ent["mk"]),
                                              _lib.ptr(ent["wv"]), fn.dim, st))
        # written IN PLACE once allocated: a captured CUDA graph of the sampler holds these pointers (diffusion.py)
        if ws:
            rows = sum(w.shape[0] for w in ws)
            if self._tproj_w is None or self._tproj_w.shape[0] != rows or self._tproj_w.device != ws[0].device:
                self._tproj_w = torch.empty(rows, ws[0].shape[1], device=ws[0].device, dtype=torch.float32)
                self._tproj_b = torch.empty(rows, device=ws[0].device, dtype=torch.float32)
            torch.cat(ws, 0, out=self._tproj_w)
            torch.cat(bs, 0, out=self._tproj_b)
        else:
            self._tproj_w = self._tproj_b = None
        self._prepared_versions = ver

    # ------------------------------------------------------------------ kernel wrappers
    def _launch_conv(self, name: str, npix: int, fn, *args):
        """``fn(*args)``: the launch of conv ``name`` with ``npix`` output pixels.  While ``_conv_timing`` is a list
        (bench.py's roofline pass) it also appends ``(name, algorithmic FLOPs, (start, end) CUDA events)``."""
        timing = self._conv_timing
        if timing is None:
            _lib.check(fn(*args))
            return
        pc = self._convs[name]
        # algorithmic K: init_conv's packing pads it to 7 or 49 taps of 64 channels; an Upsample counts as the reference's
        # 3x3 conv on the up-sampled tensor, whatever its phase decomposition launches
        k = pc.w.shape[1] if pc.kind < 2 else 49 * self.channels
        ev = (torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True))
        timing.append((name, 2.0 * npix * pc.cout * k, ev))
        ev[0].record()
        _lib.check(fn(*args))
        ev[1].record()

    def _conv(self, name: str, src0: Tensor, src1: Optional[Tensor] = None, residual: Optional[Tensor] = None,
              stats: Optional[Tensor] = None) -> Tensor:
        pc = self._convs[name]
        n, h, w, c0 = src0.shape
        c1 = src1.shape[-1] if src1 is not None else 0
        if pc.mode == 1:
            h, w = h // 2, w // 2
        out = torch.empty(n, h, w, pc.cout, device=src0.device, dtype=BF16)
        self._launch_conv(name, n * h * w, self._lib.fd_conv_igemm, _lib.ptr(src0), c0, _lib.ptr(src1), c1, _lib.ptr(pc.w),
                          _lib.ptr(pc.bias), _lib.ptr(residual), _lib.ptr(out), _lib.ptr(stats), n, h, w, pc.cout,
                          pc.kh, pc.kw, pc.pad[0], pc.pad[1], pc.mode, self._st)
        return out

    def _conv_gnsilu_in(self, name: str, src: Tensor, in_stats: Tensor, norm, ss: Optional[Tensor], ss_off: int,
                        stats: Optional[Tensor]) -> Tensor:
        pc = self._convs[name]
        n, h, w, _ = src.shape
        out = torch.empty(n, h, w, pc.cout, device=src.device, dtype=BF16)
        ss_ptr = ss.data_ptr() + 4 * ss_off if ss is not None else None
        self._launch_conv(name, n * h * w, self._lib.fd_conv3x3_gnsilu_in, _lib.ptr(src), _lib.ptr(in_stats),
                          _lib.ptr(norm.weight), _lib.ptr(norm.bias), ss_ptr, ss.shape[1] if ss is not None else 0, self.GN_EPS,
                          _lib.ptr(pc.w), _lib.ptr(pc.bias), None, _lib.ptr(out), _lib.ptr(stats), n, h, w, self._st)
        return out

    def _conv_res_gn(self, name: str, src0: Tensor, src1: Optional[Tensor], raw: Tensor, raw_stats: Tensor, norm) -> Tensor:
        """res_conv(x) + silu(GroupNorm(raw)) (:212-214) in one launch: the GroupNorm apply rides in the conv's epilogue."""
        pc = self._convs[name]
        n, h, w, c0 = src0.shape
        c1 = src1.shape[-1] if src1 is not None else 0
        out = torch.empty(n, h, w, pc.cout, device=src0.device, dtype=BF16)
        self._launch_conv(name, n * h * w, self._lib.fd_conv_igemm_rt, _lib.ptr(src0), c0, _lib.ptr(src1), c1, _lib.ptr(pc.w),
                          _lib.ptr(pc.bias), _lib.ptr(raw), _lib.ptr(raw_stats), _lib.ptr(norm.weight), _lib.ptr(norm.bias),
                          self.GN_EPS, _lib.ptr(out), n, h, w, pc.cout, pc.kh, pc.kw, pc.pad[0], pc.pad[1], self._st)
        return out

    def _gn_silu(self, x: Tensor, stats: Tensor, norm, ss: Optional[Tensor], ss_off: int,
                 residual: Optional[Tensor], exact: bool = False) -> Tensor:
        n, h, w, c = x.shape
        out = torch.empty_like(x)
        ss_ptr = ss.data_ptr() + 4 * ss_off if ss is not None else None
        # inference forward: the one-MUFU SiLU of the fused kernels; the training forward (exact=True from
        # unet_train._t_gn_silu; grad mode cannot tell the two apart, it is off inside autograd.Function.forward) keeps the
        # exp form its parity tests were pinned on
        fn = self._lib.fd_gn_silu if exact else self._lib.fd_gn_silu_fast
        _lib.check(fn(_lib.ptr(x), _lib.ptr(stats), _lib.ptr(norm.weight), _lib.ptr(norm.bias), ss_ptr,
                      ss.shape[1] if ss is not None else 0, _lib.ptr(residual), _lib.ptr(out), n, h * w, c, self.GN_EPS, self._st))
        return out

    def _chan_ln(self, x: Tensor, g: Tensor, residual: Optional[Tensor] = None) -> Tensor:
        n, h, w, c = x.shape
        out = torch.empty_like(x)
        _lib.check(self._lib.fd_chan_layernorm(_lib.ptr(x), _lib.ptr(g), _lib.ptr(residual), _lib.ptr(out), n * h * w, c,
                                               self.LN_EPS, self._st))
        return out

    def _conv_res_gn_head(self, name: str, src0: Tensor, src1: Optional[Tensor], raw: Tensor, raw_stats: Tensor, norm,
                          head: tuple) -> Tensor:
        """_conv_res_gn followed by final_conv and the un-pad crop (:416-417) in the same launch: fd_conv_igemm_rt_head."""
        pc = self._convs[name]
        n, h, w, c0 = src0.shape
        c1 = src1.shape[-1] if src1 is not None else 0
        fc, h0, w0, pt, pl = head
        out = torch.empty(n, self.out_dim, h0, w0, device=src0.device, dtype=torch.float32)
        self._launch_conv(name, n * h * w, self._lib.fd_conv_igemm_rt_head, _lib.ptr(src0), c0, _lib.ptr(src1), c1,
                          _lib.ptr(pc.w), _lib.ptr(pc.bias), _lib.ptr(raw), _lib.ptr(raw_stats), _lib.ptr(norm.weight),
                          _lib.ptr(norm.bias), self.GN_EPS, _lib.ptr(fc.weight), _lib.ptr(fc.bias), self.out_dim, _lib.ptr(out),
                          n, h, w, h0, w0, pt, pl, self._st)
        return out

    def _upsample(self, i: int, x: Tensor) -> Tensor:
        """Upsample ``ups.{i}.3`` (nearest x2 + 3x3 conv, :89-93) as the four phase convolutions of fd_conv_igemm_up."""
        pc = self._convs[f"ups.{i}.3"]
        n, h, w, c = x.shape
        out = torch.empty(n, 2 * h, 2 * w, pc.cout, device=x.device, dtype=BF16)
        self._launch_conv(f"ups.{i}.3", n * 4 * h * w, self._lib.fd_conv_igemm_up, _lib.ptr(x), c, _lib.ptr(self._up_w[i]),
                          _lib.ptr(pc.bias), _lib.ptr(out), n, h, w, pc.cout, self._st)
        return out

    def _final_conv_crop(self, x: Tensor, frame: Tuple[int, int, int, int]) -> Tensor:
        """final_conv (:361,417) on the padded frame, storing only the H0 x W0 window at (pad_top, pad_left) of
        ``frame = (H0, W0, pad_top, pad_left)``: InputPadder.unpad folded into the store."""
        n, h, w, _ = x.shape
        H0, W0, pt, pl = frame
        fc = self.final_conv
        out = torch.empty(n, self.out_dim, H0, W0, device=x.device, dtype=torch.float32)
        _lib.check(self._lib.fd_final_conv_crop(_lib.ptr(x), _lib.ptr(fc.weight), _lib.ptr(fc.bias), _lib.ptr(out), n, h, w,
                                                self.dim, self.out_dim, pt, pl, H0, W0, self._st))
        return out

    def _resnet(self, name: str, rb: _ResnetBlock, x0: Tensor, x1: Optional[Tensor], ss: Optional[Tensor],
                head: Optional[tuple] = None) -> Tensor:
        """ResnetBlock.forward (:202-214).  head = (final_conv, H0, W0, pad_top, pad_left): also apply the output head."""
        st1, st2 = self._next_stats(), self._next_stats()
        h1 = self._conv(name + ".block1.proj", x0, x1, stats=st1)
        pc2 = self._convs[name + ".block2.proj"]
        if h1.shape[-1] == 64 and pc2.cout == 64 and h1.shape[2] >= 128:
            # 64 -> 64 at full resolution: GroupNorm + scale/shift + SiLU of h1 is applied to the input strips inside the
            # conv (fd_conv3x3_gnsilu_in), the activated tensor never goes through HBM.  Measured on the DDIM-50 benchmark:
            # 7.08-7.11 vs 6.96 flows/s for the separate gn_silu pass (DESIGN.md section 6)
            h2 = self._conv_gnsilu_in(name + ".block2.proj", h1, st1, rb.block1.norm, ss, self._tproj_off[name], st2)
        else:
            a1 = self._gn_silu(h1, st1, rb.block1.norm, ss, self._tproj_off[name], None)
            h2 = self._conv(name + ".block2.proj", a1, stats=st2)
        if (name + ".res_conv") in self._convs:
            # block2's GroupNorm + SiLU rides in the res_conv's epilogue: no second gn_silu pass for the 9 ResnetBlocks with a
            # res_conv (ups.*, final_res_block), 4.4 GB less HBM traffic per batch-8 forward at 440x1024
            if head is not None:
                return self._conv_res_gn_head(name + ".res_conv", x0, x1, h2, st2, rb.block2.norm, head)
            return self._conv_res_gn(name + ".res_conv", x0, x1, h2, st2, rb.block2.norm)
        assert x1 is None
        return self._gn_silu(h2, st2, rb.block2.norm, None, 0, x0)

    def _linear_attention(self, name: str, res, x: Tensor) -> Tensor:
        """Residual(PreNorm(LinearAttention)) (:81-87,127-135,229-244)."""
        n, h, w, c = x.shape
        ent = self._la_tc.get(name)
        if ent is not None:
            # C in {64, 128}: two tcgen05 / TMA passes over x (fd_linattn_tc), no LayerNorm output, qkv or attention tensor
            # in HBM
            fn = res.fn.fn
            out = torch.empty_like(x)
            ws = torch.empty(self._lib.fd_linattn_tc_workspace_floats(n, h * w, c), device=x.device, dtype=torch.float32)
            _lib.check(self._lib.fd_linattn_tc(_lib.ptr(x), _lib.ptr(ent["wk"]), _lib.ptr(ent["sk"]), _lib.ptr(ent["mk"]),
                                               _lib.ptr(ent["wq"]), _lib.ptr(ent["sq"]), _lib.ptr(ent["wv"]),
                                               _lib.ptr(fn.to_out[0].weight), _lib.ptr(fn.to_out[0].bias), _lib.ptr(fn.to_out[1].g),
                                               _lib.ptr(out), _lib.ptr(ws), n, h * w, c, self.LN_EPS, self._st))
            return out
        y = self._chan_ln(x, res.fn.norm.g)
        qkv = self._conv(name + ".to_qkv", y)
        att = torch.empty(n, h, w, 128, device=x.device, dtype=BF16)
        ws = torch.empty(self._lib.fd_linattn_workspace_floats(n, h * w), device=x.device, dtype=torch.float32)
        _lib.check(self._lib.fd_linattn(_lib.ptr(qkv), _lib.ptr(att), _lib.ptr(ws), n, h * w, self._st))
        o = self._conv(name + ".to_out", att)
        return self._chan_ln(o, res.fn.fn.to_out[1].g, residual=x)

    def _attention(self, name: str, res, x: Tensor) -> Tensor:
        """Residual(PreNorm(Attention)) (:246-268)."""
        n, h, w, c = x.shape
        y = self._chan_ln(x, res.fn.norm.g)
        qkv = self._conv(name + ".to_qkv", y)
        att = torch.empty(n, h, w, 128, device=x.device, dtype=BF16)
        _lib.check(self._lib.fd_attention(_lib.ptr(qkv), _lib.ptr(att), n, h * w, self._st))
        return self._conv(name + ".to_out", att, residual=x)

    def _next_stats(self) -> Tensor:
        s = self._stats[self._stats_i]
        self._stats_i += 1
        return s

    # ------------------------------------------------------------------ forward
    def forward(self, x: Tensor, external_cond: Optional[Tensor] = None, time: Optional[Tensor] = None,
                nan_mask: bool = False, return_taps: bool = False):
        """``Unet.forward(x, external_cond, time)`` (:363-417): x (B,Cx,H,W) fp32, cond (B,Cc,H,W) fp32, time (B,)
        int64 -> (B,out_dim,H,W) fp32.  ``nan_mask`` folds UnetWithWarp's NaN -> 0 + mask channel
        (flow_diffuser.py:39-45) into the input packing.

        With autograd enabled (training_step) the call is one ``UnetFunction`` node whose backward runs the backward
        kernels (unet_train.py); under ``torch.no_grad()`` (sampling, validation) it is the inference path."""
        if torch.is_grad_enabled() and not return_taps and any(p.requires_grad for p in self.parameters()):
            if len(self.downs) != 4:
                raise NotImplementedError(
                    "the backward kernels cover the four-level UNets (flow_diffuser, flow_learner); the three-level autoencoder "
                    "UNets (flow_pred.py:23-37) are used frozen (flow_diffuser.py:93-94): call them under torch.no_grad() or "
                    "set requires_grad_(False)")
            return UnetFunction.apply(self, x, external_cond, time, nan_mask, *self.parameters())
        with _lib.nvtx_range("unet.forward"), torch.no_grad():
            self._begin(x, external_cond, time)
            blocks = _InferBlocks(self, {} if return_taps else None)
            out = self._walk(blocks, x, external_cond, time, nan_mask)
            if return_taps:
                return out, {k: (v if v.dim() == 2 else v.permute(0, 3, 1, 2).float()) for k, v in blocks.taps.items()}
            return out

    def _begin(self, x: Tensor, external_cond: Optional[Tensor], time: Optional[Tensor]):
        """Input checks, weight preparation and the launch stream: the start of both forwards."""
        _lib.require_cuda(x, external_cond, time)
        if self.time_in and time is None:
            raise ValueError("when Unet takes time arg, time argument must be passed in")      # :378-379
        self.prepare()
        self._lib = _lib.load()
        self._st = _lib.stream()

    def _walk(self, blocks, x: Tensor, external_cond: Optional[Tensor], time: Optional[Tensor], nan_mask: bool):
        """The body of ``Unet.forward`` (:363-417) for both forwards.  ``blocks`` runs the blocks: ``_InferBlocks`` (fused
        kernels, nothing kept) or ``unet_train._TrainBlocks`` (records the tape for the backward).  ``blocks.group``
        marks where a gradient bucket of the training backward starts; ``blocks.tap`` offers an activation to
        ``return_taps``."""
        lib, st = self._lib, self._st
        B, Cx, H0, W0 = x.shape
        Cc = external_cond.shape[1] if external_cond is not None else 0
        assert Cx + int(nan_mask) + Cc == self.channels, (Cx, nan_mask, Cc, self.channels)
        dev = x.device
        x = x.detach().float().contiguous()
        cond = external_cond.detach().float().contiguous() if external_cond is not None else None
        # three 2x pixel-unshuffle downsamples (:95-99) need H, W % 8 == 0 (436 -> 440): replicate-pad like the
        # repo's own InputPadder(mode='sintel') (future/raft_utils.py:7-25) and crop the prediction back -- both folded
        # into the first / last kernel (the input packing clamps its reads, the output head writes the window only)
        mult = 2 ** (len(self.downs) - 1)                # 8, or 4 for the three-level autoencoder UNets (flow_pred.py:23-37)
        ph, pw = (-H0) % mult, (-W0) % mult
        pt, pl = ph // 2, pw // 2
        H, W = H0 + ph, W0 + pw

        blocks.group("front")
        # time embedding (:319-324) and every block's (scale, shift) (:206-208); none at all for Unet(time_in=False)
        ss = None
        if self.time_in:
            temb = blocks.time_embedding(time.to(torch.int64).contiguous())
            blocks.tap("temb", temb)
            J = self._tproj_w.shape[0]
            ss = torch.empty(B, J, device=dev, dtype=torch.float32)
            _lib.check(lib.fd_time_proj(_lib.ptr(temb), _lib.ptr(self._tproj_w), _lib.ptr(self._tproj_b), _lib.ptr(ss), B,
                                        self.time_dim, J, st))
        self._stats = torch.zeros(2 * len(self._resblocks), B, 8, 2, device=dev, dtype=torch.float64)
        self._stats_i = 0

        # init_conv 7x7 (:297,374) as a 7x1 conv over the horizontally unrolled input
        packed = torch.empty(B, H, W, 64, device=dev, dtype=BF16)
        pack = lib.fd_pack_input_wide if self._wide_input else lib.fd_pack_input_pad
        _lib.check(pack(_lib.ptr(x), _lib.ptr(cond), _lib.ptr(packed), B, Cx, Cc, H0, W0, pt, pl, H, W, int(nan_mask), st))
        h = r = blocks.init_conv(packed)
        del packed
        blocks.tap("init_conv", h)

        skips: List[Tensor] = []
        n_levels = len(self.downs)
        for i, (b1, b2, attn, _) in enumerate(self.downs):
            if i >= 2:
                blocks.group(f"downs.{i}")
            h = blocks.resnet(f"downs.{i}.0", b1, h, None, ss)
            skips.append(h)
            if i == 0:
                blocks.tap("downs.0.0", h)
            h = blocks.resnet(f"downs.{i}.1", b2, h, None, ss)
            h = blocks.linear_attention(f"downs.{i}.2", attn, h)
            if i == 0:
                blocks.tap("downs.0.2", h)
            skips.append(h)
            h = blocks.conv(f"downs.{i}.3", h)
        blocks.group("mid")
        h = blocks.resnet("mid_block1", self.mid_block1, h, None, ss)
        blocks.tap("mid_block1", h)
        h = blocks.attention("mid_attn", self.mid_attn, h)
        blocks.tap("mid_attn", h)
        h = blocks.resnet("mid_block2", self.mid_block2, h, None, ss)
        for i, (b1, b2, attn, _) in enumerate(self.ups):
            if i <= 2:
                blocks.group(("ups.0", "ups.1", "ups.23")[i])
            h = blocks.resnet(f"ups.{i}.0", b1, h, skips.pop(), ss)
            h = blocks.resnet(f"ups.{i}.1", b2, h, skips.pop(), ss)
            h = blocks.linear_attention(f"ups.{i}.2", attn, h)
            h = blocks.upsample(i, h) if i < n_levels - 1 else blocks.conv(f"ups.{i}.3", h)
        blocks.group("final")
        out = blocks.final(h, r, ss, (H0, W0, pt, pl))
        self._stats = None
        return out


class _InferBlocks:
    """``Unet._walk``'s blocks for the inference forward (sampling, validation): the fused kernels.  ``taps`` is None, or
    the dict that collects ``return_taps``' activations."""

    def __init__(self, unet: Unet, taps: Optional[Dict[str, Tensor]]):
        self.unet, self.taps = unet, taps
        self.init_conv = partial(unet._conv, "init_conv")
        self.conv, self.resnet, self.upsample = unet._conv, unet._resnet, unet._upsample
        self.linear_attention, self.attention = unet._linear_attention, unet._attention

    def group(self, name: str):
        pass

    def tap(self, name: str, h: Tensor):
        if self.taps is not None:
            self.taps[name] = h

    def time_embedding(self, time: Tensor) -> Tensor:
        u = self.unet
        tm = u.time_mlp
        temb = torch.empty(time.shape[0], u.time_dim, device=time.device, dtype=torch.float32)
        _lib.check(u._lib.fd_time_embed(_lib.ptr(time), _lib.ptr(tm[1].weight), _lib.ptr(tm[1].bias), _lib.ptr(tm[3].weight),
                                        _lib.ptr(tm[3].bias), _lib.ptr(temb), time.shape[0], u.dim, u.time_dim, u._st))
        return temb

    def final(self, h: Tensor, r: Tensor, ss: Optional[Tensor], frame: Tuple[int, int, int, int]) -> Tensor:
        u = self.unet
        if (self.taps is None and u.dim == 64 and u.out_dim <= 4 and
                "final_res_block.res_conv" in u._convs and u._convs["final_res_block.res_conv"].kh == 1):
            # final ResnetBlock's res_conv + residual + final_conv + crop in one launch: the last 64-channel activation
            # (461 MB at batch 8, 440x1024) is neither written nor re-read.  return_taps needs that activation: two launches
            return u._resnet("final_res_block", u.final_res_block, h, r, ss, head=(u.final_conv,) + frame)
        h = u._resnet("final_res_block", u.final_res_block, h, r, ss)
        self.tap("final_res_block", h)
        return u._final_conv_crop(h, frame)
