"""Optimiser and gradient exchange of the training step.

Reference: ``torch.optim.Adam(lr, weight_decay)`` (flow_diffuser.py:129-134: L2-in-gradient decay, not AdamW),
Lightning's ``gradient_clip_val`` (global L2 norm, exp_base.py:192,205) and ``DDPStrategy``'s gradient
all-reduce (exp_base.py:198).

``FusedAdam`` keeps the parameters it owns as views of ONE flat fp32 buffer (plus flat ``exp_avg`` /
``exp_avg_sq``), so a step is two launches of ``libflowdiff.so``: ``fd_sumsq`` (gradient norm, stays on the
device) and ``fd_adam_step`` (clip coefficient + decay + Adam, i.e. the whole post-reduce pass is one kernel).

Gradient exchange: ``GradSync`` is DDP's bucketed all-reduce.  The UNet's backward announces each of its eight
contiguous gradient buckets as soon as the backward has walked past the bucket's layers (``unet_train.GRAD_GROUPS``,
reverse layer order); the bucket is all-reduced over NCCL right away, asynchronously, while the rest of the backward
keeps the SMs busy.  90 % of the 143 MB sit in the deep levels, which finish first; only the last bucket (init_conv,
time MLP, the two full-resolution levels: ~2 MB) is exchanged after the last backward kernel.  Measured in round 1
with ONE all-reduce after the backward: 0.28 ms (N = 1) -> 1.86 ms (N = 8) for all-reduce + clip + Adam of a 55 ms step.
``allreduce_gradients`` is the un-overlapped single-collective form (gradient accumulation, foreign modules).

Weight EMA (opt-in, ``ema_params``): the averaged weights live in a third flat buffer at the parameters' offsets, and on
the steps the schedule (``ema_weight``) selects, ``fd_adam_ema_step`` replaces ``fd_adam_step`` and updates them from the
freshly written parameters in the same pass: 36 instead of 28 bytes per parameter, no extra launch."""
from __future__ import annotations

import os
from typing import Callable, Iterable, Optional

import torch
import torch.distributed as dist

from . import _lib


def ema_weight(k: int, beta: float, after: int, every: int) -> Optional[float]:
    """Weight ``w`` of the EMA update ``ema <- lerp(ema, p, w)`` after optimiser step ``k`` (1-based, counted after the
    step), or None when step ``k`` leaves the EMA alone.  Up to step ``after`` the EMA copies the weights (w = 1); then
    every ``every`` steps it decays with ema_pytorch's warm-up at inv_gamma = 1, power = 2/3:
    ``d = min(beta, 1 - (1 + j) ** (-2/3))``, ``w = 1 - d``, with ``j = k - after``.  float64 throughout."""
    if k <= after:
        return 1.0
    j = k - after
    if j % every != 0:
        return None
    return 1.0 - min(float(beta), 1.0 - (1.0 + j) ** (-2.0 / 3.0))


class FusedAdam(torch.optim.Optimizer):
    """Drop-in for ``torch.optim.Adam(params, lr, betas, eps, weight_decay)`` (same update, same state names).

    ``max_grad_norm`` > 0 folds ``clip_grad_norm_`` into the step; ``grad_scale`` multiplies the gradients first
    (``1 / world_size`` after a SUM all-reduce).  ``on_step`` is called after every step (the UNet uses it to
    invalidate its packed bf16 weights).

    ``ema_params``: tensors aligned one-to-one (shape and order) with the parameters this optimiser updates; they keep an
    exponential moving average of them on the schedule of ``ema_weight(step, ema_decay, ema_update_after_step,
    ema_update_every)``.  ``ema_updated`` tells ``on_step`` whether the last step changed them."""

    def __init__(self, params: Iterable[torch.nn.Parameter], lr: float = 1e-3, betas=(0.9, 0.999), eps: float = 1e-8,
                 weight_decay: float = 0.0, max_grad_norm: float = 0.0, on_step: Optional[Callable[[], None]] = None,
                 ema_params: Optional[Iterable[torch.Tensor]] = None, ema_decay: float = 0.9999,
                 ema_update_after_step: int = 100, ema_update_every: int = 10):
        defaults = dict(lr=lr, betas=tuple(betas), eps=eps, weight_decay=weight_decay)
        super().__init__(params, defaults)
        if len(self.param_groups) != 1:
            raise ValueError("FusedAdam keeps one flat buffer: pass a single parameter group")
        self.ema_params = list(ema_params) if ema_params is not None else None
        if self.ema_params is not None:
            if not 0.0 <= float(ema_decay) < 1.0 or int(ema_update_after_step) < 0 or int(ema_update_every) < 1:
                raise ValueError("need 0 <= ema_decay < 1, ema_update_after_step >= 0 and ema_update_every >= 1")
            params_ = self._params()
            if len(params_) != len(self.ema_params) or any(p.shape != e.shape for p, e in zip(params_, self.ema_params)):
                raise ValueError("ema_params must match the optimised parameters one-to-one in shape and order")
        self.ema_decay, self.ema_update_after_step = float(ema_decay), int(ema_update_after_step)
        self.ema_update_every = int(ema_update_every)
        self.ema_updated = False                         # whether the last step() changed the EMA
        self._flat_ema: Optional[torch.Tensor] = None
        self.max_grad_norm = float(max_grad_norm)
        self.grad_scale = 1.0
        self.on_step = on_step
        self._flat_p: Optional[torch.Tensor] = None
        self._offsets = None
        self._reduced: Optional[torch.Tensor] = None     # flat gradient already exchanged by allreduce_gradients
        self._presynced = False                          # GradSync exchanged p.grad during the backward
        self.step_count = 0

    # ------------------------------------------------------------------ flat storage
    def _params(self):
        return [p for p in self.param_groups[0]["params"] if p.requires_grad]

    def _flatten(self):
        params = self._params()
        dev = params[0].device
        for p in params + (self.ema_params or []):
            if not p.is_cuda or p.dtype != torch.float32:
                raise _lib.FlowDiffError("FusedAdam updates fp32 CUDA parameters (no CPU fallback)")
        offs, off = [], 0
        for p in params:
            offs.append(off)
            off += (p.numel() + 3) // 4 * 4
        flat = torch.zeros(off, device=dev, dtype=torch.float32)
        for p, o in zip(params, offs):
            view = flat[o:o + p.numel()].view_as(p)
            view.copy_(p.data)
            p.data = view                      # the module's parameters now alias the flat buffer
        self._flat_p, self._offsets, self._n = flat, offs, off
        if self.ema_params is not None:          # same offsets: one kernel index addresses a parameter and its average
            flat_e = torch.zeros(off, device=dev, dtype=torch.float32)
            for e, o in zip(self.ema_params, offs):
                view = flat_e[o:o + e.numel()].view_as(e)
                view.copy_(e.data)
                e.data = view
            self._flat_ema = flat_e
        self._flat_g = torch.zeros(off, device=dev, dtype=torch.float32)
        m = torch.zeros(off, device=dev, dtype=torch.float32)
        v = torch.zeros(off, device=dev, dtype=torch.float32)
        self._sumsq = torch.zeros(1, device=dev, dtype=torch.float32)
        for p, o in zip(params, offs):         # torch.optim-compatible state views (state_dict / checkpoints)
            old = self.state.get(p)            # state restored by load_state_dict (resume) moves into the flat buffers
            mv, vv = m[o:o + p.numel()].view_as(p), v[o:o + p.numel()].view_as(p)
            step = torch.tensor(0.0)
            if old:
                mv.copy_(old["exp_avg"])
                vv.copy_(old["exp_avg_sq"])
                step = torch.as_tensor(old["step"]).detach().float().cpu().clone()
                self.step_count = int(step)
            self.state[p] = {"step": step, "exp_avg": mv, "exp_avg_sq": vv}
        self._m, self._v = m, v

    def load_state_dict(self, state_dict):
        super().load_state_dict(state_dict)
        self._flat_p = None                    # re-flatten on the next step: picks the restored moments up

    def _still_flat(self) -> bool:
        if self._flat_p is None:
            return False
        base = self._flat_p.data_ptr()
        if not all(p.data_ptr() == base + 4 * o for p, o in zip(self._params(), self._offsets)):
            return False
        if self.ema_params is None:
            return True
        base = self._flat_ema.data_ptr()
        return all(e.data_ptr() == base + 4 * o for e, o in zip(self.ema_params, self._offsets))

    def flat_gradient(self) -> torch.Tensor:
        """The gradients as one flat tensor laid out like the parameters (zero-copy when ``p.grad`` already are
        consecutive views of one buffer, as ``UnetFunction.backward`` returns them)."""
        params = self._params()
        g0 = params[0].grad
        if g0 is not None:
            base = g0.data_ptr()
            if all(p.grad is not None and p.grad.data_ptr() == base + 4 * o and p.grad.is_contiguous()
                   for p, o in zip(params, self._offsets)):
                st = g0.untyped_storage()
                start = (base - st.data_ptr()) // 4
                if start * 4 + self._n * 4 <= st.nbytes():
                    return torch.empty(0, device=g0.device, dtype=torch.float32).set_(st, start, (self._n,))
        self._flat_g.zero_()
        for p, o in zip(params, self._offsets):
            if p.grad is not None:
                self._flat_g[o:o + p.numel()].view_as(p).copy_(p.grad)
        return self._flat_g

    # ------------------------------------------------------------------ step
    @torch.no_grad()
    def step(self, closure=None):
        loss = None
        if closure is not None:
            with torch.enable_grad():
                loss = closure()
        if not self._still_flat():
            self._flatten()
        lib = _lib.load(check_device=True)
        g = self._reduced if self._reduced is not None else self.flat_gradient()
        self._reduced = None
        self._presynced = False
        grp = self.param_groups[0]
        self.step_count += 1
        st = _lib.stream()
        sumsq = None
        if self.max_grad_norm > 0:
            self._sumsq.zero_()
            _lib.check(lib.fd_sumsq(_lib.ptr(g), self._n, _lib.ptr(self._sumsq), st))
            sumsq = self._sumsq
        b1, b2 = grp["betas"]
        w = None
        if self.ema_params is not None:
            w = ema_weight(self.step_count, self.ema_decay, self.ema_update_after_step, self.ema_update_every)
        args = (float(grp["lr"]), float(b1), float(b2), float(grp["eps"]), float(grp["weight_decay"]), self.step_count,
                _lib.ptr(sumsq), self.max_grad_norm, float(self.grad_scale))
        if w is None:
            _lib.check(lib.fd_adam_step(_lib.ptr(self._flat_p), _lib.ptr(g), _lib.ptr(self._m), _lib.ptr(self._v), self._n,
                                        *args, st))
        else:
            _lib.check(lib.fd_adam_ema_step(_lib.ptr(self._flat_p), _lib.ptr(g), _lib.ptr(self._m), _lib.ptr(self._v),
                                            _lib.ptr(self._flat_ema), self._n, *args, w, st))
        self.ema_updated = w is not None
        for p in self._params():
            self.state[p]["step"] += 1
        if self.on_step is not None:
            self.on_step()
        return loss

    def grad_norm(self) -> torch.Tensor:
        """Global L2 norm of the (scaled) gradient seen by the last step (device scalar)."""
        return self._sumsq.sqrt() * self.grad_scale


class GradSync:
    """Bucketed, overlapped gradient all-reduce (DDPStrategy's exchange, exp_base.py:198).

    ``attach(unet)`` registers it as the UNet's ``grad_sync``: during ``UnetFunction.backward`` the UNet calls
    ``bucket_ready(flat, lo, hi)`` when elements [lo, hi) of its flat gradient buffer are final, and ``finish(flat)``
    after its last kernel.  Each bucket is SUM-all-reduced asynchronously (NCCL runs it on its own stream, ordered
    after the kernels launched so far); ``finish`` makes the launching stream wait for all of them.  The 1/world mean
    is folded into the optimiser's ``grad_scale``.  ``comm_dtype=torch.bfloat16`` exchanges a bf16 copy of each bucket
    (half the bytes; the reference's DDP exchanges fp32, which is the default here)."""

    def __init__(self, optimizer: Optional["FusedAdam"] = None, group=None, comm_dtype: Optional[torch.dtype] = None):
        self.optimizer, self.group = optimizer, group
        self.comm_dtype = comm_dtype if comm_dtype not in (None, torch.float32) else None
        self._pending = []
        self._stage: Optional[torch.Tensor] = None
        self.buckets_last_backward = 0
        self.bytes_last_backward = 0

    def world(self) -> int:
        if not (dist.is_available() and dist.is_initialized()):
            return 1
        return dist.get_world_size(self.group)

    def attach(self, unet) -> "GradSync":
        unet.grad_sync = self
        return self

    @staticmethod
    def detach(unet) -> None:
        unet.grad_sync = None

    def bucket_ready(self, flat: torch.Tensor, lo: int, hi: int) -> None:
        if self.world() == 1:
            return
        if not self._pending:
            self.buckets_last_backward = self.bytes_last_backward = 0
        t = flat[lo:hi]
        if self.comm_dtype is not None:
            if self._stage is None or self._stage.numel() != flat.numel() or self._stage.device != flat.device:
                self._stage = torch.empty(flat.numel(), device=flat.device, dtype=self.comm_dtype)
            buf = self._stage[lo:hi]
            buf.copy_(t)
        else:
            buf = t
        work = dist.all_reduce(buf, op=dist.ReduceOp.SUM, group=self.group, async_op=True)
        self._pending.append((work, lo, hi, buf))
        self.buckets_last_backward += 1
        self.bytes_last_backward += buf.numel() * buf.element_size()

    def finish(self, flat: torch.Tensor) -> None:
        if not self._pending:
            return
        for work, lo, hi, buf in self._pending:
            work.wait()                          # stream-orders the launching stream after the collective
            if self.comm_dtype is not None:
                flat[lo:hi].copy_(buf)
        self._pending = []
        if self.optimizer is not None:
            self.optimizer.grad_scale = 1.0 / self.world()
            self.optimizer._presynced = True     # allreduce_gradients() must not exchange this gradient again


def allreduce_gradients(optimizer: FusedAdam, group=None) -> None:
    """DDP's exchange step in one collective: SUM all-reduce of the flat gradient over NCCL (gloo in the CPU tests); the
    1/world mean is folded into the optimiser's ``grad_scale``.  No-op when ``GradSync`` already exchanged this
    gradient bucket by bucket during the backward."""
    if int(os.environ.get("WORLD_SIZE", "1")) > 1 and not (dist.is_available() and dist.is_initialized()):
        raise RuntimeError("WORLD_SIZE > 1 but torch.distributed is not initialised: the replicas would train "
                           "independently (call dist.init_process_group before the first training step)")
    if not (dist.is_available() and dist.is_initialized()):
        return
    world = dist.get_world_size(group)
    if world == 1:
        return
    if getattr(optimizer, "_presynced", False):
        optimizer._presynced = False
        return
    if not optimizer._still_flat():
        optimizer._flatten()
    g = optimizer.flat_gradient()
    dist.all_reduce(g, op=dist.ReduceOp.SUM, group=group)
    optimizer._reduced = g                      # the next step() consumes exactly this buffer
    optimizer.grad_scale = 1.0 / world


def allreduce_flat(t: torch.Tensor, group=None) -> torch.Tensor:
    """SUM all-reduce + mean of any flat tensor (host-logic helper, used by the gloo tests)."""
    if dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1:
        dist.all_reduce(t, op=dist.ReduceOp.SUM, group=group)
        t /= dist.get_world_size(group)
    return t
