"""Diffusion process around the UNet: schedule tables, forward noising, DDPM / DDIM sampling and the
NaN-aware x0 loss -- the ``ConditionalDiffusion`` surface of the reference
(denoising_diffusion.py:463-993) for the configuration flow_diffuser uses
(objective ``pred_x0``, sigmoid schedule, ``noise_space='image'``, no self-conditioning,
``auto_normalize=False``; flow_diffuser.py:117-127).

Differences from the reference, all forced by SURVEY.md's "seven facts":
  * ``image_size`` may be ``(H, W)``; nothing asserts square inputs (:986-987 could not run 436x1024);
  * ``sampling_timesteps`` is honoured and ``ddim_sample`` accepts ``additional_tgt`` (:732,784 raise);
  * the per-step scheduler math is ONE fused launch (``fd_ddim_step`` / ``fd_ddpm_step``) whose scalars
    are computed on the host from the fp32 tables exactly as the reference's 0-d tensor ops do;
  * ``return_all_timesteps`` writes every state straight into one preallocated buffer.
"""
from __future__ import annotations

import math
from typing import List, Optional, Sequence, Tuple, Union

import torch
from torch import nn

from . import _lib
from . import warp as W

Tensor = torch.Tensor


def sigmoid_beta_schedule(timesteps: int, start: float = -3, end: float = 3, tau: float = 1) -> Tensor:
    """float64 sigmoid schedule (denoising_diffusion.py:448-461)."""
    t = torch.linspace(0, timesteps, timesteps + 1, dtype=torch.float64) / timesteps
    lo, hi = torch.tensor(start / tau).sigmoid(), torch.tensor(end / tau).sigmoid()
    ac = (hi - ((t * (end - start) + start) / tau).sigmoid()) / (hi - lo)
    ac = ac / ac[0]
    return torch.clip(1 - ac[1:] / ac[:-1], 0, 0.999)


def ddim_time_pairs(total: int, steps: int) -> List[Tuple[int, int]]:
    """The integer DDIM grid (:737-739): fp32 linspace(-1, T-1, S+1) truncated to int, reversed."""
    times = list(reversed(torch.linspace(-1, total - 1, steps=steps + 1).int().tolist()))
    return list(zip(times[:-1], times[1:]))


def dpmpp_coeffs(alphas_cumprod: Sequence[float], times: Sequence[int], i: int, order: int):
    """Coefficients of step ``i`` of the multistep DPM-Solver++ (data prediction; Lu et al., arXiv:2211.01095) on the
    grid ``times`` (descending, ending at -1): ``x_next = cx*x + c0*D0 + c1*D1 + c2*D2`` with D0 the clamped prediction at
    ``times[i]`` and D1 / D2 those at ``times[i-1]`` / ``times[i-2]``.  float64 from the fp32 ``alphas_cumprod`` table.
    The step uses order ``min(order, i + 1)``; the final step (to -1) returns D0: ``(0, 1, 0, 0, last=1)``.
    Order 1 is DDIM with eta = 0: ``cx = sigma_t / sigma_s``, ``c0 = alpha_t - alpha_s * sigma_t / sigma_s``."""
    s, t = int(times[i]), int(times[i + 1])
    if t < 0:
        return 0.0, 1.0, 0.0, 0.0, 1
    k = min(int(order), i + 1)

    def alpha_sigma_lambda(tt):
        a = float(alphas_cumprod[tt])
        al, sg = math.sqrt(a), math.sqrt(1.0 - a)
        return al, sg, math.log(al) - math.log(sg)

    _, sigma_s, lam_s = alpha_sigma_lambda(s)
    alpha_t, sigma_t, lam_t = alpha_sigma_lambda(t)
    h = lam_t - lam_s
    phi1 = math.expm1(-h)
    cx, c0, c1, c2 = sigma_t / sigma_s, -alpha_t * phi1, 0.0, 0.0
    if k >= 2:
        lam_1 = alpha_sigma_lambda(int(times[i - 1]))[2]
        r0 = (lam_s - lam_1) / h
        if k == 2:                                 # - alpha_t*phi1/2 * (D0 - D1)/r0
            c0 += -0.5 * alpha_t * phi1 / r0
            c1 = 0.5 * alpha_t * phi1 / r0
        else:                                      # + alpha_t*phi2*Dd1 - alpha_t*phi3*Dd2
            lam_2 = alpha_sigma_lambda(int(times[i - 2]))[2]
            r1 = (lam_1 - lam_2) / h
            phi2 = phi1 / h + 1.0
            phi3 = phi2 / h - 0.5
            f = r0 / (r0 + r1)
            m = 1.0 / (r0 + r1)
            # E0 = (D0 - D1)/r0, E1 = (D1 - D2)/r1, Dd1 = E0 + f*(E0 - E1), Dd2 = m*(E0 - E1), expanded in D0, D1, D2
            c0 += alpha_t * phi2 * (1.0 + f) / r0 - alpha_t * phi3 * m / r0
            c1 = (alpha_t * phi2 * (-(1.0 + f) / r0 - f / r1) + alpha_t * phi3 * m * (1.0 / r0 + 1.0 / r1))
            c2 = alpha_t * phi2 * f / r1 - alpha_t * phi3 * m / r1
    return cx, c0, c1, c2, 0


class _SqErrSums(torch.autograd.Function):
    """(sum over non-NaN pairs of (a-b)^2, their count) with the gradient wrt ``a`` (warp.py:260-271 under autograd)."""

    @staticmethod
    def forward(ctx, a: Tensor, b: Tensor):
        a, b = a.detach().float().contiguous(), b.detach().float().contiguous()
        lib = _lib.load()
        n = a.numel()
        sums = torch.empty(3, device=a.device, dtype=torch.float32)
        ws = torch.empty(lib.fd_nan_mse_workspace_floats(1, 1, n), device=a.device, dtype=torch.float32)
        _lib.check(lib.fd_nan_mse_fwd(_lib.ptr(a), _lib.ptr(b), _lib.ptr(sums), _lib.ptr(ws), 1, 1, n, n, n, _lib.stream()))
        ctx.save_for_backward(a, b)
        num, den = sums[0].clone(), sums[1].clone()
        ctx.mark_non_differentiable(den)
        return num, den

    @staticmethod
    def backward(ctx, gnum: Tensor, _gden):
        a, b = ctx.saved_tensors
        n = a.numel()
        ga = torch.empty_like(a)
        lib = _lib.load()
        # the kernel scales by 2 * upstream / sums[1]: the upstream gradient stays on the device as sums[1] = 1 / g (reading
        # it on the host would be a device-to-host sync at the head of every backward pass)
        unit = torch.zeros(3, device=a.device, dtype=torch.float32)
        unit[1] = 1.0 / gnum.detach().float()
        _lib.check(lib.fd_nan_mse_bwd(_lib.ptr(a), _lib.ptr(b), _lib.ptr(unit), 1.0, _lib.ptr(ga), 1, 1, n, n, n, n,
                                      _lib.stream()))
        return ga, None


class ConditionalDiffusion(nn.Module):
    BUFFERS = ("betas", "alphas_cumprod", "alphas_cumprod_prev", "sqrt_alphas_cumprod",
               "sqrt_one_minus_alphas_cumprod", "log_one_minus_alphas_cumprod", "sqrt_recip_alphas_cumprod",
               "sqrt_recipm1_alphas_cumprod", "posterior_variance", "posterior_log_variance_clipped",
               "posterior_mean_coef1", "posterior_mean_coef2", "loss_weight")

    def __init__(self, model: nn.Module, image_size: Union[int, Sequence[int]], timesteps: int = 1000,
                 sampling_timesteps: Optional[int] = None, objective: str = "pred_x0", beta_schedule: str = "sigmoid",
                 ddim_sampling_eta: float = 0.0, auto_normalize: bool = False, min_snr_loss_weight: bool = True,
                 min_snr_gamma: float = 5.0, conditioned: bool = True, channels: int = 2, noise_space: str = "image",
                 sampler: Optional[str] = None, solver_order: int = 2):
        super().__init__()
        if objective != "pred_x0" or beta_schedule != "sigmoid" or noise_space != "image" or auto_normalize:
            raise NotImplementedError("flow_diffuser uses objective=pred_x0, sigmoid schedule, image noise space, "
                                      "auto_normalize=False (flow_diffuser.py:117-127); nothing else is on the hot path")
        if sampler not in (None, "dpmpp"):
            raise ValueError(f"sampler must be null (DDIM / DDPM as the reference) or 'dpmpp', not {sampler!r}")
        if int(solver_order) not in (1, 2, 3):
            raise ValueError(f"solver_order must be 1, 2 or 3, not {solver_order}")
        if sampler == "dpmpp" and float(ddim_sampling_eta) > 0:
            raise NotImplementedError("sampler='dpmpp' is the deterministic solver: ddim_sampling_eta must be 0")
        self.sampler = sampler           # None: DDIM when sampling_timesteps < timesteps, else DDPM; "dpmpp": DPM-Solver++
        self.solver_order = int(solver_order)
        self.model = model
        self.channels = channels
        self.conditioned = conditioned
        self.noise_space = noise_space
        self.objective = objective
        self.image_size = (image_size, image_size) if isinstance(image_size, int) else tuple(int(v) for v in image_size)
        self.self_condition = False
        self._graphs = {}          # CUDA graphs of the DDIM / DPM-Solver++ loops, keyed by sampler and shapes
        self.graph_replayed_launches = 0   # kernels executed through graph replays (not seen by fd_launch_count)

        betas = sigmoid_beta_schedule(timesteps)
        alphas = 1.0 - betas
        ac = torch.cumprod(alphas, dim=0)
        ac_prev = torch.nn.functional.pad(ac[:-1], (1, 0), value=1.0)
        self.num_timesteps = int(betas.shape[0])
        self.sampling_timesteps = int(sampling_timesteps) if sampling_timesteps is not None else self.num_timesteps
        assert self.sampling_timesteps <= self.num_timesteps
        self.is_ddim_sampling = self.sampling_timesteps < self.num_timesteps
        self.ddim_sampling_eta = float(ddim_sampling_eta)

        post_var = betas * (1.0 - ac_prev) / (1.0 - ac)
        snr = ac / (1 - ac)
        table = {
            "betas": betas, "alphas_cumprod": ac, "alphas_cumprod_prev": ac_prev,
            "sqrt_alphas_cumprod": ac.sqrt(), "sqrt_one_minus_alphas_cumprod": (1.0 - ac).sqrt(),
            "log_one_minus_alphas_cumprod": (1.0 - ac).log(), "sqrt_recip_alphas_cumprod": (1.0 / ac).sqrt(),
            "sqrt_recipm1_alphas_cumprod": (1.0 / ac - 1).sqrt(), "posterior_variance": post_var,
            "posterior_log_variance_clipped": post_var.clamp(min=1e-20).log(),
            "posterior_mean_coef1": betas * ac_prev.sqrt() / (1.0 - ac),
            "posterior_mean_coef2": (1.0 - ac_prev) * alphas.sqrt() / (1.0 - ac),
            "loss_weight": (snr.clone().clamp_(max=min_snr_gamma) if min_snr_loss_weight else snr),   # registered, unused (:975-980)
        }
        for name in self.BUFFERS:
            self.register_buffer(name, table[name].to(torch.float32))
        # host copies: the per-step scalars are looked up here, never read back from the device
        self._host = {k: table[k].to(torch.float32) for k in self.BUFFERS}

    @property
    def device(self):
        return self.betas.device

    def normalize(self, x):      # auto_normalize=False -> identity (:585)
        return x

    def unnormalize(self, x):
        return x

    # ------------------------------------------------------------------ forward process
    def q_sample(self, x_start: Tensor, t: Tensor, noise: Optional[Tensor] = None) -> Tensor:
        """:806-812 as one launch."""
        if noise is None:
            noise = torch.randn_like(x_start)
        x_start, noise = x_start.float().contiguous(), noise.float().contiguous()
        _lib.require_cuda(x_start, noise, t)
        out = torch.empty_like(x_start)
        lib = _lib.load()
        B = x_start.shape[0]
        t = t.to(torch.int64).contiguous()
        _lib.check(lib.fd_q_sample(_lib.ptr(x_start), _lib.ptr(noise), _lib.ptr(t), _lib.ptr(self.sqrt_alphas_cumprod),
                                   _lib.ptr(self.sqrt_one_minus_alphas_cumprod), _lib.ptr(out), B,
                                   x_start.numel() // B, _lib.stream()))
        return out

    # ------------------------------------------------------------------ model call
    def model_with_condition(self, x, t, x_self_cond=None, external_cond=None, additional_tgt=None):
        assert self.conditioned == torch.is_tensor(external_cond)
        from .unet import Unet
        if isinstance(self.model, Unet):
            return self.model(x, external_cond, t)
        return self.model(x, external_cond, t, None, additional_out=additional_tgt is not None)

    # ------------------------------------------------------------------ reverse process
    def _ddim_scalars(self, time: int, time_next: int):
        """Host-side fp32 replica of the 0-d tensor arithmetic at :757-761."""
        h = self._host
        recip, recipm1 = float(h["sqrt_recip_alphas_cumprod"][time]), float(h["sqrt_recipm1_alphas_cumprod"][time])
        if time_next < 0:
            return recip, recipm1, 0.0, 0.0, 0.0, 1
        alpha, alpha_next = h["alphas_cumprod"][time], h["alphas_cumprod"][time_next]
        sigma = self.ddim_sampling_eta * ((1 - alpha / alpha_next) * (1 - alpha_next) / (1 - alpha)).sqrt()
        c = (1 - alpha_next - sigma ** 2).sqrt()
        return recip, recipm1, float(alpha_next.sqrt()), float(c), float(sigma), 0

    def _split_model_out(self, out: Tensor, additional_tgt):
        if additional_tgt is None:
            return out, None
        k = additional_tgt.shape[1]
        return out[:, :-k].contiguous(), out[:, -k:]

    @torch.no_grad()
    def ddim_sample(self, shape, return_all_timesteps: bool = False, external_cond: Optional[Tensor] = None,
                    additional_tgt: Optional[Tensor] = None, x_T: Optional[Tensor] = None,
                    noises: Optional[Sequence[Tensor]] = None):
        """:731-774.  ``x_T`` / ``noises`` inject the random draws (parity runs); otherwise they come from
        the device generator in the reference's order (x_T first, then one draw per step, used only if eta > 0)."""
        lib = _lib.load(check_device=True)
        dev = self.device
        B = shape[0]
        pairs = ddim_time_pairs(self.num_timesteps, self.sampling_timesteps)
        img = (x_T.to(dev).float().contiguous().clone() if x_T is not None else torch.randn(shape, device=dev))
        n = img.numel()
        traj = None
        if return_all_timesteps:
            traj = torch.empty((len(pairs) + 1,) + tuple(img.shape), device=dev, dtype=torch.float32)
            traj[0].copy_(img)
        additionals = [None]
        eta = self.ddim_sampling_eta
        for i, (time, time_next) in enumerate(pairs):
            t = torch.full((B,), time, device=dev, dtype=torch.long)
            out = self.model_with_condition(img, t, None, external_cond, additional_tgt)
            out, add = self._split_model_out(out, additional_tgt)
            additionals.append(add)
            recip, recipm1, san, c, sigma, last = self._ddim_scalars(time, time_next)
            noise = None
            if not last:
                if noises is not None:
                    noise = noises[i].to(dev).float().contiguous()
                elif eta > 0:
                    noise = torch.randn_like(img)
            nxt = traj[i + 1] if traj is not None else img
            _lib.check(lib.fd_ddim_step(_lib.ptr(img), _lib.ptr(out), _lib.ptr(noise) if sigma != 0.0 else None,
                                        _lib.ptr(nxt), None, n, recip, recipm1, san, c, sigma, last, _lib.stream()))
            img = nxt
        ret = traj.transpose(0, 1) if traj is not None else img      # time axis at dim 1 like torch.stack(imgs, 1)
        return (ret, additionals) if additional_tgt is not None else ret

    @torch.no_grad()
    def p_sample_loop(self, shape, return_all_timesteps: bool = False, external_cond: Optional[Tensor] = None,
                      additional_tgt: Optional[Tensor] = None, x_T: Optional[Tensor] = None,
                      noises: Optional[Sequence[Tensor]] = None):
        """:700-729 + p_sample :677-698 + q_posterior :613-623 (ancestral DDPM)."""
        lib = _lib.load(check_device=True)
        dev = self.device
        B = shape[0]
        h = self._host
        img = (x_T.to(dev).float().contiguous().clone() if x_T is not None else torch.randn(shape, device=dev))
        n = img.numel()
        T = self.num_timesteps
        traj = None
        if return_all_timesteps:
            traj = torch.empty((T + 1,) + tuple(img.shape), device=dev, dtype=torch.float32)
            traj[0].copy_(img)
        additionals = [None]
        for i, time in enumerate(reversed(range(T))):
            t = torch.full((B,), time, device=dev, dtype=torch.long)
            out = self.model_with_condition(img, t, None, external_cond, additional_tgt)
            out, add = self._split_model_out(out, additional_tgt)
            additionals.append(add)
            noise = None
            if time > 0:
                noise = noises[i].to(dev).float().contiguous() if noises is not None else torch.randn_like(img)
            sigma = float((0.5 * h["posterior_log_variance_clipped"][time]).exp())
            nxt = traj[i + 1] if traj is not None else img
            _lib.check(lib.fd_ddpm_step(_lib.ptr(img), _lib.ptr(out), _lib.ptr(noise), _lib.ptr(nxt), None, n,
                                        float(h["posterior_mean_coef1"][time]), float(h["posterior_mean_coef2"][time]),
                                        sigma, _lib.stream()))
            img = nxt
        ret = traj.transpose(0, 1) if traj is not None else img
        return (ret, additionals) if additional_tgt is not None else ret

    @torch.no_grad()
    def dpmpp_sample(self, shape, return_all_timesteps: bool = False, external_cond: Optional[Tensor] = None,
                     additional_tgt: Optional[Tensor] = None, x_T: Optional[Tensor] = None):
        """Multistep DPM-Solver++ (orders 1-3, ``self.solver_order``) on the DDIM time grid, with the contract and return
        shapes of ``ddim_sample``.  One fused launch per step (``fd_dpmpp_step``) clamps the prediction, writes it into
        the history slot the next steps read, and applies the update; two rotating slots hold D_{i-1} and D_{i-2}
        (order 3 overwrites the older one in the same pass that reads it).  Order 1 is DDIM with eta = 0."""
        if self.ddim_sampling_eta > 0:
            raise NotImplementedError("sampler='dpmpp' is the deterministic solver: ddim_sampling_eta must be 0")
        lib = _lib.load(check_device=True)
        dev = self.device
        B = shape[0]
        pairs = ddim_time_pairs(self.num_timesteps, self.sampling_timesteps)
        times = [p[0] for p in pairs] + [pairs[-1][1]]
        ac = self._host["alphas_cumprod"].tolist()
        img = (x_T.to(dev).float().contiguous().clone() if x_T is not None else torch.randn(shape, device=dev))
        n = img.numel()
        traj = None
        if return_all_timesteps:
            traj = torch.empty((len(pairs) + 1,) + tuple(img.shape), device=dev, dtype=torch.float32)
            traj[0].copy_(img)
        hist = (torch.empty_like(img), torch.empty_like(img))
        additionals = [None]
        for i, (time, _) in enumerate(pairs):
            t = torch.full((B,), time, device=dev, dtype=torch.long)
            out = self.model_with_condition(img, t, None, external_cond, additional_tgt)
            out, add = self._split_model_out(out, additional_tgt)
            additionals.append(add)
            cx, c0, c1, c2, last = dpmpp_coeffs(ac, times, i, self.solver_order)
            d_out = hist[i % 2]                 # D_{i-2}'s slot: read (order 3) and overwritten with D_i in one pass
            d1 = hist[(i + 1) % 2] if c1 != 0.0 else None
            d2 = d_out if c2 != 0.0 else None
            nxt = traj[i + 1] if traj is not None else img
            _lib.check(lib.fd_dpmpp_step(_lib.ptr(img), _lib.ptr(out), _lib.ptr(d1), _lib.ptr(d2), _lib.ptr(nxt),
                                         _lib.ptr(d_out), n, cx, c0, c1, c2, last, _lib.stream()))
            img = nxt
        ret = traj.transpose(0, 1) if traj is not None else img
        return (ret, additionals) if additional_tgt is not None else ret

    @torch.no_grad()
    def _sample_graphed(self, fn, shape, return_all_timesteps: bool, external_cond: Tensor, x_T: Optional[Tensor]):
        """A whole deterministic sampling loop -- eta = 0 DDIM or DPM-Solver++, ``fn`` -- (S UNet forwards + S fused
        updates, ~8k launches at S = 50) as ONE CUDA graph: captured once per (sampler, shape, device), replayed with the
        inputs copied into static buffers.  Neither sampler draws per-step noise, so only x_T is random and it is drawn
        outside the graph; the DPM-Solver++ history buffers are allocated inside the capture and live with the graph."""
        dev = self.device
        key = (fn.__name__, self.solver_order if fn == self.dpmpp_sample else None,
               tuple(shape), bool(return_all_timesteps), tuple(external_cond.shape), dev.index)
        if x_T is None:
            x_T = torch.randn(shape, device=dev)
        # The graph holds raw pointers: to the packed bf16 weights and the concatenated time-MLP weights (both rewritten
        # IN PLACE by prepare(), so calling it here before every replay is what keeps a replay after an optimiser step or
        # a checkpoint load current) and to the parameter storages themselves (biases, GroupNorm / LayerNorm gains, the
        # time MLP), which move when an optimiser flattens them or a module is moved: then the graph is re-captured.
        self.model.prepare()
        ptrs = hash(tuple(p.data_ptr() for p in self.model.parameters()))
        entry = self._graphs.get(key)
        if entry is not None and entry[5] != ptrs:
            entry = None
            del self._graphs[key]
        if entry is None:
            s_cond = external_cond.detach().float().contiguous().clone()
            s_x = x_T.detach().to(dev).float().contiguous().clone()
            side = torch.cuda.Stream(device=dev)
            side.wait_stream(torch.cuda.current_stream(dev))
            with torch.cuda.stream(side):        # eager warm-up: lazy one-time initialisation must not be captured
                fn(shape, return_all_timesteps, s_cond, x_T=s_x)
            torch.cuda.current_stream(dev).wait_stream(side)
            graph = torch.cuda.CUDAGraph()
            lib = _lib.load()
            n0 = lib.fd_launch_count()
            with torch.cuda.graph(graph):
                s_out = fn(shape, return_all_timesteps, s_cond, x_T=s_x)
            entry = (graph, s_cond, s_x, s_out, int(lib.fd_launch_count() - n0), ptrs)
            self._graphs[key] = entry
        graph, s_cond, s_x, s_out, n_kernels, _ = entry
        s_cond.copy_(external_cond)
        s_x.copy_(x_T)
        graph.replay()
        self.graph_replayed_launches += n_kernels
        return s_out.clone()

    @torch.no_grad()
    def sample(self, batch_size: int = 16, return_all_timesteps: bool = False, external_cond: Optional[Tensor] = None,
               additional_tgt: Optional[Tensor] = None, image_size: Optional[Sequence[int]] = None,
               use_cuda_graph: bool = False, **kw):
        """:776-784.  The spatial size follows ``external_cond`` when given, else ``image_size``."""
        if external_cond is not None:
            assert external_cond.shape[0] == batch_size
            hw = tuple(external_cond.shape[-2:])
        else:
            hw = tuple(image_size) if image_size is not None else self.image_size
        shape = (batch_size, self.channels) + hw
        from .unet import Unet
        if self.sampler == "dpmpp":
            if use_cuda_graph and additional_tgt is None and external_cond is not None and isinstance(self.model, Unet):
                return self._sample_graphed(self.dpmpp_sample, shape, return_all_timesteps, external_cond, kw.get("x_T"))
            return self.dpmpp_sample(shape, return_all_timesteps=return_all_timesteps, external_cond=external_cond,
                                     additional_tgt=additional_tgt, **kw)
        if (use_cuda_graph and self.is_ddim_sampling and self.ddim_sampling_eta == 0.0 and additional_tgt is None
                and external_cond is not None and kw.get("noises") is None and isinstance(self.model, Unet)):
            return self._sample_graphed(self.ddim_sample, shape, return_all_timesteps, external_cond, kw.get("x_T"))
        fn = self.ddim_sample if self.is_ddim_sampling else self.p_sample_loop
        return fn(shape, return_all_timesteps=return_all_timesteps, external_cond=external_cond,
                  additional_tgt=additional_tgt, **kw)

    # ------------------------------------------------------------------ loss
    def p_losses(self, x_start: Tensor, t: Tensor, noise: Optional[Tensor] = None, external_cond: Optional[Tensor] = None,
                 additional_tgt=None, additional_weight=None, model_out_override=None) -> Tensor:
        """:823-891 (value only in this round; the backward kernels are the next build step)."""
        x = self.q_sample(x_start, t, noise)
        if model_out_override is None:
            model_out = self.model_with_condition(x, t, None, external_cond, additional_tgt)
            model_out, additional_out = self._split_model_out(model_out, additional_tgt)
        else:
            model_out, additional_out = model_out_override
        target = x_start
        if additional_tgt is not None:
            return self._loss(model_out, target, t, additional_tgt, external_cond, additional_out, additional_weight)
        if target.shape[1] == 5:
            return self._loss(model_out[:, :3], target[:, :3], t, target[:, 3:], external_cond, model_out[:, 3:], 0.0)
        return self._loss(model_out[:, :3], target[:, :3], t)

    def _loss(self, image_out, target, t=None, flow_tgt=None, external_cond=None, flow_out=None, additional_weight=None):
        """:893-983: level 1 = NaN-aware squared error; with a flow target, pyramid levels 2,4,8,16 compare the
        splat of ``external_cond`` along the predicted flow with the splat of the target along zero flow, each
        weighted by level^4; everything is pooled by one nanmean.  No SNR weighting, flow term disabled."""
        image_out, target = image_out.contiguous(), target.contiguous()
        sums = [self._sq_err_sums(image_out, target, 1.0)]
        if flow_tgt is not None:
            for level in (2, 4, 8, 16):
                a = self.model._warp(external_cond, flow_out, scale=level)
                b = self.model._warp(target, torch.zeros_like(flow_out), scale=level)
                sums.append(self._sq_err_sums(a, b, float(level) ** 4))
        num = torch.stack([s[0] for s in sums]).sum()
        den = torch.stack([s[1] for s in sums]).sum()
        return num / den

    @staticmethod
    def _sq_err_sums(a: Tensor, b: Tensor, weight: float):
        num, den = _SqErrSums.apply(a, b)
        return num * weight, den

    def forward(self, img: Tensor, external_cond: Optional[Tensor] = None, *args, t: Optional[Tensor] = None, **kwargs):
        """:985-993: t ~ randint(0, T, (B,)) then p_losses (RNG order: randint, then randn_like inside)."""
        b = img.shape[0]
        if t is None:
            t = torch.randint(0, self.num_timesteps, (b,), device=img.device).long()
        return self.p_losses(img, t, *args, external_cond=external_cond, **kwargs)
