"""``FlowDiffuser``: the algorithm class of ``algorithm=flow_diffuser``
(reference: algorithms/diffusion_animation/flow_diffuser.py:65-365) on the sm_100a kernels.

Same constructor (``FlowDiffuser(cfg.algorithm)``), same methods and metric keys
(``configure_optimizers / preprocess / loss / sample / training_step / validation_step``), same
parameter names (``unet.*``, ``_model.*``, ``model.*`` aliases and the 13 schedule buffers), so the
experiment runner that drives the reference class (experiments/exp_base.py:120-214) drives this one.

New optional config keys (SURVEY.md section 8b): ``sampling_timesteps`` (DDIM when < ``timesteps``),
``image_size`` as ``[H, W]``, ``return_all_timesteps`` (default true like the reference), ``sampler`` (null: the
reference's DDIM / DDPM; ``dpmpp``: multistep DPM-Solver++ on the DDIM grid) with ``solver_order`` (1-3), and
``ema_decay`` (null: off) with ``ema_update_after_step`` / ``ema_update_every``: an exponential moving average of the UNet
weights (``ema_unet``), kept by the fused optimiser step and used for sampling and validation.

When ``pytorch_lightning`` is importable the class derives from ``LightningModule``; otherwise from a
minimal stand-in with the attributes the reference touches (``log_dict``, ``log``, ``global_step``,
``logger``, ``device``).
"""
from __future__ import annotations

import copy
import os
import random
from typing import Optional, Sequence, Tuple

import torch
from torch import nn

from . import warp as W
from .diffusion import ConditionalDiffusion
from .unet import Unet

Tensor = torch.Tensor

try:  # pragma: no cover - not installed in the build image
    import pytorch_lightning as pl
    _Base = pl.LightningModule
except Exception:  # noqa: BLE001
    class _Base(nn.Module):
        """The slice of LightningModule that flow_diffuser.py uses."""

        global_step = 0
        logger = None

        def __init__(self):
            super().__init__()
            self.logged = {}

        @property
        def device(self):
            for p in self.parameters():
                return p.device
            return torch.device("cpu")

        def log_dict(self, d, **kwargs):
            for k, v in d.items():
                self.logged[k] = v.detach() if torch.is_tensor(v) else v

        def log(self, k, v, **kwargs):
            self.log_dict({k: v})


def _cfg_get(cfg, key, default=None):
    try:
        v = getattr(cfg, key)
    except (AttributeError, KeyError):
        return default
    return default if v is None else v


class Augmentor:
    """Training-time augmentation (augmentation.py:6-76), host-side torch/torchvision like the reference (kept as the
    executable specification of ``augment.GpuAugmentor``, which FlowDiffuser uses on CUDA batches):
    per item, (a) photometric jitter / grayscale / blur applied to both frames with jitter parameters drawn
    ONCE at construction, (b) horizontal flip negating the last flow channel, vertical flip negating the
    second-last, (c) random resized crop rescaling the flow by crop/size (square inputs, as in the reference)."""

    def __init__(self):
        import torchvision.transforms as T
        lim = 0.1
        deltas = [(random.random() - 0.5) * 2 * lim for _ in range(4)]
        ranges = [(b + d, b + d + 0.01) for b, d in zip((1, 1, 1, 0), deltas)]
        self._jitter = T.ColorJitter(*ranges)
        self._gray = T.Grayscale(3)
        self._blur = T.GaussianBlur(3, random.random() * 0.5)
        self._T = T

    @staticmethod
    def _both_frames(fn, pair: Tensor) -> Tensor:
        return torch.cat([fn(half) for half in torch.chunk(pair, 2, dim=1)], dim=1)

    def _photometric(self, pair: Tensor) -> Tensor:
        if torch.rand(1) < 0.4:
            pair = self._both_frames(self._jitter, pair)
        if torch.rand(1) < 0.1:
            pair = self._both_frames(self._gray, pair)
        if torch.rand(1) < 0.2:
            pair = self._both_frames(self._blur, pair)
        return pair

    def _geometric(self, item: Tensor) -> Tensor:
        TF = self._T.functional
        if torch.rand(1) < 0.3:
            torch.rand(1)      # the wrapped RandomHorizontalFlip(p=1.0) draws its own number (augmentation.py:34-37)
            item = TF.hflip(item)
            item[:, -1] = -item[:, -1]
        if torch.rand(1) < 0.3:
            torch.rand(1)      # RandomVerticalFlip(p=1.0), :39-42
            item = TF.vflip(item)
            item[:, -2] = -item[:, -2]
        if torch.rand(1) < 0.15:
            # the reference resizes to (W, W) and scales both flow channels by crop/W (:44-50), which only works
            # for square frames; the same rule per axis keeps it identical there and valid for H != W
            H, Wd = item.shape[-2:]
            top, left, h, w = self._T.RandomResizedCrop.get_params(item, [0.8, 1.0], [0.9, 1.1])
            scale = torch.tensor([h / H, w / Wd], dtype=item.dtype, device=item.device)
            item[:, -2:] = item[:, -2:] * scale[None, :, None, None]
            item = TF.resized_crop(item, top, left, h, w, (H, Wd), antialias=False)
        return item

    def __call__(self, batch):
        img, tgt, flow = batch
        frames = torch.cat([self._photometric(x) for x in torch.chunk(torch.cat((img, tgt), 1), img.shape[0], 0)], 0)
        full = torch.cat((frames, flow), dim=1)
        full = torch.cat([self._geometric(x.clone()) for x in torch.chunk(full, full.shape[0], 0)], 0)
        return full[:, :3], full[:, 3:6], full[:, 6:]


def logged_stats(prefix: str, name: str, x: Tensor):
    """The four logged scalars of a tensor (flow_diffuser.py:223-231, 264-279; flow_learner.py likewise): min, max, mean and
    the mean over positions of the unbiased std over the batch axis -- one pass over x (fd_tensor_stats) instead of seven
    eager reductions; the results stay on the device (no host synchronisation in the step)."""
    from . import _lib
    _lib.require_cuda(x)
    x = x.detach().float().contiguous()
    lib = _lib.load()
    inner = x.numel() // x.shape[0]
    out = torch.empty(4, device=x.device, dtype=torch.float32)
    ws = torch.empty(lib.fd_tensor_stats_workspace_floats(inner), device=x.device, dtype=torch.float32)
    _lib.check(lib.fd_tensor_stats(_lib.ptr(x), x.shape[0], inner, _lib.ptr(out), _lib.ptr(ws), _lib.stream()))
    return {f"{prefix}/{name}_min": out[0], f"{prefix}/{name}_max": out[1], f"{prefix}/{name}_mean": out[2],
            f"{prefix}/{name}_std": out[3]}


class UnetWithWarp(nn.Module):
    """flow_diffuser.py:20-63: predicts the flow with the UNet (NaN-safe input) and forward-splats the
    conditioning frame along it; ``full_output`` appends the flow (target='joint')."""

    def __init__(self, cfg, unet: Unet, full_output: bool, nan_safe: bool = True):
        super().__init__()
        self.cfg = cfg
        self.flow_max = cfg.flow_max
        self.dim = cfg.latent_dim if cfg.latent else 3
        self.model = unet
        self.full_output = full_output
        self.nan_safe = nan_safe
        if cfg.zero_init:
            with torch.no_grad():
                self.model.final_conv.weight.zero_()
                self.model.final_conv.bias.zero_()

    def _warp(self, image: Tensor, flow: Tensor, **kwargs) -> Tensor:
        return W.warp(image[:, :self.dim], None, flow * self.flow_max, mode="forward", **kwargs)

    def forward(self, x, external_cond=None, t=None, self_cond=None, additional_out: bool = False):
        flow = self.model(x, external_cond, t, nan_mask=self.nan_safe)     # NaN -> 0 + mask channel fused into packing
        src = external_cond if external_cond is not None else torch.nan_to_num(x[:, :self.dim], nan=0.0)
        out = self._warp(src, flow[:, :2])
        if self.full_output:
            out = torch.cat((out, flow), dim=1)
        return torch.cat((out, flow), dim=1) if additional_out else out


class FlowDiffuser(_Base):
    backward_supported = True    # training_step's loss carries the UnetFunction autograd node (unet_train.py)

    def __init__(self, cfg):
        super().__init__()
        self.cfg = cfg
        self.flow_max = cfg.flow_max
        self.latent_max = cfg.latent_max
        self.is_diffusion = cfg.is_diffusion
        self.latent = cfg.latent
        self.target = cfg.target
        if self.latent:
            # flow_diffuser.py:81-95: a frozen Autoencoder whose weights come from the FlowPred run named by cfg.ae.  The
            # reference fetches that checkpoint from wandb; here it is read from the same local path the reference caches
            # it under, or from cfg.ae_checkpoint -- absent both, the autoencoder keeps its initialisation (and says so).
            from .flow_pred import Autoencoder, load_autoencoder
            self.ae = Autoencoder(cfg)
            path = _cfg_get(cfg, "ae_checkpoint")
            if not path:
                cached = os.path.join("outputs", "loaded_checkpoints", "diffusion_control", str(_cfg_get(cfg, "ae", "")), "model.ckpt")
                path = cached if os.path.exists(cached) else None
            self.ae_loaded = load_autoencoder(self.ae, path)
            if not self.ae_loaded:
                import warnings
                warnings.warn("latent mode without an autoencoder checkpoint (algorithm.ae_checkpoint): randomly initialised "
                              "encoder / decoder")
            for p_ in self.ae.parameters():
                p_.requires_grad = False
        if not self.is_diffusion:
            raise NotImplementedError("is_diffusion=false (plain regression) is not on the flow_diffuser hot path")
        self._augmentor: Optional[Augmentor] = None
        self.dim = cfg.latent_dim if self.latent else 3                                  # flow_diffuser.py:98
        unet_dims = {"target": self.dim + 1, "joint": self.dim + 3}.get(self.target, 2)
        self.unet = Unet(64, channels=self.dim + unet_dims, out_dim=2)
        if self.target in ("target", "joint"):
            self._model = UnetWithWarp(cfg, self.unet, full_output=self.target == "joint")
        else:
            self._model = self.unet
        # (flow_diffuser.py:122: in latent mode the reference passes latent_dim whatever the target -- kept: it is the channel
        # count of the sampler's initial noise, so latent sampling works for target='target' exactly as far as it does there)
        channels = cfg.latent_dim if self.latent else 2 + int(self.target == "target") + 3 * int(self.target == "joint")

        def diffusion(net):
            return ConditionalDiffusion(
                net, _cfg_get(cfg, "image_size", 128), objective="pred_x0", channels=channels, auto_normalize=False,
                noise_space="image" if cfg.noiser == "image" else "flow", timesteps=cfg.timesteps,
                sampling_timesteps=_cfg_get(cfg, "sampling_timesteps"), min_snr_loss_weight=True,
                sampler=_cfg_get(cfg, "sampler"), solver_order=int(_cfg_get(cfg, "solver_order", 2)))

        self.model = diffusion(self._model)
        ema_decay = _cfg_get(cfg, "ema_decay")
        self.ema_decay = None if ema_decay is None else float(ema_decay)
        if self.ema_decay is not None:
            # the averaged UNet: registered (its 276 tensors ride in state_dict as ema_unet.*) but outside self.model, so
            # the optimiser never sees it.  Its sampler is NOT registered (no state_dict keys); ema_model points its schedule
            # tables at self.model's, and it keeps its own CUDA-graph cache.
            self.ema_unet = copy.deepcopy(self.unet).requires_grad_(False)
            net = UnetWithWarp(cfg, self.ema_unet, full_output=self.target == "joint") \
                if self.target in ("target", "joint") else self.ema_unet
            object.__setattr__(self, "_ema_diffusion", diffusion(net))
        self.return_all_timesteps = bool(_cfg_get(cfg, "return_all_timesteps", True))
        self.use_cuda_graph = bool(_cfg_get(cfg, "use_cuda_graph", False))

    @property
    def augmentor(self):
        """The reference builds its Augmentor in ``__init__`` (flow_diffuser.py:101); here it is the GPU implementation
        (``gpu_augment: false`` in the algorithm config selects the per-item torchvision path)."""
        if self._augmentor is None:
            if bool(_cfg_get(self.cfg, "gpu_augment", True)):
                from .augment import GpuAugmentor
                self._augmentor = GpuAugmentor()
            else:
                self._augmentor = Augmentor()
        return self._augmentor

    @property
    def ema_model(self) -> ConditionalDiffusion:
        """The ``ConditionalDiffusion`` over the EMA network (``ema_decay`` set), sharing ``self.model``'s schedule tables
        wherever the module has been moved."""
        if self.ema_decay is None:
            raise ValueError("this FlowDiffuser keeps no weight EMA (algorithm.ema_decay is null)")
        ema = self.__dict__["_ema_diffusion"]
        for name in ConditionalDiffusion.BUFFERS:
            setattr(ema, name, getattr(self.model, name))
        return ema

    def _diffusion(self, use_ema: Optional[bool]) -> ConditionalDiffusion:
        """None: the EMA network when there is one, else the online one."""
        if use_ema is None:
            use_ema = self.ema_decay is not None
        return self.ema_model if use_ema else self.model

    def configure_optimizers(self):
        """flow_diffuser.py:129-134: Adam(lr, weight_decay) over the model's parameters -- here the fused flat-buffer
        implementation with the same update rule; ``clipping`` (experiment.training.clipping, exp_base.py:192) can be
        folded into the step by setting ``optimizer.max_grad_norm``.  With ``ema_decay`` set the same step keeps
        ``ema_unet`` as the weights' moving average."""
        from .optim import FusedAdam
        ema = {}
        if self.ema_decay is not None:
            ema = dict(ema_params=list(self.ema_unet.parameters()), ema_decay=self.ema_decay,
                       ema_update_after_step=int(_cfg_get(self.cfg, "ema_update_after_step", 100)),
                       ema_update_every=int(_cfg_get(self.cfg, "ema_update_every", 10)))

        def invalidate():
            self.unet.weights_epoch += 1
            if opt.ema_updated:
                self.ema_unet.weights_epoch += 1

        opt = FusedAdam(self.model.parameters(), lr=self.cfg.lr, weight_decay=self.cfg.weight_decay,
                        max_grad_norm=float(_cfg_get(self.cfg, "clipping", 0.0) or 0.0), on_step=invalidate, **ema)
        self.optimizers = opt
        return opt

    # ------------------------------------------------------------------ data
    def preprocess(self, batch, aug: bool = True):
        """flow_diffuser.py:136-168: returns (diffusion target, cond, normalised flow)."""
        if aug:
            batch = self.augmentor(batch)
        img, tgt, flow = batch
        flow = torch.clamp(flow / self.flow_max, -1.0, 1.0)
        if self.latent:                                                                 # flow_diffuser.py:143-148
            img = torch.clamp(self.ae.encode(img) / self.latent_max, -1.0, 1.0)
        else:
            img = 2 * img - 1.0
        if self.target == "target":
            first = W.warp(img, None, flow * self.flow_max, mode="forward")
        elif self.target == "joint":
            first = torch.cat((W.warp(img, None, flow * self.flow_max, mode="forward"), flow), dim=1)
        else:
            first = flow
        return first, img, flow

    # ------------------------------------------------------------------ loss / sampling
    def loss(self, tgt, cond, flow, override=None, **kw):
        """The training loss, always of the online network."""
        return self._loss(self.model, tgt, cond, flow, override, **kw)

    def _loss(self, diffusion, tgt, cond, flow, override=None, **kw):
        if self.cfg.target == "target":
            return diffusion(tgt, external_cond=cond, additional_tgt=flow, additional_weight=self.cfg.flow_weight,
                             model_out_override=override, **kw)
        return diffusion(tgt, external_cond=cond, model_out_override=override, **kw)

    @torch.no_grad()
    def sample(self, cond, flow, use_ema: Optional[bool] = None, **kw) -> Tuple[Tensor, Tensor]:
        """flow_diffuser.py:189-215: (samples, flows); with ``return_all_timesteps`` the flows keep a time axis at dim 1.
        ``use_ema``: None samples the EMA network when ``ema_decay`` is set and the online one otherwise; False always
        the online network."""
        model = self._diffusion(use_ema)
        bsz = flow.shape[0]
        all_t = self.return_all_timesteps
        if self.cfg.target == "target":
            samples, flow = model.sample(batch_size=bsz, external_cond=cond, additional_tgt=flow,
                                         return_all_timesteps=all_t, **kw)
        elif self.cfg.target == "joint":
            joint = model.sample(batch_size=bsz, external_cond=cond, return_all_timesteps=all_t, **kw)
            samples, flow = (joint[:, :, :self.dim], joint[:, :, self.dim:]) if all_t else (joint[:, :self.dim], joint[:, self.dim:])
        else:
            flow = model.sample(batch_size=bsz, external_cond=cond, return_all_timesteps=all_t,
                                use_cuda_graph=self.use_cuda_graph, **kw)
            last = flow[:, -1] if all_t else flow
            samples = W.warp(cond[:, :self.dim], None, last.contiguous(), mode="forward")
        return samples, flow

    # ------------------------------------------------------------------ steps
    @staticmethod
    def _stats(prefix: str, name: str, x: Tensor):
        return logged_stats(prefix, name, x)

    def training_step(self, batch, batch_idx):
        batch = self.preprocess(batch)
        loss = self.loss(*batch)
        tgt, cond, flow = batch
        self.log_dict({"train/loss": loss, **self._stats("train", "cond", cond), **self._stats("train", "flow", flow)})
        return loss

    @torch.no_grad()
    def validation_step(self, batch, batch_idx):
        """flow_diffuser.py:237-349 (scalar metrics; image logging when a logger is attached).  Every metric is of the EMA
        network when ``ema_decay`` is set."""
        img, tgt, flow = batch
        model = self._diffusion(None)
        tgt_, cond, flow_ = self.preprocess(batch, aug=False)
        loss = self._loss(model, tgt_, cond, flow_)
        keep = self.return_all_timesteps
        self.return_all_timesteps = True
        try:
            samples, p_flows = self.sample(cond, flow_)
        finally:
            self.return_all_timesteps = keep
        if self.target == "target":
            samples = samples[:, -1]
            p_flows = p_flows[-1] * self.flow_max
        elif self.target == "joint":
            samples = samples[:, -1]
            p_flows = p_flows[:, -1] * self.flow_max
        else:
            p_flows = p_flows[:, -1]
        mse_tgt = self.ae.encode(tgt) if self.latent else tgt                           # flow_diffuser.py:255
        mse = W.nan_mse(samples.contiguous(), mse_tgt.contiguous() * 1.0) if torch.isnan(samples).any() else \
            torch.nn.functional.mse_loss(samples, mse_tgt)
        metrics = {"val/loss": loss, "val/mse": mse, **self._stats("val", "cond", cond), **self._stats("val", "flow", flow),
                   **self._stats("val", "samples", torch.nan_to_num(samples)), **self._stats("val", "p_flow", p_flows)}
        if self.target in ("target", "joint"):
            warped = W.warp(cond[:, :self.dim], None, flow_ * self.flow_max, mode="forward")
            override = (warped, flow_) if self.target == "target" else (torch.cat((warped, flow_), dim=1), None)
            metrics["val/ideal_loss"] = self._loss(model, tgt_, cond, flow_, override=override)
            last = model.model(tgt_, cond, torch.zeros((img.shape[0],), device=img.device, dtype=torch.long), None,
                                    additional_out=True)[:, -2:]
            metrics["val/last_step"] = torch.nn.functional.mse_loss(last, flow_)
        self.log_dict(metrics, sync_dist=True)
        if getattr(self, "logger", None) is not None and hasattr(self.logger, "log_image"):
            import torchvision
            bsz = img.shape[0]
            flos = torchvision.utils.flow_to_image(torch.cat((flow, p_flows, flow - p_flows), dim=0)) / 255.0
            shown = torch.nan_to_num(samples)
            if self.latent:                                                             # flow_diffuser.py:304-309
                shown = self.ae.decode(shown * self.latent_max, img)
                self.logger.log_image(key="dec_gt", images=list(torch.chunk(self.ae(img, flow), bsz)), step=self.global_step)
            for key, val in (("original", img), ("target", tgt), ("gt_flow", flos[:bsz]), ("target_p", flos[bsz:2 * bsz]),
                             ("difference", flos[2 * bsz:]), ("samples", shown)):
                self.logger.log_image(key=key, images=list(torch.chunk(val, bsz)), step=self.global_step)
        return None
