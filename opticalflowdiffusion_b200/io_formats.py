"""Wire / file formats either side of the flow_diffuser path (SURVEY.md section 8f, row N3), host-side like the
reference:

* Middlebury ``.flo`` optical flow files as the reference's Sintel loader reads them (datasets/animation/sintel.py:59-65:
  float32 magic, int32 width, int32 height, then h*w*2 float32 in (h, w, [u, v]) order) -- reader and writer;
* ``InputPadder`` (algorithms/diffusion_animation/future/raft_utils.py:7-25): replicate-pad to multiples of 8, the
  'sintel' mode splits the padding evenly, any other mode pads the bottom only;
* Lightning-style checkpoints: ``{"state_dict": ...}`` whose keys carry the reference's triple aliasing of the UNet
  (``unet.*``, ``_model.*`` / ``_model.model.*``, ``model.model.*`` / ``model.model.model.*``, SURVEY.md section 5) plus
  the 13 schedule buffers -- ``load_checkpoint`` accepts any one alias family (or all), ``save_checkpoint`` writes all;
  a model with a weight EMA adds ``ema_unet.*``;
* ``SintelFlowDataset``: (frame_t, frame_t+1, flow_t) triples in the (img, tgt, flow) convention of FlowDiffuser.preprocess
  (flow_diffuser.py:136-168) from an MPI-Sintel tree at a configurable root (the reference hard-codes a private path).
"""
from __future__ import annotations

import os
import re
from typing import Dict, List, Optional, Sequence, Tuple

import numpy as np
import torch
import torch.nn.functional as F

FLO_MAGIC = 202021.25


def read_flo(path: str) -> np.ndarray:
    """(h, w, 2) float32, channel 0 = u (dx), 1 = v (dy) -- exactly ``SintelDataset.load_flow`` (sintel.py:59-65),
    plus a magic-number check the reference skips."""
    with open(path, "rb") as f:
        magic = float(np.fromfile(f, np.float32, count=1)[0])
        if magic != FLO_MAGIC:
            raise ValueError(f"{path}: bad .flo magic {magic} (expected {FLO_MAGIC})")
        w = int(np.fromfile(f, np.int32, count=1)[0])
        h = int(np.fromfile(f, np.int32, count=1)[0])
        data = np.fromfile(f, np.float32, count=h * w * 2)
        if data.size != h * w * 2:
            raise ValueError(f"{path}: truncated .flo ({data.size} of {h * w * 2} values)")
        return data.reshape(h, w, 2)


def write_flo(path: str, flow) -> None:
    """flow: (h, w, 2) array or (2, h, w) tensor in pixels."""
    if torch.is_tensor(flow):
        flow = flow.detach().cpu().float().numpy()
    flow = np.asarray(flow, dtype=np.float32)
    if flow.ndim == 3 and flow.shape[0] == 2 and flow.shape[-1] != 2:
        flow = np.transpose(flow, (1, 2, 0))
    assert flow.ndim == 3 and flow.shape[-1] == 2, flow.shape
    h, w = flow.shape[:2]
    with open(path, "wb") as f:
        np.array([FLO_MAGIC], np.float32).tofile(f)
        np.array([w, h], np.int32).tofile(f)
        np.ascontiguousarray(flow).tofile(f)


class InputPadder:
    """Pads images such that dimensions are divisible by 8 (raft_utils.py:7-25)."""

    def __init__(self, dims: Sequence[int], mode: str = "sintel"):
        self.ht, self.wd = dims[-2:]
        pad_ht = (((self.ht // 8) + 1) * 8 - self.ht) % 8
        pad_wd = (((self.wd // 8) + 1) * 8 - self.wd) % 8
        if mode == "sintel":
            self._pad = [pad_wd // 2, pad_wd - pad_wd // 2, pad_ht // 2, pad_ht - pad_ht // 2]
        else:
            self._pad = [pad_wd // 2, pad_wd - pad_wd // 2, 0, pad_ht]

    def pad(self, *inputs):
        return [F.pad(x, self._pad, mode="replicate") for x in inputs]

    def unpad(self, x):
        ht, wd = x.shape[-2:]
        c = [self._pad[2], ht - self._pad[3], self._pad[0], wd - self._pad[1]]
        return x[..., c[0]:c[1], c[2]:c[3]]


# ------------------------------------------------------------------------------------------------
# checkpoints
# ------------------------------------------------------------------------------------------------
_UNET_PREFIXES = ("model.model.model.", "_model.model.", "model.model.", "_model.", "unet.")
_EMA_PREFIX = "ema_unet."


def _split_unet_key(key: str, unet_keys) -> Optional[str]:
    for pre in _UNET_PREFIXES:
        if key.startswith(pre) and key[len(pre):] in unet_keys:
            return key[len(pre):]
    return None


def load_checkpoint(algo, path_or_dict, strict: bool = True) -> Dict[str, List[str]]:
    """Load a Lightning ``.ckpt`` (or a bare state_dict) of the reference's FlowDiffuser into ``algo``.  The reference
    registers the same UNet under up to three names; a checkpoint that carries only one of them (e.g. after
    ``rewrite_checkpoint_for_compatibility``) still loads.  Returns {"missing": [...], "unexpected": [...]}, plus:

    * ``"ema_initialised"`` when ``algo`` keeps a weight EMA: True when the checkpoint has no ``ema_unet.*`` keys (every
      reference checkpoint), so the EMA starts from the loaded UNet weights; False when the EMA was restored from it;
    * ``"ignored"``: the ``ema_unet.*`` keys of a checkpoint loaded into a model without EMA (present only when any)."""
    ck = torch.load(path_or_dict, map_location="cpu", weights_only=False) if isinstance(path_or_dict, (str, os.PathLike)) \
        else path_or_dict
    sd = ck.get("state_dict", ck)
    own = algo.state_dict()
    unet_keys = set(algo.unet.state_dict().keys())
    ema = getattr(algo, "ema_unet", None)
    unet_vals: Dict[str, torch.Tensor] = {}
    other: Dict[str, torch.Tensor] = {}
    unexpected: List[str] = []
    ignored: List[str] = []
    for k, v in sd.items():
        sub = _split_unet_key(k, unet_keys)
        if sub is not None:
            prev = unet_vals.get(sub)
            if prev is not None and not torch.equal(prev, v):
                raise ValueError(f"checkpoint aliases of unet.{sub} disagree")
            unet_vals[sub] = v
        elif k in own:
            other[k] = v
        elif ema is None and k.startswith(_EMA_PREFIX):
            ignored.append(k)
        else:
            unexpected.append(k)
    missing = sorted(unet_keys - set(unet_vals))
    algo.unet.load_state_dict(unet_vals, strict=False)
    ema_init = ema is not None and not any(k.startswith(_EMA_PREFIX) for k in other)
    buf_missing = []
    with torch.no_grad():
        for k, v in other.items():
            own[k].copy_(v)
        if ema_init:
            for e, p in zip(ema.state_dict().values(), algo.unet.state_dict().values()):
                e.copy_(p)
    for k in own:
        if _split_unet_key(k, unet_keys) is None and k not in other and not (ema_init and k.startswith(_EMA_PREFIX)):
            buf_missing.append(k)
    missing += buf_missing
    if strict and (missing or unexpected):
        raise KeyError(f"checkpoint mismatch: missing {missing[:5]}{'...' if len(missing) > 5 else ''}, "
                       f"unexpected {unexpected[:5]}{'...' if len(unexpected) > 5 else ''}")
    for net in (algo.unet, ema):
        if getattr(net, "weights_epoch", None) is not None:
            net.weights_epoch += 1            # packed bf16 weights must be rebuilt
    out = {"missing": missing, "unexpected": unexpected}
    if ema is not None:
        out["ema_initialised"] = ema_init
    if ignored:
        out["ignored"] = ignored
    return out


def save_checkpoint(algo, path: str, optimizer=None, global_step: int = 0, epoch: int = 0) -> None:
    """Lightning-shaped checkpoint: all alias keys of the module's state_dict, optimizer state, counters."""
    ck = {"state_dict": {k: v.detach().cpu().clone() for k, v in algo.state_dict().items()},
          "global_step": int(global_step), "epoch": int(epoch), "pytorch-lightning_version": "2.0.0 (layout only)"}
    if optimizer is not None:
        ck["optimizer_states"] = [optimizer.state_dict()]
    torch.save(ck, path)


# ------------------------------------------------------------------------------------------------
# MPI-Sintel
# ------------------------------------------------------------------------------------------------
class SintelFlowDataset(torch.utils.data.Dataset):
    """``root/training/{clean|final}/<scene>/frame_XXXX.png`` + ``root/training/flow/<scene>/frame_XXXX.flo``.
    Items: (img, tgt, flow) with img = frame t, tgt = frame t+1 in [0,1] (3,H,W) and flow = flow t (2,H,W) in pixels,
    channel 0 = u -- the convention of the reference's FlyingChairs / KITTI loaders that FlowDiffuser.preprocess consumes.
    Scenes whose name hashes into ``val_fraction`` form the validation split (the reference's split file is private)."""

    def __init__(self, cfg, split: str = "training", device=None):
        import cv2
        self._cv2 = cv2
        self.root = str(cfg.root)
        self.render = str(getattr(cfg, "render", "clean"))
        size = getattr(cfg, "image_size", None)
        self.size: Optional[Tuple[int, int]] = None
        if size:
            w, h = (int(x) for x in str(size).split(","))          # the reference writes "W,H" (sintel.py:14)
            self.size = (w, h)
        val_fraction = float(getattr(cfg, "val_fraction", 0.1))
        frames_dir = os.path.join(self.root, "training", self.render)
        if not os.path.isdir(frames_dir):
            raise FileNotFoundError(f"no MPI-Sintel tree at {frames_dir}")
        self.items: List[Tuple[str, str, str]] = []
        for scene in sorted(os.listdir(frames_dir)):
            is_val = (sum(scene.encode()) % 100) < 100 * val_fraction
            if (split == "training") == is_val:
                continue
            pngs = sorted(f for f in os.listdir(os.path.join(frames_dir, scene)) if re.match(r"frame_\d+\.png$", f))
            for a, b in zip(pngs[:-1], pngs[1:]):
                flo = os.path.join(self.root, "training", "flow", scene, a[:-4] + ".flo")
                if os.path.exists(flo):
                    self.items.append((os.path.join(frames_dir, scene, a), os.path.join(frames_dir, scene, b), flo))

    def __len__(self):
        return len(self.items)

    def _image(self, path: str) -> torch.Tensor:
        cv2 = self._cv2
        img = cv2.cvtColor(cv2.imread(path), cv2.COLOR_BGR2RGB)
        if self.size is not None:
            img = cv2.resize(img, self.size)
        return torch.from_numpy(img).permute(2, 0, 1).float() / 255.0

    def __getitem__(self, i):
        a, b, flo = self.items[i]
        flow = read_flo(flo)
        if self.size is not None:
            h, w = flow.shape[:2]
            flow = self._cv2.resize(flow, self.size)               # like the reference (sintel.py:81); then rescale the vectors
            flow = flow * np.array([self.size[0] / w, self.size[1] / h], np.float32)
        return self._image(a), self._image(b), torch.from_numpy(np.ascontiguousarray(flow)).permute(2, 0, 1).contiguous()
