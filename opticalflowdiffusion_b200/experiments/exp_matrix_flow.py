"""``experiment=matrix_flow`` runner for ``algorithm=flow_diffuser``: the slice of
experiments/exp_base.py:47-59,120-238 + exp_99.py:18-45 that drives the hot path.

The reference builds a ``pl.Trainer`` (DDP when more than one GPU is visible, exp_base.py:198).
Lightning is not part of this path's contract, so the loop here is explicit: one process per GPU
(torchrun), batch-sharded data, ``validation`` / ``sample`` tasks run the CUDA sampling path, ``evaluate`` scores K sampled
flows per image against the ground truth over a whole split (``evaluation.FlowScores``); ``train`` is
``training_step`` -> ``loss.backward()`` (the UnetFunction backward kernels) -> one NCCL all-reduce of the flat
gradient (DDPStrategy's exchange, exp_base.py:198) -> fused clip + Adam."""
from __future__ import annotations

import os
from typing import Optional

import torch
import torch.distributed as dist

from ..datasets import SyntheticSintelDataset
from ..io_formats import SintelFlowDataset, load_checkpoint
from ..flow_diffuser import FlowDiffuser
from ..flow_learner import FlowLearner
from ..parallel import init_distributed, reduce_metrics, shard_range, sync_module_from_rank0


class MatrixFlowExperiment:
    compatible_algorithms = dict(flow_diffuser=FlowDiffuser, flow_learner=FlowLearner)      # exp_99.py:22-28
    compatible_datasets = dict(synthetic_sintel=SyntheticSintelDataset, sintel=SintelFlowDataset)

    def __init__(self, cfg, logger=None, ckpt_path: Optional[str] = None):
        self.cfg, self.logger, self.ckpt_path = cfg, logger, ckpt_path
        self.rank = int(os.environ.get("RANK", 0))
        self.world = int(os.environ.get("WORLD_SIZE", 1))
        self.local_rank = int(os.environ.get("LOCAL_RANK", 0))
        self.algo = self._build_model()

    def _build_model(self):
        name = self.cfg.algorithm.name
        if name not in self.compatible_algorithms:
            raise ValueError(f"algorithm '{name}' is outside the flow_diffuser hot path "
                             f"(have: {sorted(self.compatible_algorithms)})")
        algo = self.compatible_algorithms[name](self.cfg.algorithm)
        self._resume = None
        if self.ckpt_path:
            load_checkpoint(algo, self.ckpt_path)        # Lightning .ckpt or bare state_dict, any alias family
            ck = torch.load(self.ckpt_path, map_location="cpu", weights_only=False)
            if isinstance(ck, dict) and "optimizer_states" in ck:
                self._resume = {"optimizer": ck["optimizer_states"][0], "global_step": int(ck.get("global_step", 0)),
                                "epoch": int(ck.get("epoch", 0))}
        algo.logger = self.logger
        return algo

    def _build_dataset(self, split: str):
        if split not in ("training", "validation", "test"):
            raise NotImplementedError(f"split '{split}' is not implemented")
        return self.compatible_datasets[self.cfg.dataset.name](self.cfg.dataset, split=split)

    def _loader(self, split: str, section):
        ds = self._build_dataset(split)
        sampler = None
        if self.world > 1:      # batch-sharded data parallelism: each rank sees a disjoint slice, no collective
            sampler = torch.utils.data.DistributedSampler(ds, num_replicas=self.world, rank=self.rank,
                                                          shuffle=bool(section.data.shuffle))
        return torch.utils.data.DataLoader(ds, batch_size=int(section.data.batch_size), sampler=sampler,
                                           shuffle=bool(section.data.shuffle) and sampler is None, num_workers=0)

    def exec_task(self, task: str):
        if task == "train":
            return self.train()
        if task in ("validation", "validate", "test"):
            return self.validate()
        if task == "evaluate":
            return self.evaluate()
        raise ValueError(f"Specified task '{task}' not implemented for class {self.__class__.__name__}.")

    def train(self, max_steps: Optional[int] = None):
        """exp_base.py:178-214 without Lightning: epochs over the training loader; gradient clipping
        (experiment.training.clipping, :192) and accumulate_grad_batches (:203) as configured."""
        from ..optim import GradSync, allreduce_gradients
        dev = torch.device("cuda", self.local_rank)
        torch.cuda.set_device(dev)
        distributed = init_distributed(dev)          # WORLD_SIZE > 1: one NCCL process group (DDPStrategy, exp_base.py:198)
        self.algo.to(dev)
        sync_module_from_rank0(self.algo)            # identical replicas, as DDP broadcasts at construction
        self._synced = True
        self.algo.train()
        opt = self.algo.configure_optimizers()
        tr = self.cfg.experiment.training
        clip = tr.get("clipping") if hasattr(tr, "get") else getattr(tr, "clipping", None)
        if clip:
            opt.max_grad_norm = float(clip)
        accum = int(tr.optim.accumulate_grad_batches)
        epochs = int(self.cfg.experiment.epochs)
        unet = getattr(self.algo, "unet", None)
        unet = getattr(unet, "model", unet)          # FlowLearner wraps its UNet
        if distributed and accum == 1 and hasattr(unet, "forward_train"):
            # bucketed all-reduce overlapped with the backward; with gradient accumulation the exchange happens once per
            # optimiser step instead (allreduce_gradients below), like DDP under no_sync()
            GradSync(opt).attach(unet)
        if epochs < 0 and max_steps is None:
            max_steps = tr.get("max_steps") if hasattr(tr, "get") else None
            if max_steps is None:
                raise ValueError("experiment.epochs = -1 means 'train until stopped' (Lightning max_epochs=-1): give "
                                 "experiment.training.max_steps or train(max_steps=...)")
            max_steps = int(max_steps)
        from collections import deque
        losses, step, epoch = deque(maxlen=1024), 0, 0
        # checkpoint / resume (exp_base.py:184-190,213: ModelCheckpoint(every_n_train_steps) + fit(ckpt_path=...))
        ck_cfg = tr.get("checkpointing") if hasattr(tr, "get") else None
        every = int(ck_cfg.get("every_n_train_steps", 0)) if ck_cfg else 0
        ck_dir = os.path.join(str(self.cfg.get("output_dir", "outputs")), "checkpoints")
        if self._resume is not None:
            opt.load_state_dict(self._resume["optimizer"])
            step, epoch = self._resume["global_step"], self._resume["epoch"]
            self.algo.global_step = step
        start_step = step
        while (epochs < 0 or epoch < epochs) and (max_steps is None or step - start_step < max_steps):
            loader = self._loader("training", tr)
            if hasattr(loader.sampler, "set_epoch"):
                loader.sampler.set_epoch(epoch)
            n_batches = len(loader)
            for i, batch in enumerate(loader):
                loss = self.algo.training_step(tuple(t.to(dev, non_blocking=True) for t in batch), i)
                (loss / accum).backward()
                if (i + 1) % accum == 0 or i + 1 == n_batches:      # a short last window is stepped, not carried over
                    allreduce_gradients(opt)
                    opt.step()
                    opt.zero_grad(set_to_none=True)
                    step += 1
                    self.algo.global_step = step
                    losses.append(loss.detach())
                    if len(losses) == losses.maxlen and step % 256 == 0:
                        losses = deque((float(x) for x in losses), maxlen=losses.maxlen)    # bounded, off the device
                    if every > 0 and step % every == 0 and self.rank == 0:
                        from ..io_formats import save_checkpoint
                        os.makedirs(ck_dir, exist_ok=True)
                        save_checkpoint(self.algo, os.path.join(ck_dir, f"step_{step:07d}.ckpt"), optimizer=opt,
                                        global_step=step, epoch=epoch)
                    if max_steps is not None and step - start_step >= max_steps:
                        break
            epoch += 1
        return {"train/loss": [float(x) for x in losses], "steps": step - start_step, "global_step": step}

    @torch.no_grad()
    def validate(self, max_batches: Optional[int] = None):
        dev = torch.device("cuda", self.local_rank)
        torch.cuda.set_device(dev)
        distributed = init_distributed(dev)
        self.algo.to(dev)
        if distributed and not getattr(self, "_synced", False):
            sync_module_from_rank0(self.algo)
            self._synced = True
        limit = max_batches or int(self.cfg.experiment.validation.limit_batch)
        out = {}
        for i, batch in enumerate(self._loader("validation", self.cfg.experiment.validation)):
            if i >= limit:
                break
            self.algo.validation_step(tuple(t.to(dev) for t in batch), i)
            out = {k: float(v) for k, v in self.algo.logged.items()} if hasattr(self.algo, "logged") else {}
        return reduce_metrics(out, device=dev)     # sync_dist=True semantics for the scalars

    @torch.no_grad()
    def evaluate(self, max_batches: Optional[int] = None):
        """End-point error of ``experiment.evaluation.num_samples`` sampled flows per image against the ground truth over
        ``experiment.evaluation.split``: each rank scores the contiguous ``shard_range`` of the split's indices, unshuffled
        (no DistributedSampler: it pads by repeating images), and one fp64 SUM all-reduce gives every rank the same
        dataset-level metrics (``evaluation.FlowScores``).  ``limit_batch`` / ``max_batches`` cap the batches per rank."""
        from ..evaluation import FlowScores
        if not hasattr(self.algo, "evaluate_step"):
            raise NotImplementedError(f"algorithm '{self.cfg.algorithm.name}' has no evaluate_step")
        dev = torch.device("cuda", self.local_rank)
        torch.cuda.set_device(dev)
        distributed = init_distributed(dev)
        self.algo.to(dev)
        if distributed and not getattr(self, "_synced", False):
            sync_module_from_rank0(self.algo)
            self._synced = True
        ev = self.cfg.experiment.evaluation
        K, seed = int(ev.num_samples), int(ev.seed)
        limit = max_batches or ev.get("limit_batch")
        ds = self._build_dataset(str(ev.split))
        mine = shard_range(len(ds), self.rank, self.world)
        loader = torch.utils.data.DataLoader(torch.utils.data.Subset(ds, list(mine)), batch_size=int(ev.data.batch_size),
                                             shuffle=False, num_workers=0)
        scores = FlowScores(K, device=dev)
        start = mine.start
        for i, batch in enumerate(loader):
            if limit is not None and i >= int(limit):
                break
            n = batch[0].shape[0]
            rows = self.algo.evaluate_step(tuple(t.to(dev) for t in batch), range(start, start + n), K, seed,
                                           max_batch=ev.get("max_sample_batch"))
            scores.update(rows)
            start += n
        return scores.metrics()
