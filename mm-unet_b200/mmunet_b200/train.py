"""Minimal synthetic-data trainer for MM_Net: the caller of the hot path that produces the "MM-UNet train img/s" half of
the headline metric (SURVEY.md section 8 row f1).  It restates the parts of the reference training stack that decide what
one step costs - nothing else (no datasets, metrics, checkpoints, logging):

  loss        monai DiceFocalLoss(smooth_nr=0, smooth_dr=1e-5, sigmoid=True)      train.py:231-233
  optimizer   timm create_optimizer_v2("adamw", lr 1e-3, wd 0.05, betas (.9,.95)) train.py:197-199, config.yml:1-11
              (timm's default filter: biases and 1-D tensors are not decayed)
  schedule    LinearWarmupCosineAnnealingLR stepped per epoch, closed form        src/optimizer.py:20-100, train.py:65
  step        forward -> loss -> backward -> optimizer.step -> zero_grad           train.py:36-54
  data-parallel  one process per GPU, gradients all-reduced (mean) by torch DDP over NCCL in ~25 MB buckets that
              overlap the rest of the backward (train.py:252-253 via accelerate).  The parameters MM_Net never touches
              (`MM_Net.unused_parameters()`) are frozen instead of paying for find_unused_parameters.

Synthetic DRIVE-shaped batches: x ~ N(0,1) (B,3,S,S), target ~ Bernoulli(0.1) (B,1,S,S)  (SURVEY.md section 8d).
"""
from __future__ import annotations

import contextlib
import math
import os

import torch
import torch.distributed as dist
import torch.nn.functional as F

from . import _lib
from .mm_net import MM_Net


def dice_focal_loss(logits, target, gamma: float = 2.0, smooth_nr: float = 0.0, smooth_dr: float = 1e-5,
                    lambda_dice: float = 1.0, lambda_focal: float = 1.0):
    """monai.losses.DiceFocalLoss(sigmoid=True, to_onehot_y=False, smooth_nr=0, smooth_dr=1e-5) with its defaults
    (include_background, reduction="mean", gamma=2, no class weights): soft Dice per (sample, channel) over the
    spatial dims + sigmoid focal loss, both averaged."""
    logits = logits.float()
    target = target.float()
    p = torch.sigmoid(logits)
    dims = tuple(range(2, logits.dim()))
    inter = (p * target).sum(dims)
    denom = p.sum(dims) + target.sum(dims)
    dice = (1.0 - (2.0 * inter + smooth_nr) / (denom + smooth_dr)).mean()
    bce = logits - logits * target - F.logsigmoid(logits)                 # = BCE-with-logits, element-wise
    invprobs = F.logsigmoid(-logits * (target * 2 - 1))                   # log(1 - p_t)
    focal = ((invprobs * gamma).exp() * bce).mean()
    return lambda_dice * dice + lambda_focal * focal


def warmup_cosine_lr(epoch: int, base_lr: float, warmup_epochs: int, max_epochs: int, warmup_start_lr: float = 0.0,
                     eta_min: float = 0.0) -> float:
    """Closed form used when the scheduler is stepped with an explicit epoch (src/optimizer.py:86-100, train.py:65)."""
    if epoch < warmup_epochs:
        return warmup_start_lr + epoch * (base_lr - warmup_start_lr) / max(1, warmup_epochs - 1)
    return eta_min + 0.5 * (base_lr - eta_min) * (1 + math.cos(math.pi * (epoch - warmup_epochs) / (max_epochs - warmup_epochs)))


def make_optimizer(model, lr=1e-3, weight_decay=0.05, betas=(0.9, 0.95), capturable=False):
    decay, no_decay = [], []
    for name, p in model.named_parameters():
        if not p.requires_grad:
            continue
        (no_decay if (p.ndim <= 1 or name.endswith(".bias")) else decay).append(p)
    groups = [{"params": no_decay, "weight_decay": 0.0}, {"params": decay, "weight_decay": weight_decay}]
    fused = all(p.is_cuda for g in groups for p in g["params"])
    if capturable:      # CUDA-graph capture: the step counter and the learning rate live on the device
        lr = torch.tensor(float(lr), device=groups[1]["params"][0].device)
    return torch.optim.AdamW(groups, lr=lr, betas=betas, fused=fused, capturable=capturable)


CUBLAS_DETERMINISTIC_CONFIGS = (":4096:8", ":16:8")


def check_deterministic_cublas():
    """Under torch.use_deterministic_algorithms(True) (strict, not warn_only) torch refuses cuBLAS calls unless CUBLAS_WORKSPACE_CONFIG
    is one of CUBLAS_DETERMINISTIC_CONFIGS, and MM_Net's projections use cuBLAS.  Raise here, at construction, instead of in the first
    step (or in the middle of a CUDA-graph capture).  The variable must be set before the process first uses cuBLAS."""
    if (torch.are_deterministic_algorithms_enabled() and not torch.is_deterministic_algorithms_warn_only_enabled()
            and os.environ.get("CUBLAS_WORKSPACE_CONFIG") not in CUBLAS_DETERMINISTIC_CONFIGS):
        raise RuntimeError("Trainer: torch.use_deterministic_algorithms(True) needs CUBLAS_WORKSPACE_CONFIG=:4096:8 (or :16:8) in the "
                           "environment before the process first uses cuBLAS; it is "
                           f"{os.environ.get('CUBLAS_WORKSPACE_CONFIG')!r}")


class Trainer:
    """One rank of a (possibly data-parallel) synthetic-data MM_Net training job.

    graph=True (default): after `graph_warmup` eager steps the whole step - forward, loss, backward (with DDP's bucketed
    NCCL all-reduces), AdamW - is captured once into a CUDA graph and replayed; the ~10 k kernel launches of a step then
    cost one host call instead of ~200 ms of Python / dispatcher time (the eager step is CPU-bound on a B200)."""

    def __init__(self, image_size=512, batch_per_rank=16, dtype="bf16", device=None, seed=50, lr=1e-3, weight_decay=0.05,
                 warmup_epochs=2, max_epochs=3000, ddp=None, channels_last=False, graph=True, graph_warmup=None):
        self.rank = dist.get_rank() if dist.is_initialized() else 0
        self.world = dist.get_world_size() if dist.is_initialized() else 1
        self.device = torch.device(device if device is not None else f"cuda:{int(os.environ.get('LOCAL_RANK', 0))}")
        self.autocast_dtype = {"bf16": torch.bfloat16, "fp16": torch.float16, "fp32": None, "f32": None}[dtype]
        self.image_size, self.batch = image_size, batch_per_rank
        self.channels_last = channels_last
        self.is_cuda = self.device.type == "cuda"       # "cpu" only works with the tests' oracle stand-ins for the Mamba ops
        if self.is_cuda:
            check_deterministic_cublas()
        self.stream = torch.cuda.Stream(self.device) if self.is_cuda else None    # all training work runs on this side stream
        torch.manual_seed(seed)                                           # same initial weights on every rank (train.py:160)
        net = MM_Net(num_classes=1).to(self.device)
        frozen = set(net.unused_parameters())
        for name, p in net.named_parameters():
            if name in frozen:
                p.requires_grad_(False)
        if channels_last:
            net = net.to(memory_format=torch.channels_last)
        self.net = net.train()
        use_ddp = (self.world > 1) if ddp is None else ddp
        self.use_graph = self.is_cuda and bool(int(os.environ.get("MMU_TRAIN_GRAPH", "1" if graph else "0")))
        with (torch.cuda.stream(self.stream) if self.is_cuda else contextlib.nullcontext()):   # DDP is built on the stream it is captured on
            self.model = (torch.nn.parallel.DistributedDataParallel(net, device_ids=[self.device.index] if self.is_cuda else None,
                                                                    bucket_cap_mb=25, gradient_as_bucket_view=True,
                                                                    broadcast_buffers=False)
                          if use_ddp else net)
        self.opt = make_optimizer(net, lr, weight_decay, capturable=self.use_graph)
        self.base_lr, self.warmup_epochs, self.max_epochs = lr, warmup_epochs, max_epochs
        self.set_epoch(0)
        self.gen = torch.Generator(device="cpu").manual_seed(1234 + self.rank)
        self.graph = None
        self.graph_warmup = graph_warmup if graph_warmup is not None else (11 if use_ddp else 3)
        self.steps_done = 0
        self.hot_path_launches = 0
        S, B = image_size, batch_per_rank
        self.x_dev = torch.empty(B, 3, S, S, device=self.device)
        if channels_last:
            self.x_dev = self.x_dev.contiguous(memory_format=torch.channels_last)
        self.y_dev = torch.empty(B, 1, S, S, device=self.device, dtype=torch.uint8)
        self.loss_dev = torch.zeros((), device=self.device)
        if self.is_cuda:
            self.copy_stream = torch.cuda.Stream(self.device)
            self.stage = [(torch.empty_like(self.x_dev), torch.empty_like(self.y_dev)) for _ in range(2)]
            self.stage_ready = [torch.cuda.Event() for _ in range(2)]
            self.stage_free = [torch.cuda.Event() for _ in range(2)]
            for e in self.stage_free:
                e.record(self.stream)

    def set_epoch(self, epoch: int):
        lr = warmup_cosine_lr(epoch, self.base_lr, self.warmup_epochs, self.max_epochs)
        for g in self.opt.param_groups:
            if torch.is_tensor(g["lr"]):
                g["lr"].fill_(lr)
            else:
                g["lr"] = lr

    def synthetic_batch(self, pinned=True):
        """Host-side batch (pinned): image fp32 (B,3,S,S), vessel mask uint8 (B,1,S,S)."""
        S, B = self.image_size, self.batch
        x = torch.randn(B, 3, S, S, generator=self.gen)
        y = (torch.rand(B, 1, S, S, generator=self.gen) < 0.1).to(torch.uint8)
        return (x.pin_memory(), y.pin_memory()) if (pinned and self.is_cuda) else (x, y)

    def _fwd_bwd_opt(self):
        if self.autocast_dtype is not None:
            with torch.autocast(self.device.type, dtype=self.autocast_dtype):
                logits = self.model(self.x_dev)
        else:
            logits = self.model(self.x_dev)
        loss = dice_focal_loss(logits, self.y_dev)
        loss.backward()
        self.opt.step()
        self.loss_dev.copy_(loss.detach())

    def step(self, x_host, y_host):
        """One optimisation step from HOST tensors; returns the loss as a device scalar (no host sync)."""
        if not self.is_cuda:
            self.x_dev.copy_(x_host)
            self.y_dev.copy_(y_host)
            self._fwd_bwd_opt()
            self.opt.zero_grad(set_to_none=True)
            self.steps_done += 1
            return self.loss_dev
        cur = torch.cuda.current_stream(self.device)
        self.stream.wait_stream(cur)
        # host -> device on a copy stream into one of two staging sets: the copy of step i overlaps the kernels of step i-1
        # (the host runs ahead of the GPU); the training stream then moves the batch into the graph's static inputs (D2D).
        k = self.steps_done % 2
        with torch.cuda.stream(self.copy_stream):
            self.copy_stream.wait_event(self.stage_free[k])
            self.stage[k][0].copy_(x_host, non_blocking=True)
            self.stage[k][1].copy_(y_host, non_blocking=True)
            self.stage_ready[k].record(self.copy_stream)
        with torch.cuda.stream(self.stream):
            self.stream.wait_event(self.stage_ready[k])
            self.x_dev.copy_(self.stage[k][0], non_blocking=True)
            self.y_dev.copy_(self.stage[k][1], non_blocking=True)
            self.stage_free[k].record(self.stream)
            if self.graph is not None:
                self.graph.replay()
            elif self.use_graph and self.steps_done >= self.graph_warmup:
                self.opt.zero_grad(set_to_none=True)
                g = torch.cuda.CUDAGraph()
                with torch.cuda.graph(g, stream=self.stream):
                    self._fwd_bwd_opt()
                    self.opt.zero_grad(set_to_none=True)      # gradients live in the graph's private pool
                self.graph = g
                g.replay()                                    # capture does not execute: run the step once
            else:
                n0 = _lib.launch_count()
                self._fwd_bwd_opt()
                self.opt.zero_grad(set_to_none=True)
                self.hot_path_launches = _lib.launch_count() - n0      # C-ABI kernel launches of one step (what a graph replays)
        cur.wait_stream(self.stream)
        self.steps_done += 1
        return self.loss_dev
