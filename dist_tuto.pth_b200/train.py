"""Distributed synchronous SGD (layer L6): the tutorial's ``run(rank, size)``.

Parity: train_dist.py:103-127 / tuto.md:283-303 --
``torch.manual_seed(1234)``; ``partition_dataset()``; ``Net()``;
``SGD(lr=0.01, momentum=0.5)``; 10 epochs; per batch
zero_grad -> forward -> nll_loss -> backward -> average_gradients -> step;
per epoch ``print('Rank ', rank, ', epoch ', epoch, ': ', mean_loss)``.

Fixes: D4 (loss accumulated detached, on device, read once per epoch); replicas
are made identical by an explicit parameter broadcast, not only by equal seeds.

Engines:
  * ``engine="torch"``  -- torch ops + ``average_gradients`` (CPU/gloo plumbing
    path, BASELINE.json config #1; also runs on CUDA).
  * ``engine="fused"``  -- the B200 path: one fused sm_100a forward+backward
    kernel, one fused peer-memory all-reduce + SGD kernel, replayed as a CUDA
    graph (``ops/convnet_fused.py``).  Default on CUDA for per-GPU batches < 2048 (the reference's 128 // world).
  * ``engine="batched"`` -- the throughput path for large per-GPU batches (BASELINE B1 "large-batch variant"): conv2
    forward / data gradient / weight gradient and fc1 as implicit GEMMs on tcgen05 (``ops/convnet_batched.py``), same
    fused exchange + SGD kernel.  ``auto`` picks it from 2048 samples per GPU up (measured: 1.1x the per-sample engine at
    1024, 2.5x at 4096, 2.7x at 16384 -- profiles/REPORT_r2.md section 2).
"""
from __future__ import annotations

import collections
import time
from math import ceil
from typing import Callable, Optional

import torch
import torch.nn.functional as F

from . import comm
from .data import partition_dataset
from .models.convnet import Net
from .ops.optim import FlatSGD
from .utils import say
from .utils.checkpoint import load_checkpoint, restore_optimizer, save_checkpoint
from .utils.trace import NullTracer, Tracer
from .parallel.ddp import GradBucket, average_gradients, broadcast_parameters

__all__ = ["run", "train", "TrainConfig", "BATCHED_FROM"]

BATCHED_FROM = 2048      # per-GPU batch from which engine="auto" takes the batched tensor-core engine


class TrainConfig:
    """Literal defaults of the reference, exposed as fields (SURVEY §5 config row)."""

    def __init__(self, epochs: int = 10, lr: float = 0.01, momentum: float = 0.5, seed: int = 1234,
                 global_batch: int = 128, engine: str = "auto", device: Optional[str] = None,
                 max_steps: Optional[int] = None, dataset=None, log: Callable[..., None] = say,
                 p_drop: float = 0.5, checkpoint: Optional[str] = None, resume: Optional[str] = None,
                 checkpoint_every: Optional[int] = None, trace: Optional[str] = None):
        self.epochs, self.lr, self.momentum, self.seed = epochs, lr, momentum, seed
        self.global_batch, self.engine, self.device = global_batch, engine, device
        self.max_steps, self.dataset, self.log, self.p_drop = max_steps, dataset, log, p_drop
        # checkpoint: written by rank 0 at the end (and after every `checkpoint_every`-th epoch); resume: a checkpoint to start
        # from -- parameters, momentum, step counter AND the number of completed epochs, so a resumed run does the remaining
        # epochs with the shuffles those epochs would have had (restart after a failure: spawn.py --max-restarts)
        self.checkpoint, self.resume, self.checkpoint_every = checkpoint, resume, checkpoint_every
        # trace: path of a Chrome / Perfetto trace (utils/trace.py) -- host spans per epoch / step phase and one device span per
        # step (torch engine) or per epoch (fused engines: their steps are launched by C++ / CUDA graphs), all ranks in one file
        self.trace = trace


def _spans_machines() -> bool:
    """True when the default group's world is the two-level one (launch.init_processes built it for a multi-machine job)."""
    try:
        from .parallel import symm
        from .parallel.hier import HierWorld
        w = symm.lookup_world(None)
        return isinstance(w, HierWorld) and w.n_nodes > 1
    except Exception:
        return False


def _pick_device(cfg: TrainConfig) -> torch.device:
    if cfg.device is not None:
        return torch.device(cfg.device)
    if torch.cuda.is_available() and comm.is_initialized() and \
            "nccl" in str(torch.distributed.get_backend()):
        return torch.device("cuda", torch.cuda.current_device())
    return torch.device("cpu")


def train(rank: int, size: int, cfg: Optional[TrainConfig] = None):
    """Run the training loop; returns a dict with per-epoch mean losses and timing."""
    cfg = cfg or TrainConfig()
    torch.manual_seed(cfg.seed)                                   # train_dist.py:105
    device = _pick_device(cfg)
    engine = cfg.engine
    tracer = Tracer(rank) if cfg.trace else NullTracer()
    multi_node = _spans_machines()
    if engine == "auto":
        # several machines: the in-kernel gradient exchange of the fused engines is a single-NVSwitch-domain protocol, the
        # bucketed engine reduces through the two-level world (parallel/hier.py)
        engine = "torch" if (device.type != "cuda" or multi_node) else \
            ("batched" if cfg.global_batch // max(size, 1) >= BATCHED_FROM else "fused")
    if multi_node and engine in ("fused", "batched"):
        raise ValueError(f"engine={engine!r} exchanges gradients inside one NVSwitch domain; this job spans several machines "
                         "(use engine='auto' or 'torch')")
    if engine not in ("torch", "fused", "batched"):
        raise ValueError(f"TrainConfig.engine must be auto / torch / fused / batched, got {engine!r}")
    fused_raw = engine in ("fused", "batched") and (cfg.dataset is None or hasattr(cfg.dataset, "images"))
    train_set, bsz = partition_dataset(cfg.dataset, global_batch=cfg.global_batch, seed=cfg.seed,
                                       **({"raw_uint8": True} if fused_raw else {}))
    num_batches = ceil(len(train_set.dataset) / float(bsz))      # train_dist.py:112
    start_steps, optimizer, resume_blob = 0, None, {}
    copies_in_flight = collections.deque()                       # torch engine on CUDA, see step_fn
    if engine == "fused":
        from .ops.convnet_fused import FusedTrainer
        trainer = FusedTrainer(bsz, lr=cfg.lr, momentum=cfg.momentum, seed=cfg.seed, device=device,
                               p_drop=cfg.p_drop, raw_uint8=fused_raw)
        if cfg.resume:
            resume_blob = load_checkpoint(cfg.resume, trainer)
            start_steps = int(resume_blob.get("steps", 0))
        step_fn, epoch_loss_fn, model = trainer.step, trainer.pop_loss_sum, trainer
    elif engine == "batched":
        from .ops.convnet_batched import BatchedTrainer
        trainer = BatchedTrainer(bsz, lr=cfg.lr, momentum=cfg.momentum, seed=cfg.seed, device=device,
                                 p_drop=cfg.p_drop, raw_uint8=fused_raw)
        if cfg.resume:
            resume_blob = load_checkpoint(cfg.resume, trainer)
            start_steps = int(resume_blob.get("steps", 0))
        recycles = hasattr(train_set, "before_recycle")
        if recycles:          # the loader's pinned staging buffers: a buffer is refilled only after its H2D copy has left it
            def _oldest_step_done():
                if copies_in_flight:
                    copies_in_flight.popleft().synchronize()
            train_set.before_recycle = _oldest_step_done

        def step_fn(data, target):
            trainer.step(data, target)
            if recycles:
                ev = torch.cuda.Event()
                ev.record(trainer.stream)
                copies_in_flight.append(ev)
        epoch_loss_fn, model = trainer.pop_loss_sum, trainer
    else:
        model = Net(cfg.p_drop).to(device)
        if cfg.resume:
            resume_blob = load_checkpoint(cfg.resume, model)
            start_steps = int(resume_blob.get("steps", 0))
        broadcast_parameters(model)
        model._grad_bucket = GradBucket(list(model.parameters()))
        # optim.SGD(lr=0.01, momentum=0.5) of train_dist.py:110, over flat buffers: update + zero_grad in one pass
        optimizer = FlatSGD(model, lr=cfg.lr, momentum=cfg.momentum)
        if cfg.resume:
            restore_optimizer(optimizer, model, resume_blob)         # momentum: FlatSGD layout or per-name (fused engine's)
        acc = torch.zeros((), device=device)

        # The native loader recycles its pinned staging buffers; the async H2D copies below must have left a buffer
        # before the prefetch thread refills it.  One event per handed-out batch, consumed in hand-out order.
        if device.type == "cuda" and hasattr(train_set, "before_recycle"):
            def _oldest_copy_done():
                if copies_in_flight:
                    copies_in_flight.popleft().synchronize()
            train_set.before_recycle = _oldest_copy_done

        step_span = tracer.device_span if device.type == "cuda" else tracer.span     # CUDA events cannot time CPU work

        def step_fn(data, target):
            with step_span("step", cat="step"):
                with tracer.span("h2d"):
                    data = data.to(device, non_blocking=True)
                    target = target.to(device, non_blocking=True)
                if device.type == "cuda" and hasattr(train_set, "before_recycle"):
                    ev = torch.cuda.Event()
                    ev.record()
                    copies_in_flight.append(ev)
                optimizer.zero_grad()                                # buckets were re-zeroed by the previous step()
                with tracer.span("forward + loss"):
                    output = model(data)
                    loss = F.nll_loss(output, target)
                    acc.add_(loss.detach())                          # epoch_loss += loss (D4 fixed)
                with tracer.span("backward"):
                    loss.backward()
                with tracer.span("average_gradients"):
                    average_gradients(model)
                with tracer.span("optimizer"):
                    optimizer.step()

        def epoch_loss_fn():
            v = float(acc.item())
            acc.zero_()
            return v

    history, steps, t0 = [], 0, time.perf_counter()
    start_epoch = 0
    if resume_blob.get("in_progress"):            # a periodic checkpoint of an unfinished run: do the REMAINING epochs
        start_epoch = min(int(resume_blob.get("epoch", 0)), cfg.epochs)
        history = list(resume_blob.get("history", []))[:start_epoch]
    # (a checkpoint of a finished run starts a new run of cfg.epochs epochs from its parameters / momentum / step counter)
    if start_epoch and hasattr(train_set, "_epoch"):
        train_set._epoch = start_epoch                                    # the loader shuffles by (seed, epoch index)
    done = False
    native_loop = engine == "fused" and hasattr(train_set, "begin_epoch") and torch.cuda.is_available()
    for epoch in range(start_epoch, cfg.epochs):
        model.train()
        nb = 0
        copies_in_flight.clear()          # the previous epoch ended with a device sync (epoch_loss_fn): nothing is pending
        with tracer.span(f"epoch {epoch}", cat="epoch", engine=engine):
            if native_loop:       # C++ executor: prefetch thread -> cudaGraphLaunch per step, no Python in the loop
                budget = None if cfg.max_steps is None else cfg.max_steps - steps
                with tracer.span("run_native (C++ executor: the whole epoch, returns drained)", cat="step"):
                    nb, _ = trainer.run_native(train_set, max_steps=budget)
                steps += nb
                done = cfg.max_steps is not None and steps >= cfg.max_steps
            else:
                batches = iter(train_set)
                while True:
                    with tracer.span("next batch", cat="data"):
                        item = next(batches, None)
                    if item is None:
                        break
                    step_fn(*item)
                    steps += 1
                    nb += 1
                    if cfg.max_steps is not None and steps >= cfg.max_steps:
                        done = True
                        batches.close() if hasattr(batches, "close") else None     # run the loader's clean-up (stops its thread)
                        break
            denom = num_batches if not done else max(nb, 1)
            with tracer.span("read epoch loss (device sync)", cat="sync"):
                loss_sum = epoch_loss_fn()
        mean_loss = loss_sum / denom
        history.append(mean_loss)
        cfg.log("Rank ", comm.get_rank(), ", epoch ", epoch, ": ", mean_loss)
        if done:
            break
        epochs_done = epoch + 1
        if cfg.checkpoint and cfg.checkpoint_every and epochs_done % cfg.checkpoint_every == 0 and epochs_done < cfg.epochs:
            if comm.get_rank() == 0:
                save_checkpoint(cfg.checkpoint, model, optimizer=optimizer, steps=start_steps + steps, history=history,
                                epoch=epochs_done, in_progress=True)
            if size > 1:
                comm.barrier()                   # nobody runs ahead into a failure before the checkpoint is on disk
    elapsed = time.perf_counter() - t0
    if cfg.checkpoint and comm.get_rank() == 0:
        save_checkpoint(cfg.checkpoint, model, optimizer=optimizer, steps=start_steps + steps, history=history,
                        epoch=max(0, len(history) - (1 if done else 0)), in_progress=False)
    trace_file = tracer.save(cfg.trace) if cfg.trace else None          # collective: rank 0 writes every rank's rows
    return {"loss": history, "steps": steps, "seconds": elapsed, "bsz": bsz,
            "samples_per_s": steps * bsz * size / max(elapsed, 1e-9), "model": model, "trace": trace_file}


def run(rank: int, size: int):
    """Distributed Synchronous SGD Example (train_dist.py:103)."""
    return train(rank, size, TrainConfig())
