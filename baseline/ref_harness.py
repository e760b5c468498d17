"""Reference arm: drive the UNMODIFIED reference scripts from ``baseline/_ref``.

Nothing from ``dist_tuto.pth_b200`` (models, kernels, engine) is on the measured path.  What is used:

  * ``train_dist.Net``                    the reference model class (train_dist.py:53-71), ``.cuda(rank)``
                                          as in its commented line :109
  * ``train_dist.partition_dataset()``    unmodified (e2e path); it finds MNIST idx files under ./data, so
                                          we point the cwd at a scratch dir holding *synthetic* idx files
                                          (there is no network; BASELINE.json prescribes synthetic 28x28)
  * ``train_dist.average_gradients``      ``--ref-avg committed``: exactly as committed (never communicates,
                                          SURVEY D1);  ``--ref-avg tutorial`` (default, the stronger
                                          baseline): the body printed in the tutorial text tuto.md:310-314
                                          -- per-parameter ``dist.all_reduce(SUM)`` + ``/= size`` on NCCL
  * the loop body of ``train_dist.run``   :118-124, verbatim order of operations, ``optim.SGD(lr=0.01,
                                          momentum=0.5)``.  ``run()`` itself cannot be timed for K steps
                                          (it is a closed 10-epoch loop), so the loop is re-issued here.

Process-group bootstrap is torchrun-env NCCL (plumbing, outside the timed region); the reference's own
``init_processes`` pins MASTER_PORT=29500 which collides with / ignores the driver-chosen port.
"""
from __future__ import annotations

import importlib.util
import json
import os
import sys
import time
import warnings

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)


def load_reference():
    sys.path.insert(0, HERE)
    import install_ref
    ok, why = install_ref.verify()          # installed beforehand by install_ref.py: the benchmark writes nothing here
    if not ok:
        return None, why
    spec = importlib.util.spec_from_file_location("ref_train_dist", os.path.join(install_ref.DST, "train_dist.py"))
    mod = importlib.util.module_from_spec(spec)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        spec.loader.exec_module(mod)
    return mod, "ok"


def tutorial_average_gradients(model, dist):
    """tuto.md:310-314 verbatim semantics (the committed function is dead code, SURVEY D1/D2)."""
    size = float(dist.get_world_size())
    for param in model.parameters():
        dist.all_reduce(param.grad.data, op=dist.ReduceOp.SUM)
        param.grad.data /= size


def run(args):
    ref, why = load_reference()
    if ref is None:
        print(json.dumps({"impl": "reference", "unavailable": why}))
        return 0
    import torch
    import torch.distributed as dist
    import torch.nn.functional as F
    import torch.optim as optim
    if not torch.cuda.is_available():
        print(json.dumps({"impl": "reference", "unavailable": "no CUDA device"}))
        return 0
    warnings.filterwarnings("ignore")
    rank = int(os.environ.get("RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    local = int(os.environ.get("LOCAL_RANK", rank))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
    os.environ.setdefault("MASTER_PORT", "29511")
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    sys.path.insert(0, ROOT)
    from bench_common import ClockSampler, aligned_start, max_over_ranks, result_line, synthetic_idx_dir  # no kernels in there

    K, W = args.steps, args.warmup
    bsz = 128 // world                                              # train_dist.py:85
    torch.manual_seed(1234)                                         # train_dist.py:105
    model = ref.Net().cuda(local)                                   # train_dist.py:107,109
    optimizer = optim.SGD(model.parameters(), lr=0.01, momentum=0.5)  # train_dist.py:110
    avg = (lambda m: ref.average_gradients(m)) if args.ref_avg == "committed" else \
        (lambda m: tutorial_average_gradients(m, dist))

    def step(data, target):
        optimizer.zero_grad()
        output = model(data)
        loss = F.nll_loss(output, target)
        loss.backward()
        avg(model)
        optimizer.step()
        return loss

    # ---------------- value: device-resident synthetic batches cycling through a pool larger than L2
    pool = max(8, (160 << 20) // (bsz * 784 * 4))
    g = torch.Generator(device=dev).manual_seed(1234 + rank)
    px = torch.randn(pool, bsz, 1, 28, 28, device=dev, generator=g)
    py = torch.randint(0, 10, (pool, bsz), device=dev, generator=g)
    for i in range(W):
        step(px[i % pool], py[i % pool])
    torch.cuda.synchronize()
    dist.barrier()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with ClockSampler(local) as clk:
        e0.record()
        for i in range(K):
            step(px[(W + i) % pool], py[(W + i) % pool])
        e1.record()
        torch.cuda.synchronize()
        dist.barrier()
        torch.cuda.synchronize()
    ms = max_over_ranks(e0.elapsed_time(e1), dev)
    value = 128 // world * world * K / (ms / 1e3)

    # ---------------- e2e: the reference's own partition_dataset() + DataLoader + .cuda(rank) + loss read
    cwd = os.getcwd()
    scratch = synthetic_idx_dir(rank)
    os.chdir(scratch)
    try:
        train_set, bsz2 = ref.partition_dataset()                    # unmodified (train_dist.py:74-91)
    finally:
        os.chdir(cwd)
    it = iter(train_set)

    def next_batch():
        nonlocal it
        try:
            return next(it)
        except StopIteration:
            it = iter(train_set)
            return next(it)

    for _ in range(W):
        d, t = next_batch()
        step(d.cuda(local), t.cuda(local)).item()
    t0 = aligned_start(dev)                      # barrier + synchronize + common start instant (same as our arm)
    h2d = 0
    for _ in range(K):
        d, t = next_batch()
        h2d = d.numel() * d.element_size() + t.numel() * t.element_size()
        step(d.cuda(local), t.cuda(local)).item()                    # train_dist.py:117 enabled + loss read
    torch.cuda.synchronize()
    e2e_ms = max_over_ranks((time.perf_counter() - t0) * 1e3, dev)
    e2e = bsz2 * world * K / (e2e_ms / 1e3)
    if rank == 0:
        print(result_line(impl="reference", value=value, ms=ms, n_gpus=world, steps=K, warmup=W, clocks=clk.summary(),
                          e2e_value=e2e, h2d=h2d, d2h=4, gpu_launches=0, dtype="fp32",
                          extra_config={"engine": "reference Net + torch.optim.SGD + per-parameter NCCL all_reduce",
                                        "ref_avg": args.ref_avg,
                                        "l2": f"inputs cycle through a {pool * bsz * 784 * 4 >> 20} MB device pool (> L2)",
                                        "e2e_path": "reference partition_dataset()/DataLoader on synthetic idx files, "
                                                    ".cuda(rank), loss.item() per step"}))
    dist.barrier()
    dist.destroy_process_group()
    return 0
