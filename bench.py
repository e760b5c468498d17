#!/usr/bin/env python
"""Headline benchmark (driver contract): MNIST-ConvNet synchronous data-parallel SGD, samples/s.

    python bench.py --gpus N --steps K --warmup W [--impl ours|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
        bench.py --gpus N --steps K --warmup W

Config = BASELINE.json #2 / train_dist.py: global batch 128 (``128 // N`` per GPU -> strong scaling), SGD lr 0.01
momentum 0.5, dropout on, synthetic 28x28 data, random-init weights.

``value``  : device-timed (CUDA events, max over ranks) training throughput of the fused engine -- full step =
             forward + loss + backward + peer-memory gradient all-reduce + SGD, nothing skipped -- on batches
             cycling through a device pool larger than L2.
``e2e``    : the same metric through the public API a user calls (``partition_dataset()`` -> native loader ->
             ``FusedTrainer.run_native``, i.e. what ``train()`` runs per epoch): every step copies its batch (uint8
             pixels + labels) from pinned host memory to the device and the running loss back to pinned host memory.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--ref-avg", default="tutorial", choices=["tutorial", "committed"])
    ap.add_argument("--graph-chunk", type=int, default=50)
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--large-batch", type=int, default=4096,
                    help="per-GPU batch of the extra large-batch (throughput, weak-scaling) measurement; 0 = skip")
    ap.add_argument("--loader-buffers", type=int, default=24, help="pinned ring depth of the native loader (e2e arm)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps write what they computed (the trained parameters by name and the running "
                         "[loss sum, #correct]) as DIR/<name>.npy, float32; inputs are seeded, so runs with the same "
                         "arguments can be compared array for array.  Gradient sums use float atomics: after the ~500 "
                         "steps of the default run two runs differed by up to 2.4e-3 in a weight (B200, 1000 W)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be >= 1")
    return args


def gpu_smi_id(torch, dev):
    """What to pass to ``nvidia-smi --id=``: the device's UUID (robust against CUDA_VISIBLE_DEVICES), else its index."""
    try:
        u = str(torch.cuda.get_device_properties(dev).uuid)
        return u if u.startswith("GPU-") else "GPU-" + u
    except Exception:
        return dev.index


def large_batch_arm(torch, b2, LB, rank, size, dev, max_over_ranks, steps):
    """Device-timed samples/s of ``steps`` full training steps at per-GPU batch ``LB`` (weak scaling) on the batched
    tcgen05 engine."""
    from dist_tuto.pth_b200.ops.convnet_batched import BatchedTrainer
    tr = BatchedTrainer(LB, lr=0.01, momentum=0.5, seed=1234, device=dev, p_drop=0.5, raw_uint8=True)
    npool = min(steps, 64) + 1                  # graphs are reused round-robin beyond 64 steps
    g = torch.Generator(device=dev).manual_seed(99 + rank)
    xs = torch.randint(0, 256, (npool, LB, 1, 28, 28), dtype=torch.uint8, device=dev, generator=g)
    ys = torch.randint(0, 10, (npool, LB), device=dev, generator=g)
    st = tr.stream
    with torch.cuda.stream(st):
        for i in range(3):
            tr._kernels(xs[i], ys[i], LB)
    st.synchronize()
    graphs = []
    for i in range(npool):
        gr = torch.cuda.CUDAGraph()
        with torch.cuda.graph(gr, stream=st):
            tr._kernels(xs[i], ys[i], LB)
        graphs.append(gr)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    with torch.cuda.stream(st):
        for gr in graphs:
            gr.replay()
    st.synchronize()
    b2.barrier()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with torch.cuda.stream(st):
        flush.fill_(1)
        graphs[0].replay()                      # pre-roll (untimed): ranks aligned by its exchange
        e0.record(st)
        for i in range(steps):
            graphs[1 + i % (npool - 1)].replay()
        e1.record(st)
    st.synchronize()
    ms = max_over_ranks(e0.elapsed_time(e1), dev)
    loss = float(tr.loss_acc[0].item())
    out = {"per_gpu_batch": LB, "global_batch": LB * size, "scaling": "weak", "steps": steps, "us_per_step": ms / steps * 1e3,
           "samples_per_s": LB * size * steps / (ms / 1e3), "dtype": "bf16 tensor-core operands (tcgen05), fp32 accumulate / master weights",
           "engine": "batched: conv2 fwd/dgrad/wgrad + fc1 on tcgen05 with TMA-fed operands, fused all-reduce+SGD kernel",
           "launches_per_step": tr.gpu_launches_per_step, "loss_finite": loss == loss,
           "l2": f"L2 flushed before the pre-roll; the timed steps cycle through {npool - 1} batches "
                 f"({(npool - 1) * LB * 784 / 2**20:.0f} MB) not touched since"}
    del graphs, tr
    return out


def dump_outputs(out_dir, arrays):
    """Write every tensor as ``out_dir/<name>.npy`` in float32."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    for name, t in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), t.detach().float().cpu().numpy())


def ours(args):
    import torch
    import dist_tuto.pth_b200 as b2
    from bench_common import ClockSampler, aligned_start, max_over_ranks, result_line
    from dist_tuto.pth_b200.data import SyntheticMNIST
    from dist_tuto.pth_b200.ops.convnet_fused import FusedTrainer, unpack_params

    K, W = args.steps, max(args.warmup, 3)

    def body(rank, size):
        dev = torch.device("cuda", torch.cuda.current_device())
        bsz = 128 // size
        tr = FusedTrainer(bsz, lr=0.01, momentum=0.5, seed=1234, device=dev, p_drop=0.5, raw_uint8=True)
        # ------------------------------------------------------------ value: device-timed
        # Layout of the measured stream (nothing but graph launches between the two events, no host sync inside):
        #     [L2 flush] [pre-roll graph: G untimed steps] e0 [timed graphs: exactly K steps] e1
        # * every graph is replayed once beforehand (upload + instantiate cost is not timed);
        # * e0 is recorded ON THE STREAM behind the pre-roll steps: every step ends with the cross-GPU gradient
        #   exchange, so by the time e0 fires all ranks are aligned to within one exchange and the host is already
        #   ~G steps ahead with its launches -- inter-process start skew cannot sit inside e0 -> e1;
        # * the batches of the timed graphs are not touched between the L2 flush (256 MB written) and their step.
        batch_bytes = bsz * 784 * 4
        G = max(1, min(args.graph_chunk, K))
        n_full, rem = divmod(K, G)
        n_timed = min(n_full, 64)                    # graphs are reused round-robin beyond 64 chunks
        n_graphs = n_timed + 1                       # + the pre-roll graph
        pool = n_graphs * G + rem
        g = torch.Generator(device=dev).manual_seed(1234 + rank)
        px = torch.randn(pool, bsz, 1, 28, 28, device=dev, generator=g)
        py = torch.randint(0, 10, (pool, bsz), device=dev, generator=g)
        flush_buf = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
        st = tr.stream
        with torch.cuda.stream(st):
            for i in range(W):
                tr._kernels(px[i % pool], py[i % pool], bsz)
        st.synchronize()

        def capture(first, count):
            gr = torch.cuda.CUDAGraph()
            with torch.cuda.graph(gr, stream=st):
                for i in range(count):
                    tr._kernels(px[first + i], py[first + i], bsz)
            return gr

        graphs = [capture(j * G, G) for j in range(n_graphs)]          # graphs[0] = pre-roll
        tail = capture(n_graphs * G, rem) if rem else None
        with torch.cuda.stream(st):
            for gr in graphs + ([tail] if tail is not None else []):   # untimed: uploads every graph that is timed later
                gr.replay()
        st.synchronize()
        b2.barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        smi_id = gpu_smi_id(torch, dev)            # physical GPU (UUID): CUDA_VISIBLE_DEVICES re-numbers the logical index
        with ClockSampler(smi_id) as clk:
            with torch.cuda.stream(st):
                flush_buf.fill_(1)                                     # L2 flush: 256 MB > 126 MB L2
                graphs[0].replay()                                     # pre-roll (untimed)
                e0.record(st)
                for s in range(n_full):
                    graphs[1 + s % n_timed].replay()
                if tail is not None:
                    tail.replay()
                e1.record(st)
            st.synchronize()
            b2.barrier()
            torch.cuda.synchronize()
        if args.dump_outputs and rank == 0:        # replicas are identical: rank 0 holds what every caller receives
            dump_outputs(args.dump_outputs, {**unpack_params(tr.params), "loss_acc": tr.loss_acc})
        ms = max_over_ranks(e0.elapsed_time(e1), dev)
        value = bsz * size * K / (ms / 1e3)
        clocks = clk.summary()
        if clocks["samples"] < 3:
            # the timed region (K x ~30 us) is shorter than one nvidia-smi query: sample the clocks under the SAME load by
            # replaying the timed graphs for ~0.6 s (not part of any reported time)
            reps = min(100000, max(8, int(600.0 / max(ms / K * G, 1e-3))))   # same count on every rank (ms is the max over ranks)
            with ClockSampler(smi_id) as probe:
                with torch.cuda.stream(st):
                    for s in range(reps):
                        graphs[s % n_graphs].replay()
                st.synchronize()
            b2.barrier()
            clocks = dict(probe.summary(), in_timed_region=clocks["samples"],
                          note="timed region shorter than one nvidia-smi query; sampled while replaying the timed graphs right after it")
        l2_note = (f"L2 flushed (256 MB written) right before the pre-roll; the K timed steps read {min(K, n_timed * G + rem)} distinct "
                   f"batches ({min(K, n_timed * G + rem) * batch_bytes / 2**20:.1f} MB) not touched since the flush")
        loss_dev = float(tr.loss_acc[0].item())
        assert loss_dev == loss_dev, "loss is NaN"

        # ------------------------------------------------------------ e2e: public API, pinned H2D + loss D2H per step
        e2e, h2d = None, bsz * 784 * 1 + bsz * 8          # raw uint8 pixels (normalised in-kernel) + int64 labels
        exec_chunk = 1
        if not args.no_e2e:
            ds = SyntheticMNIST(n=60000, seed=1234)
            loader, bsz2 = b2.partition_dataset(ds, raw_uint8=True, num_buffers=args.loader_buffers)
            assert bsz2 == bsz

            # the call a user makes (train.py does exactly this per epoch): the C++ executor drives
            # prefetch thread -> [H2D batch from the pinned ring, convnet_step, allreduce_sgd, D2H loss] per step.
            # Warm-up and timed steps are consecutive steps of the SAME epoch (steady state of train()'s loop: the
            # once-per-epoch index shuffle / prefetch-thread start is not inside a 20-step window, as it is not
            # inside 468 of the 469 steps of an epoch); a new epoch starts only when the current one runs dry.
            state = {"fresh": True}

            def advance(n):
                done = 0
                while done < n:                          # an epoch has 60000/128 = 468 full batches
                    d, fin = tr.run_native(loader, max_steps=n - done, new_epoch=state["fresh"])
                    state["fresh"] = fin
                    done += d

            advance(W)
            tr._executors[id(loader)][0].reset_stats()
            t0 = aligned_start(dev)                      # barrier + synchronize, then all ranks leave at the same instant
            advance(K)
            seen = tr.last_loss_cumulative()             # host copy of the last step's D2H loss
            torch.cuda.synchronize()
            e2e_ms = max_over_ranks((time.perf_counter() - t0) * 1e3, dev)
            e2e = bsz * size * K / (e2e_ms / 1e3)
            assert seen == seen
            ex = tr._executors[id(loader)][0]
            host_stats = {k: (round(v, 1) if isinstance(v, float) else v) for k, v in ex.stats().items()}
            host_stats["flag_mode"] = bool(ex.flag_mode())
            exec_chunk = getattr(tr, "exec_chunk", 1) if ex.chunking() else 1
        # ------------------------------------------------------------ extra key: BASELINE.md B1 "large-batch variant"
        # Same network / optimizer / data-parallel exchange at a throughput-sized per-GPU batch (weak scaling), run by the
        # batched tensor-core engine (csrc/convnet_batched.cu).  Not the headline: `value` above stays global batch 128.
        large = None
        if args.large_batch > 0:
            try:
                large = large_batch_arm(torch, b2, args.large_batch, rank, size, dev, max_over_ranks, K)
            except Exception as e:      # never take the headline down
                large = {"error": f"{type(e).__name__}: {e}"[:300]}
        if rank == 0:
            sym = tr.symm.describe() if tr.symm is not None else {"world": 1}
            print(result_line(impl="ours", value=value, ms=ms, n_gpus=size, steps=K, warmup=W, clocks=clocks,
                              e2e_value=e2e, h2d=h2d, d2h=8, gpu_launches=tr.gpu_launches_per_step * K, dtype="fp32",
                              extra_config={"engine": ("ONE kernel per step: fused convnet_step (cluster-per-sample for small per-GPU batches) whose tail does the gradient exchange + SGD; CUDA graph, PDL"
                                                       if tr.fused_tail else "fused convnet_step (cluster-per-sample for small per-GPU batches) + allreduce_sgd kernels, CUDA graph, PDL"),
                                            "precision": "fp32 SIMT forward/backward (>= the required bf16); " + ("bf16" if tr.wire_bf16 else "fp32") + " gradients on the wire; fp32 accumulate + SGD",
                                            "cluster_ctas_per_sample": tr.cluster,
                                            "gradient_exchange": ("push: flag-in-data stores into peer inboxes, local reduce" if tr.inbox_handle is not None
                                                                  else ("barrier + peer loads" if size > 1 else "none (1 GPU)")),
                                            "l2": l2_note,
                                            "timing": "CUDA events on the launch stream: [L2 flush][pre-roll graph, untimed] e0 [K steps] e1, "
                                                      "enqueued back to back; max over ranks.  e2e: host clock from a common start instant (barrier + "
                                                      "synchronize, then all ranks spin to an agreed CLOCK_MONOTONIC time) to this rank's synchronize "
                                                      "after its K-th loss read-back; max over ranks",
                                            "graph_chunk": G, "symm": sym,
                                            "e2e_path": "partition_dataset(raw_uint8) -> C++ prefetch thread -> C++ StepExecutor: per step one H2D "
                                                        "(uint8 batch + labels, pinned), 2 kernels, one D2H (loss); "
                                                        + (f"chunks of {exec_chunk} steps = 3 graph launches on 3 streams ({exec_chunk} H2D nodes | {2 * exec_chunk} kernels | {exec_chunk} D2H nodes)"
                                                           if exec_chunk > 1 else ("plain PDL stream launches; flag mode: stream memory ops instead of cross-stream events"
                                                                                   if (not args.no_e2e and host_stats.get("flag_mode")) else
                                                                                   "plain PDL stream launches, 3 streams ordered by events (9 driver calls per step)")),
                                            "e2e_host_us": host_stats if not args.no_e2e else None,
                                            "large_batch": large}),
                  flush=True)

    rank = int(os.environ.get("RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    if world != args.gpus and "RANK" in os.environ:
        print(f"[bench] WORLD_SIZE={world} overrides --gpus {args.gpus}", file=sys.stderr)
    if "RANK" not in os.environ and args.gpus > 1:
        # convenience: self-launch N local ranks
        b2.launch(body, size=args.gpus, backend="b200", join_timeout_s=1800)
        return 0
    kw = {}
    if "MASTER_PORT" in os.environ:
        kw = dict(master_addr=os.environ.get("MASTER_ADDR", "127.0.0.1"), master_port=int(os.environ["MASTER_PORT"]))
    else:
        kw = dict(master_port=b2.find_free_port())
    b2.init_processes(rank, world, body, backend="b200", **kw)
    return 0


def main():
    args = parse()
    if args.impl == "reference":
        sys.path.insert(0, os.path.join(ROOT, "baseline"))
        try:
            import ref_harness
            return ref_harness.run(args)
        except Exception as e:  # the arm must never take the driver down
            if int(os.environ.get("RANK", 0)) == 0:
                print(json.dumps({"impl": "reference", "unavailable": f"{type(e).__name__}: {e}"[:300]}))
            return 0
    return ours(args)


if __name__ == "__main__":
    sys.exit(main())
