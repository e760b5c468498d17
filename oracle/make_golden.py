"""Record what the original tutorial's ``train_dist.py`` computes, as small golden vectors for the test suite.

    python oracle/make_golden.py <directory holding the original train_dist.py>

The original script is loaded unmodified and run on CPU in fp32: the initial weights of its ``Net`` under
``torch.manual_seed(1234)`` (what its ``run()`` seeds), an eval-mode forward, a few steps of its training loop body
(``zero_grad``, forward, ``nll_loss``, ``backward``, ``average_gradients``, ``SGD(lr=0.01, momentum=0.5).step()``) with
dropout off so that the steps are reproducible elsewhere, and the index shards of its ``DataPartitioner``.  The result
goes to ``tests/golden/reference_convnet.npz`` (about 0.4 MB) together with the SHA-256 of the script it came from."""
import hashlib
import importlib.util
import os
import sys
import tempfile
import warnings

import numpy as np
import torch
import torch.distributed as dist
import torch.nn.functional as F

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
OUT = os.path.join(ROOT, "tests", "golden", "reference_convnet.npz")
BATCH, STEPS, DATA_SEED = 16, 4, 2024


def load(src_dir):
    path = os.path.join(src_dir, "train_dist.py")
    spec = importlib.util.spec_from_file_location("ref_train_dist", path)
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    with open(path, "rb") as f:
        return mod, hashlib.sha256(f.read()).hexdigest()


def main(src_dir):
    warnings.simplefilter("ignore")
    torch.use_deterministic_algorithms(True)
    ref, sha = load(src_dir)
    with tempfile.TemporaryDirectory() as tmp:      # its average_gradients() asks the process group for the world size
        dist.init_process_group("gloo", init_method=f"file://{tmp}/rdzv", rank=0, world_size=1)
        try:
            torch.manual_seed(1234)
            model = ref.Net()
            init = [p.detach().clone() for p in model.parameters()]
            g = torch.Generator().manual_seed(DATA_SEED)
            xs = torch.randn(STEPS, BATCH, 1, 28, 28, generator=g)
            ys = torch.randint(0, 10, (STEPS, BATCH), generator=g)
            model.eval()
            with torch.no_grad():
                logp = model(xs[0])
            optimizer = torch.optim.SGD(model.parameters(), lr=0.01, momentum=0.5)
            losses = []
            for data, target in zip(xs, ys):
                optimizer.zero_grad()
                loss = F.nll_loss(model(data), target)
                loss.backward()
                ref.average_gradients(model)
                optimizer.step()
                losses.append(float(loss))
            final = [p.detach().clone() for p in model.parameters()]
        finally:
            dist.destroy_process_group()
    shards3 = ref.DataPartitioner(list(range(6000)), [1.0 / 3] * 3).partitions
    shards2 = ref.DataPartitioner(list(range(60000)), [0.5, 0.5]).partitions
    out = {"train_dist_sha256": np.array(sha), "x": xs.numpy(), "y": ys.numpy(), "eval_logp": logp.numpy(),
           "losses": np.array(losses, dtype=np.float32),
           "init": torch.cat([p.reshape(-1) for p in init]).numpy(),
           "final": torch.cat([p.reshape(-1) for p in final]).numpy(),
           "shards_6000_w3": np.array(shards3, dtype=np.int32),
           "shards_60000_w2_head": np.array([s[:256] for s in shards2], dtype=np.int32)}
    os.makedirs(os.path.dirname(OUT), exist_ok=True)
    np.savez_compressed(OUT, **out)
    print(f"wrote {OUT} ({os.path.getsize(OUT)} bytes); losses {losses}")


if __name__ == "__main__":
    if len(sys.argv) != 2:
        sys.exit(__doc__)
    main(sys.argv[1])
