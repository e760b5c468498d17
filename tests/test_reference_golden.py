"""Parity with the original tutorial's ``train_dist.py`` through stored vectors (tests/golden/reference_convnet.npz,
recorded by oracle/make_golden.py from the unmodified script): the seeded initial weights, an eval forward, four SGD steps
of its training loop with dropout off, and its DataPartitioner shards."""
import os

import numpy as np
import pytest
import torch
import torch.nn.functional as F

import dist_tuto.pth_b200 as b2
from dist_tuto.pth_b200 import data as D

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
G = np.load(os.path.join(ROOT, "tests", "golden", "reference_convnet.npz"))


def _flat(net):
    return torch.cat([p.detach().reshape(-1) for p in net.parameters()]).cpu()


def test_partitioner_shards_match_reference():
    assert D.DataPartitioner(list(range(6000)), [1.0 / 3] * 3).partitions == G["shards_6000_w3"].tolist()
    head = [p[:256] for p in D.DataPartitioner(range(60000), [0.5, 0.5]).partitions]
    assert head == G["shards_60000_w2_head"].tolist()


def test_seeded_init_and_eval_forward_match_reference():
    torch.manual_seed(1234)
    net = b2.Net().eval()
    assert torch.equal(_flat(net), torch.from_numpy(G["init"]))
    with torch.no_grad():
        out = net(torch.from_numpy(G["x"][0]))
    assert torch.allclose(out, torch.from_numpy(G["eval_logp"]), atol=1e-5)


def test_sgd_steps_match_reference_cpu():
    torch.manual_seed(1234)
    net = b2.Net().eval()                            # dropout off, as the stored trajectory
    opt = b2.FlatSGD(net, lr=0.01, momentum=0.5)
    losses = []
    for x, y in zip(torch.from_numpy(G["x"]), torch.from_numpy(G["y"])):
        opt.zero_grad()
        loss = F.nll_loss(net(x), y)
        loss.backward()
        opt.step()
        losses.append(float(loss.detach()))
    assert losses == pytest.approx(G["losses"].tolist(), rel=1e-5)
    assert torch.allclose(_flat(net), torch.from_numpy(G["final"]), atol=1e-6)


@pytest.mark.gpu
@pytest.mark.timeout(600)
def test_fused_trainer_steps_match_reference():
    from dist_tuto.pth_b200.ops.convnet_fused import FusedTrainer, unpack_params
    dev = torch.device("cuda", 0)
    tr = FusedTrainer(G["x"].shape[1], lr=0.01, momentum=0.5, seed=1234, device=dev, p_drop=0.0)
    for x, y in zip(torch.from_numpy(G["x"]), torch.from_numpy(G["y"])):
        tr.step(x.pin_memory(), y.pin_memory())
    got = tr.pop_loss_sum()
    assert abs(got - float(G["losses"].sum())) < 1e-4 * float(G["losses"].sum())
    views = unpack_params(tr.params)
    flat = torch.cat([views[n].reshape(-1).cpu() for n, _ in b2.Net().named_parameters()])
    assert torch.allclose(flat, torch.from_numpy(G["final"]), atol=2e-5, rtol=1e-4)
