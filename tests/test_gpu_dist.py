"""GPU side of the row-sharded training path (SURVEY.md §8(e)): the K2b `row_offset` form on one GPU (shards emulated
back to back), and -- when the box has >= 2 GPUs -- a real 2-rank NCCL step against the unsharded CUDA model."""
import os
import socket

import pytest
import torch
import torch.nn.functional as F

from conftest import ROOT

pytestmark = pytest.mark.gpu
DEV = "cuda"


def test_sharded_k2_forward_backward_equals_unsharded():
    from sngnn_b200 import synth, graph as G, functional as SF
    n, c, k, thr = 6000, 32, 10, 0.0
    ei = synth.make_graph(n, 70000, seed=4, symmetric=True, hub_offset=3.0).to(DEV)
    g = G.prepare(ei, n, True)
    torch.manual_seed(1)
    h = torch.randn(n, c, device=DEV)
    w = torch.randn(n, c, device=DEV)
    h0 = h.clone().requires_grad_(True)
    out_ref = SF.edge_topk_agg(h0, g, k, thr)
    (out_ref * w).sum().backward()
    h1 = h.clone().requires_grad_(True)
    outs = []
    for lo, hi in ((0, 2500), (2500, 2501), (2501, 6000)):              # three ragged shards, one after the other
        outs.append(SF.ShardedEdgeTopkAgg.apply(h1, g.row_slice(lo, hi), lo, k, thr))
    out = torch.cat(outs)
    (out * w).sum().backward()                                           # h1.grad = sum of the shards' contributions
    assert torch.equal(out, out_ref)
    scale = h0.grad.abs().max()
    assert ((h1.grad - h0.grad).abs().max() / scale) < 1e-5              # FP32 atomics: order differs between the two runs


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _worker(rank, ws, port, kind, ret):
    import sys
    sys.path.insert(0, ROOT)
    import torch.distributed as dist
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=ws, device_id=dev)
    from sngnn_b200 import dist as D, synth
    import sngnn_b200.models as M
    n, fd, hid, ncls, k, thr = 5001, 24, 32, 5, 6, 0.1
    x = synth.make_features(n, fd, "clustered", seed=1).to(dev)
    ei = synth.make_graph(n, 50000, seed=2, symmetric=True, hub_offset=3.0).to(dev)
    y = synth.make_labels(n, ncls, seed=3).to(dev)
    torch.manual_seed(7)
    if kind == "SNGNN_Plus_Plus":
        model = M.SNGNN_Plus_Plus(fd, hid, ncls, n, 2, k, thr, 0.5, 1, 0.0)
    else:
        model = M.SNGNN_Plus(fd, hid, ncls, n, 2, k, thr, 1, 0.0)
    model = model.to(dev).train()
    lo, hi = D.shard_bounds(n, ws, rank)
    logp = D.sharded_forward(model, x[lo:hi].contiguous(), ei, n)
    (F.nll_loss(logp, y[lo:hi], reduction="sum") / n).backward()
    D.allreduce_grads(model.parameters())
    grads = {name: p.grad.clone() for name, p in model.named_parameters()}
    model.zero_grad()
    ref = model(synth.GraphData(x, ei))                                    # unsharded CUDA model, same parameters
    F.nll_loss(ref, y).backward()
    torch.testing.assert_close(logp.detach(), ref.detach()[lo:hi], rtol=1e-5, atol=2e-6)
    for name, p in model.named_parameters():
        err = (grads[name] - p.grad).abs().max() / (p.grad.abs().max() + 1e-12)
        assert err < 1e-4, (kind, name, float(err))
    ret[rank] = True
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
@pytest.mark.parametrize("kind", ["SNGNN_Plus_Plus", "SNGNN_Plus"])
def test_two_rank_nccl_training_step_equals_unsharded(kind):
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    ret = ctx.Manager().dict()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, 2, port, kind, ret)) for r in range(2)]
    for p in procs:
        p.start()
    for p in procs:
        p.join(300)
        assert p.exitcode == 0, f"worker exited with {p.exitcode}"
    assert dict(ret) == {0: True, 1: True}


@pytest.mark.parametrize("kind", ["SNGNN_Plus_Plus", "SNGNN_Plus", "SNGNN"])
def test_sharded_forward_world1_equals_model(kind):
    """sharded_forward with a single rank (no process group) runs the sharded code path -- the fused ++ shard kernel, the
    scatter backward, the row-block gradient assembly -- on one GPU; it must reproduce model(data) and its gradients."""
    from sngnn_b200 import dist as D, synth
    import sngnn_b200.models as M
    n, fd, hid, ncls, k, thr = 4001, 24, 32, 5, 6, 0.1
    x = synth.make_features(n, fd, "clustered", seed=1).to(DEV)
    ei = synth.make_graph(n, 40000, seed=2, symmetric=True, hub_offset=3.0).to(DEV)
    y = synth.make_labels(n, ncls, seed=3).to(DEV)
    torch.manual_seed(7)
    if kind == "SNGNN_Plus_Plus":
        model = M.SNGNN_Plus_Plus(fd, hid, ncls, n, 2, k, thr, 0.5, 1, 0.0)
    elif kind == "SNGNN_Plus":
        model = M.SNGNN_Plus(fd, hid, ncls, n, 2, k, thr, 1, 0.0)
    else:
        model = M.SNGNN(fd, hid, ncls, 2)
        model.dropout = torch.nn.Dropout(0.0)
    model = model.to(DEV).train()
    logp = D.sharded_forward(model, x, ei, n)
    F.nll_loss(logp, y).backward()
    grads = {name: p.grad.clone() for name, p in model.named_parameters()}
    model.zero_grad()
    ref = model(synth.GraphData(x, ei))
    F.nll_loss(ref, y).backward()
    torch.testing.assert_close(logp.detach(), ref.detach(), rtol=1e-5, atol=2e-6)
    for name, p in model.named_parameters():
        err = (grads[name] - p.grad).abs().max() / (p.grad.abs().max() + 1e-12)
        assert err < 2e-5, (kind, name, float(err))
