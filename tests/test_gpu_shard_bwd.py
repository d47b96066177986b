"""Deterministic backward of row shards: sng_edge_bwd in its row-shard form, through the shard's own transpose index.
One shard [0, n) must reproduce the whole graph's backward bit for bit; ragged shards (an empty one included) must add up
to it within FP32 reordering and repeat bit for bit; sharded training steps must repeat bit for bit."""
import os
import socket

import pytest
import torch

from conftest import ROOT

pytestmark = pytest.mark.gpu
DEV = "cuda"
N = 3000


def _hub_graph(seed, symmetric, shift=0):
    """make_graph + forced target rows with in-degree > 1024 and in (32, 1024]; shift > 0 drops every edge from a source
    below it (sources are then shifted by min(src) = shift, which needs the self loops removed)."""
    from sngnn_b200 import synth
    ei = synth.make_graph(N, 12 * N, seed=seed, symmetric=symmetric, hub_offset=3.0)
    gen = torch.Generator().manual_seed(seed)
    extra = []
    for hnode, d in ((shift + 3, 1500), (shift + 17, 200)):
        src = torch.randperm(N, generator=gen)[:d]
        src = src[src != hnode]
        extra.append(torch.stack([src, torch.full_like(src, hnode)]))
    ex = torch.cat(extra, 1)
    if symmetric:
        ex = torch.cat([ex, ex.flip(0)], 1)
    ei = torch.cat([ei, ex, torch.tensor([[shift], [0]])], 1)
    ei = ei[:, ei[0] >= shift]
    key = torch.unique(ei[0] * N + ei[1])
    return torch.stack([key // N, key % N]).to(DEV)


def _prepared(seed=11, symmetric=True, shift=0):
    from sngnn_b200 import graph as G
    g = G.prepare(_hub_graph(seed, symmetric, shift), N, True)
    deg = (g.rowptr_in[1:] - g.rowptr_in[:-1]).cpu()
    assert bool(((deg > 32) & (deg <= 1024)).any()) and bool((deg > 1024).any()) and g.src_shift == shift
    return g


def _data(c, seed=1):
    torch.manual_seed(seed)
    return torch.randn(N, c, device=DEV), torch.randn(N, c, device=DEV)


GRID = [(4, 10, 0.0), (4, 0, None), (32, 10, 0.0), (32, 0, None), (64, 10, 0.0), (128, 6, -1.0), (128, 0, None), (256, 10, 0.0)]


@pytest.mark.parametrize("c,k,thr", GRID)
def test_whole_range_shard_reproduces_edge_agg_backward(c, k, thr):
    from sngnn_b200 import functional as SF
    g = _prepared()
    h, w = _data(c)
    h0 = h.clone().requires_grad_(True)
    out0 = SF.edge_topk_agg(h0, g, k, thr)
    (out0 * w).sum().backward()
    h1 = h.clone().requires_grad_(True)
    out1 = SF.ShardedEdgeTopkAgg.apply(h1, g.row_slice(0, N), 0, k, thr)
    (out1 * w).sum().backward()
    assert torch.equal(out1, out0)
    assert torch.equal(h1.grad, h0.grad)


def _shard_grads(g, h, w, k, thr, bounds):
    """Each shard's contribution to dL/dh, one shard after the other on this GPU."""
    from sngnn_b200 import functional as SF
    parts = []
    for lo, hi in bounds:
        hs = h.clone().requires_grad_(True)
        (SF.ShardedEdgeTopkAgg.apply(hs, g.row_slice(lo, hi), lo, k, thr) * w[lo:hi]).sum().backward()
        parts.append(hs.grad)
    return parts


BOUNDS = ((0, 1200), (1200, 1200), (1200, 1201), (1201, N))          # ragged, an empty shard and a 1-row shard


@pytest.mark.parametrize("c,k,thr", GRID)
@pytest.mark.parametrize("shift", [0, 5])
def test_ragged_shards_add_up_and_repeat(c, k, thr, shift):
    from sngnn_b200 import functional as SF
    g = _prepared(symmetric=shift == 0, shift=shift)
    h, w = _data(c)
    h0 = h.clone().requires_grad_(True)
    (SF.edge_topk_agg(h0, g, k, thr) * w).sum().backward()
    p1 = _shard_grads(g, h, w, k, thr, BOUNDS)
    p2 = _shard_grads(g, h, w, k, thr, BOUNDS)
    for a, b in zip(p1, p2):
        assert torch.equal(a, b)
    assert int(p1[1].abs().max()) == 0                                   # the empty shard contributes zero
    total = p1[0]
    for p in p1[1:]:
        total = total + p
    assert float((total - h0.grad).abs().max() / h0.grad.abs().max()) < 1e-5


def _fused_operands(c):
    torch.manual_seed(5)
    return (torch.randn(N, c, device=DEV) * 0.1, torch.randn(c, device=DEV), torch.full((1,), 0.3, device=DEV), None)


def _fused_shard_bwd(g, h, gg, k, thr, fuse, bounds):
    """(dh contributions, dbeta parts) of the fused SNGNN++ pass on each shard: sng_edge_fwd with the fused epilogue on the
    shard's rows, then sng_edge_bwd in its row-shard form with beta / diff (what dist._ShardedFusedAgg runs)."""
    from sngnn_b200 import functional as SF
    dhs, dbs = [], []
    for lo, hi in bounds:
        s = g.row_slice(lo, hi)
        _, ss, sw, sq, sc, inv, diff = SF._edge_fwd(h, s, lo, k, thr, True, fuse, want_q=True)
        dh, dwt, db = SF.edge_bwd(h, inv, gg[lo:hi].contiguous(), s, k, ss, sw, sq, sc, fuse[2], diff, row_offset=lo)
        assert dwt is None
        dhs.append(dh)
        dbs.append(db)
    return dhs, dbs


@pytest.mark.parametrize("c", [4, 32, 128])
def test_fused_shard_backward_repeats_and_matches_unsharded(c):
    from sngnn_b200 import functional as SF
    g = _prepared()
    assert g.symmetric
    h, gg = _data(c)
    k, thr = 10, 0.0
    fuse = _fused_operands(c)
    _, ss, sw, sq, sc, inv, diff = SF._edge_fwd(h, g, 0, k, thr, True, fuse, want_q=True)
    dh_ref, _, db_ref = SF.edge_bwd(h, inv, gg, g, k, ss, sw, sq, sc, fuse[2], diff)
    d1, b1 = _fused_shard_bwd(g, h, gg, k, thr, fuse, BOUNDS)
    d2, b2 = _fused_shard_bwd(g, h, gg, k, thr, fuse, BOUNDS)
    for a, b in zip(d1 + b1, d2 + b2):
        assert torch.equal(a, b)
    dh = d1[0] + d1[1] + d1[2] + d1[3]
    db = b1[0] + b1[1] + b1[2] + b1[3]
    assert float((dh - dh_ref).abs().max() / dh_ref.abs().max()) < 1e-5
    assert float((db - db_ref).abs()) <= 1e-5 * float((diff * gg).abs().sum())      # condition-aware: dbeta is a long sum


def _model(kind, n, fd, hid, ncls, k, thr):
    import sngnn_b200.models as M
    torch.manual_seed(7)
    if kind == "SNGNN_Plus_Plus":
        return M.SNGNN_Plus_Plus(fd, hid, ncls, n, 2, k, thr, 0.5, 1, 0.0)
    if kind == "SNGNN_Plus":
        return M.SNGNN_Plus(fd, hid, ncls, n, 2, k, thr, 1, 0.0)
    model = M.SNGNN(fd, hid, ncls, 2)
    model.dropout = torch.nn.Dropout(0.0)
    return model


def _sharded_step(model, x_local, ei, n, y_local, scale):
    from sngnn_b200 import dist as D, functional as SF
    model.zero_grad()
    logp = D.sharded_forward(model, x_local, ei, n)
    (SF.nll_loss(logp, y_local) * scale).backward()
    D.allreduce_grads(model.parameters())
    return {name: p.grad.clone() for name, p in model.named_parameters()}


@pytest.mark.parametrize("kind", ["SNGNN_Plus_Plus", "SNGNN_Plus", "SNGNN"])
def test_sharded_forward_world1_gradients_repeat(kind):
    from sngnn_b200 import synth
    n, fd, hid, ncls, k, thr = 4001, 24, 32, 5, 6, 0.1
    x = synth.make_features(n, fd, "clustered", seed=1).to(DEV)
    ei = synth.make_graph(n, 40000, seed=2, symmetric=True, hub_offset=3.0).to(DEV)
    y = synth.make_labels(n, ncls, seed=3).to(DEV)
    model = _model(kind, n, fd, hid, ncls, k, thr).to(DEV).train()
    g1 = _sharded_step(model, x, ei, n, y, 1.0)
    g2 = _sharded_step(model, x, ei, n, y, 1.0)
    for name in g1:
        assert torch.equal(g1[name], g2[name]), name


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
    import torch.nn.functional as F
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=ws, device_id=dev)
    from sngnn_b200 import dist as D, synth
    n, fd, hid, ncls, k, thr = 5001, 24, 32, 5, 6, 0.1
    x = synth.make_features(n, fd, "clustered", seed=1).to(dev)
    ei = synth.make_graph(n, 50000, seed=2, symmetric=True, hub_offset=3.0).to(dev)
    y = synth.make_labels(n, ncls, seed=3).to(dev)
    model = _model(kind, n, fd, hid, ncls, k, thr).to(dev).train()
    lo, hi = D.shard_bounds(n, ws, rank)
    g1 = _sharded_step(model, x[lo:hi].contiguous(), ei, n, y[lo:hi], (hi - lo) / n)
    g2 = _sharded_step(model, x[lo:hi].contiguous(), ei, n, y[lo:hi], (hi - lo) / n)
    for name in g1:
        assert torch.equal(g1[name], g2[name]), (kind, name)
    model.zero_grad()
    F.nll_loss(model(synth.GraphData(x, ei)), y).backward()               # unsharded CUDA model, same parameters
    for name, p in model.named_parameters():
        err = (g1[name] - p.grad).abs().max() / (p.grad.abs().max() + 1e-12)
        assert err < 1e-4, (kind, name, float(err))
    ret[rank] = True
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
@pytest.mark.parametrize("kind", ["SNGNN_Plus_Plus", "SNGNN_Plus"])
def test_two_rank_nccl_gradients_repeat(kind):
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
