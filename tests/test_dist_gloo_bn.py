"""gloo tests (CPU) of BatchNorm and top_k <= 0 in the row-sharded training step (sngnn_b200/dist.py): FP64 CPU stand-ins
replace the four BatchNorm launch helpers and the aggregation / ++ fusion kernels, so what is under test is the partitioning,
the all-reduce of the statistics, the running buffers and the gradient bookkeeping -- against the unsharded oracle."""
import os
import socket
import types

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp
import torch.nn.functional as F

from conftest import ROOT


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _bn_fwd_stats(z):
    a = z.clamp_min(0)
    return torch.stack([a.sum(0), (a * a).sum(0)]).double()


def _bn_fwd_apply(z, sums, n_total, eps, gamma, beta, mean=None, rstd=None):
    if sums is not None:
        mean = sums[0] / n_total
        rstd = (sums[1] / n_total - mean * mean).clamp_min(0).add(eps).rsqrt()
    return (z.clamp_min(0) - mean) * rstd * gamma + beta, mean, rstd


def _bn_bwd_stats(z, g, mean, rstd):
    ahat = (z.clamp_min(0) - mean) * rstd
    return torch.stack([g.sum(0), (g * ahat).sum(0)]).double()


def _bn_bwd_apply(z, g, sums, n_total, gamma, mean, rstd):
    ahat = (z.clamp_min(0) - mean) * rstd
    if sums is not None:
        g = g - sums[0] / n_total - ahat * sums[1] / n_total
    return torch.where(z > 0, gamma * rstd * g, torch.zeros_like(g))


BN_OPS = types.SimpleNamespace(bn_fwd_stats=_bn_fwd_stats, bn_fwd_apply=_bn_fwd_apply, bn_bwd_stats=_bn_bwd_stats, bn_bwd_apply=_bn_bwd_apply)


def _make_model(kind, fd, hid, ncls, n, k, thr, bn, layers=3):
    import sngnn_b200.models as M
    if kind == "SNGNN":
        model = M.SNGNN(fd, hid, ncls, layers, bn=bn)
        model.dropout = torch.nn.Dropout(0.0)
    elif kind == "SNGNN_Plus":
        model = M.SNGNN_Plus(fd, hid, ncls, n, layers, k, thr, 1, 0.0, bn=bn)
    else:
        model = M.SNGNN_Plus_Plus(fd, hid, ncls, n, layers, k, thr, 0.5, 1, 0.0, bn=bn)
    return model.double()


def _case(kind, k, n, ws, rank, training, momentum):
    """One sharded step, in training or in eval mode (the running statistics, forward and backward), against the oracle; returns
    the running buffers and the gradients for the cross-rank comparison."""
    from sngnn_b200 import dist as D, synth
    from oracle import sn_ref
    fd, hid, ncls, thr, layers = 10, 8, 3, 0.0, 3
    x = synth.make_features(n, fd, "clustered", seed=1).double()
    ei = synth.make_graph(n, 5 * n, seed=2, hub_offset=2.0)
    y = synth.make_labels(n, ncls, seed=3)
    torch.manual_seed(7)                                          # same replicated parameters on every rank
    model = _make_model(kind, fd, hid, ncls, n, k, thr, True, layers)
    for bn in model.bns:                                          # non-trivial affine parameters and running buffers
        bn.momentum = momentum
        bn.weight.data.uniform_(0.5, 1.5)
        bn.bias.data.uniform_(-0.5, 0.5)
        bn.running_mean.uniform_(-1, 1)
        bn.running_var.uniform_(0.5, 2)
        bn.num_batches_tracked.fill_(3)
    model.train(training)
    sd0 = {kk: v.detach().clone() for kk, v in model.state_dict().items()}
    lo, hi = D.shard_bounds(n, ws, rank)
    rsl = kind != "SNGNN"
    pe = sn_ref.process_edges(ei, n, rsl)

    def agg(h_all, shard, row_offset, top_k, th):
        return sn_ref.sn_aggregate(h_all, pe, top_k, th)[row_offset:row_offset + shard.n]

    def fuse(out1, w_w, w_b, beta, bias, shard, nn_, lo_):
        out0 = sn_ref.structural_term(pe, w_w, w_b, nn_)[lo_:lo_ + out1.size(0)]
        out0 = F.pad(out0, (0, out1.size(1) - out0.size(1)))
        out = beta * out0 + (1 - beta) * out1
        return out if bias is None else out + F.pad(bias, (0, out1.size(1) - bias.numel()))

    logp = D.sharded_forward(model, x[lo:hi].clone(), ei, n, agg=agg, fuse=fuse, bn_ops=BN_OPS)
    sd = {kk: v.clone().requires_grad_(v.is_floating_point() and "running" not in kk) for kk, v in sd0.items()}
    bns = []
    for l in range(layers - 1):
        rm, rv = sd[f"bns.{l}.running_mean"], sd[f"bns.{l}.running_var"]
        mom = 1.0 / 4 if momentum is None else momentum          # num_batches_tracked 3 -> 4: the cumulative average
        bns.append(lambda t, l=l, rm=rm, rv=rv, mom=mom: F.batch_norm(t, rm, rv, sd[f"bns.{l}.weight"], sd[f"bns.{l}.bias"], training, mom, 1e-5))
    ref = sn_ref.stack_forward(kind, sn_ref.params_from_state_dict(sd, layers), x, ei, top_k=k, thr=thr, remove_self_loops=rsl, bns=bns)
    assert torch.allclose(logp.detach(), ref.detach()[lo:hi], rtol=1e-9, atol=1e-11), (kind, k, training)
    bufs = []
    for l, bn in enumerate(model.bns):
        assert torch.allclose(bn.running_mean, sd[f"bns.{l}.running_mean"], rtol=1e-12, atol=1e-14)
        assert torch.allclose(bn.running_var, sd[f"bns.{l}.running_var"], rtol=1e-12, atol=1e-14)
        assert int(bn.num_batches_tracked) == (4 if training else 3)
        bufs += [bn.running_mean, bn.running_var, bn.num_batches_tracked.double().reshape(1)]
    loss = F.nll_loss(logp, y[lo:hi], reduction="sum") / n
    loss.backward()
    D.allreduce_grads(model.parameters())
    F.nll_loss(ref, y).backward()
    for name, p in model.named_parameters():
        g_ref = sd[name].grad
        assert p.grad is not None and torch.allclose(p.grad, g_ref, rtol=1e-8, atol=1e-11), (kind, k, name, (p.grad - g_ref).abs().max())
    if k <= 0:                                                    # out_1 = 0: lin gets a zero, not a missing, gradient
        assert all(conv.lin.weight.grad.abs().sum() == 0 for conv in model.lins)
    grads = torch.cat([p.grad.reshape(-1) for p in model.parameters()])
    return torch.cat(bufs + [grads])


CASES = [("SNGNN", 2, True, 0.1), ("SNGNN_Plus", 3, True, 0.1), ("SNGNN_Plus_Plus", 3, True, None),
         ("SNGNN_Plus", 0, True, 0.1), ("SNGNN_Plus_Plus", 0, True, 0.1), ("SNGNN_Plus_Plus", 3, False, 0.1)]


def _worker(rank, ws, port, n, ret):
    import sys
    sys.path.insert(0, ROOT)
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=ws)
    for i, (kind, k, training, momentum) in enumerate(CASES):
        state = _case(kind, k, n, ws, rank, training, momentum)
        every = [torch.empty_like(state) for _ in range(ws)]
        dist.all_gather(every, state)
        assert all(torch.equal(e, state) for e in every), (kind, k, training, "buffers / gradients differ across ranks")
    ret[rank] = True
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.parametrize("ws,n", [(2, 41), (3, 4)])
def test_sharded_batch_norm_and_top_k_zero_match_unsharded_oracle(ws, n):
    """BatchNorm (training with momentum 0.1 and None, and eval mode, each with its backward) and top_k = 0 in the sharded step of the three models: rows,
    every gradient after allreduce_grads (gamma / beta counted once) and the running buffers equal the oracle's, identically
    on every rank.  (3, 4): shard_bounds gives the last rank no rows, and it still joins every all-reduce."""
    from sngnn_b200 import dist as D
    assert D.shard_bounds(n, ws, ws - 1)[1] - D.shard_bounds(n, ws, ws - 1)[0] == (0 if ws == 3 else 20)
    ctx = mp.get_context("spawn")
    ret = ctx.Manager().dict()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, ws, port, n, ret)) for r in range(ws)]
    for p in procs:
        p.start()
    for p in procs:
        p.join(300)
        assert p.exitcode == 0, f"worker exited with {p.exitcode}"
    assert dict(ret) == {r: True for r in range(ws)}


def test_sharded_batch_norm_rejections_come_before_any_kernel():
    from sngnn_b200 import dist as D
    n = 20
    ei = torch.stack([torch.arange(n), torch.arange(n).roll(1)])
    model = _make_model("SNGNN_Plus", 8, 4, 3, 1, 2, 0.0, True).train()
    with pytest.raises(ValueError, match="Expected more than 1 value per channel when training"):
        D.sharded_forward(model, torch.randn(1, 8, dtype=torch.float64), ei[:, :0], 1, bn_ops=BN_OPS)
    model = _make_model("SNGNN_Plus", 8, 4, 3, n, 2, 0.0, True)
    model.bns[0] = torch.nn.BatchNorm1d(4, affine=False).double()
    with pytest.raises(NotImplementedError, match="affine=True and track_running_stats=True"):
        D.sharded_forward(model, torch.randn(n, 8, dtype=torch.float64), ei, n, bn_ops=BN_OPS)
    model = _make_model("SNGNN_Plus", 8, 4, 3, n, 2, 0.0, True)
    model.bns[1] = torch.nn.BatchNorm1d(4, track_running_stats=False).double()
    with pytest.raises(NotImplementedError, match="affine=True and track_running_stats=True"):
        D.sharded_forward(model, torch.randn(n, 8, dtype=torch.float64), ei, n, bn_ops=BN_OPS)
