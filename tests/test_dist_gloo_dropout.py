"""gloo tests (CPU) of the counter-based dropout on row shards (dist.RowDropout, sharded_forward(dropout=...)) and of the row-sharded
epoch loop (train.train_sharded).  The numpy oracle (oracle/dropout_ref.py) stands in for the two dropout kernels, FP64 CPU
stand-ins for the aggregation / ++ fusion / BatchNorm kernels: what is under test is that every rank draws the masks of the
GLOBAL rows, the gradient bookkeeping, and that the epoch statistics and the stopping decision are the same on every rank and
equal to world 1's."""
import os
import types

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp
import torch.nn.functional as F

from conftest import ROOT
from test_dist_gloo_bn import BN_OPS, _free_port

SEED, CALL0, P = 0x9E3779B97F4A7C15, 5, 0.5


def _do_fwd(z, row_offset, seed, call, p, relu):
    from oracle import dropout_ref as R
    return torch.from_numpy(R.forward(z.detach().numpy(), row_offset, seed, call, p, relu))


def _do_bwd(z, g, row_offset, seed, call, p, relu):
    from oracle import dropout_ref as R
    return torch.from_numpy(R.backward(None if z is None else z.detach().numpy(), g.detach().numpy(), row_offset, seed, call, p, relu))


DO_OPS = types.SimpleNamespace(row_dropout_fwd=_do_fwd, row_dropout_bwd=_do_bwd)


def _problem(n, fd=10, ncls=3):
    from sngnn_b200 import synth
    x = synth.make_features(n, fd, "clustered", seed=1).double()
    ei = synth.make_graph(n, 5 * n, seed=2, hub_offset=2.0)
    y = synth.make_labels(n, ncls, seed=3)
    return x, ei, y


def _model(kind, n, bn, fd=10, hid=8, ncls=3, k=3, layers=3):
    import sngnn_b200.models as M
    torch.manual_seed(7)                                          # same replicated parameters on every rank
    if kind == "SNGNN":
        model = M.SNGNN(fd, hid, ncls, layers, bn=bn)
    elif kind == "SNGNN_Plus":
        model = M.SNGNN_Plus(fd, hid, ncls, n, layers, k, 0.0, 1, P, bn=bn)
    else:
        model = M.SNGNN_Plus_Plus(fd, hid, ncls, n, layers, k, 0.0, 0.5, 1, P, bn=bn)
    model.dropout = torch.nn.Dropout(P)
    return model.double()


def _stand_ins(kind, ei, n):
    from oracle import sn_ref
    pe = sn_ref.process_edges(ei, n, kind != "SNGNN")

    def agg(h_all, shard, row_offset, top_k, th):
        return sn_ref.sn_aggregate(h_all, pe, top_k, th)[row_offset:row_offset + shard.n]

    def fuse(out1, w_w, w_b, beta, bias, shard, nn_, lo_):
        out0 = sn_ref.structural_term(pe, w_w, w_b, nn_)[lo_:lo_ + out1.size(0)]
        out0 = F.pad(out0, (0, out1.size(1) - out0.size(1)))
        out = beta * out0 + (1 - beta) * out1
        return out if bias is None else out + F.pad(bias, (0, out1.size(1) - bias.numel()))
    return agg, fuse


def _reference(kind, sd, x, ei, k, layers, bn):
    """Unsharded FP64 forward: relu [-> batch norm over all rows] -> the global masks of call CALL0 + l, scaled by 1 / (1 - p)."""
    from oracle import dropout_ref as R, sn_ref
    params = sn_ref.params_from_state_dict(sd, layers)
    n = x.size(0)
    for l, p in enumerate(params):
        if kind == "SNGNN":
            x = sn_ref.snconv(x, ei, p["lin_w"], p["lin_b"], p.get("bias"))
        elif kind == "SNGNN_Plus":
            x = sn_ref.snconv_plus(x, ei, p["lin_w"], p["lin_b"], k, 0.0, True, p.get("bias"))
        else:
            x = sn_ref.snconv_plus_plus(x, ei, p["lin_w"], p["lin_b"], p["w_w"], p["w_b"], p["beta"], k, 0.0, True, p.get("bias"))
        if l < len(params) - 1:
            x = F.relu(x)
            if bn:
                x = F.batch_norm(x, None, None, sd[f"bns.{l}.weight"], sd[f"bns.{l}.bias"], True, 0.1, 1e-5)
            keep = torch.from_numpy(R.keep_mask(n, x.size(1), 0, SEED, CALL0 + l, P))
            x = torch.where(keep, x / (1 - P), torch.zeros_like(x))
    return F.log_softmax(x, dim=1)


def _forward_case(kind, bn, n, ws, rank):
    from sngnn_b200 import dist as D
    k, layers = 3, 3
    x, ei, y = _problem(n)
    model = _model(kind, n, bn, k=k, layers=layers).train()
    if bn:
        for b in model.bns:
            b.weight.data.uniform_(0.5, 1.5)
            b.bias.data.uniform_(-0.5, 0.5)
    sd = {kk: v.detach().clone().requires_grad_(v.is_floating_point() and "running" not in kk) for kk, v in model.state_dict().items()}
    lo, hi = D.shard_bounds(n, ws, rank)
    agg, fuse = _stand_ins(kind, ei, n)
    rd = D.RowDropout(SEED, ops=DO_OPS)
    rd.calls = CALL0
    logp = D.sharded_forward(model, x[lo:hi].clone(), ei, n, agg=agg, fuse=fuse, bn_ops=BN_OPS if bn else None, dropout=rd)
    assert rd.calls == CALL0 + layers - 1                          # one call per dropout site, on every rank
    ref = _reference(kind, sd, x, ei, k, layers, bn)
    assert torch.allclose(logp.detach(), ref.detach()[lo:hi], rtol=1e-9, atol=1e-11), (kind, bn)
    (F.nll_loss(logp, y[lo:hi], reduction="sum") / n).backward()
    D.allreduce_grads(model.parameters())
    F.nll_loss(ref, y).backward()
    for name, p in model.named_parameters():
        g_ref = sd[name].grad
        assert p.grad is not None and torch.allclose(p.grad, g_ref, rtol=1e-8, atol=1e-11), (kind, bn, name, (p.grad - g_ref).abs().max())
    return torch.cat([p.grad.reshape(-1) for p in model.parameters()])


FORWARD_CASES = [("SNGNN", False), ("SNGNN_Plus", False), ("SNGNN_Plus_Plus", False), ("SNGNN_Plus", True), ("SNGNN_Plus_Plus", True)]
LOOP_CFG = dict(epochs=6, patience=2, log_every=1, lr=0.05, weight_decay=5e-4)


def _loss(out, y, mask):
    return F.nll_loss(out[mask], y[mask])


def _run_loop(n, ws, rank, log=None):
    """train.train_sharded with the stand-ins: SNGNN_Plus_Plus, dropout 0.5, the trainer's 48/32/20 split."""
    from sngnn_b200 import dist as D, synth, train as T
    x, ei, y = _problem(n)
    data = synth.GraphData(x, ei, y)
    data.train_mask, data.val_mask, data.test_mask = T.make_splits(n, 0, "cpu")
    model = _model("SNGNN_Plus_Plus", n, False)
    agg, fuse = _stand_ins("SNGNN_Plus_Plus", ei, n)
    sd = T.ShardedData(data, n, *D.shard_bounds(n, ws, rank))
    opt = torch.optim.Adam(model.parameters(), lr=LOOP_CFG["lr"], weight_decay=LOOP_CFG["weight_decay"])
    final, hist = T.train_sharded(model, sd, opt, LOOP_CFG, log, dropout=D.RowDropout(SEED, ops=DO_OPS), agg=agg, fuse=fuse,
                                  loss_fn=_loss)
    return final, hist, torch.cat([p.detach().reshape(-1) for p in model.parameters()])


def _worker(rank, ws, port, n, ret):
    import sys
    sys.path.insert(0, ROOT)
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=ws)
    for kind, bn in FORWARD_CASES:
        state = _forward_case(kind, bn, n, ws, rank)
        every = [torch.empty_like(state) for _ in range(ws)]
        dist.all_gather(every, state)
        assert all(torch.equal(e, state) for e in every), (kind, bn, "gradients differ across ranks")
    final, hist, params = _run_loop(n, ws, rank)
    every = [torch.empty_like(params) for _ in range(ws)]
    dist.all_gather(every, params)
    assert all(torch.equal(e, params) for e in every), "parameters differ across ranks after the epoch loop"
    ret[rank] = (final, hist)
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.parametrize("ws,n", [(2, 41), (3, 4)])
def test_row_dropout_on_shards_and_the_sharded_epoch_loop(ws, n):
    """sharded_forward with RowDropout at p = 0.5 (the three models, and BatchNorm) equals the unsharded FP64 forward / backward
    under the same global masks; the epoch loop gives every rank the same history and stop epoch, equal to world 1's.
    (3, 4): the last rank owns no rows (and some ranks no training rows) and still joins every collective."""
    final1, hist1, _ = _run_loop(n, 1, 0)                          # world 1: no process group
    ctx = mp.get_context("spawn")
    ret = ctx.Manager().dict()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, ws, port, n, ret)) for r in range(ws)]
    for p in procs:
        p.start()
    for p in procs:
        p.join(300)
        assert p.exitcode == 0, f"worker exited with {p.exitcode}"
    assert sorted(ret.keys()) == list(range(ws))
    assert all(ret[r] == ret[0] for r in range(ws))               # the same floats on every rank
    final, hist = ret[0]
    assert len(hist) == len(hist1) and final == final1
    for a, b in zip(hist, hist1):
        assert a == pytest.approx(b, rel=1e-9, abs=1e-12)


def test_row_dropout_counter():
    """The call index advances once per dropout site of a training forward with p > 0, never in eval mode or at p = 0."""
    from sngnn_b200 import dist as D
    n = 30
    x, ei, _ = _problem(n)
    agg, fuse = _stand_ins("SNGNN_Plus", ei, n)
    rd = D.RowDropout(-1, ops=DO_OPS)
    assert rd.seed == 2**64 - 1 and rd.calls == 0
    z = torch.randn(4, 6, dtype=torch.float64)
    assert torch.equal(rd(z, 0, P, training=False, relu=True), z.clamp_min(0)) and rd.calls == 0
    assert rd(z, 0, 0.0) is z and rd.calls == 0
    a, b = rd(z, 0, P), rd(z, 0, P)
    assert rd.calls == 2 and not torch.equal(a, b)                  # a fresh mask per call
    model = _model("SNGNN_Plus", n, False, layers=4)
    for training, p, step in ((True, P, 3), (False, P, 0), (True, 0.0, 0)):
        model.train(training)
        model.dropout.p = p
        before = rd.calls
        D.sharded_forward(model, x, ei, n, agg=agg, fuse=fuse, dropout=rd)
        assert rd.calls == before + step, (training, p)
    model.train()
    model.dropout.p = 0.0                                           # inactive RowDropout == the default path
    assert torch.equal(D.sharded_forward(model, x, ei, n, agg=agg, fuse=fuse, dropout=rd), D.sharded_forward(model, x, ei, n, agg=agg, fuse=fuse))
