"""GPU side of BatchNorm on row shards (sng_bn_*: fused ReLU + BatchNorm statistics / apply, forward and backward) and of
top_k <= 0 in the sharded step: the kernels against an FP64 autograd reference, shards emulated back to back on one GPU,
world-1 sharded_forward against model(data) and the golden BatchNorm run, and -- with >= 2 GPUs -- a 2-rank NCCL step."""
import copy
import os
import socket

import pytest
import torch
import torch.nn.functional as F

from conftest import ROOT, load_golden, golden_inputs, golden_grad

pytestmark = pytest.mark.gpu
DEV = "cuda"
EPS = 1e-5


def _inputs(n, c, ld, seed):
    g = torch.Generator().manual_seed(seed)
    zbuf = torch.randn(n, ld, generator=g) + torch.linspace(-1, 1, c).repeat(1, ld // c + 1)[:, :ld]   # mixed-sign channels
    zbuf[:, c:] = float("nan")                                      # columns beyond c must never be read
    gamma, beta = torch.rand(c, generator=g) + 0.5, torch.randn(c, generator=g)
    gy = torch.randn(n, c, generator=g)
    return zbuf.to(DEV)[:, :c], gamma.to(DEV), beta.to(DEV), gy.to(DEV)


def _rel(a, b, scale=None):
    scale = b.double().abs().max() if scale is None else scale
    return float((a.double() - b.double()).abs().max() / (scale + 1e-30))


@pytest.mark.parametrize("n,c,ld", [(2, 3, 3), (1000, 4, 8), (4097, 8, 12), (100003, 32, 36), (30000, 100, 128), (5000, 512, 516),
                                    (77777, 32, 32)])
def test_bn_kernels_match_fp64_autograd(n, c, ld):
    from sngnn_b200 import functional as SF
    z, gamma, beta, gy = _inputs(n, c, ld, n + c)
    assert z.stride(0) == ld
    sums = SF.bn_fwd_stats(z)
    y, mean, rstd = SF.bn_fwd_apply(z, sums, n, EPS, gamma, beta)
    bsums = SF.bn_bwd_stats(z, gy, mean, rstd)
    dz = SF.bn_bwd_apply(z, gy, bsums, n, gamma, mean, rstd)

    z64 = z.double().requires_grad_(True)
    w64, b64 = gamma.double().requires_grad_(True), beta.double().requires_grad_(True)
    a64 = F.relu(z64)
    y64 = F.batch_norm(a64, None, None, w64, b64, True, 0.0, EPS)
    y64.backward(gy.double())
    mean64, var64 = a64.detach().mean(0), a64.detach().var(0, unbiased=False)
    # dz is a difference of terms of size |gamma rstd g| that cancel almost exactly for tiny n (n = 2: dz is rounding noise)
    dz_scale = (gamma.double() * (var64 + EPS).rsqrt() * gy.double()).abs().max()
    for name, got, ref, scale in (("y", y, y64.detach(), None), ("mean", mean, mean64, None), ("rstd", rstd, (var64 + EPS).rsqrt(), None),
                                  ("dz", dz, z64.grad, dz_scale), ("dgamma", bsums[1], w64.grad, None), ("dbeta", bsums[0], b64.grad, None)):
        assert _rel(got, ref, scale) < 1e-5, (name, _rel(got, ref, scale))


def test_bn_kernels_on_emulated_shards():
    """Ragged shards (one empty) back to back: the local sums add up to the whole's within FP64 rounding; given the same global
    sums, the per-shard outputs concatenate to the whole's bit for bit; repeated calls are bit-identical."""
    from sngnn_b200 import functional as SF
    n, c = 100001, 32
    z, gamma, beta, gy = _inputs(n, c, 40, 5)
    bounds = [(0, 40000), (40000, 40000), (40000, 40001), (40001, n)]
    sums = SF.bn_fwd_stats(z)
    assert torch.equal(sums, SF.bn_fwd_stats(z))
    parts = [SF.bn_fwd_stats(z[lo:hi]) for lo, hi in bounds]
    assert torch.equal(parts[1], torch.zeros_like(parts[1]))                  # an empty shard writes zero sums
    torch.testing.assert_close(sum(parts), sums, rtol=1e-12, atol=1e-9)
    y, mean, rstd = SF.bn_fwd_apply(z, sums, n, EPS, gamma, beta)
    bsums = SF.bn_bwd_stats(z, gy, mean, rstd)
    assert torch.equal(bsums, SF.bn_bwd_stats(z, gy, mean, rstd))
    bparts = [SF.bn_bwd_stats(z[lo:hi], gy[lo:hi], mean, rstd) for lo, hi in bounds]
    assert torch.equal(bparts[1], torch.zeros_like(bparts[1]))
    torch.testing.assert_close(sum(bparts), bsums, rtol=1e-12, atol=1e-9)
    dz = SF.bn_bwd_apply(z, gy, bsums, n, gamma, mean, rstd)
    ys, dzs = [], []
    for lo, hi in bounds:
        ys_, mean_s, rstd_s = SF.bn_fwd_apply(z[lo:hi], sums, n, EPS, gamma, beta)
        assert torch.equal(mean_s, mean) and torch.equal(rstd_s, rstd)
        ys.append(ys_)
        dzs.append(SF.bn_bwd_apply(z[lo:hi], gy[lo:hi], bsums, n, gamma, mean, rstd))
    assert torch.equal(torch.cat(ys), y) and torch.equal(torch.cat(dzs), dz)
    y2, _, _ = SF.bn_fwd_apply(z, sums, n, EPS, gamma, beta)
    assert torch.equal(y2, y) and torch.equal(SF.bn_bwd_apply(z, gy, bsums, n, gamma, mean, rstd), dz)


def _model(kind, fd, hid, ncls, n, k, thr, bn, layers=3):
    import sngnn_b200.models as M
    torch.manual_seed(7)
    if kind == "SNGNN":
        m = M.SNGNN(fd, hid, ncls, layers, bn=bn)
        m.dropout = torch.nn.Dropout(0.0)
    elif kind == "SNGNN_Plus":
        m = M.SNGNN_Plus(fd, hid, ncls, n, layers, k, thr, 1, 0.0, bn=bn)
    else:
        m = M.SNGNN_Plus_Plus(fd, hid, ncls, n, layers, k, thr, 0.5, 1, 0.0, bn=bn)
    if bn:
        for b in m.bns:
            b.weight.data.uniform_(0.5, 1.5)
            b.bias.data.uniform_(-0.5, 0.5)
    return m.to(DEV)


def _data(n=4001, fd=24, ncls=5):
    from sngnn_b200 import synth
    x = synth.make_features(n, fd, "clustered", seed=1).to(DEV)
    ei = synth.make_graph(n, 40000, seed=2, symmetric=True, hub_offset=3.0).to(DEV)
    y = synth.make_labels(n, ncls, seed=3).to(DEV)
    return x, ei, y


def _step(model, x, ei, y, sharded):
    from sngnn_b200 import dist as D, synth
    model.zero_grad()
    out = D.sharded_forward(model, x, ei, x.size(0)) if sharded else model(synth.GraphData(x, ei))
    F.nll_loss(out, y).backward()
    return out


def _compare(model, ref, logp, out):
    torch.testing.assert_close(logp.detach(), out.detach(), rtol=1e-5, atol=2e-6)
    for (name, p), q in zip(model.named_parameters(), ref.parameters()):
        assert p.grad is not None and q.grad is not None, name
        # dL/dbeta is ONE sum over N * C terms that largely cancel: two FP32 paths differ there by summation noise relative to
        # the small result (both are held to 1e-5 against FP64 by the golden run and the gloo test)
        tol = 1e-4 if name.endswith("beta") else 2e-5
        assert _rel(p.grad, q.grad) < tol if q.grad.abs().max() > 0 else p.grad.abs().max() == 0, (name, _rel(p.grad, q.grad))


def _buffers(model):
    return [b for m in model.bns for b in (m.running_mean, m.running_var, m.num_batches_tracked)]


@pytest.mark.parametrize("kind,k", [("SNGNN", 0), ("SNGNN_Plus", 6), ("SNGNN_Plus_Plus", 6), ("SNGNN_Plus", 0), ("SNGNN_Plus_Plus", 0)])
@pytest.mark.parametrize("bn", [True, False])
def test_sharded_forward_world1_matches_model(kind, k, bn):
    """world 1 (no process group): bn=True and top_k = 0 through the sharded path reproduce model(data) -- logits, every
    gradient, the running buffers -- in training and in eval mode (running statistics, backward included)."""
    if not bn and (k > 0 or kind == "SNGNN"):
        pytest.skip("covered by test_gpu_dist.py")
    x, ei, y = _data()
    ref = _model(kind, 24, 32, 5, x.size(0), k, 0.1, bn).train()
    model = copy.deepcopy(ref)
    logp = _step(model, x, ei, y, True)
    out = _step(ref, x, ei, y, False)
    _compare(model, ref, logp, out)
    if k == 0 and kind != "SNGNN":
        assert all(conv.lin.weight.grad.abs().sum() == 0 for conv in model.lins)
    if bn:
        for a, b in zip(_buffers(model), _buffers(ref)):
            torch.testing.assert_close(a, b, rtol=1e-6, atol=1e-6)
        model.eval(); ref.eval()                                    # running statistics, forward and backward
        _compare(model, ref, _step(model, x, ei, y, True), _step(ref, x, ei, y, False))
        for a, b in zip(_buffers(model), _buffers(ref)):
            torch.testing.assert_close(a, b, rtol=1e-6, atol=1e-6)


def test_sharded_forward_world1_is_bit_reproducible():
    x, ei, y = _data()
    m1 = _model("SNGNN_Plus_Plus", 24, 32, 5, x.size(0), 6, 0.1, True).train()
    m2 = copy.deepcopy(m1)
    _step(m1, x, ei, y, True)
    _step(m2, x, ei, y, True)
    for (name, p), q in zip(m1.named_parameters(), m2.parameters()):
        assert torch.equal(p.grad, q.grad), name
    for a, b in zip(_buffers(m1), _buffers(m2)):
        assert torch.equal(a, b)


def test_sharded_forward_world1_golden_batch_norm_run():
    """Run 50 of models_tiny.pt (SNGNN_Plus_Plus, hidden 8, 2 layers, bn=True) through the sharded path: golden logits, loss and
    every gradient."""
    import sngnn_b200.models as M
    from sngnn_b200 import dist as D
    g = load_golden("models_tiny.pt")
    x, ei, y = golden_inputs(g)
    run = g["runs"][50]
    cfg = run["cfg"]
    assert run["kind"] == "SNGNN_Plus_Plus" and cfg["bn"]
    n, fd = x.shape
    m = M.SNGNN_Plus_Plus(fd, cfg["hidden"], int(y.max()) + 1, n, cfg["layers"], cfg["top_k"], cfg["thr"], cfg["beta"], cfg["rsl"], 0.0,
                          bn=True)
    m.load_state_dict(run["state_dict"])
    m = m.to(DEV).train()
    mask = (torch.arange(n) % 2 == 0).to(DEV)
    yd = y.to(DEV)
    out = D.sharded_forward(m, x.to(DEV), ei.to(DEV), n)
    loss = F.nll_loss(out[mask], yd[mask])
    loss.backward()
    torch.testing.assert_close(out.detach().cpu(), run["logp"], rtol=1e-5, atol=2e-6)
    torch.testing.assert_close(loss.detach().cpu(), run["loss"], rtol=1e-5, atol=1e-6)
    for k, p in m.named_parameters():
        got, ref, scale = golden_grad(p.grad.detach().cpu(), run["grads"][k])
        err = (got - ref).abs().max().item() / (scale.item() + 1e-12)
        assert err < 1e-5, (k, err)


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _worker(rank, ws, port, kind, k, ret):
    import sys
    sys.path.insert(0, ROOT)
    import torch.distributed as dist
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=ws, device_id=dev)
    from sngnn_b200 import dist as D, synth
    import sngnn_b200.models as M
    n, fd, hid, ncls, thr = 5001, 24, 32, 5, 0.1
    x = synth.make_features(n, fd, "clustered", seed=1).to(dev)
    ei = synth.make_graph(n, 50000, seed=2, symmetric=True, hub_offset=3.0).to(dev)
    y = synth.make_labels(n, ncls, seed=3).to(dev)
    torch.manual_seed(7)
    if kind == "SNGNN_Plus_Plus":
        model = M.SNGNN_Plus_Plus(fd, hid, ncls, n, 3, k, thr, 0.5, 1, 0.0, bn=True)
    else:
        model = M.SNGNN_Plus(fd, hid, ncls, n, 3, k, thr, 1, 0.0, bn=True)
    model = model.to(dev).train()
    ref = copy.deepcopy(model)
    lo, hi = D.shard_bounds(n, ws, rank)
    logp = D.sharded_forward(model, x[lo:hi].contiguous(), ei, n)
    (F.nll_loss(logp, y[lo:hi], reduction="sum") / n).backward()
    D.allreduce_grads(model.parameters())
    out = ref(synth.GraphData(x, ei))                                      # unsharded CUDA model, same parameters
    F.nll_loss(out, y).backward()
    torch.testing.assert_close(logp.detach(), out.detach()[lo:hi], rtol=1e-5, atol=2e-6)
    for (name, p), q in zip(model.named_parameters(), ref.parameters()):
        err = (p.grad - q.grad).abs().max() / (q.grad.abs().max() + 1e-12)
        assert err < 1e-4, (kind, k, name, float(err))
    bufs = torch.cat([b.double().reshape(-1) for b in _buffers(model)])
    torch.testing.assert_close(bufs, torch.cat([b.double().reshape(-1) for b in _buffers(ref)]), rtol=1e-6, atol=1e-6)
    every = [torch.empty_like(bufs) for _ in range(ws)]
    dist.all_gather(every, bufs)
    assert all(torch.equal(e, bufs) for e in every), "running buffers differ across ranks"
    ret[rank] = True
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
@pytest.mark.parametrize("kind,k", [("SNGNN_Plus_Plus", 6), ("SNGNN_Plus", 6), ("SNGNN_Plus_Plus", 0)])
def test_two_rank_nccl_batch_norm_step_equals_unsharded(kind, k):
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    ret = ctx.Manager().dict()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, 2, port, kind, k, ret)) for r in range(2)]
    for p in procs:
        p.start()
    for p in procs:
        p.join(300)
        assert p.exitcode == 0, f"worker exited with {p.exitcode}"
    assert dict(ret) == {0: True, 1: True}
