"""The all-pairs mode's deterministic backward: the transpose of fixed-width neighbour lists (sng_list_transpose) and the
gather-form list backward (sng_list_bwd, the passes of sng_edge_bwd), on one GPU, on row shards and through
dist.sharded_forward.  Gradients are checked against FP64 autograd of the oracle, repeated runs must be bit-identical,
and a [0, N) shard must reproduce the unsharded backward bit for bit."""
import os
import socket

import pytest
import torch
import torch.nn.functional as F

from conftest import ROOT

pytestmark = pytest.mark.gpu
DEV = "cuda"
N = 1500
HUB = 7                                   # random lists: a column that more than 1,024 rows select


def _rel(a, b):
    return float((a.double() - b.double()).abs().max() / (b.double().abs().max() + 1e-30))


def _random_lists(n, k, seed, dup=True):
    """Lists with duplicates, empty rows, cnt < k, -1 padding and a hub column (the chunked source pass)."""
    gen = torch.Generator().manual_seed(seed)
    idx = torch.randint(0, n, (n, k), generator=gen, dtype=torch.int32)
    cnt = torch.randint(1, k + 1, (n,), generator=gen, dtype=torch.int32)
    cnt[::9] = 0
    cnt[1::4] = k
    if dup and k > 1:
        idx[::3, 1] = idx[::3, 0]
    idx[:, 0] = HUB                                                        # every non-empty row: 1,333 of 1,500
    idx[torch.arange(k)[None, :] >= cnt[:, None]] = -1
    return idx, cnt


def _cosines(h, idx):
    nh = F.normalize(h.double(), dim=-1, eps=1e-12)
    return torch.where(idx >= 0, (nh[:, None, :] * nh[idx.clamp(min=0).long()]).sum(-1), torch.zeros((), dtype=torch.float64, device=h.device))


def _inv_denom(kind, cnt, n):
    if kind == "candidates":
        return torch.full((cnt.numel(),), 1.0 / (n - 1), dtype=torch.float64, device=cnt.device)
    return 1.0 / cnt.clamp(min=1).double()


# ------------------------------------------------------------------------------------------ 1. transpose
@pytest.mark.parametrize("k", [1, 10, 33, 64])
@pytest.mark.parametrize("rows", [(0, N), (400, 1130), (0, 0)])
def test_list_transpose_equals_stable_argsort(k, rows):
    from sngnn_b200 import functional as SF
    lo, hi = rows
    idx, cnt = _random_lists(N, k, seed=k)
    idx, cnt = idx[lo:hi].contiguous(), cnt[lo:hi].contiguous()
    ref = SF.list_transpose(idx, cnt, N)                                    # host branch: stable argsort
    got = SF.list_transpose(idx.to(DEV), cnt.to(DEV), N)
    nnz = int(ref.rowptr_tr[-1])
    assert torch.equal(got.rowptr_tr.cpu(), ref.rowptr_tr)
    assert torch.equal(got.col_tr[:nnz].cpu(), ref.col_tr[:nnz])
    assert torch.equal(got.sel_q.cpu(), ref.sel_q)
    if hi - lo > 1100:
        assert int(ref.rowptr_tr[HUB + 1] - ref.rowptr_tr[HUB]) > 1024


def test_list_transpose_chunk_tables_match_the_host_branch():
    from sngnn_b200 import functional as SF
    idx, cnt = _random_lists(N, 10, seed=5)
    ref = SF.list_transpose(idx, cnt, N, chunk_tables=True)
    got = SF.list_transpose(idx.to(DEV), cnt.to(DEV), N, chunk_tables=True)
    assert ref.chunk_tab.size(0) > 32
    for name in ("chunk_tab", "lrows", "lrow_ptr"):
        assert torch.equal(getattr(got, name).cpu(), getattr(ref, name)), name


# ------------------------------------------------------------------------------------------ 2. single-GPU list backward
def _lists_of(source, h, k, c):
    from sngnn_b200 import simknn
    if source == "knn":
        idx, sim, cnt = simknn.build_knn(h, k, -1.0, True)
        return idx, sim, cnt
    idx, cnt = _random_lists(h.size(0), k, seed=c + k)
    idx, cnt = idx.to(DEV), cnt.to(DEV)
    return idx, _cosines(h, idx).float(), cnt


def _list_backward(h, idx, sim, cnt, inv, w, row_offset=0):
    from sngnn_b200 import functional as SF
    hd = h.clone().requires_grad_(True)
    out = SF.ListAgg.apply(hd, idx, sim, cnt, inv, row_offset)
    (out * w).sum().backward()
    return out.detach(), hd.grad


GRID2 = [(c, k) for c in (4, 32) for k in (5, 10, 33, 64)] + [(c, k) for c in (128, 256, 512) for k in (10, 64)]


@pytest.mark.parametrize("c,k", GRID2)
@pytest.mark.parametrize("source", ["knn", "random"])
@pytest.mark.parametrize("denominator", ["candidates", "selected"])
def test_list_backward_vs_fp64_autograd(c, k, source, denominator):
    from oracle import sn_ref
    torch.manual_seed(c * 100 + k)
    h = torch.randn(N, c, device=DEV)
    w = torch.randn(N, c, device=DEV)
    idx, sim, cnt = _lists_of(source, h, k, c)
    inv = _inv_denom(denominator, cnt, N)
    out, dh = _list_backward(h, idx, sim, cnt, inv.float(), w)
    out2, dh2 = _list_backward(h, idx, sim, cnt, inv.float(), w)
    assert torch.equal(out, out2) and torch.equal(dh, dh2)
    h64 = h.double().cpu().requires_grad_(True)                           # the oracle runs on the host, in FP64
    idx64 = idx.long().cpu()
    n64 = F.normalize(h64, dim=-1, eps=1e-12)
    s64 = torch.where(idx64 >= 0, (n64[:, None, :] * n64[idx64.clamp(min=0)]).sum(-1), torch.zeros((), dtype=torch.float64))
    ref = sn_ref.knn_mean_aggregate(h64, idx64, s64, cnt.long().cpu(), (1.0 / inv).cpu())
    (ref * w.double().cpu()).sum().backward()
    assert _rel(out.cpu(), ref.detach()) < 1e-5
    assert _rel(dh.cpu(), h64.grad) < 1e-5, _rel(dh.cpu(), h64.grad)


# ------------------------------------------------------------------------------------------ 3. row shards
@pytest.mark.parametrize("c", [4, 32, 128])
@pytest.mark.parametrize("denominator", ["candidates", "selected"])
def test_list_shards_reproduce_and_add_up(c, denominator):
    from sngnn_b200 import simknn
    torch.manual_seed(c)
    h = torch.randn(N, c, device=DEV)
    w = torch.randn(N, c, device=DEV)

    def run(rows):
        hd = h.clone().requires_grad_(True)
        out = simknn.allpairs_topk_agg(hd, 10, 0.0, True, denominator, rows=rows)
        lo = 0 if rows is None else rows[0]
        (out * w[lo:lo + out.size(0)]).sum().backward()
        return out.detach(), hd.grad

    out_full, dh_full = run(None)
    out_0n, dh_0n = run((0, N))
    assert torch.equal(out_0n, out_full) and torch.equal(dh_0n, dh_full)
    bounds = [(0, 0), (0, 1), (1, 700), (700, 700), (700, N)]
    parts = [run(b) for b in bounds]
    again = [run(b) for b in bounds]
    for (o, d), (o2, d2) in zip(parts, again):
        assert torch.equal(o, o2) and torch.equal(d, d2)
    assert parts[0][0].size(0) == 0 and not parts[0][1].any()
    assert torch.equal(torch.cat([o for o, _ in parts]), out_full)
    total = sum(d for _, d in parts)
    assert _rel(total, dh_full) < 1e-5


# ------------------------------------------------------------------------------------------ 4. model, world 1
def _model(kind, n, fd, hid, ncls, denominator):
    import sngnn_b200.models as M
    torch.manual_seed(7)
    if kind == "SNGNN_Plus_Plus":
        return M.SNGNN_Plus_Plus(fd, hid, ncls, n, 2, 6, 0.1, 0.5, 1, 0.0, candidates="all_pairs", denominator=denominator)
    return M.SNGNN_Plus(fd, hid, ncls, n, 2, 6, 0.1, 1, 0.0, candidates="all_pairs", denominator=denominator)


def _sharded_step(model, x_local, ei, n, y_local, scale):
    from sngnn_b200 import dist as D, functional as SF
    model.zero_grad()
    logp = D.sharded_forward(model, x_local, ei, n)
    (SF.nll_loss(logp, y_local) * scale).backward()
    D.allreduce_grads(model.parameters())
    return logp.detach(), {name: p.grad.clone() for name, p in model.named_parameters()}


@pytest.mark.parametrize("kind", ["SNGNN_Plus", "SNGNN_Plus_Plus"])
@pytest.mark.parametrize("symmetric", [True, False])
@pytest.mark.parametrize("denominator", ["candidates", "selected"])
@pytest.mark.parametrize("hid", [32, 256])
def test_sharded_forward_world1_all_pairs(kind, symmetric, denominator, hid):
    from sngnn_b200 import functional as SF, synth
    n, fd, ncls = 3001, 24, 5
    x = synth.make_features(n, fd, "clustered", seed=1).to(DEV)
    ei = synth.make_graph(n, 30000, seed=2, symmetric=symmetric, hub_offset=3.0).to(DEV)
    y = synth.make_labels(n, ncls, seed=3).to(DEV)
    model = _model(kind, n, fd, hid, ncls, denominator).to(DEV).train()
    logp, g1 = _sharded_step(model, x, ei, n, y, 1.0)
    _, g2 = _sharded_step(model, x, ei, n, y, 1.0)
    for name in g1:
        assert torch.equal(g1[name], g2[name]), name
    model.zero_grad()
    ref = model(synth.GraphData(x, ei))
    SF.nll_loss(ref, y).backward()
    assert torch.equal(logp, ref.detach())
    for name, p in model.named_parameters():
        err = (g1[name] - p.grad).abs().max() / (p.grad.abs().max() + 1e-12)
        assert err < 2e-5, (name, float(err))


# ------------------------------------------------------------------------------------------ 5. two-rank NCCL
def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _worker(rank, ws, port, kind, denominator, ret):
    import sys
    sys.path.insert(0, ROOT)
    import torch.distributed as dist
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=ws, device_id=dev)
    from sngnn_b200 import dist as D, synth
    n, fd, hid, ncls = 4001, 24, 32, 5
    x = synth.make_features(n, fd, "clustered", seed=1).to(dev)
    ei = synth.make_graph(n, 40000, seed=2, symmetric=True, hub_offset=3.0).to(dev)
    y = synth.make_labels(n, ncls, seed=3).to(dev)
    model = _model(kind, n, fd, hid, ncls, denominator).to(dev).train()
    lo, hi = D.shard_bounds(n, ws, rank)
    _, g1 = _sharded_step(model, x[lo:hi].contiguous(), ei, n, y[lo:hi], (hi - lo) / n)
    _, g2 = _sharded_step(model, x[lo:hi].contiguous(), ei, n, y[lo:hi], (hi - lo) / n)
    for name in g1:
        assert torch.equal(g1[name], g2[name]), (kind, name)
    model.zero_grad()
    F.nll_loss(model(synth.GraphData(x, ei)), y).backward()               # unsharded model, same parameters
    for name, p in model.named_parameters():
        err = (g1[name] - p.grad).abs().max() / (p.grad.abs().max() + 1e-12)
        assert err < 1e-4, (kind, name, float(err))
    ret[rank] = True
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
@pytest.mark.parametrize("kind,denominator", [("SNGNN_Plus_Plus", "candidates"), ("SNGNN_Plus", "selected")])
def test_two_rank_nccl_all_pairs_gradients_repeat(kind, denominator):
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    ret = ctx.Manager().dict()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, 2, port, kind, denominator, ret)) for r in range(2)]
    for p in procs:
        p.start()
    for p in procs:
        p.join(300)
        assert p.exitcode == 0, f"worker exited with {p.exitcode}"
    assert dict(ret) == {0: True, 1: True}
