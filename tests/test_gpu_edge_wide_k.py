"""top_k > SNG_MAX_TOPK (64) on the edge path: the per-edge form (sng_edge_fwd_wide / sng_edge_bwd_wide).

The selection rule is the oracle's (oracle.sn_ref.edge_select): S_i = {e : s_e >= thr and rank_i(e) < K}, ranks by (s desc,
position asc).  The kernels save it as one flag per in-edge; rows with more than K in-edges are cut once by a radix select.
Every comparison has the suite's two halves: (a) the selected set against the rule wherever the FP64 scores are further than
BAND from thr and from the row's K-th score, (b) values and gradients GIVEN the kernel's selection against FP64 (outputs rtol
1e-5 / atol 1e-6, 2e-6 fused; gradients 1e-5 of their largest magnitude).  The rows are those of the boundary graph of
test_gpu_edge_boundaries: in-degrees 0, <= 32, 33..1024 and > 1024, so every K below 1,057 cuts some rows and K >= max_deg
none."""
import copy
import os
import socket

import pytest
import torch
import torch.nn.functional as F

from conftest import ROOT
from test_gpu_edge_boundaries import N_BOUNDARY, _device_graph, _features, _rel

DEV = "cuda"
WIDTHS = (4, 32, 128, 512)                 # narrow register kernel, staged + chunk kernels, long-row + hub kernels (two widths)
BIG = 1 << 40                              # beyond int32: any K at or above the largest in-degree
KS = (65, 100, 1000, BIG)
THRS = (-1.0, 0.5)
BAND = 1e-6
ATOL = {False: 1e-6, True: 2e-6}


def _csr(g):
    """(src, dst) of the CSR by target on the host, in-edge position order inside each row."""
    rp = g.rowptr_in.cpu().long()
    dst = torch.repeat_interleave(torch.arange(g.n), rp[1:] - rp[:-1])
    return g.col_in.cpu().long(), dst


def _scores64(h64, src, dst):
    nrm = F.normalize(h64, dim=-1, eps=1e-12)
    return (nrm[dst] * nrm[src]).sum(-1)


def _structural(n, cp, seed):
    """(wt [N, Cp], w.bias, beta, bias) as autograd leaves on the device; w.weight = wt.t()."""
    gen = torch.Generator().manual_seed(seed)
    wt = (torch.randn(n, cp, generator=gen) * 0.1).to(DEV).requires_grad_(True)
    rest = [t.to(DEV).requires_grad_(True) for t in (torch.randn(cp, generator=gen), torch.full((1,), 0.3), torch.randn(cp, generator=gen))]
    return [wt] + rest


def _ref_out(h64, src, dst, flags, denominator, st64=None):
    """FP64 layer output given the selection `flags` (bool per CSR edge): where(flags, s, 0) through the mean, blended like
    SNGNN++ when st64 = (wt, w.bias, beta, bias) is given (in-lists = out-lists: out_0[i] = sum of wt over i's sources)."""
    n = h64.size(0)
    s = _scores64(h64, src, dst)
    w = torch.where(flags, s, torch.zeros_like(s))
    tot = torch.zeros_like(h64).index_add(0, dst, w[:, None] * h64[src])
    if denominator == "candidates":
        den = torch.zeros(n, dtype=h64.dtype).index_add(0, dst, torch.ones_like(s))
    else:
        den = torch.zeros(n, dtype=h64.dtype).index_add(0, dst, flags.to(h64.dtype))
    out1 = tot / den.clamp(min=1)[:, None]
    if st64 is None:
        return out1
    wt, wb, beta, bias = st64
    out0 = torch.zeros_like(h64).index_add(0, dst, wt[src]) + wb
    return beta * out0 + (1 - beta) * out1 + bias


def _check_selection(flags, s64, dst, n, k, thr):
    """(a): every edge where the kernel and the rule disagree lies within BAND of thr or of its row's K-th score; and
    |S_i| = min(K, #{s >= thr}) in every row without a score within BAND of thr."""
    from oracle import sn_ref
    ref = sn_ref.edge_select(s64, dst, k, thr)
    for e in (flags != ref).nonzero().flatten().tolist():
        r = int(dst[e])
        row = s64[dst == r].sort(descending=True).values
        kth = row[min(k, row.numel()) - 1]
        assert abs(float(s64[e]) - thr) < BAND or abs(float(s64[e] - kth)) < BAND, (r, e, float(s64[e]), float(kth))
    cnt = torch.zeros(n, dtype=torch.long).index_add(0, dst, flags.long())
    ncand = torch.zeros(n, dtype=torch.long).index_add(0, dst, (s64 >= thr).long())
    near = torch.zeros(n, dtype=torch.long).index_add(0, dst, ((s64 - thr).abs() < BAND).long())
    ok = near == 0
    assert torch.equal(cnt[ok], ncand[ok].clamp(max=k))
    return cnt


# ------------------------------------------------------------------------------------------ 1. forward
@pytest.mark.gpu
@pytest.mark.parametrize("denominator", ["candidates", "selected"])
@pytest.mark.parametrize("form", ["plain", "fused"])
@pytest.mark.parametrize("cp", WIDTHS)
def test_forward_selection_and_values(cp, form, denominator):
    """Training and inference outputs are bit-identical; the flags follow the rule (FP64 band); |S_i| = min(K, #candidates);
    values given the flags match FP64; denominator='selected' writes the factor it applied."""
    from sngnn_b200 import functional as SF
    _, _, g = _device_graph(True)
    n = N_BOUNDARY
    h = _features(n, cp, 21).to(DEV)
    h64 = h.double().cpu()
    src, dst = _csr(g)
    s64 = _scores64(h64, src, dst)
    deg = torch.bincount(dst, minlength=n)
    fuse = st64 = None
    if form == "fused":
        wt, wb, beta, bias = _structural(n, cp, 5)
        fuse = SF._structural_operands(wt.t(), wb, beta, bias, cp)
        st64 = tuple(t.detach().double().cpu() for t in (wt, wb, beta, bias))
    assert g.max_deg == 1057
    for k in KS:
        for thr in THRS:
            inv_denom = torch.empty(n, device=DEV) if denominator == "selected" else None
            out_t, flags, _, diff = SF._edge_fwd_wide(h, g, 0, k, thr, True, fuse, denominator=denominator, inv_denom=inv_denom)
            out_i, flags_i, _, _ = SF._edge_fwd_wide(h, g, 0, k, thr, False, fuse, denominator=denominator)
            assert torch.equal(out_t, out_i), (k, thr)
            f = flags[:g.num_edges].cpu().bool()
            kk = min(k, g.max_deg)
            assert (flags_i is None) == (kk >= g.max_deg)
            if flags_i is not None:                                    # inference keeps the flags of the cut rows
                cut = deg[dst] > kk
                assert torch.equal(flags_i[:g.num_edges].cpu().bool()[cut], f[cut])
            cnt = _check_selection(f, s64, dst, n, kk, thr)
            if inv_denom is not None:
                assert torch.equal(inv_denom.cpu(), 1.0 / cnt.clamp(min=1).float())
            ref = _ref_out(h64, src, dst, f, denominator, st64)
            torch.testing.assert_close(out_t.double().cpu(), ref, rtol=1e-5, atol=ATOL[fuse is not None])
            assert (diff is None) == (fuse is None)


def _tie_graph(cp):
    """Three hub rows whose K-th rank falls inside a block of exact ties: target 0 with 9,000 in-edges (more than the cut
    kernel's shared-memory stage), 1 with 300, 2 with 1,500.  Each takes `hi` edges from distinct sources scoring 0.82..0.98,
    `tie` duplicate edges from node 50 (the same score, bit for bit), the rest from sources scoring 0.1..0.32, in a shuffled
    edge order.  With K = 100 the rule selects the `hi` edges and the 100 - hi LOWEST positions among the ties."""
    n = 12000
    e0 = torch.zeros(cp)
    e0[0] = 1.0
    e1 = torch.zeros(cp)
    e1[1] = 1.0
    h = torch.zeros(n, cp)
    h[0:3] = e0
    h[50] = e0 + 2.0 * e1                                                  # score 1/sqrt(5)
    hi_nodes = torch.arange(100, 200)
    h[hi_nodes] = e0 + (0.2 + 0.5 * torch.arange(100.0) / 100)[:, None] * e1
    lo_nodes = torch.arange(1000, n)
    h[lo_nodes] = e0 + (3.0 + 7.0 * torch.arange(float(lo_nodes.numel())) / lo_nodes.numel())[:, None] * e1
    gen = torch.Generator().manual_seed(3)
    edges = []
    for t, deg, hi, tie in ((0, 9000, 60, 200), (1, 300, 90, 30), (2, 1500, 80, 100)):
        srcs = torch.cat([hi_nodes[:hi], torch.full((tie,), 50), lo_nodes[torch.randperm(lo_nodes.numel(), generator=gen)[:deg - hi - tie]]])
        srcs = srcs[torch.randperm(deg, generator=gen)]
        edges.append(torch.stack([srcs, torch.full_like(srcs, t)]))
    return h, torch.cat(edges, 1)


@pytest.mark.gpu
@pytest.mark.parametrize("cp", [4, 32, 128])
def test_exact_ties_at_the_cut_take_the_lowest_positions(cp):
    from sngnn_b200 import functional as SF, graph as G
    from oracle import sn_ref
    h, ei = _tie_graph(cp)
    n = h.size(0)
    eid = ei.to(DEV)
    g = G.prepare(eid, n, True)
    src, dst = _csr(g)
    s64 = _scores64(h.double(), src, dst)
    for thr in (-1.0, 0.4):
        out, flags, _, _ = SF._edge_fwd_wide(h.to(DEV), g, 0, 100, thr, True)
        f = flags[:g.num_edges].cpu().bool()
        assert torch.equal(f, sn_ref.edge_select(s64, dst, 100, thr))
        for t, hi in ((0, 60), (1, 90), (2, 80)):
            row = dst == t
            ties = (src == 50) & row
            taken = f & ties
            assert int(taken.sum()) == 100 - hi
            assert int(taken.nonzero().max()) < int((ties & ~taken).nonzero().min())          # the lowest positions
        torch.testing.assert_close(out.double().cpu(), _ref_out(h.double(), src, dst, f, "candidates"), rtol=1e-5, atol=1e-6)


# ------------------------------------------------------------------------------------------ 2. backward
def _fp64_grads(h, src, dst, f, denominator, gout, st=None):
    """FP64 autograd given the flags: the gradients of h (and of wt, w.bias, beta, bias) and sum |gout * out|, the magnitude
    that bounds the error of dL/dbeta (a signed sum of N * C terms)."""
    h64 = h.detach().double().cpu().requires_grad_(True)
    st64 = None if st is None else [t.detach().double().cpu().requires_grad_(True) for t in st]
    out = _ref_out(h64, src, dst, f, denominator, st64)
    g64 = gout.double().cpu()
    (out * g64).sum().backward()
    return [h64.grad] + ([] if st is None else [t.grad for t in st64]), float((g64 * out.detach()).abs().sum())


def _run(h, g, k, thr, st, denominator, gout):
    from sngnn_b200 import functional as SF
    leaves = [h] + ([] if st is None else st)
    for t in leaves:
        t.grad = None
    wt, wb, beta, bias = st if st is not None else (None, None, None, None)
    out = SF.EdgeWideAgg.apply(h, g, 0, k, thr, None if wt is None else wt.t(), wb, beta, bias, None, denominator)
    (out * gout).sum().backward()
    return out.detach(), [t.grad.clone() for t in leaves]


@pytest.mark.gpu
@pytest.mark.parametrize("denominator", ["candidates", "selected"])
@pytest.mark.parametrize("form", ["plain", "fused"])
@pytest.mark.parametrize("cp", WIDTHS)
def test_backward_given_the_selection_vs_fp64(cp, form, denominator):
    """Gradients of h (and, fused, of W^T, w.bias, beta, bias) match FP64 autograd given the forward's flags at 1e-5; a
    second run is bit-identical."""
    from sngnn_b200 import functional as SF
    _, _, g = _device_graph(True)
    n = N_BOUNDARY
    src, dst = _csr(g)
    h = _features(n, cp, 31).to(DEV).requires_grad_(True)
    st = _structural(n, cp, 9) if form == "fused" else None
    gout = torch.randn(n, cp, generator=torch.Generator().manual_seed(4)).to(DEV)
    for k, thr in ((100, 0.5), (1000, -1.0)):
        flags = SF._edge_fwd_wide(h.detach(), g, 0, k, thr, True)[1]
        f = flags[:g.num_edges].cpu().bool()
        out, grads = _run(h, g, k, thr, st, denominator, gout)
        out2, grads2 = _run(h, g, k, thr, st, denominator, gout)
        assert torch.equal(out, out2) and all(torch.equal(a, b) for a, b in zip(grads, grads2))
        ref, mag = _fp64_grads(h, src, dst, f, denominator, gout, st)
        for name, a, b in zip(("h", "wt", "w.bias", "beta", "bias"), grads, ref):
            scale = float(b.abs().max()) + 1e-12
            if name == "beta":             # a signed sum of N * C terms: bounded by their magnitudes, not by the total
                scale = max(scale, 1e-2 * mag)
            err = float((a.cpu().double() - b).abs().max()) / scale
            assert err < 1e-5, (k, thr, name, err)


@pytest.mark.gpu
@pytest.mark.parametrize("cp", [8, 32, 128])
@pytest.mark.parametrize("k", [65, 100])
def test_selected_edge_with_zero_score_carries_its_gradient(cp, k):
    """Row 0 has 70 in-edges: 35 sources orthogonal to it (s = 0 exactly, selected at thr = 0) and 35 at s = 0.707.  K = 100
    selects all 70 in place; K = 65 cuts the row inside the zero scores (the 30 lowest positions).  Either way the zero-score
    edges carry dL/ds_e into dL/dh_0, which FP64 autograd given the flags confirms."""
    from sngnn_b200 import functional as SF, graph as G
    from oracle import sn_ref
    n = 80
    h = torch.zeros(n, cp)
    h[0, 0] = 1.0
    h[1:36, 1] = 1.0 + torch.arange(35.0) / 35                           # orthogonal to row 0
    h[36:71, 0] = 1.0
    h[36:71, 2] = 1.0
    h[71:] = torch.randn(n - 71, cp, generator=torch.Generator().manual_seed(2))
    perm = torch.randperm(70, generator=torch.Generator().manual_seed(5))
    ei = torch.stack([torch.arange(1, 71)[perm], torch.zeros(70, dtype=torch.long)])
    g = G.prepare(ei.to(DEV), n, True)
    src, dst = _csr(g)
    s64 = _scores64(h.double(), src, dst)
    hd = h.to(DEV).requires_grad_(True)
    gout = torch.randn(n, cp, generator=torch.Generator().manual_seed(6)).to(DEV)
    flags = SF._edge_fwd_wide(hd.detach(), g, 0, k, 0.0, True)[1]
    f = flags[:g.num_edges].cpu().bool()
    assert torch.equal(f, sn_ref.edge_select(s64, dst, k, 0.0))
    zero = (s64 == 0) & f
    assert int(zero.sum()) == (35 if k == 100 else 30)
    _, (dh,) = _run(hd, g, k, 0.0, None, "candidates", gout)
    (ref,), _ = _fp64_grads(hd, src, dst, f, "candidates", gout)
    assert _rel(dh, ref) < 1e-5
    assert float(ref[0, 1].abs()) > 1e-3                                   # the zero-score edges' direction reaches dh_0


# ------------------------------------------------------------------------------------------ 3. row shards
SHARDS = ((0, 1200), (1200, 1200), (1200, 1201), (1201, 3000))      # ragged, an empty shard and a 1-row shard


@pytest.mark.gpu
@pytest.mark.parametrize("cp,k,thr", [(4, 100, 0.5), (32, 65, -1.0), (128, 1000, 0.5), (512, 100, -1.0)])
def test_row_shards(cp, k, thr):
    """A [0, N) shard reproduces the unsharded forward and backward bit for bit; ragged shards (an empty and a 1-row one
    among them) give the same rows bit for bit and contributions to dL/dh that add up to it."""
    from sngnn_b200 import functional as SF
    _, _, g = _device_graph(False)
    n = N_BOUNDARY
    h = _features(n, cp, 41).to(DEV).requires_grad_(True)
    gout = torch.randn(n, cp, generator=torch.Generator().manual_seed(8)).to(DEV)

    out = SF.edge_agg(h, g, k, thr)
    (out * gout).sum().backward()
    dh = h.grad.clone()
    h.grad = None
    out0 = SF.sharded_edge_agg(h, g.row_slice(0, n), 0, k, thr)
    (out0 * gout).sum().backward()
    assert torch.equal(out0, out) and torch.equal(h.grad, dh)
    rows, acc = [], torch.zeros_like(dh)
    for lo, hi in SHARDS:
        h.grad = None
        o = SF.sharded_edge_agg(h, g.row_slice(lo, hi), lo, k, thr)
        assert o.size(0) == hi - lo
        (o * gout[lo:hi]).sum().backward()
        rows.append(o.detach())
        acc += h.grad
    assert torch.equal(torch.cat(rows), out.detach())
    assert _rel(acc, dh) < 1e-5                                             # the shards' sums add in another order


# ------------------------------------------------------------------------------------------ 4. models, sharded training, trainer
def _model_data(symmetric, n=3000):
    from sngnn_b200 import synth
    x = synth.make_features(n, 48, "clustered", seed=1)
    ei = synth.make_graph(n, 40000, seed=2, symmetric=symmetric, hub_offset=3.0)
    y = synth.make_labels(n, 5, seed=3)
    return x, ei, y


@pytest.mark.gpu
@pytest.mark.parametrize("kind,symmetric", [("SNGNN_Plus", True), ("SNGNN_Plus", False), ("SNGNN_Plus_Plus", True),
                                            ("SNGNN_Plus_Plus", False)])
def test_models_vs_oracle_and_in_eval(kind, symmetric):
    """Both models at K = 100 (rows with up to several hundred in-edges are cut) against oracle.sn_ref.stack_forward, outputs
    and parameter gradients; under no_grad in eval mode (dropout 0) the output is the training output bit for bit."""
    import sngnn_b200.models as M
    from sngnn_b200 import graph as G, synth
    from oracle import sn_ref
    x, ei, y = _model_data(symmetric)
    n, k, thr = x.size(0), 100, 0.2
    torch.manual_seed(0)
    if kind == "SNGNN_Plus":
        model = M.SNGNN_Plus(48, 32, 5, n, 2, k, thr, 1, 0.0)
    else:
        model = M.SNGNN_Plus_Plus(48, 32, 5, n, 2, k, thr, 0.5, 1, 0.0)
    model = model.to(DEV).train()
    data = synth.GraphData(x, ei).to(DEV)
    assert G.prepare(data.edge_index, n, True).max_deg > k
    out = model(data)
    F.nll_loss(out, y.to(DEV)).backward()
    sd = {kk: v.detach().cpu().clone().requires_grad_(v.is_floating_point()) for kk, v in model.state_dict().items()}
    ref = sn_ref.stack_forward(kind, sn_ref.params_from_state_dict(sd, 2), x, ei, top_k=k, thr=thr, remove_self_loops=True)
    F.nll_loss(ref, y).backward()
    torch.testing.assert_close(out.detach().cpu(), ref.detach(), rtol=1e-5, atol=2e-6)
    for name, p in model.named_parameters():
        assert _rel(p.grad, sd[name].grad) < 1e-5, (name, _rel(p.grad, sd[name].grad))
    model.eval()
    with torch.no_grad():
        assert torch.equal(model(data), out.detach())


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["SNGNN_Plus", "SNGNN_Plus_Plus"])
def test_sharded_forward_world1_matches_model(kind):
    """world 1 (no process group): sharded_forward at K = 100 -- the per-edge form through edge_agg_sharded and, for SNGNN++ on
    a symmetric graph, the fused shard pass -- reproduces model(data), logits and every gradient, in training and in eval."""
    from test_gpu_shard_bn import _compare, _data, _model, _step
    x, ei, y = _data()
    ref = _model(kind, 24, 32, 5, x.size(0), 100, 0.1, False).train()
    model = copy.deepcopy(ref)
    _compare(model, ref, _step(model, x, ei, y, True), _step(ref, x, ei, y, False))
    model.eval()
    ref.eval()
    _compare(model, ref, _step(model, x, ei, y, True), _step(ref, x, ei, y, False))


@pytest.mark.gpu
def test_trainer_at_top_k_100_lowers_the_loss():
    from sngnn_b200 import train as T
    _, hist = T.main(["--dataset", "small", "--model", "SNGNN_Plus_Plus", "--top_k", "100", "--thr", "0.0", "--epochs", "15",
                      "--patience", "100", "--log-every", "0"], log=lambda *a: None)
    assert len(hist) == 15 and hist[-1][0] < hist[0][0]


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
    n, fd, hid, ncls, k, thr = 5001, 24, 32, 5, 100, 0.1
    x = synth.make_features(n, fd, "clustered", seed=1).to(dev)
    ei = synth.make_graph(n, 50000, seed=2, symmetric=True, hub_offset=3.0).to(dev)
    y = synth.make_labels(n, ncls, seed=3).to(dev)
    torch.manual_seed(7)
    if kind == "SNGNN_Plus_Plus":
        model = M.SNGNN_Plus_Plus(fd, hid, ncls, n, 2, k, thr, 0.5, 1, 0.0)
    else:
        model = M.SNGNN_Plus(fd, hid, ncls, n, 2, k, thr, 1, 0.0)
    model = model.to(dev).train()
    ref = copy.deepcopy(model)
    lo, hi = D.shard_bounds(n, ws, rank)
    logp = D.sharded_forward(model, x[lo:hi].contiguous(), ei, n)
    (F.nll_loss(logp, y[lo:hi], reduction="sum") / n).backward()
    D.allreduce_grads(model.parameters())
    out = ref(synth.GraphData(x, ei))
    F.nll_loss(out, y).backward()
    torch.testing.assert_close(logp.detach(), out.detach()[lo:hi], rtol=1e-5, atol=2e-6)
    for (name, p), q in zip(model.named_parameters(), ref.parameters()):
        err = (p.grad - q.grad).abs().max() / (q.grad.abs().max() + 1e-12)
        assert err < 1e-4, (kind, name, float(err))
    ret[rank] = True
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.gpu
@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
@pytest.mark.parametrize("kind", ["SNGNN_Plus", "SNGNN_Plus_Plus"])
def test_two_rank_nccl_step_equals_unsharded(kind):
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    ret = ctx.Manager().dict()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, 2, port, kind, ret)) for r in range(2)]
    for p in procs:
        p.start()
    for p in procs:
        p.join(300)
        if p.exitcode is None:
            p.terminate()
            p.join()
        assert p.exitcode == 0, f"worker exited with {p.exitcode}"
    assert dict(ret) == {0: True, 1: True}
