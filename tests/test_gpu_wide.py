"""Layers wider than 128 channels (up to SNG_MAX_CHANNELS = 512): the edge kernels hold such a row in a whole warp, several
float4 slots per lane.  CPU tests check the limit itself; GPU tests check every wide path against the FP64 oracle:
aggregation and selection, the fused SNGNN++ pass and the K4 path, bit-reproducible backward, row shards, all-pairs lists,
whole models and the trainer."""
import os
import re

import pytest
import torch
import torch.nn.functional as F

from conftest import ROOT
from parity import compare_lists

DEV = "cuda"
gpu = pytest.mark.gpu


# ------------------------------------------------------------------------------------------------ CPU
def test_max_channels_matches_the_header():
    from sngnn_b200 import _C
    with open(os.path.join(ROOT, "include", "sng.h")) as f:
        m = re.search(r"#define\s+SNG_MAX_CHANNELS\s+(\d+)", f.read())
    assert m and int(m.group(1)) == _C.MAX_CHANNELS == 512


@pytest.mark.parametrize("width", [509, 512])
def test_wide_layers_build(width):
    import sngnn_b200.models as M
    conv = M.SNConv_plus_plus(12, width, 10)
    assert conv.lin.out_features == width and conv.w.weight.shape == (width, 10)
    m = M.SNGNN_Plus_Plus(12, width, 3, 10, 2)
    assert m.lins[0].lin.out_features == width and m.lins[1].lin.in_features == width
    assert M.SNGNN_Plus(12, width, 3, 10, 2).lins[0].lin.out_features == width
    assert M.SNGNN(12, width, 3, 2).lins[0].lin.out_features == width


def test_layers_above_the_limit_are_rejected():
    import sngnn_b200.models as M
    with pytest.raises(ValueError, match="512"):
        M.SNConv_plus_plus(12, 513, 10)
    with pytest.raises(ValueError, match="512"):
        M.SNGNN_Plus_Plus(12, 513, 3, 10, 2)
    with pytest.raises(ValueError, match="512"):
        M.SNGNN(12, 513, 3, 2)


# ------------------------------------------------------------------------------------------------ GPU
def _hub_graph(n, e, seed, symmetric, hubs=(3, 17), hub_deg=(1500, 200)):
    """make_graph + forced rows with in-degree > 1024 (hub kernel) and in (32, 1024] (long-row kernel)."""
    from sngnn_b200 import synth
    ei = synth.make_graph(n, e, seed=seed, symmetric=symmetric, hub_offset=3.0)
    g = torch.Generator().manual_seed(seed)
    extra = []
    for hnode, d in zip(hubs, hub_deg):
        src = torch.randperm(n, generator=g)[:d]
        src = src[src != hnode]
        extra.append(torch.stack([src, torch.full_like(src, hnode)]))
    ex = torch.cat(extra, 1)
    if symmetric:
        ex = torch.cat([ex, ex.flip(0)], 1)
    ei = torch.cat([ei, ex], 1)
    key = torch.unique(ei[0] * n + ei[1])
    return torch.stack([key // n, key % n])


def _prepared(ei, n, rsl=True):
    from sngnn_b200 import graph as G
    g = G.prepare(ei.to(DEV), n, rsl)
    deg = (g.rowptr_in[1:] - g.rowptr_in[:-1]).cpu()
    assert bool(((deg > 32) & (deg <= 1024)).any()) and bool((deg > 1024).any())   # long-row and hub kernels both run
    return g


def _rel(a, b):
    return float((a.cpu().double() - b).abs().max() / (b.abs().max() + 1e-12))


@gpu
@pytest.mark.parametrize("c,k,thr", [(132, 10, 0.0), (256, 64, -1.0), (256, 1, -1.0), (300, 1, 0.3), (512, 10, -1.0), (512, 64, 0.0)])
def test_wide_selection_and_aggregate_vs_oracle(c, k, thr):
    """Selection lists in the FP64 band, out_1 within 1e-5, dh of sng_edge_bwd vs autograd of the oracle; the backward is
    bit-reproducible.  c = 132 / 300: ragged last slot; 256 / 512: exact multiples; 132, 256 use G = 64, 300, 512 G = 128."""
    from oracle import sn_ref
    from sngnn_b200 import functional as SF
    n = 3000
    torch.manual_seed(c + k)
    ei = _hub_graph(n, 20000, seed=c + k, symmetric=True)
    g = _prepared(ei, n)
    h = torch.randn(n, c)
    h[7] = h[3]; h[11] = 0                                   # duplicate + zero row
    cp = SF.padded_channels(c)
    w = torch.randn(n, cp, device=DEV)
    w[:, c:] = 0
    grads = []
    for _ in range(2):
        hp = F.pad(h, (0, cp - c)).to(DEV).requires_grad_(True)
        out, (sel_src, sel_w, sel_cnt) = SF.edge_topk_agg(hp, g, k, thr, return_selection=True)
        (out * w).sum().backward()
        grads.append(hp.grad)
    assert torch.equal(grads[0], grads[1])

    h64 = h.double().requires_grad_(True)
    pe = sn_ref.process_edges(ei, n, True)
    out_ref = sn_ref.sn_aggregate(h64, pe, k, thr)
    (out_ref * w[:, :c].cpu().double()).sum().backward()
    torch.testing.assert_close(out[:, :c].detach().cpu().double(), out_ref.detach(), rtol=1e-5, atol=1e-6)
    assert _rel(grads[0][:, :c], h64.grad) < 1e-5

    n64 = F.normalize(h.double(), dim=-1, eps=1e-12)
    s64 = (n64[pe[1]] * n64[pe[0]]).sum(-1)
    rank = sn_ref.edge_rank(s64, pe[1])
    selm = (rank < k) & (s64 >= thr)
    idx_ref = torch.full((n, k), -1, dtype=torch.long)
    idx_ref[pe[1][selm], rank[selm]] = pe[0][selm]
    cnt_ref = torch.zeros(n, dtype=torch.long).index_add(0, pe[1][selm], torch.ones(int(selm.sum()), dtype=torch.long))
    res = compare_lists(sel_src, sel_cnt, idx_ref, cnt_ref, lambda r, j: (n64[r] * n64[j]).sum(-1), thr)
    assert res["out_of_band"] == 0, res


@gpu
def test_wide_base_layer_select_all_vs_oracle():
    from oracle import sn_ref
    from sngnn_b200 import functional as SF
    n, c = 3000, 256
    torch.manual_seed(2)
    ei = _hub_graph(n, 20000, seed=5, symmetric=False)
    g = _prepared(ei, n, False)
    assert not g.symmetric
    h = torch.randn(n, c)
    w = torch.randn(n, c, device=DEV)
    dhs = []
    for _ in range(2):
        hp = h.to(DEV).requires_grad_(True)
        out = SF.edge_topk_agg(hp, g, None, None)
        (out * w).sum().backward()
        dhs.append(hp.grad)
    assert torch.equal(dhs[0], dhs[1])
    h64 = h.double().requires_grad_(True)
    ref = sn_ref.sn_aggregate(h64, sn_ref.process_edges(ei, n, False))
    (ref * w.cpu().double()).sum().backward()
    torch.testing.assert_close(out.detach().cpu().double(), ref.detach(), rtol=1e-5, atol=1e-6)
    assert _rel(dhs[0], h64.grad) < 1e-5


@gpu
@pytest.mark.parametrize("c,sym", [(256, True), (512, True), (256, False), (512, False)])
def test_wide_snconv_plus_plus_fused_and_k4_vs_oracle(c, sym):
    """One SNConv_plus_plus layer: the fused single pass (symmetric graph) or the K4 form (asymmetric) against the oracle with
    the kernel's selection; outputs and the gradients of x, lin, W^T, b_w, beta and bias at 1e-5, a bit-reproducible backward."""
    from oracle import sn_ref
    import sngnn_b200.models as M
    from sngnn_b200 import functional as SF
    n, fd, k, thr = 3000, 24, 10, 0.0
    torch.manual_seed(c + sym)
    ei = _hub_graph(n, 20000, seed=c + 3, symmetric=sym)
    g = _prepared(ei, n)
    assert g.symmetric == sym
    x = torch.randn(n, fd)
    conv = M.SNConv_plus_plus(fd, c, n, k, thr, 0.3, True, bias=True).to(DEV)
    with torch.no_grad():
        conv.bias.normal_()
    xd = x.to(DEV).requires_grad_(True)
    wgt = torch.randn(n, c, device=DEV)

    def run():
        conv.zero_grad()
        xd.grad = None
        SF.record_selection = []
        try:
            out = conv(xd, ei.to(DEV))
            rec = SF.record_selection
        finally:
            SF.record_selection = None
        (out * wgt).sum().backward()
        return out.detach().clone(), {kk: p.grad.detach().clone() for kk, p in conv.named_parameters()}, xd.grad.clone(), rec

    out, grads, dx, rec = run()
    out2, grads2, dx2, _ = run()
    assert torch.equal(out, out2) and torch.equal(dx, dx2)
    for kk in ("w.weight", "w.bias", "beta"):
        assert torch.equal(grads[kk], grads2[kk]), kk
    (sel_src, sel_cnt), = rec
    p64 = {kk: p.detach().cpu().double().contiguous().requires_grad_(True) for kk, p in conv.named_parameters()}
    x64 = x.double().requires_grad_(True)
    ref = sn_ref.snconv_plus_plus(x64, ei, p64["lin.weight"], p64["lin.bias"], p64["w.weight"], p64["w.bias"], p64["beta"], k, thr,
                                  True, p64["bias"], forced=(sel_src.cpu().long(), sel_cnt.cpu().long()))
    (ref * wgt.cpu().double()).sum().backward()
    torch.testing.assert_close(out.cpu().double(), ref.detach(), rtol=1e-5, atol=2e-6)
    for kk in grads:
        r = p64[kk].grad
        scale = r.abs().max() + 1e-12
        if kk == "beta":                                   # a signed sum of n * c terms: see test_gpu_edge.py
            scale = torch.maximum(scale, 1e-2 * (wgt.cpu().double().abs() * ref.detach().abs()).sum())
        assert float((grads[kk].cpu().double() - r).abs().max() / scale) < 1e-5, kk
    assert _rel(dx, x64.grad) < 1e-5


@gpu
def test_wide_row_shards_equal_the_whole_graph():
    from sngnn_b200 import functional as SF
    n, c, k, thr = 3000, 256, 10, 0.0
    ei = _hub_graph(n, 20000, seed=4, symmetric=True)
    g = _prepared(ei, n)
    torch.manual_seed(1)
    h = torch.randn(n, c, device=DEV)
    w = torch.randn(n, c, device=DEV)
    h0 = h.clone().requires_grad_(True)
    out_ref = SF.edge_topk_agg(h0, g, k, thr)
    (out_ref * w).sum().backward()
    h1 = h.clone().requires_grad_(True)
    outs = [SF.ShardedEdgeTopkAgg.apply(h1, g.row_slice(lo, hi), lo, k, thr) for lo, hi in ((0, 1200), (1200, 1201), (1201, 3000))]
    out = torch.cat(outs)
    (out * w).sum().backward()
    assert torch.equal(out, out_ref)
    assert float((h1.grad - h0.grad).abs().max() / h0.grad.abs().max()) < 1e-5      # FP32 atomics in the scatter form


@gpu
def test_wide_sharded_forward_world1_equals_model():
    from sngnn_b200 import dist as D, synth
    import sngnn_b200.models as M
    n, fd, hid, ncls, k, thr = 3001, 24, 256, 5, 6, 0.1
    x = synth.make_features(n, fd, "clustered", seed=1).to(DEV)
    ei = synth.make_graph(n, 30000, seed=2, symmetric=True, hub_offset=3.0).to(DEV)
    y = synth.make_labels(n, ncls, seed=3).to(DEV)
    torch.manual_seed(7)
    model = M.SNGNN_Plus_Plus(fd, hid, ncls, n, 2, k, thr, 0.5, 1, 0.0).to(DEV).train()
    logp = D.sharded_forward(model, x, ei, n)
    F.nll_loss(logp, y).backward()
    grads = {name: p.grad.clone() for name, p in model.named_parameters()}
    model.zero_grad()
    ref = model(synth.GraphData(x, ei))
    F.nll_loss(ref, y).backward()
    torch.testing.assert_close(logp.detach(), ref.detach(), rtol=1e-5, atol=2e-6)
    for name, p in model.named_parameters():
        err = (grads[name] - p.grad).abs().max() / (p.grad.abs().max() + 1e-12)
        assert err < 2e-5, (name, float(err))


@gpu
def test_wide_list_aggregation_vs_oracle():
    """All-pairs mode: ListAgg (sng_list_agg_fwd, scatter backward) on given lists vs knn_mean_aggregate, the list weights
    being the cosines of h (so the backward runs through them too)."""
    from oracle import sn_ref
    from sngnn_b200 import functional as SF
    n, c, k = 2000, 256, 12
    gen = torch.Generator().manual_seed(3)
    h = torch.randn(n, c, generator=gen)
    idx = torch.randint(0, n, (n, k), generator=gen)
    cnt = torch.randint(0, k + 1, (n,), generator=gen)
    idx[torch.arange(k)[None, :] >= cnt[:, None]] = -1
    denom = torch.randint(1, 40, (n,), generator=gen).double()
    nh = F.normalize(h, dim=-1)
    sim = torch.where(idx >= 0, (nh[:, None, :] * nh[idx.clamp(min=0)]).sum(-1), torch.zeros(()))
    hd = h.to(DEV).requires_grad_(True)
    out = SF.ListAgg.apply(hd, idx.to(DEV, torch.int32), sim.to(DEV), cnt.to(DEV, torch.int32), (1.0 / denom).float().to(DEV))
    w = torch.randn(n, c, generator=gen)
    (out * w.to(DEV)).sum().backward()
    h64 = h.double().requires_grad_(True)
    n64 = F.normalize(h64, dim=-1, eps=1e-12)
    s64 = (n64[:, None, :] * n64[idx.clamp(min=0)]).sum(-1)
    ref = sn_ref.knn_mean_aggregate(h64, idx, s64, cnt, denom)
    (ref * w.double()).sum().backward()
    torch.testing.assert_close(out.detach().cpu().double(), ref.detach(), rtol=1e-5, atol=1e-6)
    assert _rel(hd.grad, h64.grad) < 1e-5


@gpu
@pytest.mark.parametrize("kind,hid", [("SNGNN", 256), ("SNGNN_Plus", 300), ("SNGNN_Plus_Plus", 256)])
def test_wide_models_vs_oracle(kind, hid):
    """Two-layer models with a wide hidden layer: logits, loss and every parameter gradient vs the oracle run with the
    selection the kernels recorded."""
    from oracle import sn_ref
    from sngnn_b200 import functional as SF, synth
    import sngnn_b200.models as M
    n, fd, ncls, k, thr = 2500, 24, 5, 6, 0.1
    x = synth.make_features(n, fd, "clustered", seed=1)
    ei = synth.make_graph(n, 25000, seed=2, symmetric=True, hub_offset=3.0)
    y = synth.make_labels(n, ncls, seed=3)
    torch.manual_seed(7)
    if kind == "SNGNN":
        model = M.SNGNN(fd, hid, ncls, 2)
        model.dropout = torch.nn.Dropout(0.0)
    elif kind == "SNGNN_Plus":
        model = M.SNGNN_Plus(fd, hid, ncls, n, 2, k, thr, 1, 0.0)
    else:
        model = M.SNGNN_Plus_Plus(fd, hid, ncls, n, 2, k, thr, 0.5, 1, 0.0)
    sd0 = {kk: v.detach().clone() for kk, v in model.state_dict().items()}
    model = model.to(DEV).train()
    SF.record_selection = []
    try:
        out = model(synth.GraphData(x.to(DEV), ei.to(DEV)))
        rec = SF.record_selection
    finally:
        SF.record_selection = None
    loss = F.nll_loss(out, y.to(DEV))
    loss.backward()
    forced = [(s.cpu().long(), c.cpu().long()) for s, c in rec] if rec else None
    assert kind == "SNGNN" or len(forced) == 2
    params = {kk: v.double().contiguous().requires_grad_(True) for kk, v in sd0.items()}
    ref = sn_ref.stack_forward(kind, sn_ref.params_from_state_dict(params, 2), x.double(), ei, top_k=k, thr=thr,
                               remove_self_loops=True, forced=forced)
    loss_ref = F.nll_loss(ref, y)
    loss_ref.backward()
    torch.testing.assert_close(out.detach().cpu().double(), ref.detach(), rtol=1e-5, atol=2e-6)
    assert abs(float(loss) - float(loss_ref)) <= 1e-5 * abs(float(loss_ref)) + 1e-6
    for name, p in model.named_parameters():
        assert _rel(p.grad, params[name].grad) < 1e-5, name


@gpu
def test_train_main_with_a_wide_hidden_layer():
    from sngnn_b200 import train as T
    final, hist = T.main("--model SNGNN_Plus_Plus --dataset small --num_layers 2 --hidden_channels 256 --top_k 10 --thr 0.0 "
                         "--dropout 0.0 --epochs 4 --log-every 0".split(), log=lambda s: None)
    assert len(hist) == 4 and all(torch.isfinite(torch.tensor(h[0])) for h in hist)
    assert hist[-1][0] < hist[0][0]                       # the training loss goes down


@gpu
def test_wide_errors():
    from sngnn_b200 import functional as SF, graph as G, _C
    ei = torch.tensor([[0, 1], [1, 0]], device=DEV)
    g = G.prepare(ei, 2, True)
    with pytest.raises(RuntimeError, match="rc=-2"):                  # SNG_ERR_UNSUPPORTED
        SF._edge_fwd(torch.randn(2, 516, device=DEV), g, 0, 1, 0.0, False)
    assert "512" in _C.last_error()
    with pytest.raises(RuntimeError):
        SF.edge_topk_agg(torch.randn(2, 256, device=DEV), g, 65, 0.0)     # top_k > SNG_MAX_TOPK at any width
    assert "top_k" in _C.last_error()
