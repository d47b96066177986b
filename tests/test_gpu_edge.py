"""GPU parity of the edge-restricted path (K0, K2, K2b, K3, K4) through the C-ABI, against the CPU oracle and
the golden vectors of the reference.  Tolerances: indices exact (FP64-band rule), values 1e-5 relative."""
import pytest
import torch
import torch.nn.functional as F

from conftest import load_golden, golden_inputs, golden_state_dict, golden_grad
from parity import compare_lists

pytestmark = pytest.mark.gpu
DEV = "cuda"


def _models():
    import sngnn_b200.models as M
    return M


def _build(M, g, run, x, y):
    cfg, kind = run["cfg"], run["kind"]
    N, Fd = x.shape
    C = int(y.max()) + 1
    if kind == "SNGNN":
        m = M.SNGNN(Fd, cfg["hidden"], C, cfg["layers"], bn=cfg.get("bn", False))
        m.dropout = torch.nn.Dropout(0.0)
    elif kind == "SNGNN_Plus":
        m = M.SNGNN_Plus(Fd, cfg["hidden"], C, N, cfg["layers"], cfg["top_k"], cfg["thr"], cfg["rsl"], 0.0, bn=cfg.get("bn", False))
    else:
        m = M.SNGNN_Plus_Plus(Fd, cfg["hidden"], C, N, cfg["layers"], cfg["top_k"], cfg["thr"], cfg["beta"], cfg["rsl"], 0.0,
                              bn=cfg.get("bn", False))
    m.load_state_dict(golden_state_dict(g, run))
    return m.to(DEV).train()


@pytest.mark.parametrize("fname", ["models_tiny.pt", "models_small.pt", "models_chameleon.pt"])
def test_models_match_reference_golden(fname):
    from sngnn_b200.synth import GraphData
    M = _models()
    g = load_golden(fname)
    x, ei, y = golden_inputs(g)
    data = GraphData(x, ei).to(DEV)
    yd = y.to(DEV)
    mask = (torch.arange(x.size(0)) % 2 == 0).to(DEV)
    worst = 0.0
    for run in g["runs"]:
        m = _build(M, g, run, x, y)
        out = m(data)
        loss = F.nll_loss(out[mask], yd[mask])
        loss.backward()
        tag = f"{fname} {run['kind']} {run['cfg']}"
        torch.testing.assert_close(out.detach().cpu(), run["logp"], rtol=1e-5, atol=2e-6, msg=lambda s: f"{tag}: {s}")
        torch.testing.assert_close(loss.detach().cpu(), run["loss"], rtol=1e-5, atol=1e-6, msg=lambda s: f"{tag} loss: {s}")
        for k, p in m.named_parameters():
            got, ref, scale = golden_grad(p.grad.detach().cpu(), run["grads"][k])
            err = (got - ref).abs().max().item() / (scale.item() + 1e-12)
            worst = max(worst, err)
            assert err < 1e-5, f"{tag} grad {k}: rel-to-max err {err:.3e}"
    print(f"{fname}: worst grad error relative to max {worst:.2e}")


@pytest.mark.parametrize("n,e,c,k,thr,rsl", [(5000, 60000, 32, 10, 0.0, True), (5000, 60000, 5, 3, 0.3, False),
                                              (20000, 400000, 64, 10, -0.5, True), (3000, 30000, 2, 64, -1.0, True),
                                              (4000, 50000, 128, 7, 0.2, True),
                                              # narrow rows (C <= 4): the register kernels
                                              (5000, 60000, 2, 10, 0.0, True), (5000, 60000, 4, 3, -0.5, False), (8000, 100000, 3, 10, 0.1, True)])
def test_edge_selection_and_aggregate_vs_oracle(n, e, c, k, thr, rsl):
    """sel lists exact vs the oracle's rank rule; out_1 within 1e-5; dh via K2b vs autograd of the oracle."""
    from oracle import sn_ref
    from sngnn_b200 import synth, graph as G, functional as SF
    torch.manual_seed(n + c)
    ei = synth.make_graph(n, e, seed=n, symmetric=True, hub_offset=3.0)
    h = torch.randn(n, c)
    h[7] = h[3]; h[11] = 0                                   # duplicate + zero row
    cp = SF.padded_channels(c)
    hp = F.pad(h, (0, cp - c)).to(DEV).requires_grad_(True)
    g = G.prepare(ei.to(DEV), n, rsl)
    out, (sel_src, sel_w, sel_cnt) = SF.edge_topk_agg(hp, g, k, thr, return_selection=True)
    w = torch.randn(n, cp, device=DEV)
    w[:, c:] = 0                                              # the module slices the padding away
    (out * w).sum().backward()

    # oracle (FP32 for values, FP64 for the index band rule)
    h64 = h.double().requires_grad_(True)
    pe = sn_ref.process_edges(ei, n, rsl)
    out_ref = sn_ref.sn_aggregate(h64, pe, k, thr)
    (out_ref * w[:, :c].cpu().double()).sum().backward()
    torch.testing.assert_close(out[:, :c].detach().cpu().double(), out_ref.detach(), rtol=1e-5, atol=1e-6)
    scale = h64.grad.abs().max()
    assert ((hp.grad[:, :c].cpu().double() - h64.grad).abs().max() / scale) < 1e-5

    # selection lists
    n64 = F.normalize(h.double(), dim=-1, eps=1e-12)
    s64 = (n64[pe[1]] * n64[pe[0]]).sum(-1)
    rank = sn_ref.edge_rank(s64, pe[1])
    selm = (rank < k) & (s64 >= thr)
    idx_ref = torch.full((n, k), -1, dtype=torch.long)
    idx_ref[pe[1][selm], rank[selm]] = pe[0][selm]
    cnt_ref = torch.zeros(n, dtype=torch.long).index_add(0, pe[1][selm], torch.ones(int(selm.sum()), dtype=torch.long))
    res = compare_lists(sel_src, sel_cnt, idx_ref, cnt_ref, lambda r, j: (n64[r] * n64[j]).sum(-1), thr)
    print(res)
    assert res["out_of_band"] == 0, res
    assert res["exact"] >= 0.999 * n


def test_base_snconv_select_all_vs_oracle():
    from oracle import sn_ref
    from sngnn_b200 import synth, graph as G, functional as SF
    n, c = 6000, 12
    ei = synth.make_graph(n, 50000, seed=5, symmetric=False, hub_offset=3.0)
    h = torch.randn(n, c)
    hp = h.to(DEV).requires_grad_(True)
    g = G.prepare(ei.to(DEV), n, False)
    out = SF.edge_topk_agg(hp, g, None, None)
    w = torch.randn(n, c, device=DEV)
    (out * w).sum().backward()
    h64 = h.double().requires_grad_(True)
    ref = sn_ref.sn_aggregate(h64, sn_ref.process_edges(ei, n, False))
    (ref * w.cpu().double()).sum().backward()
    torch.testing.assert_close(out.detach().cpu().double(), ref.detach(), rtol=1e-5, atol=1e-6)
    assert ((hp.grad.cpu().double() - h64.grad).abs().max() / h64.grad.abs().max()) < 1e-5


def test_rownorm_spmm_sddmm():
    from sngnn_b200 import functional as SF, synth, graph as G
    torch.manual_seed(0)
    x = torch.randn(3000, 65, device=DEV)
    x[5] = 0
    xf, xh, inv = SF.rownorm(x, want_f32=True, want_f16=True, f16_ld=80, want_inv=True)
    ref = F.normalize(x, dim=-1)
    torch.testing.assert_close(xf, ref, rtol=1e-6, atol=1e-7)
    torch.testing.assert_close(xh[:, :65].float(), ref, rtol=1e-3, atol=1e-4)
    assert xh[:, 65:].abs().max().item() == 0
    torch.testing.assert_close(inv, 1.0 / x.norm(dim=1).clamp(min=1e-12), rtol=1e-5, atol=0)
    n, c = 4000, 32
    ei = synth.make_graph(n, 40000, seed=3).to(DEV)
    g = G.prepare(ei, n, True)
    X = torch.randn(n, c, device=DEV)
    out = SF.spmm(X, g.rowptr_in, g.col_in, n)
    pe = G.process_edges(ei, n, True)
    ref = torch.zeros(n, c, device=DEV, dtype=torch.float64).index_add(0, pe[1], X.double()[pe[0]])
    torch.testing.assert_close(out.double(), ref, rtol=1e-5, atol=1e-5)
    a, b = pe[0][:1000], pe[1][:1000]
    s = SF.sddmm_dot(F.normalize(X, dim=-1), a, b)
    nx = F.normalize(X.double(), dim=-1)
    torch.testing.assert_close(s.double(), (nx[a] * nx[b]).sum(-1), rtol=1e-5, atol=1e-6)


def test_errors_are_loud():
    from sngnn_b200 import functional as SF, graph as G, _C
    ei = torch.tensor([[0, 1], [1, 0]], device=DEV)
    g = G.prepare(ei, 2, True)
    with pytest.raises(RuntimeError):
        SF.edge_topk_agg(torch.randn(2, 4), g, 1, 0.0)                  # CPU tensor: no CPU path
    with pytest.raises(RuntimeError):
        SF.edge_topk_agg(torch.randn(2, 4, device=DEV), g, 65, 0.0)     # top_k > SNG_MAX_TOPK
    assert "top_k" in _C.last_error()


@pytest.mark.parametrize("n,e,rsl,structural,sym", [(5000, 60000, True, True, True), (5000, 60000, False, True, False),
                                                    (300, 0, True, True, False), (4097, 9000, False, False, True), (70000, 900000, True, True, True)])
def test_graph_prepare_cuda_equals_torch(n, e, rsl, structural, sym):
    """sng_graph_prepare (stable radix sort on the GPU) == the torch construction (stable argsort) of graph.py on the CPU:
    identical CSR arrays, i.e. identical in-edge POSITION order, which is the tie-break order of the selection rule."""
    from sngnn_b200 import synth, graph as G
    if e:
        ei = synth.make_graph(n, e, seed=n, symmetric=sym, hub_offset=3.0)
        extra = torch.tensor([[5, 9, 9, 7], [5, 9, 2, 7]])                       # pre-existing loops and a duplicate-prone edge
        ei = torch.cat([ei, extra, ei[:, :50]], dim=1)                           # duplicates are kept (SURVEY.md appendix A.1)
        ei = ei[:, torch.randperm(ei.size(1), generator=torch.Generator().manual_seed(1))]   # not sorted: position order matters
        if structural:
            ei = ei[:, ei[0] >= 3]                                               # min(src) = 3: the shift quirk of R models.py:125
    else:
        ei = torch.zeros(2, 0, dtype=torch.long)
    G.clear_cache()
    ref = G.prepare(ei, n, rsl)
    got = G.prepare(ei.to(DEV), n, rsl)
    assert got.num_edges == ref.num_edges and got.n == ref.n and got.src_shift == ref.src_shift
    assert got.symmetric == ref.symmetric and got.max_deg == ref.max_deg
    assert torch.equal(got.rows_long.cpu().sort().values, ref.rows_long) and torch.equal(got.rows_hub.cpu().sort().values, ref.rows_hub)
    for name in ("rowptr_in", "col_in", "rowptr_out", "col_out", "col_in_shift", "tpos"):
        a, b = getattr(got, name), getattr(ref, name)
        assert (a is None) == (b is None), name
        if a is not None:
            assert torch.equal(a.cpu(), b), name
    torch.testing.assert_close(got.inv_deg.cpu(), ref.inv_deg, rtol=1e-6, atol=0)


def _hub_graph(n, e, seed, symmetric, hubs=(3, 17), hub_deg=(1500, 200)):
    """make_graph + a few forced hub rows (in-degree > 1024 and in (32, 1024]) so every degree class of the forward runs."""
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
    key = torch.unique(ei[0] * n + ei[1])                         # coalesced, sorted row-major
    return torch.stack([key // n, key % n])


@pytest.mark.parametrize("c,k,thr,sym", [(32, 10, 0.0, True), (32, 10, 0.0, False), (5, 3, 0.2, True), (64, 40, -0.3, True), (8, 1, 0.99, True),
                                          (2, 10, 0.0, True), (2, 10, 0.0, False), (4, 5, 0.1, True), (3, 40, -0.3, True)])
def test_snconv_plus_plus_fused_and_unfused_vs_oracle(c, k, thr, sym):
    """One SNConv_plus_plus layer on a graph with short, long (> 32) and hub (> 1024) rows: the fused single pass (symmetric
    graph) and the two-kernel form (asymmetric) against the FP64 oracle -- output, every parameter gradient and dL/dx at
    1e-5, and the backward must be bit-reproducible (no float atomics)."""
    from oracle import sn_ref
    import sngnn_b200.models as M
    from sngnn_b200 import graph as G
    n, fd = 6000, 24
    torch.manual_seed(c * 7 + k)
    ei = _hub_graph(n, 60000, seed=c + k, symmetric=sym)
    x = torch.randn(n, fd)
    x[9] = x[4]
    conv = M.SNConv_plus_plus(fd, c, n, k, thr, 0.3, True, bias=True).to(DEV)
    with torch.no_grad():
        conv.bias.normal_()
    gph = G.prepare(ei.to(DEV), n, True)
    assert gph.symmetric == sym and gph.rows_hub.numel() >= 1 and gph.rows_long.numel() >= 1
    xd = x.to(DEV).requires_grad_(True)
    wgt = torch.randn(n, c, device=DEV)

    def run():
        conv.zero_grad()
        xd.grad = None
        out = conv(xd, ei.to(DEV))
        (out * wgt).sum().backward()
        return out.detach().clone(), {kk: p.grad.detach().clone() for kk, p in conv.named_parameters()}, xd.grad.detach().clone()

    out, grads, dx = run()
    out2, grads2, dx2 = run()
    assert torch.equal(out, out2) and torch.equal(dx, dx2)
    for kk in grads:
        if kk not in ("lin.weight", "lin.bias"):                          # the dense lin backward is cuBLAS (split-K may differ run to run)
            assert torch.equal(grads[kk], grads2[kk]), kk
    p64 = {kk: p.detach().cpu().double().contiguous().requires_grad_(True) for kk, p in conv.named_parameters()}
    x64 = x.double().requires_grad_(True)
    ref = sn_ref.snconv_plus_plus(x64, ei, p64["lin.weight"], p64["lin.bias"], p64["w.weight"], p64["w.bias"], p64["beta"], k, thr, True,
                                  p64["bias"])
    (ref * wgt.cpu().double()).sum().backward()
    torch.testing.assert_close(out.cpu().double(), ref.detach(), rtol=1e-5, atol=2e-6)
    for kk in grads:
        r = p64[kk].grad
        scale = r.abs().max() + 1e-12
        if kk == "beta":
            # dL/dbeta = sum((out_0 - out_1) * w) is a signed sum of n * c terms: when it cancels (narrow layers), FP32 rounding of
            # the terms (1e-7 each) bounds the error by 1e-7 of the sum of their magnitudes, not 1e-5 of the total
            scale = torch.maximum(scale, 1e-2 * (wgt.cpu().double().abs() * ref.detach().abs()).sum())
        err = (grads[kk].cpu().double() - r).abs().max() / scale
        assert err < 1e-5, (kk, float(err))
    assert ((dx.cpu().double() - x64.grad).abs().max() / (x64.grad.abs().max() + 1e-12)) < 1e-5
    # inference mode (no lists, no diff) gives the same output
    with torch.no_grad():
        out3 = conv(x.to(DEV), ei.to(DEV))
    assert torch.equal(out3, out)


def test_edge_forward_degree_classes_match_general_kernel():
    """The degree-dispatched forward (short / long / hub kernels) against the general chunked kernel on the same rows:
    identical selection lists, outputs equal to FP32 rounding."""
    from sngnn_b200 import graph as G, functional as SF
    n, c, k = 8000, 32, 10
    ei = _hub_graph(n, 90000, seed=11, symmetric=True)
    gph = G.prepare(ei.to(DEV), n, True)
    h = torch.randn(n, c, device=DEV)
    h[20] = h[21]
    out_a, ss_a, sw_a, _, sc_a, _, _ = SF._edge_fwd(h, gph, 0, k, 0.1, True)
    tab, gph.chunk_tab = gph.chunk_tab, None                              # tables unknown -> general kernel on every row
    out_b, ss_b, sw_b, _, sc_b, _, _ = SF._edge_fwd(h, gph, 0, k, 0.1, True)
    gph.chunk_tab = tab
    assert torch.equal(sc_a, sc_b) and torch.equal(ss_a, ss_b)
    torch.testing.assert_close(sw_a, sw_b, rtol=1e-6, atol=1e-7)
    torch.testing.assert_close(out_a, out_b, rtol=1e-5, atol=1e-6)


@pytest.mark.parametrize("n,c", [(1, 2), (5000, 5), (200003, 2)])
def test_nll_loss_matches_torch_and_is_reproducible(n, c):
    from sngnn_b200 import functional as SF
    torch.manual_seed(n)
    logits = torch.randn(n, c, device=DEV)
    y = torch.randint(0, c, (n,), device=DEV)
    mask = torch.rand(n, device=DEV) < 0.6
    mask[0] = True
    a = torch.log_softmax(logits, 1).requires_grad_(True)
    b = a.detach().clone().requires_grad_(True)
    la = SF.nll_loss(a, y, mask)
    lb = F.nll_loss(b[mask], y[mask])
    (la * 3.0).backward(); (lb * 3.0).backward()
    torch.testing.assert_close(la, lb, rtol=1e-5, atol=1e-6)
    torch.testing.assert_close(a.grad, b.grad, rtol=1e-5, atol=1e-9)
    assert torch.equal(SF.nll_loss(a.detach(), y, mask), la.detach())          # fixed-order reduction
    torch.testing.assert_close(SF.nll_loss(a.detach(), y), F.nll_loss(a.detach(), y), rtol=1e-5, atol=1e-6)


@pytest.mark.parametrize("n,f,c", [(1, 3, 2), (5000, 65, 32), (3001, 269, 32), (2277, 2325, 5), (4097, 128, 64), (700, 40, 16)])
def test_lin_norm_matches_linear_and_normalize(n, f, c):
    """sng_lin_norm_fwd (lin + bias + 1/norm in one pass, R: models/models.py:121-122) against F.linear / F.normalize, forward
    and backward; unsupported shapes fall back to the library GEMM with inv_norm = None."""
    from sngnn_b200 import functional as SF, _C
    torch.manual_seed(n + f)
    x = torch.randn(n, f, device=DEV, requires_grad=True)
    lin = torch.nn.Linear(f, c).to(DEV)
    cp = SF.padded_channels(c)
    h, inv = SF.lin_norm(x, lin.weight, lin.bias, cp)
    assert bool(_C.lib().sng_lin_norm_supported(f, c)) == (inv is not None)
    ref = F.linear(x, lin.weight, lin.bias)
    torch.testing.assert_close(h[:, :c], ref, rtol=2e-5, atol=2e-5)
    assert h.shape == (n, cp) and (cp == c or h[:, c:].abs().max().item() == 0)
    if inv is not None:
        torch.testing.assert_close(inv, 1.0 / ref.norm(dim=1).clamp(min=1e-12), rtol=2e-5, atol=0)
    w = torch.randn(n, cp, device=DEV)
    (h * w).sum().backward()
    gx, gw, gb = x.grad.clone(), lin.weight.grad.clone(), lin.bias.grad.clone()
    x.grad = None; lin.zero_grad()
    (ref * w[:, :c]).sum().backward()
    torch.testing.assert_close(gx, x.grad, rtol=1e-4, atol=1e-4)
    torch.testing.assert_close(gw, lin.weight.grad, rtol=1e-4, atol=1e-3)
    torch.testing.assert_close(gb, lin.bias.grad, rtol=1e-4, atol=1e-3)


@pytest.mark.parametrize("n,f,c", [(1000, 65, 32), (5000, 128, 5), (777, 32, 2), (300, 100, 7), (2000, 128, 32), (64, 7, 1),
                                   (70001, 65, 32), (33, 66, 3), (0, 16, 4)])
def test_lin_bwd_weight_gradient(n, f, c):
    """dW = g^T x and db = sum g (sng_lin_bwd) against FP64; bit-reproducible."""
    from sngnn_b200 import functional as SF
    torch.manual_seed(n + f + c)
    cp = SF.padded_channels(c)
    gh = torch.randn(n, cp, device=DEV)
    x = torch.randn(n, f, device=DEV)
    dw, db = SF.lin_bwd(gh, x, c)
    ref_w = gh[:, :c].double().t() @ x.double()
    ref_b = gh[:, :c].double().sum(0)
    scale = ref_w.abs().max().item() + 1e-12
    assert (dw.double() - ref_w).abs().max().item() / scale < 1e-5
    assert (db.double() - ref_b).abs().max().item() / (ref_b.abs().max().item() + 1e-12) < 1e-5
    dw2, db2 = SF.lin_bwd(gh, x, c)
    assert torch.equal(dw, dw2) and torch.equal(db, db2)
    # strided views (a column slice of a wider matrix) go through the leading dimensions
    wide = torch.randn(n, f + 3, device=DEV)
    dw3, _ = SF.lin_bwd(gh, wide[:, :f], c, want_bias=False)
    assert (dw3.double() - gh[:, :c].double().t() @ wide[:, :f].double()).abs().max().item() / scale < 1e-5 or n == 0


def test_lin_bwd_wide_layers_keep_the_library_gemm():
    """f > 128 is outside sng_lin_bwd (loud error from the C ABI); LinNorm.backward routes such layers to the library GEMM."""
    from sngnn_b200 import functional as SF, _C
    assert not _C.lib().sng_lin_bwd_supported(269, 32) and _C.lib().sng_lin_bwd_supported(128, 32)
    with pytest.raises(RuntimeError):
        SF.lin_bwd(torch.randn(10, 32, device=DEV), torch.randn(10, 269, device=DEV), 32)
    x = torch.randn(500, 269, device=DEV)
    w = torch.randn(32, 269, device=DEV, requires_grad=True)
    b = torch.randn(32, device=DEV, requires_grad=True)
    h, _ = SF.lin_norm(x, w, b, 32)
    h.square().sum().backward()
    ref = (2 * (x @ w.t() + b)).t() @ x
    assert (w.grad - ref).abs().max() / ref.abs().max() < 1e-5
