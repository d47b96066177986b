"""denominator='selected' on the edge-restricted path: out_1[i] = sum_{e in S_i} s_e h[src_e] / max(|S_i|, 1), computed by the
edge kernels themselves (sng_edge_fwd_denom / sng_edge_bwd_denom) in inference and training, with and without the fused
SNGNN++ epilogue.

The reference has no such option, so the formula above is the definition: _forced_selected states it in FP64 on top of the
oracle's own forced aggregation (oracle.sn_ref.sn_aggregate_forced, the in-degree mean given the selection, rescaled per row
by deg_i / max(|S_i|, 1)).  Every comparison has two halves: (a) the selection lists against the oracle's rule within the FP64
band (parity.compare_lists), (b) values and gradients GIVEN the selection at 1e-5.  The rows
are those of the boundary graph of test_gpu_edge_boundaries: in-degrees 0, <= 32, 33..1024 (chunks + merge at C <= 32, the
long-row kernel above) and > 1024 (the hub kernel at C > 32)."""
import pytest
import torch
import torch.nn.functional as F

from parity import compare_lists
from test_gpu_edge_boundaries import _device_graph, _features, _oracle_lists, _rel

DEV = "cuda"
# outputs: rtol 1e-5 and atol 1e-6, or 2e-6 for the fused SNGNN++ output (the suite's layer tolerance: at the hubs out_0 is
# an FP32 sum of over a thousand W^T rows)
ATOL = {False: 1e-6, True: 2e-6}
WIDTHS = (4, 32, 128, 512)                 # narrow register kernel, staged kernel, long-row + hub kernels (two widths)
TOP_KS = (1, 10, 64)
THRS = (-1.0, 0.5)                         # 0.5 leaves rows that have in-edges with no candidate at all


def _structural(n, cp, seed):
    """(w.weight [C, N] in transposed storage, w.bias, beta, bias) on the device, as leaves of autograd."""
    gen = torch.Generator().manual_seed(seed)
    wt = (torch.randn(n, cp, generator=gen) * 0.1).to(DEV).requires_grad_(True)
    rest = [t.to(DEV).requires_grad_(True) for t in (torch.randn(cp, generator=gen), torch.full((1,), 0.3), torch.randn(cp, generator=gen))]
    return wt, rest


def _forced_selected(h64, pe, ss, sc):
    """out_1[i] = sum_{t < sc[i]} cos(h_i, h_{ss[i,t]}) h_{ss[i,t]} / max(sc[i], 1) in FP64, autograd-capable: the oracle's forced
    in-degree mean times deg_i / max(sc[i], 1) (pe = the processed edge list, whose targets give deg_i)."""
    from oracle import sn_ref
    sc = sc.cpu().long()
    deg = torch.zeros(h64.size(0), dtype=h64.dtype).index_add(0, pe[1], torch.ones(pe.size(1), dtype=h64.dtype))
    scale = deg.clamp(min=1) / sc.clamp(min=1).to(h64.dtype)
    return sn_ref.sn_aggregate_forced(h64, pe, ss.cpu().long(), sc) * scale[:, None]


def _stack_selected(kind, params, x, ei, forced, layer_inputs):
    """oracle.sn_ref.stack_forward (no BatchNorm, no dropout, self loops removed) with each layer's out_1 given its lists
    `forced` and divided by the selected count (_forced_selected)."""
    from oracle import sn_ref
    n = x.size(0)
    pe = sn_ref.process_edges(ei, n, True)
    for l, p in enumerate(params):
        layer_inputs.append(x.detach())
        out = _forced_selected(F.linear(x, p["lin_w"], p["lin_b"]), pe, *forced[l])
        if kind == "SNGNN_Plus_Plus":
            out = p["beta"] * sn_ref.structural_term(pe, p["w_w"], p["w_b"], n) + (1 - p["beta"]) * out
        if "bias" in p:
            out = out + p["bias"]
        x = F.relu(out) if l < len(params) - 1 else out
    return F.log_softmax(x, dim=1)


def _oracle_out(h64, pe, ss, sc, st64=None):
    """Reference output given the selection (ss, sc): out_1 with denominator='selected', blended like SNGNN++ when st64 is given."""
    from oracle import sn_ref
    out1 = _forced_selected(h64, pe, ss, sc)
    if st64 is None:
        return out1
    wt64, wb64, beta64, bias64 = st64
    out0 = sn_ref.structural_term(pe, wt64.t(), wb64, h64.size(0))
    return beta64 * out0 + (1 - beta64) * out1 + bias64


# ------------------------------------------------------------------------------------------ 1. forward
@pytest.mark.gpu
@pytest.mark.parametrize("form", ["plain", "fused"])
@pytest.mark.parametrize("cp", WIDTHS)
def test_forward_every_dispatch_class(cp, form):
    """Inference equals training bit for bit; the output equals the candidates kernel rescaled by deg / max(cnt, 1) (the
    previous Python path, then K4 for SNGNN++) to rounding; a row that selects nothing outputs 0 (no NaN); lists in the FP64
    band and values given the lists at 1e-5."""
    from oracle import sn_ref
    from sngnn_b200 import functional as SF
    fused = form == "fused"
    ei, _, g = _device_graph(fused)
    n = g.n
    assert g.symmetric == fused
    pe = sn_ref.process_edges(ei, n, True)
    h = _features(n, cp, seed=cp + 3)
    hd = h.to(DEV)
    h64 = h.double()
    deg = (g.rowptr_in[1:] - g.rowptr_in[:-1]).cpu()
    st = st64 = None
    if fused:
        wt, (wb, beta, bias) = _structural(n, cp, cp)
        st = (wt.t(), wb, beta, bias)
        st64 = tuple(t.detach().cpu().double() for t in (wt, wb, beta, bias))
    for k in TOP_KS:
        for thr in THRS:
            tag = f"{form} cp={cp} k={k} thr={thr}"
            out_t, (ss, _, sc) = SF.edge_topk_agg(hd.clone().requires_grad_(True), g, k, thr, return_selection=True, structural=st,
                                                  denominator="selected")
            out_t = out_t.detach()
            with torch.no_grad():
                out_i = SF.edge_topk_agg(hd, g, k, thr, structural=st, denominator="selected")
                old = SF.edge_topk_agg(hd, g, k, thr) * (sc.clamp(min=1).float() * g.inv_deg).reciprocal()[:, None]
                if fused:
                    old = SF.PPFuse.apply(old, *st, g)
            assert torch.equal(out_t, out_i), tag
            assert bool(torch.isfinite(out_i).all()), tag
            assert _rel(out_i, old) < 1e-6, (tag, _rel(out_i, old))
            empty = (sc.cpu() == 0)
            if thr > 0:
                assert bool((empty & (deg > 0)).any()), tag
            if not fused:
                assert float(out_i[empty.to(DEV)].abs().max()) == 0, tag
            # (a) the lists against the oracle's rule, (b) the values given the lists
            idx_ref, cnt_ref, _, nrm = _oracle_lists(h64, pe, n, k, thr)
            res = compare_lists(ss, sc, idx_ref, cnt_ref, lambda r, j: (nrm[r] * nrm[j]).sum(-1), thr)
            assert res["out_of_band"] == 0, (tag, res)
            if n * k * cp > 3e7:
                continue                   # the oracle's [n, k, C] FP64 gather: the rescaled candidates output above covers it
            ref = _oracle_out(h64, pe, ss, sc, st64)
            torch.testing.assert_close(out_i.cpu().double(), ref, rtol=1e-5, atol=ATOL[fused], msg=lambda m: f"{tag}: {m}")


# ------------------------------------------------------------------------------------------ 2. backward
# (cp, top_k): pass T runs the narrow kernel (4), the staged kernel (32, k <= 32) and the general one with the per-row factor
# (32 with k > 32, and every width above 32)
BWD_CASES = [(4, 10), (32, 10), (32, 64), (128, 10), (128, 64), (512, 10)]


@pytest.mark.gpu
@pytest.mark.parametrize("form", ["plain", "fused"])
@pytest.mark.parametrize("cp,k", BWD_CASES)
def test_backward_given_the_selection_vs_fp64(cp, k, form):
    """dL/dh and, fused, dL/dW^T, dL/db_w, dL/dbeta, dL/dbias against FP64 autograd of the oracle given the selection; two
    runs bit-identical; the fused single pass agrees with EdgeAgg + K4 (PPFuse)."""
    from oracle import sn_ref
    from sngnn_b200 import functional as SF
    fused = form == "fused"
    ei, _, g = _device_graph(fused)
    n = g.n
    pe = sn_ref.process_edges(ei, n, True)
    thr = 0.0
    h = _features(n, cp, seed=cp + 7)
    up = torch.randn(n, cp, generator=torch.Generator().manual_seed(cp + 8))
    upd = up.to(DEV)

    def run(single_pass=True):
        hd = h.to(DEV).requires_grad_(True)
        leaves = [hd]
        st = None
        if fused:
            wt, rest = _structural(n, cp, cp + 9)
            leaves += [wt] + rest
            st = (wt.t(), *rest)
        if fused and not single_pass:
            out1, (ss, _, sc) = SF.edge_topk_agg(hd, g, k, thr, return_selection=True, denominator="selected")
            out = SF.PPFuse.apply(out1, *st, g)
        else:
            out, (ss, _, sc) = SF.edge_topk_agg(hd, g, k, thr, return_selection=True, structural=st, denominator="selected")
        (out * upd).sum().backward()
        return out.detach(), ss, sc, [t.grad for t in leaves], [t.detach() for t in leaves]

    out, ss, sc, grads, leaves = run()
    out2, _, _, grads2, _ = run()
    assert torch.equal(out, out2)
    for a, b in zip(grads, grads2):
        assert torch.equal(a, b)
    p64 = [t.cpu().double().requires_grad_(True) for t in leaves]
    ref = _oracle_out(p64[0], pe, ss, sc, tuple(p64[1:]) if fused else None)
    (ref * up.double()).sum().backward()
    torch.testing.assert_close(out.cpu().double(), ref.detach(), rtol=1e-5, atol=ATOL[fused])

    def check(grads, tag):
        for name, got, r in zip(["h", "wt", "w_bias", "beta", "bias"], grads, p64):
            scale = r.grad.abs().max() + 1e-12
            if name == "beta":             # a signed sum of n * C terms: bounded by their magnitudes, not by the total
                scale = torch.maximum(scale, 1e-2 * (up.double().abs() * ref.detach().abs()).sum())
            err = float((got.cpu().double() - r.grad).abs().max() / scale)
            assert err < 1e-5, (tag, name, err)

    check(grads, "single pass")
    if fused:                              # EdgeAgg + K4: the same layer in two passes
        out_k4, ss_k4, sc_k4, grads_k4, _ = run(single_pass=False)
        assert torch.equal(ss_k4, ss) and torch.equal(sc_k4, sc)
        assert _rel(out_k4, out) < 1e-5
        check(grads_k4, "EdgeAgg + K4")


# ------------------------------------------------------------------------------------------ 3. models
def _model(kind, n, fd, hid, ncls, layers, k, thr):
    import sngnn_b200.models as M
    torch.manual_seed(3)
    if kind == "SNGNN_Plus_Plus":
        return M.SNGNN_Plus_Plus(fd, hid, ncls, n, layers, k, thr, 0.3, 1, 0.0, denominator="selected")
    return M.SNGNN_Plus(fd, hid, ncls, n, layers, k, thr, 1, 0.0, denominator="selected")


@pytest.mark.gpu
@pytest.mark.parametrize("layers", [1, 2])
@pytest.mark.parametrize("kind", ["SNGNN_Plus", "SNGNN_Plus_Plus"])
def test_models_vs_oracle_and_in_eval(kind, layers, monkeypatch):
    """Logits and parameter gradients against the oracle's layer stack given each layer's lists (recorded through
    functional.record_selection; the lists themselves in the FP64 band of each layer's input); model.eval() under no_grad
    gives the training logits; on a symmetric graph SNGNN++ never runs the separate K4 kernel (functional.PPFuse)."""
    from oracle import sn_ref
    from sngnn_b200 import functional as SF, synth
    n, fd, hid, ncls, k, thr = 3000, 12, 16, 5, 6, 0.1
    ei = synth.make_graph(n, 30000, seed=21, symmetric=True, hub_offset=3.0)
    x = torch.randn(n, fd, generator=torch.Generator().manual_seed(22))
    y = torch.randint(0, ncls, (n,), generator=torch.Generator().manual_seed(23))
    data = synth.GraphData(x, ei).to(DEV)
    model = _model(kind, n, fd, hid, ncls, layers, k, thr).to(DEV).train()

    def no_k4(*_a, **_k):
        raise AssertionError("the SNGNN++ layer ran the separate K4 pass on a symmetric graph")
    monkeypatch.setattr(SF.PPFuse, "apply", no_k4)
    rec = []
    monkeypatch.setattr(SF, "record_selection", rec)
    mask = (torch.arange(n) % 2 == 0)
    out = model(data)
    F.nll_loss(out[mask.to(DEV)], y.to(DEV)[mask.to(DEV)]).backward()
    monkeypatch.setattr(SF, "record_selection", None)
    assert len(rec) == layers

    sd = {kk: v.detach().cpu().double().contiguous().requires_grad_(True) for kk, v in model.state_dict().items()}
    inputs = []
    forced = [(ss.cpu().long(), sc.cpu().long()) for ss, sc in rec]
    ref = _stack_selected(kind, sn_ref.params_from_state_dict(sd, layers), x.double(), ei, forced, inputs)
    F.nll_loss(ref[mask], y[mask]).backward()
    torch.testing.assert_close(out.detach().cpu().double(), ref.detach(), rtol=1e-5, atol=2e-6)
    for name, p in model.named_parameters():
        r = sd[name].grad
        err = float((p.grad.cpu().double() - r).abs().max() / (r.abs().max() + 1e-12))
        assert err < 1e-5, (name, err)
    pe = sn_ref.process_edges(ei, n, True)
    for l, ((ss, sc), xin) in enumerate(zip(rec, inputs)):
        h64 = F.linear(xin, sd[f"lins.{l}.lin.weight"].detach(), sd[f"lins.{l}.lin.bias"].detach())
        idx_ref, cnt_ref, _, nrm = _oracle_lists(h64, pe, n, k, thr)
        res = compare_lists(ss, sc, idx_ref, cnt_ref, lambda r, j: (nrm[r] * nrm[j]).sum(-1), thr)
        assert res["out_of_band"] == 0, (l, res)
    model.eval()
    with torch.no_grad():
        assert torch.equal(model(data), out.detach())


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["SNGNN_Plus", "SNGNN_Plus_Plus"])
def test_trainer_runs_with_selected_denominator(kind):
    """train.train validates and tests under no_grad every epoch: three epochs with denominator='selected' complete."""
    from sngnn_b200 import train as T
    cfg = dict(epochs=3, patience=100, log_every=0)
    data, ncls = T.load_data("small", 0, DEV)
    n, fd = data.x.shape
    model = _model(kind, n, fd, 16, ncls, 2, 4, 0.0).to(DEV)
    opt = torch.optim.Adam(model.parameters(), lr=0.01, weight_decay=5e-4)
    _, hist = T.train(model, data, opt, cfg)
    assert len(hist) == 3 and all(torch.isfinite(torch.tensor(h[0])) and torch.isfinite(torch.tensor(h[2])) for h in hist)


# ------------------------------------------------------------------------------------------ 4. row shards (kernel level)
SHARDS = ((0, 1200), (1200, 1200), (1200, 1201), (1201, 3000))      # ragged, an empty shard and a 1-row shard


@pytest.mark.gpu
@pytest.mark.parametrize("cp,k", [(4, 10), (32, 10), (32, 64), (128, 10)])
def test_row_shards_take_the_mode(cp, k):
    """_edge_fwd / edge_bwd with row_offset and denominator='selected': the shard [0, N) equals the whole graph bit for bit,
    the forward rows of ragged shards concatenate bit for bit, and their backward contributions add up to the whole."""
    from sngnn_b200 import functional as SF
    _, _, g = _device_graph(False)
    n, thr = g.n, 0.0
    h = _features(n, cp, seed=cp + 11).to(DEV)
    gg = torch.randn(n, cp, generator=torch.Generator().manual_seed(cp + 12)).to(DEV)

    def fwd_bwd(graph, lo):
        inv_denom = torch.empty(graph.n, device=DEV)
        out, ss, sw, sq, sc, inv, _ = SF._edge_fwd(h, graph, lo, k, thr, True, want_q=True, denominator="selected", inv_denom=inv_denom)
        dh, _, _ = SF.edge_bwd(h, inv, gg[lo:lo + graph.n].contiguous(), graph, k, ss, sw, sq, sc, row_offset=lo, inv_denom=inv_denom)
        return out, inv_denom, dh, sc

    out_ref, inv_ref, dh_ref, sc_ref = fwd_bwd(g, 0)
    assert torch.equal(inv_ref, 1.0 / sc_ref.clamp(min=1).float())      # the factor of every row, as an IEEE division
    out_w, inv_w, dh_w, _ = fwd_bwd(g.row_slice(0, n), 0)
    assert torch.equal(out_w, out_ref) and torch.equal(inv_w, inv_ref) and torch.equal(dh_w, dh_ref)
    parts = [fwd_bwd(g.row_slice(lo, hi), lo) for lo, hi in SHARDS]
    assert torch.equal(torch.cat([p[0] for p in parts]), out_ref)
    assert torch.equal(torch.cat([p[1] for p in parts]), inv_ref)
    assert int(parts[1][2].abs().max()) == 0                            # the empty shard contributes zero
    total = sum(p[2] for p in parts)
    assert float((total - dh_ref).abs().max() / dh_ref.abs().max()) < 1e-5
