"""The wide all-pairs build (top_k > SNG_KNN_MAX_TOPK: sng_simknn_wide_count + sng_simknn_wide_select) and the list
aggregation at list widths above 64: lists against the oracle rule, the prefix property against K1, rows that need the exact
scan, determinism and row shards, ListAgg forward / backward against FP64, and both models in the all-pairs mode."""
import pytest
import torch
import torch.nn.functional as F

from parity import compare_lists, check_tie_order

pytestmark = pytest.mark.gpu
DEV = "cuda"
ALL = 2 ** 40                                            # threshold-only: every neighbour with cosine >= thr


def _features(n, d, kind, seed):
    from sngnn_b200 import synth
    return synth.make_features(n, d, kind, seed=seed, dup_frac=0.01, zero_rows=3)


def _k_eff(n, k, rs):
    return min(k, n - (1 if rs else 0))


def _oracle(x, k, thr, rs, q_lo=0, q_hi=None):
    from oracle import sn_ref
    return sn_ref.simknn_allpairs(x.double(), _k_eff(x.size(0), k, rs), thr, rs, q_lo, q_hi, dtype=torch.float64)


def _score64(x):
    from oracle import sn_ref
    n64 = sn_ref.rownorm(x.double())
    return lambda r, j: (n64[r] * n64[j]).sum(-1)


def _check(x, k, thr, rs, out, q_lo=0, q_hi=None):
    idx, sim, cnt = out[:3]
    n = x.size(0)
    assert idx.shape == (idx.size(0), _k_eff(n, k, rs)) and idx.dtype == torch.int32
    idx_ref, sim_ref, cnt_ref = _oracle(x, k, thr, rs, q_lo, q_hi)
    score = _score64(x)
    res = compare_lists(idx, cnt, idx_ref, cnt_ref, lambda r, j: score(r + q_lo, j), thr)
    assert res["out_of_band"] == 0, res
    assert check_tie_order(idx, sim, cnt)
    kk = idx.size(1)
    same = (idx.cpu().long() == idx_ref) & (torch.arange(kk)[None, :] < cnt.cpu()[:, None])
    if same.any():
        assert (sim.cpu().double()[same] - sim_ref[same]).abs().max() < (2e-6 if x.size(1) <= 512 else 1e-5)
    return res


CASES = [(3000, 65, 100, -1.0, True, "normal"), (3000, 65, 256, 0.5, True, "clustered"), (2000, 8, 1000, -1.0, False, "normal"),
         (2000, 128, ALL, 0.9, True, "clustered"), (1500, 512, 65, 0.5, False, "clustered"), (1200, 2325, 100, 0.5, True, "binary"),
         (2500, 65, ALL, 0.5, True, "binary"), (4000, 65, 100, 0.9, False, "binary"), (1000, 8, 256, 0.9, True, "clustered"),
         (2000, 65, ALL, -1.0, True, "clustered")]


@pytest.mark.parametrize("n,d,k,thr,rs,kind", CASES)
def test_wide_build_matches_oracle(n, d, k, thr, rs, kind):
    from sngnn_b200 import simknn
    x = _features(n, d, kind, seed=5 * n + d)
    out = simknn.build_knn(x.to(DEV), k, thr, rs, return_fallback=True)
    torch.cuda.synchronize()
    res = _check(x, k, thr, rs, out)
    print(f"wide n={n} d={d} k={k} thr={thr} rs={rs} {kind}: {res} exact_rows={int(out[3][0])}")


@pytest.mark.parametrize("n,d,k,thr,kind", [(20000, 65, 100, -1.0, "clustered"), (36000, 65, 256, 0.0, "normal"), (20000, 128, 1000, 0.5, "clustered")])
def test_seeded_wide_build_matches_oracle(n, d, k, thr, kind):
    """Databases large enough for the seed pass (the emission threshold then comes from the sample's group maxima)."""
    from sngnn_b200 import simknn
    x = _features(n, d, kind, seed=n + k)
    out = simknn.build_knn(x.to(DEV), k, thr, True, return_fallback=True)
    torch.cuda.synchronize()
    lo, hi = n // 3, n // 3 + 600
    res = _check(x, k, thr, True, tuple(t[lo:hi] for t in out[:3]), lo, hi)
    print(f"seeded wide n={n} k={k}: {res} exact_rows={int(out[3][0])}")


@pytest.mark.parametrize("n,d,thr", [(3000, 65, -1.0), (20000, 65, 0.0)])
def test_first_64_entries_equal_the_k64_build(n, d, thr):
    from sngnn_b200 import simknn
    x = _features(n, d, "clustered", seed=n).to(DEV)
    i64, s64, c64 = simknn.build_knn(x, 64, thr, True)
    iw, sw, cw = simknn.build_knn(x, 100, thr, True)
    rows = cw >= 64
    assert rows.any()
    assert torch.equal(iw[rows, :64], i64[rows]) and torch.equal(sw[rows, :64], s64[rows])
    assert torch.equal(torch.minimum(cw, torch.full_like(cw, 64)), c64)


@pytest.mark.parametrize("n,d,pats,k", [(3000, 40, 5, 100), (40000, 24, 2, 100)])
def test_massive_ties_and_duplicates_go_through_the_exact_scan(n, d, pats, k):
    """A few distinct rows repeated thousands of times: with two patterns (one all-zero) every non-zero row ties at cosine 1
    with ~20,000 columns, more candidates than a block sorts, so those rows take the exact scan; zero rows are answered by rule."""
    from sngnn_b200 import simknn
    g = torch.Generator().manual_seed(n)
    p = torch.randn(pats, d, generator=g)
    p[0] = 0
    x = p[torch.randint(0, pats, (n,), generator=g)]
    out = simknn.build_knn(x.to(DEV), k, -1.0, True, return_fallback=True)
    torch.cuda.synchronize()
    if n > 20000:
        assert int(out[3][0]) > 0
    lo, hi = (0, n) if n <= 5000 else (n // 2, n // 2 + 400)
    _check(x, k, -1.0, True, tuple(t[lo:hi] for t in out[:3]), lo, hi)


def test_lists_wider_than_a_block_sort():
    """Threshold-only at thr = -1 on 20,000 rows: every list holds 19,999 entries, more than the 16,384 a block sorts in
    shared memory, so rows are ranked in global memory."""
    from sngnn_b200 import simknn
    n, d = 20000, 16
    x = _features(n, d, "normal", seed=3)
    xf, xh = simknn.normalize_operands(x.to(DEV))
    lo, hi = 5000, 5040
    out = simknn.build_knn_normalized(xf, xh, d, ALL, -1.0, True, lo, hi)
    torch.cuda.synchronize()
    assert out[0].shape == (hi - lo, n - 1) and bool((out[2] == n - 1).all())
    _check(x, ALL, -1.0, True, out, lo, hi)


def test_deterministic_and_row_shards_equal_the_full_build():
    from sngnn_b200 import simknn
    n, d, k = 3000, 65, 100
    x = _features(n, d, "clustered", seed=9).to(DEV)
    full = simknn.build_knn(x, k, 0.2, True)
    again = simknn.build_knn(x, k, 0.2, True)
    for a, b in zip(full, again):
        assert torch.equal(a, b)
    parts = [simknn.build_knn(x, k, 0.2, True, q_lo=lo, q_hi=hi) for lo, hi in ((0, 1000), (1000, 1001), (1001, 3000))]
    for t in range(3):
        assert torch.equal(full[t], torch.cat([p[t] for p in parts]))
    h = torch.randn(n, 16, device=DEV)
    empty = simknn.allpairs_topk_agg(h, k, 0.2, True, rows=(700, 700))
    assert empty.shape == (0, 16)


# ------------------------------------------------------------------------------------------ ListAgg at k > 64
def _rel(a, b):
    return float((a.double() - b.double()).abs().max() / (b.double().abs().max() + 1e-30))


@pytest.mark.parametrize("c", [4, 32, 128])
@pytest.mark.parametrize("k", [100, 1000])
@pytest.mark.parametrize("denominator", ["candidates", "selected"])
def test_list_agg_forward_backward_vs_fp64(c, k, denominator):
    from sngnn_b200 import functional as SF, simknn
    from oracle import sn_ref
    n = 2000
    torch.manual_seed(c + k)
    h = torch.randn(n, c, device=DEV)
    w = torch.randn(n, c, device=DEV)
    idx, sim, cnt = simknn.build_knn(h, k, 0.0, True)
    inv = (torch.full((n,), 1.0 / (n - 1), device=DEV) if denominator == "candidates" else 1.0 / cnt.clamp(min=1).float())

    def run():
        hd = h.clone().requires_grad_(True)
        out = SF.ListAgg.apply(hd, idx, sim, cnt, inv, 0)
        (out * w).sum().backward()
        return out.detach(), hd.grad

    out, dh = run()
    out2, dh2 = run()
    assert torch.equal(out, out2) and torch.equal(dh, dh2)
    h64 = h.double().cpu().requires_grad_(True)
    idx64 = idx.long().cpu()
    n64 = F.normalize(h64, dim=-1, eps=1e-12)
    s64 = torch.where(idx64 >= 0, (n64[:, None, :] * n64[idx64.clamp(min=0)]).sum(-1), torch.zeros((), dtype=torch.float64))
    ref = sn_ref.knn_mean_aggregate(h64, idx64, s64, cnt.long().cpu(), (1.0 / inv.double()).cpu())
    (ref * w.double().cpu()).sum().backward()
    assert _rel(out.cpu(), ref.detach()) < 1e-5
    assert _rel(dh.cpu(), h64.grad) < 1e-5


@pytest.mark.parametrize("denominator", ["candidates", "selected"])
def test_list_agg_shards_add_up(denominator):
    from sngnn_b200 import simknn
    n, c, k = 1500, 32, 100
    torch.manual_seed(1)
    h = torch.randn(n, c, device=DEV)
    w = torch.randn(n, c, device=DEV)

    def run(rows):
        hd = h.clone().requires_grad_(True)
        out = simknn.allpairs_topk_agg(hd, k, 0.0, True, denominator, rows=rows)
        lo = 0 if rows is None else rows[0]
        (out * w[lo:lo + out.size(0)]).sum().backward()
        return out.detach(), hd.grad

    out_full, dh_full = run(None)
    parts = [run(b) for b in ((0, 0), (0, 700), (700, 700), (700, n))]
    assert not parts[0][1].any()
    assert torch.equal(torch.cat([o for o, _ in parts]), out_full)
    assert _rel(sum(d for _, d in parts), dh_full) < 1e-5


# ------------------------------------------------------------------------------------------ models
def test_allpairs_conv_at_k100_matches_the_oracle():
    """SNConv_plus(candidates='all_pairs', top_k=100) == the reference conv run on the complete graph."""
    import sngnn_b200.models as M
    from oracle import sn_ref
    torch.manual_seed(0)
    n, fd, c, k, thr = 700, 24, 8, 100, 0.1
    x = torch.randn(n, fd)
    conv = M.SNConv_plus(fd, c, n, k, thr, True, candidates="all_pairs").to(DEV)
    out = conv(x.to(DEV), torch.zeros(2, 0, dtype=torch.long, device=DEV))
    src = torch.arange(n).repeat(n); dst = torch.arange(n).repeat_interleave(n)
    keep = src != dst
    ei = torch.stack([src[keep], dst[keep]])
    h = F.linear(x, conv.lin.weight.detach().cpu(), conv.lin.bias.detach().cpu())
    ref = sn_ref.sn_aggregate(h, ei, k, thr)
    torch.testing.assert_close(out.detach().cpu(), ref, rtol=1e-4, atol=1e-6)


@pytest.mark.parametrize("kind", ["SNGNN_Plus", "SNGNN_Plus_Plus"])
@pytest.mark.parametrize("denominator", ["candidates", "selected"])
def test_models_at_k100_world1_sharded_and_eval(kind, denominator):
    """Both models with candidates='all_pairs', top_k=100: world-1 sharded_forward equals model(data), logits and gradients;
    under no_grad in eval mode the output is the training output bit for bit."""
    import sngnn_b200.models as M
    from sngnn_b200 import dist as D, functional as SF, synth
    n, fd, hid, ncls = 2001, 24, 32, 5
    x = synth.make_features(n, fd, "clustered", seed=1).to(DEV)
    ei = synth.make_graph(n, 20000, seed=2, symmetric=True, hub_offset=3.0).to(DEV)
    y = synth.make_labels(n, ncls, seed=3).to(DEV)
    torch.manual_seed(7)
    if kind == "SNGNN_Plus_Plus":
        model = M.SNGNN_Plus_Plus(fd, hid, ncls, n, 2, 100, 0.1, 0.5, 1, 0.0, candidates="all_pairs", denominator=denominator)
    else:
        model = M.SNGNN_Plus(fd, hid, ncls, n, 2, 100, 0.1, 1, 0.0, candidates="all_pairs", denominator=denominator)
    model = model.to(DEV).train()
    logp = D.sharded_forward(model, x, ei, n)
    SF.nll_loss(logp, y).backward()
    g1 = {name: p.grad.clone() for name, p in model.named_parameters()}
    model.zero_grad()
    ref = model(synth.GraphData(x, ei))
    SF.nll_loss(ref, y).backward()
    assert torch.equal(logp.detach(), ref.detach())
    for name, p in model.named_parameters():
        assert _rel(g1[name], p.grad) < 2e-5, name
    model.eval()
    with torch.no_grad():
        assert torch.equal(model(synth.GraphData(x, ei)), ref.detach())
