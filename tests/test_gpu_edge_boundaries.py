"""The edge kernels at their dispatch boundaries: sng_edge_fwd / sng_edge_bwd and sng_list_agg_fwd / sng_list_bwd.

The kernels branch on three axes, and each branch has its own masks and its own tie-break code:
  * channel width: G = group_lanes(c) float4 slots per row, the smallest power of two >= c / 4.  When c / 4 is not a power
    of two (a "ragged" width: 12, 20, 100, 132, ...) the last lanes or slots of a row hold no data;
  * degree class: at c <= 32 rows of <= 32 in-edges run the staged kernel and longer rows are cut into 32-edge chunks that
    a merge kernel combines (a register tournament for top_k <= 16, sorted insertion above, two winners per lane above 32);
    at c > 32 the long-row kernel runs every row and rows of more than 1,024 in-edges go to the hub kernel.  The
    backward's source pass splits on out-degrees the same way;
  * top_k: the staged pass T of the backward runs up to top_k = 32, the general kernel above.
This file puts rows exactly at those boundaries and checks every width class, exact and ragged, against the FP64 oracle:
  A. _boundary_graph: rows with in- and out-degrees 0, 1, 31 | 32 | 33, 63 | 64 | 65, 1023 | 1024 | 1025 and 1057, and
     duplicate edges (the construction is checked on the host, without a GPU);
  B. width x path: EdgeAgg, the fused and the two-kernel (K4) SNGNN++ layer, row shards and the list aggregation;
  C. exact score ties (scaled twin rows, orthogonal neighbours, duplicate edges): the selection ORDER is asserted index for
     index against the oracle's rank rule (score desc, edge position asc) -- no FP64 band;
  D. leading dimensions > c through the C ABI, NaN in the input padding and a sentinel in the output padding: the results
     must equal the ld == c call bit for bit;
  E. the staged forms against the general kernels on the same rows.
Tolerances are those of the rest of the suite: out within rtol 1e-5 / atol 1e-6 of FP64, gradients within 1e-5 of their
largest magnitude, backward passes bit-reproducible."""
import functools

import pytest
import torch
import torch.nn.functional as F

from parity import compare_lists

DEV = "cuda"
N_BOUNDARY = 3000
PLANTED = (0, 1, 31, 32, 33, 63, 64, 65, 1023, 1024, 1025, 1057)   # 1057 = 33 chunks, the last one a single edge
DUP_DEGREES = (33, 65, 1025)                                        # planted rows whose first two edges share their source

# an exact and a ragged width of every lane-group size G: 1 (4), 2 (8), 4 (12, 16), 8 (20, 28), 16 (36, 40), 32 (68, 100, 124),
# 64 (132, 252), 128 (260, 508)
WIDTHS = (4, 8, 12, 16, 20, 28, 36, 40, 68, 100, 124, 132, 252, 260, 508)


def _rel(a, b):
    a, b = a.detach().cpu().double(), b.detach().cpu().double()
    return float((a - b).abs().max() / (b.abs().max() + 1e-30))


# ------------------------------------------------------------------------------------------ A. the boundary graph
def _planted_nodes(n):
    """(targets, sources): the node planted with in-degree PLANTED[i] is targets[i]; in an asymmetric graph the node planted
    with out-degree PLANTED[i] is sources[i].  Both sit at the top of the id range, so node 0 keeps its out-edge (src shift 0)
    and the hubs come last: targets[-2] (1025 edges) and targets[-1] (1057)."""
    m = len(PLANTED)
    return list(range(n - m, n)), list(range(n - 2 * m, n - m))


def _boundary_graph(n, seed, symmetric, rsl):
    """edge_index [2, E] of a sparse synth.make_graph background in which every edge touching a planted node is replaced by
    exactly the planted ones: target rows whose in-degree after graph.prepare(ei, n, rsl) is each of PLANTED (in-degree 0
    only with rsl: otherwise the appended self loop counts) and, for an asymmetric graph, source rows with those
    out-degrees (pass S of the backward dispatches on them).  The rows of DUP_DEGREES hold one duplicate edge each, which
    prepare keeps.  A symmetric graph is sorted row-major, so its in-lists equal its out-lists (the fused SNGNN++ pass); an
    asymmetric one is shuffled, so edge-position order differs from source-id order."""
    from sngnn_b200 import synth
    targets, sources = _planted_nodes(n)
    pool = n - 2 * len(PLANTED)                                   # planted edges connect planted nodes to nodes [0, pool)
    ei = synth.make_graph(n, 4 * n, seed=seed, symmetric=symmetric)
    ei = ei[:, (ei < pool).all(0)]
    gen = torch.Generator().manual_seed(seed)
    loop = 0 if rsl else 1
    extra = []
    for d, t, s in zip(PLANTED, targets, sources):
        if d - loop < 0:
            continue
        for node, incoming in ((t, True),) + ((() if symmetric else ((s, False),))):
            nb = torch.randperm(pool, generator=gen)[:d - loop]
            if d in DUP_DEGREES:
                nb[1] = nb[0]
            me = torch.full_like(nb, node)
            extra.append(torch.stack([nb, me]) if incoming else torch.stack([me, nb]))
    ex = torch.cat(extra, 1)
    if symmetric:
        ex = torch.cat([ex, ex.flip(0)], 1)
    ei = torch.cat([ei, ex], 1)
    if symmetric:
        ei = ei[:, torch.argsort(ei[0] * n + ei[1], stable=True)]
    else:
        ei = ei[:, torch.randperm(ei.size(1), generator=gen)]
    return ei.contiguous()


def _chunks_of(tab, ptr, rows, r):
    i = rows.tolist().index(r)
    return tab[int(ptr[i]):int(ptr[i + 1])]


@pytest.mark.parametrize("symmetric,rsl", [(True, True), (False, True), (True, False), (False, False)])
def test_boundary_graph_plants_every_degree_class(symmetric, rsl):
    """Host construction of graph.prepare on the boundary graph: every planted in-degree (and out-degree) is present, the
    degree lists and the chunk tables of both passes cut each planted row into 32 ... 32, tail edges, only the planted
    rows are hubs, duplicates are kept, and the symmetric flag (the fused SNGNN++ pass) is what the builder promises."""
    from sngnn_b200 import graph as G
    n = N_BOUNDARY
    ei = _boundary_graph(n, 7, symmetric, rsl)
    g = G.prepare(ei, n, rsl)
    assert g.symmetric == symmetric and g.src_shift == 0
    targets, sources = _planted_nodes(n)
    deg_in = (g.rowptr_in[1:] - g.rowptr_in[:-1]).long()
    deg_out = (g.rowptr_out[1:] - g.rowptr_out[:-1]).long()
    planted = [(d, t, t if symmetric else s) for d, t, s in zip(PLANTED, targets, sources) if rsl or d > 0]
    assert len(planted) == len(PLANTED) - (0 if rsl else 1)
    long_rows, hub_rows = set(g.rows_long.tolist()), set(g.rows_hub.tolist())
    assert hub_rows == {t for d, t, _ in planted if d > 1024}
    for d, t, s in planted:
        assert int(deg_in[t]) == d and int(deg_out[s]) == d, (d, int(deg_in[t]), int(deg_out[s]))
        assert (t in long_rows) == (32 < d <= 1024) and (t in hub_rows) == (d > 1024), d
        src = g.col_in[int(g.rowptr_in[t]):int(g.rowptr_in[t + 1])]
        assert (src.unique().numel() < d) == (d in DUP_DEGREES), d
        want = [32] * (d // 32) + ([d % 32] if d % 32 else [])
        if d <= 32:
            assert t not in g.lrows.tolist() and s not in g.lrows_out.tolist()
            continue
        ch = _chunks_of(g.chunk_tab, g.lrow_ptr, g.lrows, t)
        assert ch[:, 1].tolist() == want, d
        assert ch[:, 0].tolist() == [int(g.rowptr_in[t]) + 32 * i for i in range(len(want))]
        assert (ch[:, 2] == t).all() and (ch[:, 3] == 0).all()
        cho = _chunks_of(g.chunk_tab_out, g.lrow_ptr_out, g.lrows_out, s)
        assert cho[:, 1].tolist() == want, d
        assert cho[:, 0].tolist() == [int(g.rowptr_out[s]) + 32 * i for i in range(len(want))]
    if rsl:
        assert int(deg_in[targets[0]]) == 0


@functools.lru_cache(maxsize=None)
def _device_graph(symmetric, rsl=True):
    """(edge_index on the host, edge_index on the GPU, its PreparedGraph) of the boundary graph.  The device tensor is kept
    alive here, so graph.prepare's cache keeps returning the same PreparedGraph."""
    from sngnn_b200 import graph as G
    ei = _boundary_graph(N_BOUNDARY, 11 if symmetric else 13, symmetric, rsl)
    eid = ei.to(DEV)
    return ei, eid, G.prepare(eid, N_BOUNDARY, rsl)


def _features(n, c, seed):
    """Rows of width c with every column non-zero: the kernels see a ragged width, not a zero-padded narrower one."""
    x = torch.randn(n, c, generator=torch.Generator().manual_seed(seed))
    return torch.where(x == 0, torch.ones_like(x), x)


def _cases(cp):
    """(top_k, thr) runs of a width: both sides of every top_k boundary at the narrow end, fewer at the wide end; None =
    select all."""
    if cp <= 32:
        ks = [(k, thr) for k in (1, 16, 17, 32, 33, 64) for thr in (0.0, -1.0)]
    elif cp <= 128:
        ks = [(k, (0.0, -1.0)[i % 2]) for i, k in enumerate((1, 16, 17, 32, 33, 64))]
    else:
        ks = [(17, 0.0), (33, -1.0), (64, 0.0)]
    return ks + [(None, None)]


def _oracle_lists(h64, pe, n, k, thr):
    """The oracle's selection (R: models/models.py:145-154): idx [n, k] source ids in rank order (-1 padded), cnt [n], and
    epos [n, k] = the position of each selected edge in the processed edge list."""
    from oracle import sn_ref
    nrm = F.normalize(h64.detach(), dim=-1, eps=1e-12)
    s = (nrm[pe[1]] * nrm[pe[0]]).sum(-1)
    rank = sn_ref.edge_rank(s, pe[1])
    sel = (rank < k) & (s >= thr)
    idx = torch.full((n, k), -1, dtype=torch.long)
    epos = torch.full((n, k), -1, dtype=torch.long)
    idx[pe[1][sel], rank[sel]] = pe[0][sel]
    epos[pe[1][sel], rank[sel]] = sel.nonzero().flatten()
    cnt = torch.zeros(n, dtype=torch.long).index_add_(0, pe[1][sel], torch.ones(int(sel.sum()), dtype=torch.long))
    return idx, cnt, epos, nrm


# ------------------------------------------------------------------------------------------ B. width x path
@pytest.mark.gpu
@pytest.mark.parametrize("cp", WIDTHS)
def test_edge_agg_every_width_and_degree_class_vs_fp64(cp):
    """EdgeAgg (sng_edge_fwd + sng_edge_bwd) on the asymmetric boundary graph, at both sides of every top_k boundary and
    select-all: out and dL/dh against FP64 autograd of the oracle, the backward bit-reproducible, the lists within the FP64
    band, and the row of in-degree 0 empty (count 0, -1 padding, out = 0)."""
    from oracle import sn_ref
    from sngnn_b200 import functional as SF
    ei, _, g = _device_graph(False)
    n = g.n
    pe = sn_ref.process_edges(ei, n, True)
    h = _features(n, cp, seed=cp)
    w = torch.randn(n, cp, generator=torch.Generator().manual_seed(cp + 1))
    wd = w.to(DEV)
    z = _planted_nodes(n)[0][0]
    for k, thr in _cases(cp):
        tag = f"cp={cp} k={k} thr={thr}"

        def run():
            hd = h.to(DEV).requires_grad_(True)
            out, (ss, sw, sc) = SF.edge_topk_agg(hd, g, k, thr, return_selection=True)
            (out * wd).sum().backward()
            return out.detach(), ss, sc, hd.grad

        out, ss, sc, dh = run()
        out2, _, _, dh2 = run()
        assert torch.equal(out, out2) and torch.equal(dh, dh2), tag
        h64 = h.double().requires_grad_(True)
        ref = sn_ref.sn_aggregate(h64, pe, k, thr)
        (ref * w.double()).sum().backward()
        torch.testing.assert_close(out.cpu().double(), ref.detach(), rtol=1e-5, atol=1e-6, msg=lambda m: f"{tag}: {m}")
        assert _rel(dh, h64.grad) < 1e-5, (tag, _rel(dh, h64.grad))
        assert float(out[z].abs().max()) == 0, tag
        if k is None:
            continue
        idx_ref, cnt_ref, _, nrm = _oracle_lists(h64, pe, n, k, thr)
        res = compare_lists(ss, sc, idx_ref, cnt_ref, lambda r, j: (nrm[r] * nrm[j]).sum(-1), thr)
        assert res["out_of_band"] == 0 and res["exact"] >= n - 3, (tag, res)
        assert int(sc[z]) == 0 and bool((ss[z] == -1).all()), tag


# output widths of the layer tests: C = 3, 6, 10, 18 are padded to Cp = 4, 8, 12, 20 (the padding columns of h are zero);
# the others reach the kernels as they are
LAYER_WIDTHS = (3, 6, 10, 12, 18, 20, 28, 36, 68, 100, 132, 260, 508)


@pytest.mark.gpu
@pytest.mark.parametrize("form", ["fused", "k4"])
@pytest.mark.parametrize("c", LAYER_WIDTHS)
def test_snconv_plus_plus_every_width_vs_fp64(c, form):
    """One SNConv_plus_plus layer: the fused single pass on the symmetric boundary graph, the two-kernel form (EdgeAgg, then
    sng_pp_fuse_fwd / _bwd) on the asymmetric one.  Output and the gradients of x, lin, W^T, b_w, beta and bias against FP64
    autograd; the backward bit-reproducible; a row with no in- and no out-edges gives beta b_w + bias."""
    from oracle import sn_ref
    import sngnn_b200.models as M
    from sngnn_b200 import functional as SF
    ei, eid, g = _device_graph(form == "fused")
    assert g.symmetric == (form == "fused")
    n, fd = g.n, 16
    cp = SF.padded_channels(c)
    z = _planted_nodes(n)[0][0]
    x = _features(n, fd, seed=c + 100)
    wgt = torch.randn(n, c, generator=torch.Generator().manual_seed(c + 200))
    cases = [(1, -1.0), (16, 0.0), (17, -1.0), (32, 0.0), (33, -1.0), (64, 0.0)] if cp <= 32 else [(17, 0.0), (33, -1.0)]
    if cp <= 32 and form == "k4":
        cases = cases[1::2]
    elif cp <= 32:
        cases = cases[0::2] + [(17, 0.0)]
    for k, thr in cases:
        tag = f"{form} c={c} k={k} thr={thr}"
        torch.manual_seed(c * 7 + k)
        conv = M.SNConv_plus_plus(fd, c, n, k, thr, 0.3, True, bias=True).to(DEV)
        with torch.no_grad():
            conv.bias.normal_()
        xd = x.to(DEV).requires_grad_(True)
        wd = wgt.to(DEV)

        def run():
            conv.zero_grad()
            xd.grad = None
            out = conv(xd, eid)
            (out * wd).sum().backward()
            return out.detach().clone(), {kk: p.grad.detach().clone() for kk, p in conv.named_parameters()}, xd.grad.detach().clone()

        out, grads, dx = run()
        out2, grads2, dx2 = run()
        assert torch.equal(out, out2) and torch.equal(dx, dx2), tag
        for kk in grads:
            if kk not in ("lin.weight", "lin.bias"):                          # the dense lin backward may be a library GEMM
                assert torch.equal(grads[kk], grads2[kk]), (tag, kk)
        with torch.no_grad():
            torch.testing.assert_close(out[z], conv.beta * conv.w.bias + conv.bias, rtol=1e-6, atol=1e-7, msg=lambda m: f"{tag}: {m}")
        p64 = {kk: p.detach().cpu().double().contiguous().requires_grad_(True) for kk, p in conv.named_parameters()}
        x64 = x.double().requires_grad_(True)
        ref = sn_ref.snconv_plus_plus(x64, ei, p64["lin.weight"], p64["lin.bias"], p64["w.weight"], p64["w.bias"], p64["beta"], k, thr,
                                      True, p64["bias"])
        (ref * wgt.double()).sum().backward()
        torch.testing.assert_close(out.cpu().double(), ref.detach(), rtol=1e-5, atol=2e-6, msg=lambda m: f"{tag}: {m}")
        for kk in grads:
            r = p64[kk].grad
            scale = r.abs().max() + 1e-12
            if kk == "beta":                                                  # a signed sum of n c terms (see test_gpu_edge.py)
                scale = torch.maximum(scale, 1e-2 * (wgt.double().abs() * ref.detach().abs()).sum())
            err = float((grads[kk].cpu().double() - r).abs().max() / scale)
            assert err < 1e-5, (tag, kk, err)
        assert _rel(dx, x64.grad) < 1e-5, (tag, _rel(dx, x64.grad))


@pytest.mark.gpu
@pytest.mark.parametrize("cp,k,thr", [(12, 17, 0.0), (20, 33, -1.0), (28, 16, 0.0), (36, 16, -1.0), (100, 33, 0.0), (132, 64, -1.0)])
def test_sharded_edge_agg_ragged_shards(cp, k, thr):
    """ShardedEdgeTopkAgg on ragged row shards of the asymmetric boundary graph: a boundary just before the 1025-edge hub,
    shards of one row.  Every shard's output equals the unsharded rows bit for bit, and the contributions to dL/dh add up to
    the unsharded gradient."""
    from sngnn_b200 import functional as SF
    _, _, g = _device_graph(False)
    n = g.n
    targets, _ = _planted_nodes(n)
    hub = targets[PLANTED.index(1025)]
    h = _features(n, cp, seed=cp + 300).to(DEV)
    w = torch.randn(n, cp, generator=torch.Generator().manual_seed(cp + 301)).to(DEV)
    h0 = h.clone().requires_grad_(True)
    out0 = SF.edge_topk_agg(h0, g, k, thr)
    (out0 * w).sum().backward()
    for bounds in ([(0, hub), (hub, n)], [(0, hub), (hub, hub + 1), (hub + 1, n)], [(0, 1), (1, n - 1), (n - 1, n)]):
        total = torch.zeros_like(h)
        for lo, hi in bounds:
            hs = h.clone().requires_grad_(True)
            out = SF.ShardedEdgeTopkAgg.apply(hs, g.row_slice(lo, hi), lo, k, thr)
            assert torch.equal(out.detach(), out0.detach()[lo:hi]), (bounds, lo, hi)
            (out * w[lo:hi]).sum().backward()
            total += hs.grad
        assert _rel(total, h0.grad) < 1e-5, (bounds, _rel(total, h0.grad))


N_LIST = 1200


def _boundary_lists(n, k, seed):
    """Lists idx [n, k] / cnt [n] with duplicates, empty rows, cnt < k and -1 padding; column 0 is in every non-empty list
    (more than 1,024 entries: a chunked source row), column 1 in exactly 33 lists and column 2 in exactly 32."""
    gen = torch.Generator().manual_seed(seed)
    idx = torch.randint(3, n, (n, k), generator=gen, dtype=torch.int32)
    cnt = torch.randint(1, k + 1, (n,), generator=gen, dtype=torch.int32)
    cnt[::11] = 0
    cnt[1::5] = k
    if k > 2:
        idx[::3, 2] = idx[::3, 1]                                           # duplicate entries
    idx[:, 0] = 0
    if k > 1:
        many = (cnt >= 2).nonzero().flatten()
        idx[many[:33], 1] = 1
        idx[many[33:65], 1] = 2
    idx[torch.arange(k)[None, :] >= cnt[:, None]] = -1
    return idx, cnt


@pytest.mark.gpu
@pytest.mark.parametrize("cp", WIDTHS)
def test_list_agg_every_width_vs_fp64(cp):
    """ListAgg (sng_list_agg_fwd + sng_list_bwd) at every width class on lists with duplicates, cnt < k and source rows of
    32, 33 and > 1,024 entries: out and dL/dh against FP64 autograd of the oracle, bit-reproducible."""
    from oracle import sn_ref
    from sngnn_b200 import functional as SF
    n = N_LIST
    h = _features(n, cp, seed=cp + 400)
    w = torch.randn(n, cp, generator=torch.Generator().manual_seed(cp + 401))
    for k in ((16, 17, 33) if cp <= 128 else (17, 64)):
        tag = f"cp={cp} k={k}"
        idx, cnt = _boundary_lists(n, k, seed=cp + k)
        col = torch.bincount(idx[idx >= 0].long(), minlength=n)
        assert int(col[0]) > 1024 and int(col[1]) == 33 and int(col[2]) == 32, tag
        h64 = h.double().requires_grad_(True)
        n64 = F.normalize(h64, dim=-1, eps=1e-12)
        s64 = torch.where(idx >= 0, (n64[:, None, :] * n64[idx.long().clamp(min=0)]).sum(-1), torch.zeros((), dtype=torch.float64))
        inv = 1.0 / cnt.clamp(min=1).double()
        args = (idx.to(DEV), s64.detach().float().to(DEV), cnt.to(DEV), inv.float().to(DEV))

        def run():
            hd = h.to(DEV).requires_grad_(True)
            out = SF.ListAgg.apply(hd, *args)
            (out * w.to(DEV)).sum().backward()
            return out.detach(), hd.grad

        out, dh = run()
        out2, dh2 = run()
        assert torch.equal(out, out2) and torch.equal(dh, dh2), tag
        ref = sn_ref.knn_mean_aggregate(h64, idx.long(), s64, cnt.long(), 1.0 / inv)
        (ref * w.double()).sum().backward()
        torch.testing.assert_close(out.cpu().double(), ref.detach(), rtol=1e-5, atol=1e-6, msg=lambda m: f"{tag}: {m}")
        assert _rel(dh, h64.grad) < 1e-5, (tag, _rel(dh, h64.grad))


# ------------------------------------------------------------------------------------------ C. exact selection order
# Rank groups of the designed candidates of a tie row, best first: every group is one score, so its members are exact ties
# and rank by edge position.  Group 7 covers ranks 15-17 (both sides of the tournament / insertion switch at top_k 16 | 17),
# group 14 ranks 30-33 (top_k 32 | 33, pass T staged | general), group 27 ranks 62-64 (top_k = 64).
TIE_GROUPS = (2, 3, 2, 2, 2, 2, 2, 3, 2, 2, 2, 2, 2, 2, 4, 2, 3, 2, 2, 2, 2, 2, 3, 2, 2, 4, 2, 3, 2)
TWIN = (1.0, 2.0, 4.0, 0.5)                     # scale factors of a group's members: power-of-two scaling keeps the cosine exact

# tie rows: (name, in-degree, designed candidates, {group: edge positions it must contain}); candidates beyond the designed
# ones score below all of them (and below 0)
TIE_ROWS = (
    ("short", 32, 32, {0: [0, 31], 7: [16, 17, 1]}),                    # one warp of the staged kernel: lane 0 vs lane 31
    ("short20", 20, 20, {0: [19, 3], 1: [0, 18]}),
    ("chunks", 97, 66, {0: [31, 32], 1: [63, 64, 0], 2: [96, 33], 7: [30, 34, 95], 14: [62, 65, 1]}),   # across chunk boundaries
    ("long", 300, 66, {0: [290, 5], 1: [160, 161], 7: [31, 32, 299], 14: [63, 64, 250, 0], 27: [95, 96, 2]}),
    # hub (> 1,024 edges): warp w of the hub kernel scans chunks w, w + 8, ...: group 0 is one warp's chunks 1 and 9,
    # group 1 two warps, group 2 the tail chunk and warp 7
    ("hub", 1100, 66, {0: [40, 296], 1: [10, 50], 2: [1099, 250], 7: [300, 5, 1090], 14: [31, 32, 520, 800], 27: [64, 63, 1000]}),
)
DUP_ROW = ("dup", 40, {0: [31, 32], 1: [5, 6], 2: [0, 39]})            # each group is ONE source node listed twice
ORTH_ROWS = (("orth", 70), ("orth_hub", 1030))                         # every score exactly 0


def _level_vectors(t, m, gen, lo=0.95, step=0.012):
    """m unit vectors of cosine lo - step * l with t (l = 0 .. m-1), in FP64."""
    th = t / t.norm()
    u = torch.randn(m, t.numel(), generator=gen, dtype=torch.float64)
    u = u - (u @ th)[:, None] * th[None, :]
    u = u / u.norm(dim=1, keepdim=True)
    cos = lo - step * torch.arange(m, dtype=torch.float64)
    return cos[:, None] * th[None, :] + (1 - cos ** 2).sqrt()[:, None] * u


def _tie_problem(cp, twins, seed=0):
    """A graph (rsl=True) whose target rows hold exact score ties at chosen edge positions, with features of width cp.
    Returns (edge_index [2, E], h [n, cp], info) with info = {row name: (target node, [source node per edge position])} and
    info["twins"] = [(node, factor, group id)] of every twin member.  twins=False makes the members of a group exact copies
    instead of power-of-two multiples."""
    gen = torch.Generator().manual_seed(seed)
    names = [r[0] for r in TIE_ROWS] + [DUP_ROW[0]] + [r[0] for r in ORTH_ROWS] + ["empty"]
    n_src = sum(r[1] for r in TIE_ROWS) + DUP_ROW[1] + sum(r[1] for r in ORTH_ROWS)
    n = len(names) + n_src
    h = torch.zeros(n, cp, dtype=torch.float64)
    info, twin_members = {}, []
    nxt = len(names)                                                    # targets first: min(src) > 0, a non-zero source shift
    edges = []
    for ti, (name, deg, m, forced) in enumerate(TIE_ROWS):
        t = torch.randn(cp, generator=gen, dtype=torch.float64)
        h[ti] = t
        sizes = list(TIE_GROUPS)
        while sum(sizes) > m:
            sizes[-1] -= 1
            if sizes[-1] == 0:
                sizes.pop()
        sizes[-1] += m - sum(sizes)
        used = {p for ps in forced.values() for p in ps}
        free = [p for p in torch.randperm(deg, generator=gen).tolist() if p not in used]
        levels = _level_vectors(t, len(sizes), gen)
        srcs = [None] * deg
        for gi, size in enumerate(sizes):
            pos = list(forced.get(gi, []))
            assert len(pos) <= size
            while len(pos) < size:
                pos.append(free.pop())
            fac = [TWIN[i] for i in torch.randperm(size, generator=gen).tolist()] if size <= 4 else [1.0] * size
            for p, f in zip(pos, fac):
                h[nxt] = levels[gi].float().double() * (f if twins else 1.0)
                twin_members.append((nxt, f if twins else 1.0, (ti, gi)))
                srcs[p] = nxt
                nxt += 1
        fill = _level_vectors(-t, len(free), gen, lo=0.9, step=0.7 / max(len(free), 1))   # cosines in (-0.9, -0.2]: never selected
        for p, v in zip(free, fill):
            h[nxt] = v
            srcs[p] = nxt
            nxt += 1
        info[name] = (ti, srcs)
        edges += [(s, ti) for s in srcs]
    # duplicate edges: each group is one source listed at two positions
    ti = names.index(DUP_ROW[0])
    name, deg, groups = DUP_ROW
    t = torch.randn(cp, generator=gen, dtype=torch.float64)
    h[ti] = t
    levels = _level_vectors(t, deg, gen)
    srcs = [None] * deg
    lv = 0
    for gi in sorted(groups):
        for p in groups[gi]:
            srcs[p] = nxt
        h[nxt] = levels[lv]
        lv += 1
        nxt += 1
    for p in range(deg):
        if srcs[p] is None:
            srcs[p] = nxt
            h[nxt] = levels[lv]
            lv += 1
            nxt += 1
    info[name] = (ti, srcs)
    edges += [(s, ti) for s in srcs]
    # orthogonal neighbours: the target's support is column 0, every neighbour's a few of the other columns (integers)
    for name, deg in ORTH_ROWS:
        ti = names.index(name)
        h[ti, 0] = 3.0
        srcs = []
        for _ in range(deg):
            cols = 1 + torch.randperm(cp - 1, generator=gen)[:3]
            h[nxt, cols] = torch.randint(1, 6, (3,), generator=gen).double()
            srcs.append(nxt)
            nxt += 1
        info[name] = (ti, srcs)
        edges += [(s, ti) for s in srcs]
    info["empty"] = (names.index("empty"), [])
    info["twins"] = twin_members
    ei = torch.tensor(edges, dtype=torch.long).t().contiguous()
    return ei, h[:nxt].float(), info


def test_tie_problem_ties_are_exact_in_fp64():
    """Host check of the tie construction: the members of every rank group score bit-identically in FP64 (scaled twins),
    the groups rank in their designed order, the orthogonal rows score exactly 0, and the designed groups straddle the
    top_k boundaries they are meant to."""
    from oracle import sn_ref
    for cp in (12, 100):
        ei, h, info = _tie_problem(cp, twins=True)
        n = h.size(0)
        pe = sn_ref.process_edges(ei, n, True)
        assert torch.equal(pe, ei)                                          # no self loops, position order kept
        nrm = F.normalize(h.double(), dim=-1, eps=1e-12)
        s = (nrm[pe[1]] * nrm[pe[0]]).sum(-1)
        by_group = {}
        for node, _, grp in info["twins"]:
            t = grp[0]
            by_group.setdefault(grp, []).append(float((nrm[node] * nrm[t]).sum()))
        for grp, vals in by_group.items():
            assert len(set(vals)) == 1, (cp, grp, vals)
        for (t, gi), vals in by_group.items():
            if (t, gi + 1) in by_group:
                assert vals[0] > by_group[(t, gi + 1)][0] + 1e-3
        rank = sn_ref.edge_rank(s, pe[1])
        for name, deg, m, forced in TIE_ROWS:
            t, srcs = info[name]
            r = rank[pe[1] == t]
            for gi, pos in forced.items():                                  # forced members of a group take consecutive ranks
                rs = sorted(int(r[p]) for p in pos)
                assert rs == sorted(rs) and rs[-1] - rs[0] < TIE_GROUPS[gi], (name, gi, rs)
        for name, _ in ORTH_ROWS:
            t, _ = info[name]
            assert bool((s[pe[1] == t] == 0).all())
    starts = torch.cumsum(torch.tensor((0,) + TIE_GROUPS), 0)
    assert (starts[7], starts[8]) == (15, 18) and (starts[14], starts[15]) == (30, 34) and (starts[27], starts[28]) == (62, 65)


@pytest.mark.gpu
@pytest.mark.parametrize("cp", [12, 28, 36, 100, 260])
def test_tie_order_is_exact(cp):
    """Exact ties, where every kernel breaks them differently -- the staged warp (lowest lane), the chunk merge (tournament
    for top_k <= 16, sorted insertion above), the long-row kernel's running list, the hub kernel's 8 warps -- and at the
    k-th place: sel_src, sel_cnt and sel_q must EQUAL the oracle's rank rule (score desc, edge position asc), out and dL/dh
    must match the FP64 oracle (a twin picked in the wrong order changes them).  Orthogonal neighbours (every score 0) at
    thr = 0 are all selected, in position order; duplicate edges are told apart by sel_q; a row without in-edges selects
    nothing.  At c <= 32 the general kernel (no chunk tables) must give the same lists."""
    from oracle import sn_ref
    from sngnn_b200 import graph as G, functional as SF
    ei, h, info = _tie_problem(cp, twins=True)
    n = h.size(0)
    g = G.prepare(ei.to(DEV), n, True)
    _, _, _, _, _, inv, _ = SF._edge_fwd(h.to(DEV), g, 0, 1, 0.0, True)
    inv = inv.cpu()
    by_group = {}
    for node, f, grp in info["twins"]:
        by_group.setdefault(grp, set()).add(float(inv[node]) * f)
    twins = all(len(v) == 1 for v in by_group.values())                 # rsqrtf(4^m x) == rsqrtf(x) / 2^m on this device
    if not twins:
        ei, h, info = _tie_problem(cp, twins=False)
        g = G.prepare(ei.to(DEV), n, True)
    print(f"cp={cp}: scaled twins {'exact' if twins else 'NOT exact: exact copies used'}")
    pe = sn_ref.process_edges(ei, n, True)
    order = torch.argsort(pe[1], stable=True)
    bypos = torch.empty_like(order)
    bypos[order] = torch.arange(order.numel())
    tpos = g.tpos.cpu().long()
    w = torch.randn(n, cp, generator=torch.Generator().manual_seed(cp))
    wd = w.to(DEV)
    for k in (1, 16, 17, 32, 33, 64):
        for thr in (0.0, -1.0):
            tag = f"cp={cp} k={k} thr={thr}"
            h64 = h.double().requires_grad_(True)
            idx, cnt, epos, _ = _oracle_lists(h64, pe, n, k, thr)
            q_ref = torch.where(idx >= 0, tpos[bypos[epos.clamp(min=0)]], torch.zeros_like(idx))
            runs = [None] if cp > 32 else [None, "general"]
            for form in runs:
                tab = g.chunk_tab
                if form == "general":
                    g.chunk_tab = None
                try:
                    out, ss, sw, sq, sc, _, _ = SF._edge_fwd(h.to(DEV), g, 0, k, thr, True, want_q=True)
                finally:
                    g.chunk_tab = tab
                assert torch.equal(sc.cpu().long(), cnt), (tag, form, (sc.cpu().long() != cnt).nonzero().flatten()[:8])
                bad = (ss.cpu().long() != idx).any(1).nonzero().flatten()
                assert bad.numel() == 0, (tag, form, [(int(r), ss[r].tolist(), idx[r].tolist()) for r in bad[:2]])
                assert torch.equal(torch.where(idx >= 0, sq.cpu().long(), 0), q_ref), (tag, form)
            for name, deg in ORTH_ROWS:                                     # s = 0 >= thr: all selected in position order
                t, srcs = info[name]
                assert int(cnt[t]) == min(k, deg) and idx[t, :min(k, deg)].tolist() == srcs[:min(k, deg)], tag
            t, srcs = info[DUP_ROW[0]]
            assert int(idx[t, 0]) == srcs[31] and (k == 1 or (int(idx[t, 1]) == srcs[31] and epos[t, 0] < epos[t, 1])), tag
            t = info["empty"][0]
            assert int(cnt[t]) == 0 and bool((idx[t] == -1).all())
            hd = h.to(DEV).requires_grad_(True)
            out = SF.edge_topk_agg(hd, g, k, thr)
            (out * wd).sum().backward()
            ref = sn_ref.sn_aggregate(h64, pe, k, thr)
            (ref * w.double()).sum().backward()
            torch.testing.assert_close(out.detach().cpu().double(), ref.detach(), rtol=1e-5, atol=1e-6, msg=lambda m: f"{tag}: {m}")
            assert _rel(hd.grad, h64.grad) < 1e-5, (tag, _rel(hd.grad, h64.grad))
            assert float(out[info["empty"][0]].abs().max()) == 0


# ------------------------------------------------------------------------------------------ D. leading dimensions
SENT = -7.25                                                            # sentinel of every output's padding columns


def _padded(x, ld, fill=float("nan")):
    out = torch.full((x.size(0), ld), fill, dtype=x.dtype, device=x.device)
    out[:, :x.size(1)] = x
    return out


def _edge_fwd_ld(h, graph, k, thr, fuse, ldh, ldo, ldw):
    """sng_edge_fwd as functional._edge_fwd calls it, but with h / wt in rows of ldh / ldw floats (NaN beyond c) and out /
    diff in rows of ldo floats (SENT beyond c)."""
    from sngnn_b200 import _C
    n, c = h.shape
    hp = _padded(h, ldh)
    out = torch.full((n, ldo), SENT, device=DEV)
    ss = sw = sc = sq = diff = None
    if k > 0:
        ss = torch.empty(n, k, dtype=torch.int32, device=DEV)
        sw = torch.empty(n, k, device=DEV)
        sc = torch.empty(n, dtype=torch.int32, device=DEV)
        sq = torch.empty(n, k, dtype=torch.int32, device=DEV)
    inv = torch.empty(n, device=DEV)
    wt = bw = beta = bias = None
    if fuse is not None:
        wt, bw, beta, bias = fuse
        wt = _padded(wt, ldw)
        diff = torch.full((n, ldo), SENT, device=DEV)
    tab, ws, wbytes = graph.chunk_tab, None, 0
    n_chunks = -1 if tab is None else int(tab.size(0))
    if n_chunks > 0 and c <= 32:
        wbytes = _C.lib().sng_edge_fwd_workspace_bytes(n_chunks, c, k)
        ws = torch.empty(wbytes, dtype=torch.uint8, device=DEV)
    n_lrows = 0 if tab is None else int(graph.lrows.numel())
    _C.call("sng_edge_fwd", hp, _C.ptr(hp), n, n, 0, c, ldh, _C.ptr(graph.rowptr_in), _C.ptr(graph.col_in), _C.ptr(graph.tpos),
            _C.ptr(tab), n_chunks, _C.ptr(graph.lrows), _C.ptr(graph.lrow_ptr), n_lrows, _C.ptr(graph.rows_hub), int(graph.rows_hub.numel()),
            _C.ptr(ws), wbytes, k, float(thr if thr is not None else 0.0), _C.ptr(out), ldo, _C.ptr(ss), _C.ptr(sw), _C.ptr(sq), _C.ptr(sc),
            _C.ptr(inv), 0, _C.ptr(wt), ldw, _C.ptr(bw), _C.ptr(beta), _C.ptr(bias), _C.ptr(diff))
    return out, ss, sw, sq, sc, inv, diff


def _edge_bwd_ld(h, inv, g, graph, k, ss, sw, sq, sc, beta, diff, ld, ldg, lddiff, lddw):
    """sng_edge_bwd as functional.edge_bwd calls it, with h / g / diff in rows of ld / ldg / lddiff floats (NaN beyond c), the
    dn_target workspace all NaN, and dh / dW^T in rows of ld / lddw floats (SENT beyond c)."""
    from sngnn_b200 import _C
    n, cp = h.shape
    fused = beta is not None
    hp, gp = _padded(h, ld), _padded(g, ldg)
    dp = _padded(diff, lddiff) if fused else None
    coef = torch.empty(max(graph.num_edges, 1) * 2, device=DEV)
    dnt = torch.full((n, ld), float("nan"), device=DEV)
    dh = torch.full((n, ld), SENT, device=DEV)
    dbeta = dwt = part = None
    if fused:
        dbeta = torch.empty(1, device=DEV)
        part = torch.empty(_C.PARTIALS, device=DEV)
        dwt = torch.full((n, lddw), SENT, device=DEV)
    tab = graph.chunk_tab_out if cp <= 32 else None
    n_chunks = -1 if tab is None else int(tab.size(0))
    cpart = None
    if n_chunks > 0:
        cg = 4
        while cg < cp:
            cg *= 2
        cpart = torch.empty(n_chunks * 3 * cg, device=DEV)
    _C.call("sng_edge_bwd", hp, _C.ptr(hp), _C.ptr(inv), _C.ptr(gp), n, n, 0, cp, ld, ldg,
            _C.ptr(graph.rowptr_in), _C.ptr(graph.col_in), _C.ptr(graph.tpos), _C.ptr(graph.rowptr_tr), _C.ptr(graph.col_tr),
            graph.src_shift, graph.num_edges, k, _C.ptr(ss), _C.ptr(sw), _C.ptr(sq), _C.ptr(sc), _C.ptr(beta), _C.ptr(dp), lddiff,
            _C.ptr(dbeta), _C.ptr(coef), _C.ptr(dnt), _C.ptr(part), _C.ptr(dh), _C.ptr(dwt), lddw,
            _C.ptr(tab), n_chunks, _C.ptr(graph.lrows_out if tab is not None else None),
            _C.ptr(graph.lrow_ptr_out if tab is not None else None), 0 if tab is None else int(graph.lrows_out.numel()), _C.ptr(cpart))
    return dh, dwt, dbeta


def _same_with_sentinel(padded, ref, what):
    c = ref.size(1)
    assert torch.equal(padded[:, :c], ref), (what, _rel(padded[:, :c], ref))
    assert bool((padded[:, c:] == SENT).all()), f"{what}: a kernel wrote into the padding columns"


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["plain", "fused"])
@pytest.mark.parametrize("cp", [12, 28, 36, 100, 132, 260])
def test_edge_kernels_leading_dimensions(cp, mode):
    """sng_edge_fwd / sng_edge_bwd with ld > c on both boundary graphs (staged kernels at G <= 8, general and hub kernels
    above; plain and fused epilogue; top_k on both sides of 32 and select-all): every output equals the ld == c call bit
    for bit and no kernel reads the NaN input padding or writes the output padding."""
    from sngnn_b200 import functional as SF
    _, _, graph = _device_graph(mode == "fused")
    n = graph.n
    gen = torch.Generator().manual_seed(cp + 500)
    h = _features(n, cp, seed=cp + 501).to(DEV)
    g = torch.randn(n, cp, generator=gen).to(DEV)
    fuse = None
    if mode == "fused":
        fuse = (torch.randn(n, cp, generator=gen).to(DEV), torch.randn(cp, generator=gen).to(DEV), torch.full((1,), 0.3, device=DEV),
                torch.randn(cp, generator=gen).to(DEV))
    for k, thr in ((17, 0.0), (33, -1.0), (0, None)):
        tag = f"{mode} cp={cp} k={k}"
        ref = SF._edge_fwd(h, graph, 0, k, thr, True, fuse, want_q=True)
        got = _edge_fwd_ld(h, graph, k, thr, fuse, cp + 4, cp + 8, cp + 8)
        _same_with_sentinel(got[0], ref[0], f"{tag} out")
        for a, b, what in zip(got[1:6], ref[1:6], ("sel_src", "sel_w", "sel_q", "sel_cnt", "inv_norm")):
            assert (a is None) == (b is None) and (a is None or torch.equal(a, b)), (tag, what)
        if fuse is not None:
            _same_with_sentinel(got[6], ref[6], f"{tag} diff")
        _, ss, sw, sq, sc, inv, diff = ref
        beta = fuse[2] if fuse is not None else None
        dh_ref, dwt_ref, db_ref = SF.edge_bwd(h, inv, g, graph, k, ss, sw, sq, sc, beta, diff)
        dh, dwt, db = _edge_bwd_ld(h, inv, g, graph, k, ss, sw, sq, sc, beta, diff, cp + 8, cp + 4, cp + 4, cp + 8)
        _same_with_sentinel(dh, dh_ref, f"{tag} dh")
        if fuse is not None:
            _same_with_sentinel(dwt, dwt_ref, f"{tag} dwt")
            assert torch.equal(db, db_ref), tag


@pytest.mark.gpu
@pytest.mark.parametrize("cp", [12, 28, 36, 100, 132, 260])
def test_list_spmm_and_pp_fuse_leading_dimensions(cp):
    """sng_list_agg_fwd, sng_list_bwd, sng_spmm_fwd and sng_pp_fuse_fwd with ld > c (NaN input padding, sentinel output
    padding) equal their ld == c calls bit for bit."""
    from sngnn_b200 import _C, functional as SF
    gen = torch.Generator().manual_seed(cp + 600)
    n, k = N_LIST, 33
    h = _features(n, cp, seed=cp + 601).to(DEV)
    g = torch.randn(n, cp, generator=gen).to(DEV)
    idx, cnt = _boundary_lists(n, k, seed=cp)
    idx, cnt = idx.to(DEV), cnt.to(DEV)
    _, _, inv = SF.rownorm(h, want_f32=False, want_inv=True)
    sim = torch.where(idx >= 0, torch.rand(n, k, generator=gen).to(DEV), torch.zeros((), device=DEV))
    inv_denom = 1.0 / cnt.clamp(min=1).float()
    ld, ldo = cp + 4, cp + 8
    # list aggregation, forward
    ref = SF.ListAgg.apply(h, idx, sim, cnt, inv_denom)
    out = torch.full((n, ldo), SENT, device=DEV)
    hp = _padded(h, ld)
    _C.call("sng_list_agg_fwd", hp, _C.ptr(hp), n, cp, ld, k, _C.ptr(idx), _C.ptr(sim), _C.ptr(cnt), _C.ptr(inv_denom), _C.ptr(out), ldo)
    _same_with_sentinel(out, ref, f"cp={cp} list_agg_fwd")
    # list backward
    dh_ref = SF.list_bwd(h, inv, g, idx, sim, cnt, inv_denom)
    tr = SF.list_transpose(idx, cnt, n, chunk_tables=cp <= 32)
    n_chunks = -1 if tr.chunk_tab is None else int(tr.chunk_tab.size(0))
    cpart = None
    if n_chunks > 0:
        cg = 4
        while cg < cp:
            cg *= 2
        cpart = torch.empty(n_chunks * 3 * cg, device=DEV)
    gp = _padded(g, ldo)
    coef = torch.empty(n * k * 2, device=DEV)
    dnt = torch.full((n, ld), float("nan"), device=DEV)
    dh = torch.full((n, ld), SENT, device=DEV)
    _C.call("sng_list_bwd", hp, _C.ptr(hp), _C.ptr(inv), _C.ptr(gp), n, n, 0, cp, ld, ldo, k, _C.ptr(idx), _C.ptr(sim), _C.ptr(cnt),
            _C.ptr(inv_denom), _C.ptr(tr.sel_q), _C.ptr(tr.rowptr_tr), _C.ptr(tr.col_tr), _C.ptr(coef), _C.ptr(dnt), _C.ptr(dh),
            _C.ptr(tr.chunk_tab), n_chunks, _C.ptr(tr.lrows), _C.ptr(tr.lrow_ptr), 0 if tr.lrows is None else int(tr.lrows.numel()),
            _C.ptr(cpart))
    _same_with_sentinel(dh, dh_ref, f"cp={cp} list_bwd")
    # K3 and K4 over the symmetric boundary graph's CSR
    _, _, graph = _device_graph(True)
    ng = graph.n
    x = _features(ng, cp, seed=cp + 602).to(DEV)
    val = torch.rand(graph.num_edges, generator=gen).to(DEV)
    rowscale = torch.rand(ng, generator=gen).to(DEV)
    bias = torch.randn(cp, generator=gen).to(DEV)
    ref = torch.empty(ng, cp, device=DEV)
    _C.call("sng_spmm_fwd", x, _C.ptr(x), ng, cp, cp, _C.ptr(graph.rowptr_in), _C.ptr(graph.col_in), _C.ptr(val), _C.ptr(rowscale),
            _C.ptr(bias), _C.ptr(ref), cp)
    xp = _padded(x, ld)
    out = torch.full((ng, ldo), SENT, device=DEV)
    _C.call("sng_spmm_fwd", xp, _C.ptr(xp), ng, cp, ld, _C.ptr(graph.rowptr_in), _C.ptr(graph.col_in), _C.ptr(val), _C.ptr(rowscale),
            _C.ptr(bias), _C.ptr(out), ldo)
    _same_with_sentinel(out, ref, f"cp={cp} spmm_fwd")
    out1 = torch.randn(ng, cp, generator=gen).to(DEV)
    b_w, beta = torch.randn(cp, generator=gen).to(DEV), torch.full((1,), 0.3, device=DEV)
    out0_ref, out_ref = SF.pp_fuse_fwd(out1, x, b_w, beta, bias, graph.rowptr_out, graph.col_out)
    o1p = _padded(out1, ld)
    out0, out = torch.full((ng, ld), SENT, device=DEV), torch.full((ng, ld), SENT, device=DEV)
    _C.call("sng_pp_fuse_fwd", xp, _C.ptr(xp), ng, cp, ld, _C.ptr(graph.rowptr_out), _C.ptr(graph.col_out), _C.ptr(b_w), _C.ptr(beta),
            _C.ptr(o1p), _C.ptr(bias), _C.ptr(out0), _C.ptr(out))
    _same_with_sentinel(out0, out0_ref, f"cp={cp} pp_fuse_fwd out0")
    _same_with_sentinel(out, out_ref, f"cp={cp} pp_fuse_fwd out")


# ------------------------------------------------------------------------------------------ E. staged vs general forms
@pytest.mark.gpu
@pytest.mark.parametrize("cp", [12, 20, 28])
def test_staged_forms_match_general_kernels_at_ragged_widths(cp):
    """At ragged widths of <= 32 channels, on the asymmetric boundary graph: the forward with the chunk tables (staged
    kernel, chunk pass, merge) selects exactly what the general kernels select on every row (no tables: long-row and hub
    kernels), and the backward's staged source pass (by-source chunk tables) agrees with the unstaged one to FP32
    summation order."""
    from sngnn_b200 import functional as SF
    _, _, graph = _device_graph(False)
    n = graph.n
    h = _features(n, cp, seed=cp + 700).to(DEV)
    g = torch.randn(n, cp, generator=torch.Generator().manual_seed(cp + 701)).to(DEV)
    for i, k in enumerate((16, 17, 32, 33, 64)):
        thr = (0.0, -1.0)[i % 2]
        tag = f"cp={cp} k={k} thr={thr}"
        out_a, ss_a, sw_a, sq_a, sc_a, inv, _ = SF._edge_fwd(h, graph, 0, k, thr, True, want_q=True)
        tab, graph.chunk_tab = graph.chunk_tab, None
        try:
            out_b, ss_b, sw_b, sq_b, sc_b, _, _ = SF._edge_fwd(h, graph, 0, k, thr, True, want_q=True)
        finally:
            graph.chunk_tab = tab
        assert torch.equal(sc_a, sc_b) and torch.equal(ss_a, ss_b) and torch.equal(sq_a, sq_b), tag
        torch.testing.assert_close(sw_a, sw_b, rtol=1e-6, atol=1e-7)
        torch.testing.assert_close(out_a, out_b, rtol=1e-5, atol=1e-6)
        dh_a, _, _ = SF.edge_bwd(h, inv, g, graph, k, ss_a, sw_a, sq_a, sc_a)
        tab, graph.chunk_tab_out = graph.chunk_tab_out, None
        try:
            dh_b, _, _ = SF.edge_bwd(h, inv, g, graph, k, ss_a, sw_a, sq_a, sc_a)
        finally:
            graph.chunk_tab_out = tab
        assert _rel(dh_a, dh_b) < 1e-6, (tag, _rel(dh_a, dh_b))
