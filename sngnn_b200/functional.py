"""Autograd functions over the C-ABI kernels (include/sng.h).  torch is used for memory, streams and the
dense `lin` GEMM only; every sparse / selection / aggregation step is a libsng.so call.

Channel padding: the edge kernels want 16-byte feature rows, so the layer output width C is padded to
Cp = 4*ceil(C/4) by zero-padding the `lin` weights (zero columns change neither norms nor dot products).
"""
import torch
import torch.nn.functional as F

from . import _C


# Test / benchmark hook: set to a list and every EdgeAgg forward in training mode appends its (sel_src, sel_cnt) -- the
# selection lists of the layers in call order (the parity gates compare them with the oracle's rule).  None = off.
record_selection = None


def padded_channels(c):
    return (c + 3) // 4 * 4


class LinNorm(torch.autograd.Function):
    """h [N, Cp] = x W^T + b (channels zero-padded to Cp) and inv_norm = 1 / max(||h_i||, 1e-12) in ONE pass over x
    (sng_lin_norm_fwd; R: models/models.py:121-122).  Backward is the dense layer's: three library GEMMs / reductions."""

    @staticmethod
    def forward(ctx, x, weight, bias, cp):
        _C.require_cuda(x, weight, bias)
        x = x.contiguous().float()
        w = weight.contiguous()
        n, f = x.shape
        c = w.size(0)
        h = torch.empty(n, cp, dtype=torch.float32, device=x.device)
        inv = torch.empty(n, dtype=torch.float32, device=x.device)
        _C.call("sng_lin_norm_fwd", x, _C.ptr(x), n, f, f, _C.ptr(w), c, f, _C.ptr(None if bias is None else bias.contiguous()), _C.ptr(h), _C.ptr(inv))
        ctx.save_for_backward(x, w)
        ctx.has_bias, ctx.c = bias is not None, c
        ctx.mark_non_differentiable(inv)
        return h, inv

    @staticmethod
    def backward(ctx, gh, _ginv):
        x, w = ctx.saved_tensors
        dx = gh[:, :ctx.c] @ w if ctx.needs_input_grad[0] else None
        want_b = ctx.has_bias and ctx.needs_input_grad[2]
        if ctx.needs_input_grad[1] and _C.lib().sng_lin_bwd_supported(x.size(1), ctx.c):
            dw, db = lin_bwd(gh, x, ctx.c, want_b)
        else:
            g = gh[:, :ctx.c]
            dw = g.t() @ x if ctx.needs_input_grad[1] else None
            db = g.sum(0) if want_b else None
        return dx, dw, db, None


def lin_bwd(gh, x, c, want_bias=True):
    """(dW [c, f], db [c] | None) = (gh[:, :c]^T x, column sums of gh[:, :c]) in one streaming pass (sng_lin_bwd): the weight
    gradient of `self.lin` (R: models/models.py:121).  The library GEMM runs this N-long reduction with a [c, f] output as one
    skinny kernel at a fraction of the memory bandwidth; fixed-order partial sums make the result bit-reproducible."""
    _C.require_cuda(gh, x)
    if gh.stride(1) != 1:
        gh = gh.contiguous()
    if x.stride(1) != 1:
        x = x.contiguous()
    n, f = x.shape
    dw = torch.empty(c, f, dtype=torch.float32, device=x.device)
    db = torch.empty(c, dtype=torch.float32, device=x.device) if want_bias else None
    nb = _C.lib().sng_lin_bwd_workspace_bytes(n, f, c)
    ws = torch.empty(nb, dtype=torch.uint8, device=x.device)
    _C.call("sng_lin_bwd", x, _C.ptr(gh), gh.stride(0), _C.ptr(x), x.stride(0), n, f, c, _C.ptr(dw), f, _C.ptr(db), _C.ptr(ws), nb)
    return dw, db


def lin_norm(x, weight, bias, cp):
    """(h [N, Cp], inv_norm [N] | None): the fused kernel when the shape is supported, else library GEMM (inv_norm = None: the
    aggregation call then computes it)."""
    if x.is_cuda and _C.lib().sng_lin_norm_supported(x.size(1), weight.size(0)):
        return LinNorm.apply(x, weight, bias, cp)
    return linear_padded(x, weight, bias, cp), None


def linear_padded(x, weight, bias, cp):
    """h = x @ W^T + b with the output width zero-padded to `cp` (R: models/models.py:121,237,324)."""
    c = weight.size(0)
    if cp != c:
        weight = F.pad(weight, (0, 0, 0, cp - c))
        bias = None if bias is None else F.pad(bias, (0, cp - c))
    return F.linear(x, weight, bias)


def _check_h(h):
    _C.require_cuda(h)
    if h.dtype != torch.float32 or h.dim() != 2 or h.size(1) % 4 != 0:
        raise RuntimeError("expected a float32 [N, 4m] tensor")
    return h.contiguous()


_DENOMINATORS = {"candidates": 0, "selected": 1}


def _edge_fwd(h_all, graph, row_offset, k, thr, train, fuse=None, want_q=False, inv_norm=None, denominator="candidates",
              inv_denom=None):
    """sng_edge_fwd_denom on the target rows of `graph` (a PreparedGraph or a row shard of one).  fuse = (wt [N, Cp], b_w [Cp],
    beta [1], bias [Cp] | None) gathers the structural term and blends in the same pass (symmetric graphs only).
    denominator='selected' divides each row by its selected count instead of its in-degree; inv_denom [graph.n] (optional)
    then receives the factor each row was scaled by, the input of edge_bwd in that mode."""
    c = h_all.size(1)
    n = graph.n
    dev = h_all.device
    out = torch.empty(n, c, dtype=torch.float32, device=dev)
    sel_src = sel_w = sel_cnt = sel_q = diff = None
    if train and k > 0:
        sel_src = torch.empty(n, k, dtype=torch.int32, device=dev)
        sel_w = torch.empty(n, k, dtype=torch.float32, device=dev)
        sel_cnt = torch.empty(n, dtype=torch.int32, device=dev)
        if want_q:
            sel_q = torch.empty(n, k, dtype=torch.int32, device=dev)
    inv_ready = inv_norm is not None                      # produced with h by sng_lin_norm_fwd
    if not inv_ready:
        inv_norm = torch.empty(h_all.size(0), dtype=torch.float32, device=dev)
    wt = bw = beta = bias = None
    if fuse is not None:
        wt, bw, beta, bias = fuse
        if train:
            diff = torch.empty_like(out)
    tab, ws, wbytes = graph.chunk_tab, None, 0
    n_chunks = -1 if tab is None else int(tab.size(0))
    if n_chunks > 0 and c <= 32:
        wbytes = _C.lib().sng_edge_fwd_workspace_bytes(n_chunks, c, k)
        ws = torch.empty(wbytes, dtype=torch.uint8, device=dev)
    n_lrows = 0 if tab is None else int(graph.lrows.numel())
    n_hub = 0 if graph.rows_hub is None else int(graph.rows_hub.numel())
    _C.call("sng_edge_fwd_denom", h_all, _C.ptr(h_all), h_all.size(0), n, row_offset, c, c, _C.ptr(graph.rowptr_in), _C.ptr(graph.col_in),
            _C.ptr(graph.tpos if want_q else None), _C.ptr(tab), n_chunks, _C.ptr(graph.lrows), _C.ptr(graph.lrow_ptr), n_lrows,
            _C.ptr(graph.rows_hub), n_hub, _C.ptr(ws), wbytes, k,
            float(thr if thr is not None else 0.0), _C.ptr(out), c, _C.ptr(sel_src), _C.ptr(sel_w), _C.ptr(sel_q), _C.ptr(sel_cnt),
            _C.ptr(inv_norm), int(inv_ready), _C.ptr(wt), c, _C.ptr(bw), _C.ptr(beta), _C.ptr(bias), _C.ptr(diff),
            _DENOMINATORS[denominator], _C.ptr(inv_denom))
    return out, sel_src, sel_w, sel_q, sel_cnt, inv_norm, diff


def _padded_wt(w_weight, cp):
    """W^T [N, Cp] of the structural weight [C, N].  The modules keep that parameter in transposed storage
    (models.SNConv_plus_plus), so this is a view of the parameter itself when C is a multiple of 4, and a small padded copy
    otherwise; a parameter in plain [C, N] storage costs a transpose copy per call.  Nothing is cached."""
    c = w_weight.size(0)
    wt = w_weight.detach().t()
    if cp != c:
        wt = F.pad(wt, (0, cp - c))
    return wt.contiguous()


def _structural_operands(w_weight, w_bias, beta, bias, cp):
    """(wt [N, Cp], b_w [Cp], beta [1], bias [Cp] | None): the SNGNN++ structural parameters, detached, padded to Cp."""
    c = w_weight.size(0)
    return (_padded_wt(w_weight, cp), F.pad(w_bias.detach(), (0, cp - c)).contiguous(), beta.detach().contiguous(),
            None if bias is None else F.pad(bias.detach(), (0, cp - c)).contiguous())


def _weight_grad(dwt, c):
    """dL/dw.weight [C, N] from dL/dW^T [N, Cp]: a view in the parameter's own (transposed) storage."""
    return (dwt if dwt.size(1) == c else dwt[:, :c]).t()


class EdgeAgg(torch.autograd.Function):
    """The similarity-navigated aggregation of one layer: out_1 of R: models/models.py:132 / :239 / :326 and -- when the
    structural parameters are given and the graph's in-lists equal its out-lists -- the whole of
    R: models/models.py:124-136 (out = beta (A W^T + b_w) + (1 - beta) out_1 + bias) in the same pass over the edges.
    Forward sng_edge_fwd, backward sng_edge_bwd (two gather passes, no float atomics, bit-reproducible).  With
    denominator='selected' out_1 divides by each row's selected count; the backward reuses the forward's per-row factors."""

    @staticmethod
    def forward(ctx, h, graph, top_k, thr, w_weight, w_bias, beta, bias, inv_norm=None, denominator="candidates"):
        h = _check_h(h)
        n, cp = h.shape
        if n != graph.n:
            raise RuntimeError(f"h has {n} rows but the graph has {graph.n} nodes")
        k = int(top_k) if top_k is not None else 0
        fused = w_weight is not None
        train = any(ctx.needs_input_grad)
        fuse = None
        if fused:
            _C.require_cuda(h, w_weight, w_bias, beta, bias)
            c = w_weight.size(0)
            if w_weight.size(1) != n:
                raise RuntimeError(f"w.weight is [{c},{w_weight.size(1)}] but the graph has {n} nodes "
                                   "(R builds w = Linear(num_nodes, out_channels), models.py:95)")
            if not graph.symmetric:
                raise RuntimeError("the fused SNGNN++ pass needs a graph whose in-lists equal its out-lists")
            fuse = _structural_operands(w_weight, w_bias, beta, bias, cp)
            ctx.c = c
        inv_denom = torch.empty(n, dtype=torch.float32, device=h.device) if train and k > 0 and denominator == "selected" else None
        out, sel_src, sel_w, sel_q, sel_cnt, inv_norm, diff = _edge_fwd(h, graph, 0, k, thr, train, fuse, want_q=True, inv_norm=inv_norm,
                                                                        denominator=denominator, inv_denom=inv_denom)
        ctx.graph, ctx.k, ctx.fused, ctx.has_bias = graph, k, fused, bias is not None
        if record_selection is not None and sel_cnt is not None:
            record_selection.append((sel_src, sel_cnt))
        ctx.save_for_backward(h, sel_src, sel_w, sel_q, sel_cnt, inv_norm, diff, beta if fused else None, inv_denom)
        if sel_cnt is not None:
            ctx.mark_non_differentiable(sel_src, sel_w, sel_cnt)
        return out, sel_src, sel_w, sel_cnt

    @staticmethod
    def backward(ctx, g, *_):
        h, sel_src, sel_w, sel_q, sel_cnt, inv_norm, diff, beta, inv_denom = ctx.saved_tensors
        graph, k, fused = ctx.graph, ctx.k, ctx.fused
        g = g.contiguous()
        dh, dwt, dbeta = edge_bwd(h, inv_norm, g, graph, k, sel_src, sel_w, sel_q, sel_cnt, beta if fused else None, diff,
                                  inv_denom=inv_denom)
        if not fused:
            return dh, None, None, None, None, None, None, None, None, None
        c = ctx.c
        gsum = g.sum(0)[:c]
        return dh, None, None, None, _weight_grad(dwt, c), gsum * beta, dbeta, (gsum if ctx.has_bias else None), None, None


def _bwd_buffers(h, graph, fused):
    """Outputs and workspaces of sng_edge_bwd_denom / sng_edge_bwd_wide: (coef, dn_target, dh, dbeta, dwt, partials, the
    by-source chunk table (c <= 32) and its size, chunk partials)."""
    cp = h.size(1)
    n = graph.n
    dev = h.device
    coef = torch.empty(max(graph.num_edges, 1) * 2, dtype=torch.float32, device=dev)
    dnt = torch.empty(n, cp, dtype=torch.float32, device=dev)
    dh = torch.empty_like(h)
    dbeta = dwt = part = None
    if fused:
        dbeta = torch.empty(1, dtype=torch.float32, device=dev)
        part = torch.empty(_C.PARTIALS, dtype=torch.float32, device=dev)
        if not graph.is_shard:
            dwt = torch.empty(n, cp, dtype=torch.float32, device=dev)
    tab = graph.chunk_tab_out if cp <= 32 else None
    n_chunks = -1 if tab is None else int(tab.size(0))
    cpart = None
    if n_chunks > 0:
        cg = 4
        while cg < cp:
            cg *= 2
        cpart = torch.empty(n_chunks * 3 * cg, dtype=torch.float32, device=dev)
    return coef, dnt, dh, dbeta, dwt, part, tab, n_chunks, cpart


def edge_bwd(h, inv_norm, g, graph, k, sel_src, sel_w, sel_q, sel_cnt, beta=None, diff=None, *, row_offset=0, inv_denom=None):
    """sng_edge_bwd_denom: dL/dh [N, Cp] of the aggregation -- two gather passes, no float atomics -- and, with `beta` (the fused
    SNGNN++ epilogue), dL/dW^T [N, Cp] and dL/dbeta.  `g` = dL/dout.  inv_denom = the per-row factors _edge_fwd wrote under
    denominator='selected' (None: 1 / max(in-degree, 1)).
    Row shard (`graph` = PreparedGraph.row_slice(lo, hi), row_offset = lo, `h` / `inv_norm` of all N nodes, `g` / `diff` / the
    lists of the shard's rows): dh is the shard's contribution to dL/dh of every node and dbeta its part of dL/dbeta, both
    bit-reproducible; dL/dW^T is not computed (None): the caller assembles it from the g0 of every shard."""
    n_total, cp = h.shape
    n = graph.n
    fused = beta is not None
    coef, dnt, dh, dbeta, dwt, part, tab, n_chunks, cpart = _bwd_buffers(h, graph, fused)
    _C.call("sng_edge_bwd_denom", h, _C.ptr(h), _C.ptr(inv_norm), _C.ptr(g), n_total, n, int(row_offset), cp, cp, cp,
            _C.ptr(graph.rowptr_in), _C.ptr(graph.col_in),
            _C.ptr(graph.tpos), _C.ptr(graph.rowptr_tr), _C.ptr(graph.col_tr), graph.src_shift, graph.num_edges, k,
            _C.ptr(sel_src), _C.ptr(sel_w), _C.ptr(sel_q), _C.ptr(sel_cnt), _C.ptr(beta), _C.ptr(diff if fused else None), cp,
            _C.ptr(dbeta), _C.ptr(coef), _C.ptr(dnt), _C.ptr(part), _C.ptr(dh), _C.ptr(dwt), cp,
            _C.ptr(tab), n_chunks, _C.ptr(graph.lrows_out if tab is not None else None),
            _C.ptr(graph.lrow_ptr_out if tab is not None else None), 0 if tab is None else int(graph.lrows_out.numel()), _C.ptr(cpart),
            _C.ptr(inv_denom))
    return dh, dwt, dbeta


def edge_agg_bwd_scatter(h_all, inv_norm, g, rowptr, col, n, row_offset, k, sel_src, sel_w, sel_cnt, inv_denom):
    """sng_edge_agg_bwd (scatter form, FP32 atomics): no layer uses it; the timing scripts compare the gather forms with it.
    `g` = dL/dout of target rows [row_offset, row_offset + n) of `h_all`; returns their contribution to dL/dh_all (the
    contributions of different row ranges add).  k > 0: selection lists + inv_denom; k == 0: every edge of rowptr / col."""
    n_total, c = h_all.shape
    g = g.contiguous()
    dval, dnrm, dh = torch.zeros_like(h_all), torch.zeros_like(h_all), torch.empty_like(h_all)
    _C.call("sng_edge_agg_bwd", h_all, _C.ptr(h_all), _C.ptr(inv_norm), _C.ptr(g), n_total, n, row_offset, c, c, _C.ptr(rowptr),
            _C.ptr(col), k, _C.ptr(sel_src), _C.ptr(sel_w), _C.ptr(sel_cnt), _C.ptr(inv_denom), _C.ptr(dval), _C.ptr(dnrm), _C.ptr(dh))
    return dh


def edge_topk_agg_rows(h_all, shard, row_offset, top_k=None, thr=None):
    """Forward-only K2 on a row shard: targets [row_offset, row_offset + shard.n) of `h_all` (all nodes, e.g. after an
    all-gather), `shard` = PreparedGraph.row_slice(lo, hi).  Returns (out [shard.n, C], sel_src, sel_w, sel_cnt)."""
    h_all = _check_h(h_all)
    out, sel_src, sel_w, _, sel_cnt, _, _ = _edge_fwd(h_all, shard, int(row_offset), int(top_k) if top_k is not None else 0, thr, True)
    return out, sel_src, sel_w, sel_cnt


class ShardedEdgeTopkAgg(torch.autograd.Function):
    """K2 / K2b on a ROW SHARD: forward computes out_1 for target rows [row_offset, row_offset + shard.n) from `h_all` (all
    nodes); backward returns this shard's contribution to dL/dh_all [N, C] -- contributions of different shards add
    (SURVEY.md §8(e): the caller reduce-scatters them, see dist.AllGatherRows).  The backward is sng_edge_bwd in its
    row-shard form, through the shard's own transpose index: no float atomics, bit-reproducible."""

    @staticmethod
    def forward(ctx, h_all, shard, row_offset, top_k, thr):
        h_all = _check_h(h_all)
        k = int(top_k) if top_k is not None else 0
        out, sel_src, sel_w, sel_q, sel_cnt, inv_norm, _ = _edge_fwd(h_all, shard, int(row_offset), k, thr, ctx.needs_input_grad[0],
                                                                     want_q=True)
        ctx.shard, ctx.k, ctx.row_offset = shard, k, int(row_offset)
        ctx.save_for_backward(h_all, sel_src, sel_w, sel_q, sel_cnt, inv_norm)
        return out

    @staticmethod
    def backward(ctx, g):
        h_all, sel_src, sel_w, sel_q, sel_cnt, inv_norm = ctx.saved_tensors
        dh, _, _ = edge_bwd(h_all, inv_norm, g.contiguous(), ctx.shard, ctx.k, sel_src, sel_w, sel_q, sel_cnt, row_offset=ctx.row_offset)
        return dh, None, None, None, None


def edge_topk_agg(h, graph, top_k=None, thr=None, return_selection=False, structural=None, inv_norm=None, denominator="candidates"):
    """out_1 (structural=None) or the fused SNGNN++ layer output (structural = (w.weight, w.bias, beta, bias)).
    inv_norm = 1 / max(||h_i||, 1e-12) when the caller already has it (lin_norm), else it is computed here.
    denominator = 'candidates' (mean over the in-degree, PyG aggr='mean') | 'selected' (mean over the selected neighbours;
    needs top_k > 0)."""
    w_weight, w_bias, beta, bias = structural if structural is not None else (None, None, None, None)
    out, sel_src, sel_w, sel_cnt = EdgeAgg.apply(h, graph, top_k, thr, w_weight, w_bias, beta, bias, inv_norm, denominator)
    if return_selection:
        return out, (sel_src, sel_w, sel_cnt)
    return out


# ------------------------------------------------------------------------------------------ per-edge form (top_k > SNG_MAX_TOPK)
def per_edge_form(top_k):
    """True when `top_k` asks for more neighbours than the selection lists of sng_edge_fwd hold (SNG_MAX_TOPK): the layer then
    runs the per-edge form (sng_edge_fwd_wide / sng_edge_bwd_wide), which saves one flag per in-edge instead of [N, top_k]
    lists.  The one place where the models and the sharded forward choose between the two forms."""
    return top_k is not None and int(top_k) > _C.MAX_TOPK


def _edge_fwd_wide(h_all, graph, row_offset, top_k, thr, train, fuse=None, inv_norm=None, denominator="candidates", inv_denom=None):
    """sng_edge_fwd_wide on the target rows of `graph` (a PreparedGraph or a row shard of one), arguments as _edge_fwd.
    Returns (out, sel_flag [num_edges] uint8 | None, inv_norm, diff); sel_flag is written for every edge in training (the
    backward's input) and exists in inference only when some row needs a cut.  Any top_k > SNG_MAX_TOPK: every value at or
    above the largest in-degree selects the same set, so it is clamped there before the call."""
    c = h_all.size(1)
    n = graph.n
    dev = h_all.device
    k = max(_C.MAX_TOPK + 1, min(int(top_k), graph.max_deg))
    out = torch.empty(n, c, dtype=torch.float32, device=dev)
    flags = None
    if train or k < graph.max_deg:
        flags = torch.empty(max(graph.num_edges, 1), dtype=torch.uint8, device=dev)
    inv_ready = inv_norm is not None
    if not inv_ready:
        inv_norm = torch.empty(h_all.size(0), dtype=torch.float32, device=dev)
    wt = bw = beta = bias = diff = None
    if fuse is not None:
        wt, bw, beta, bias = fuse
        if train:
            diff = torch.empty_like(out)
    tab = graph.chunk_tab
    n_chunks = -1 if tab is None else int(tab.size(0))
    wbytes = _C.lib().sng_edge_fwd_wide_workspace_bytes(n_chunks if c <= 32 else 0, c, graph.num_edges, graph.max_deg)
    ws = torch.empty(wbytes, dtype=torch.uint8, device=dev) if wbytes else None
    n_lrows = 0 if tab is None else int(graph.lrows.numel())
    n_hub = 0 if graph.rows_hub is None else int(graph.rows_hub.numel())
    _C.call("sng_edge_fwd_wide", h_all, _C.ptr(h_all), h_all.size(0), n, row_offset, c, c, _C.ptr(graph.rowptr_in), _C.ptr(graph.col_in),
            graph.num_edges, _C.ptr(tab), n_chunks, _C.ptr(graph.lrows), _C.ptr(graph.lrow_ptr), n_lrows, _C.ptr(graph.rows_hub), n_hub,
            _C.ptr(ws), wbytes, k, graph.max_deg, float(thr if thr is not None else 0.0), _C.ptr(out), c, _C.ptr(flags), int(bool(train)),
            _C.ptr(inv_norm), int(inv_ready), _C.ptr(wt), c, _C.ptr(bw), _C.ptr(beta), _C.ptr(bias), _C.ptr(diff),
            _DENOMINATORS[denominator], _C.ptr(inv_denom))
    return out, flags, inv_norm, diff


def edge_bwd_wide(h, inv_norm, g, graph, flags, beta=None, diff=None, *, row_offset=0, inv_denom=None):
    """sng_edge_bwd_wide: the backward of _edge_fwd_wide from its training flags -- edge_bwd's two gather passes, no float
    atomics, bit-reproducible; outputs and row-shard convention as edge_bwd."""
    n_total, cp = h.shape
    n = graph.n
    fused = beta is not None
    coef, dnt, dh, dbeta, dwt, part, tab, n_chunks, cpart = _bwd_buffers(h, graph, fused)
    _C.call("sng_edge_bwd_wide", h, _C.ptr(h), _C.ptr(inv_norm), _C.ptr(g), n_total, n, int(row_offset), cp, cp, cp,
            _C.ptr(graph.rowptr_in), _C.ptr(graph.col_in), _C.ptr(graph.tpos), _C.ptr(graph.rowptr_tr), _C.ptr(graph.col_tr),
            graph.src_shift, graph.num_edges, _C.ptr(flags), _C.ptr(inv_denom), _C.ptr(beta), _C.ptr(diff if fused else None), cp,
            _C.ptr(dbeta), _C.ptr(coef), _C.ptr(dnt), _C.ptr(part), _C.ptr(dh), _C.ptr(dwt), cp,
            _C.ptr(tab), n_chunks, _C.ptr(graph.lrows_out if tab is not None else None),
            _C.ptr(graph.lrow_ptr_out if tab is not None else None), 0 if tab is None else int(graph.lrows_out.numel()), _C.ptr(cpart))
    return dh, dwt, dbeta


class EdgeWideAgg(torch.autograd.Function):
    """EdgeAgg for top_k > SNG_MAX_TOPK (the per-edge form): the same layer outputs -- out_1, or with the structural parameters
    the fused SNGNN++ layer on a graph whose in-lists equal its out-lists -- and the same gradients.  With row_offset / a
    row shard of the graph, `h` holds every node and the backward returns the shard's contribution to dL/dh (fused: whole
    graphs only; dist._ShardedFusedAgg assembles dL/dw.weight of a shard)."""

    @staticmethod
    def forward(ctx, h, graph, row_offset, top_k, thr, w_weight, w_bias, beta, bias, inv_norm=None, denominator="candidates"):
        h = _check_h(h)
        n, cp = h.shape
        if not graph.is_shard and n != graph.n:
            raise RuntimeError(f"h has {n} rows but the graph has {graph.n} nodes")
        fused = w_weight is not None
        train = any(ctx.needs_input_grad)
        fuse = None
        if fused:
            _C.require_cuda(h, w_weight, w_bias, beta, bias)
            if graph.is_shard or not graph.symmetric:
                raise RuntimeError("the fused SNGNN++ pass needs a whole graph whose in-lists equal its out-lists")
            if w_weight.size(1) != n:
                raise RuntimeError(f"w.weight is [{w_weight.size(0)},{w_weight.size(1)}] but the graph has {n} nodes "
                                   "(R builds w = Linear(num_nodes, out_channels), models.py:95)")
            fuse = _structural_operands(w_weight, w_bias, beta, bias, cp)
            ctx.c = w_weight.size(0)
        inv_denom = torch.empty(graph.n, dtype=torch.float32, device=h.device) if train and denominator == "selected" else None
        out, flags, inv_norm, diff = _edge_fwd_wide(h, graph, int(row_offset), top_k, thr, train, fuse, inv_norm, denominator, inv_denom)
        ctx.graph, ctx.row_offset, ctx.fused, ctx.has_bias = graph, int(row_offset), fused, bias is not None
        ctx.save_for_backward(h, flags, inv_norm, diff, beta if fused else None, inv_denom)
        return out

    @staticmethod
    def backward(ctx, g):
        h, flags, inv_norm, diff, beta, inv_denom = ctx.saved_tensors
        g = g.contiguous()
        dh, dwt, dbeta = edge_bwd_wide(h, inv_norm, g, ctx.graph, flags, beta, diff, row_offset=ctx.row_offset, inv_denom=inv_denom)
        if not ctx.fused:
            return dh, None, None, None, None, None, None, None, None, None, None
        c = ctx.c
        gsum = g.sum(0)[:c]
        return dh, None, None, None, None, _weight_grad(dwt, c), gsum * beta, dbeta, (gsum if ctx.has_bias else None), None, None


def edge_agg(h, graph, top_k, thr, structural=None, inv_norm=None, denominator="candidates"):
    """The edge-candidate aggregation of the models at any top_k > 0: edge_topk_agg (selection lists) up to SNG_MAX_TOPK, the
    per-edge form (EdgeWideAgg) above.  Arguments as edge_topk_agg."""
    if not per_edge_form(top_k):
        return edge_topk_agg(h, graph, top_k, thr, structural=structural, inv_norm=inv_norm, denominator=denominator)
    w_weight, w_bias, beta, bias = structural if structural is not None else (None, None, None, None)
    return EdgeWideAgg.apply(h, graph, 0, top_k, thr, w_weight, w_bias, beta, bias, inv_norm, denominator)


def sharded_edge_agg(h_all, shard, row_offset, top_k, thr):
    """out_1 of target rows [row_offset, row_offset + shard.n) from `h_all` (all nodes), differentiable: ShardedEdgeTopkAgg
    up to SNG_MAX_TOPK, the per-edge form above (denominator='candidates')."""
    if per_edge_form(top_k):
        return EdgeWideAgg.apply(h_all, shard, int(row_offset), top_k, thr, None, None, None, None)
    return ShardedEdgeTopkAgg.apply(h_all, shard, row_offset, top_k, thr)


class ListTranspose:
    """By-source index of fixed-width neighbour lists (sng_list_transpose): rowptr_tr [n_total + 1] / col_tr = for every source
    node, the LOCAL rows of the lists that hold it, ordered by (row, rank); sel_q [nq, k] = position of entry (i, t) in col_tr
    (-1 for padding); chunk_tab / lrows / lrow_ptr = the degree tables of sng_list_bwd's staged source pass (None when not
    asked for)."""
    __slots__ = ("rowptr_tr", "col_tr", "sel_q", "chunk_tab", "lrows", "lrow_ptr")


def list_transpose(idx, cnt, n_total, chunk_tables=False):
    """Transpose of the lists idx [nq, k] / cnt [nq] (entries t < cnt[i] are node ids < n_total, the rest padding).
    CUDA tensors: sng_list_transpose (a stable radix sort), and with `chunk_tables` the chunk tables over rowptr_tr, which
    read two counts back (one host synchronisation).  CPU tensors (the host-logic tests): the same construction in torch."""
    from .graph import PreparedGraph
    nq, k = idx.shape
    t = ListTranspose()
    t.chunk_tab = t.lrows = t.lrow_ptr = None
    dev = idx.device
    if not idx.is_cuda:
        valid = (torch.arange(k)[None, :] < cnt[:, None]).reshape(-1)
        key = torch.where(valid, idx.reshape(-1).long(), torch.full_like(valid, n_total, dtype=torch.long))
        perm = torch.argsort(key, stable=True)
        nnz = int(valid.sum())
        rowptr = torch.zeros(n_total + 1, dtype=torch.int64)
        torch.cumsum(torch.bincount(key[valid], minlength=n_total), 0, out=rowptr[1:])
        t.rowptr_tr = rowptr.to(torch.int32)
        t.col_tr = (perm[:nnz] // k).to(torch.int32)
        sel_q = torch.full((nq * k,), -1, dtype=torch.int32)
        sel_q[perm[:nnz]] = torch.arange(nnz, dtype=torch.int32)
        t.sel_q = sel_q.reshape(nq, k)
    else:
        _C.require_cuda(idx, cnt)
        idx, cnt = idx.contiguous(), cnt.contiguous()
        t.rowptr_tr = torch.empty(n_total + 1, dtype=torch.int32, device=dev)
        t.col_tr = torch.empty(max(nq * k, 1), dtype=torch.int32, device=dev)
        t.sel_q = torch.empty(nq, k, dtype=torch.int32, device=dev)
        wbytes = _C.lib().sng_list_transpose_workspace_bytes(nq, k, n_total)
        if wbytes == 0:
            raise RuntimeError(f"sng_list_transpose_workspace_bytes rejected nq={nq} k={k} n_total={n_total}")
        ws = torch.empty(wbytes, dtype=torch.uint8, device=dev)
        _C.call("sng_list_transpose", idx, _C.ptr(idx), _C.ptr(cnt), nq, k, n_total, _C.ptr(t.rowptr_tr), _C.ptr(t.col_tr),
                _C.ptr(t.sel_q), _C.ptr(ws), wbytes)
    if chunk_tables:
        rp = t.rowptr_tr.long()
        deg = rp[1:] - rp[:-1]
        long_rows = deg > 32
        n_long, n_chunks = (int(v) for v in torch.stack([long_rows.sum(), torch.where(long_rows, (deg + 31) // 32, 0).sum()]).tolist())
        slot = torch.where(long_rows, torch.cumsum(long_rows, 0) - 1, n_long)          # rank among the long rows; n_long = discard
        lr = torch.zeros(n_long + 1, dtype=torch.int64, device=dev).scatter_(0, slot, torch.arange(n_total, device=dev))[:n_long]
        t.chunk_tab, t.lrow_ptr = PreparedGraph._chunk_tables(t.rowptr_tr, lr, n_chunks)
        t.lrows = lr.to(torch.int32).contiguous()
    return t


def list_bwd(h_all, inv_norm, g, idx, sim, cnt, inv_denom, row_offset=0):
    """sng_list_bwd: dL/dh [N, Cp] of the list aggregation out[i] = inv_denom[i] sum_t sim[i, t] h[idx[i, t]] with sim the
    cosines of h -- sng_edge_bwd's two gather passes through the lists' transpose (built here), no float atomics.  The
    lists are rows [row_offset, row_offset + n) of `h_all` (all N nodes); dh is their contribution to dL/dh of every node."""
    n_total, cp = h_all.shape
    n, k = idx.shape
    dev = h_all.device
    tr = list_transpose(idx, cnt, n_total, chunk_tables=cp <= 32)
    n_chunks = -1 if tr.chunk_tab is None else int(tr.chunk_tab.size(0))
    cpart = None
    if n_chunks > 0:
        cg = 4
        while cg < cp:
            cg *= 2
        cpart = torch.empty(n_chunks * 3 * cg, dtype=torch.float32, device=dev)
    coef = torch.empty(max(n * k, 1) * 2, dtype=torch.float32, device=dev)
    dnt = torch.empty(n, cp, dtype=torch.float32, device=dev)
    dh = torch.empty_like(h_all)
    _C.call("sng_list_bwd", h_all, _C.ptr(h_all), _C.ptr(inv_norm), _C.ptr(g), n_total, n, int(row_offset), cp, cp, cp,
            k, _C.ptr(idx), _C.ptr(sim), _C.ptr(cnt), _C.ptr(inv_denom), _C.ptr(tr.sel_q), _C.ptr(tr.rowptr_tr), _C.ptr(tr.col_tr),
            _C.ptr(coef), _C.ptr(dnt), _C.ptr(dh), _C.ptr(tr.chunk_tab), n_chunks, _C.ptr(tr.lrows), _C.ptr(tr.lrow_ptr),
            0 if tr.lrows is None else int(tr.lrows.numel()), _C.ptr(cpart))
    return dh


class ListAgg(torch.autograd.Function):
    """Mean aggregation over an explicit neighbour list (all-pairs mode): forward sng_list_agg_fwd, backward sng_list_bwd
    (two gather passes through the lists' transpose, no float atomics, bit-reproducible).  With `row_offset` the lists are
    rows [row_offset, row_offset + len(idx)) of `h`, which holds every node (a row shard): the backward then returns this
    shard's contribution to dL/dh of every node -- contributions of different shards add (dist.AllGatherRows)."""

    @staticmethod
    def forward(ctx, h, idx, sim, cnt, inv_denom, row_offset=0):
        h = _check_h(h)
        n, c = h.shape
        nq = idx.size(0)
        if row_offset < 0 or row_offset + nq > n:
            raise RuntimeError(f"lists of rows [{row_offset}, {row_offset + nq}) but h has {n} rows")
        out = torch.empty(nq, c, dtype=h.dtype, device=h.device)
        if nq:
            _C.call("sng_list_agg_fwd", h, _C.ptr(h), nq, c, c, idx.size(1), _C.ptr(idx), _C.ptr(sim), _C.ptr(cnt),
                    _C.ptr(inv_denom), _C.ptr(out), c)
        ctx.row_offset = int(row_offset)
        ctx.save_for_backward(h, idx, sim, cnt, inv_denom)
        return out

    @staticmethod
    def backward(ctx, g):
        h, idx, sim, cnt, inv_denom = ctx.saved_tensors
        _, _, inv_norm = rownorm(h, want_f32=False, want_inv=True)
        idx, sim, cnt, inv_denom = idx.contiguous(), sim.contiguous(), cnt.contiguous(), inv_denom.contiguous()
        dh = list_bwd(h, inv_norm, g.contiguous(), idx, sim, cnt, inv_denom, ctx.row_offset)
        return dh, None, None, None, None, None


def spmm(x, rowptr, col, n_rows, val=None, rowscale=None, bias=None):
    """K3: out[i] = rowscale[i] * sum_e val[e] x[col[e]] + bias (no autograd; used inside backward passes)."""
    x = _check_h(x)
    c = x.size(1)
    out = torch.empty(n_rows, c, dtype=x.dtype, device=x.device)
    _C.call("sng_spmm_fwd", x, _C.ptr(x), n_rows, c, c, _C.ptr(rowptr), _C.ptr(col), _C.ptr(val), _C.ptr(rowscale),
            _C.ptr(bias), _C.ptr(out), c)
    return out


class PPFuse(torch.autograd.Function):
    """out = beta*(A @ W^T + b_w) + (1-beta)*out_1 (+bias)  --  R: models/models.py:124-136 (K4)."""

    @staticmethod
    def forward(ctx, out1, w_weight, w_bias, beta, bias, graph):
        out1 = _check_h(out1)
        n, cp = out1.shape
        c = w_weight.size(0)
        if w_weight.size(1) != n:
            raise RuntimeError(f"w.weight is [{c},{w_weight.size(1)}] but the graph has {n} nodes "
                               "(R builds w = Linear(num_nodes, out_channels), models.py:95)")
        out0, out = pp_fuse_fwd(out1, *_structural_operands(w_weight, w_bias, beta, bias, cp), graph.rowptr_out, graph.col_out)
        ctx.graph, ctx.c, ctx.has_bias = graph, c, bias is not None
        ctx.save_for_backward(out0, out1, beta)
        return out

    @staticmethod
    def backward(ctx, g):
        out0, out1, beta = ctx.saved_tensors
        graph, c = ctx.graph, ctx.c
        n, cp = out1.shape
        g = g.contiguous()
        dbeta = torch.empty(1, dtype=torch.float32, device=g.device)
        part = torch.empty(_C.PARTIALS, dtype=torch.float32, device=g.device)
        g0, dout1, dwt = torch.empty_like(g), torch.empty_like(g), torch.empty_like(g)
        # dL/dW^T = A^T g0: row t gathers g0 over the (shifted) sources of t's in-edges
        _C.call("sng_pp_fuse_bwd", g, _C.ptr(out0), _C.ptr(out1), _C.ptr(g), _C.ptr(beta), n, cp, cp, _C.ptr(graph.rowptr_in),
                _C.ptr(graph.col_in_shift), _C.ptr(dbeta), _C.ptr(part), _C.ptr(g0), _C.ptr(dout1), _C.ptr(dwt))
        db_w = g0.sum(0)[:c]
        dbias = g.sum(0)[:c] if ctx.has_bias else None
        return dout1, _weight_grad(dwt, c), db_w, dbeta, dbias, None


def pp_fuse_fwd(out1, wt, b_w, beta, bias, rowptr_out, col_out):
    """sng_pp_fuse_fwd (K4) on the rows of out1 [n, Cp]: (out0 = A W^T + b_w with A's rows given by rowptr_out / col_out,
    out = beta out0 + (1 - beta) out1 + bias).  The operands are those of _structural_operands; a shard may have no rows."""
    n, cp = out1.shape
    out0, out = torch.empty_like(out1), torch.empty_like(out1)
    if n:
        _C.call("sng_pp_fuse_fwd", out1, _C.ptr(wt), n, cp, cp, _C.ptr(rowptr_out), _C.ptr(col_out), _C.ptr(b_w), _C.ptr(beta),
                _C.ptr(out1), _C.ptr(bias), _C.ptr(out0), _C.ptr(out))
    return out0, out


def pp_beta_grad(out0, out1, g):
    """dL/dbeta [1] = sum((out0 - out1) g) of the K4 blend, summed in a fixed order (sng_pp_beta_grad); 0 for no rows."""
    dbeta = torch.zeros(1, dtype=torch.float32, device=g.device)
    if g.numel():
        part = torch.empty(_C.PARTIALS, dtype=torch.float32, device=g.device)
        _C.call("sng_pp_beta_grad", g, _C.ptr(out0), _C.ptr(out1), _C.ptr(g), g.numel(), _C.ptr(dbeta), _C.ptr(part))
    return dbeta


def _bn_rows(t):
    """A float32 CUDA [n, c] tensor with unit column stride (a column slice of a padded tensor is fine); else a contiguous copy."""
    _C.require_cuda(t)
    if t.dtype != torch.float32 or t.dim() != 2:
        raise RuntimeError("expected a float32 [N, C] tensor")
    return t if t.stride(1) == 1 and t.stride(0) >= t.size(1) else t.contiguous()


def _bn_workspace(n, c, dev):
    nb = _C.lib().sng_bn_workspace_bytes(n, c)
    if nb == 0:
        raise RuntimeError(f"sng_bn_workspace_bytes rejected c={c} (1 <= c <= {_C.MAX_CHANNELS})")
    return torch.empty(nb, dtype=torch.uint8, device=dev), nb


def bn_fwd_stats(z):
    """sng_bn_fwd_stats: FP64 [2, C] = (sum of a, sum of a^2) over the rows of z [n, C], a = relu(z); zeros for n = 0."""
    z = _bn_rows(z)
    n, c = z.shape
    sums = torch.empty(2, c, dtype=torch.float64, device=z.device)
    ws, nb = _bn_workspace(n, c, z.device)
    _C.call("sng_bn_fwd_stats", z, _C.ptr(z), n, c, max(z.stride(0), c), _C.ptr(sums), _C.ptr(ws), nb)
    return sums


def bn_fwd_apply(z, sums, n_total, eps, gamma, beta, mean=None, rstd=None):
    """sng_bn_fwd_apply: (y [n, C] = gamma (relu(z) - mean) rstd + beta, mean [C], rstd [C]).  Training: `sums` = the global
    bn_fwd_stats over n_total rows, mean / rstd are computed (biased variance).  Eval: sums = None, mean / rstd given."""
    z = _bn_rows(z)
    n, c = z.shape
    if sums is None:
        mean, rstd = mean.float().contiguous(), rstd.float().contiguous()
    else:
        mean = torch.empty(c, dtype=torch.float32, device=z.device)
        rstd = torch.empty(c, dtype=torch.float32, device=z.device)
    y = torch.empty(n, c, dtype=torch.float32, device=z.device)
    _C.call("sng_bn_fwd_apply", z, _C.ptr(z), n, c, max(z.stride(0), c), _C.ptr(sums), int(n_total), float(eps),
            _C.ptr(gamma.detach().contiguous()), _C.ptr(beta.detach().contiguous()), _C.ptr(mean), _C.ptr(rstd), _C.ptr(y), c)
    return y, mean, rstd


def bn_bwd_stats(z, g, mean, rstd):
    """sng_bn_bwd_stats: FP64 [2, C] = (sum of g, sum of g * ahat) over the rows, ahat = (relu(z) - mean) rstd; zeros for n = 0."""
    z, g = _bn_rows(z), _bn_rows(g)
    n, c = z.shape
    sums = torch.empty(2, c, dtype=torch.float64, device=z.device)
    ws, nb = _bn_workspace(n, c, z.device)
    _C.call("sng_bn_bwd_stats", z, _C.ptr(z), _C.ptr(g), n, c, max(z.stride(0), c), max(g.stride(0), c), _C.ptr(mean), _C.ptr(rstd),
            _C.ptr(sums), _C.ptr(ws), nb)
    return sums


def bn_bwd_apply(z, g, sums, n_total, gamma, mean, rstd):
    """sng_bn_bwd_apply: dL/dz [n, C] of y = batch_norm(relu(z)) from the global bn_bwd_stats `sums` over n_total rows
    (sums = None: eval-mode statistics, dz = 1[z > 0] gamma rstd g)."""
    z, g = _bn_rows(z), _bn_rows(g)
    n, c = z.shape
    dz = torch.empty(n, c, dtype=torch.float32, device=z.device)
    _C.call("sng_bn_bwd_apply", z, _C.ptr(z), _C.ptr(g), n, c, max(z.stride(0), c), max(g.stride(0), c), _C.ptr(sums), int(n_total),
            _C.ptr(gamma.detach().contiguous()), _C.ptr(mean), _C.ptr(rstd), _C.ptr(dz), c)
    return dz


def row_dropout_fwd(z, row_offset, seed, call, p, relu):
    """sng_row_dropout_fwd: y [n, C] = keep ? a / (1 - p) : 0, a = relu(z) if `relu` else z, for the rows [row_offset, row_offset + n)
    of a layer; the keep bit of element (row, channel) depends only on (seed, call, global row, channel)."""
    z = _bn_rows(z)
    n, c = z.shape
    y = torch.empty(n, c, dtype=torch.float32, device=z.device)
    _C.call("sng_row_dropout_fwd", z, _C.ptr(z), n, c, max(z.stride(0), c), int(row_offset), int(seed), int(call), float(p), int(relu),
            _C.ptr(y), c)
    return y


def row_dropout_bwd(z, g, row_offset, seed, call, p, relu):
    """sng_row_dropout_bwd: dL/dz [n, C] = keep && (!relu || z > 0) ? g / (1 - p) : 0, the mask regenerated from its counters
    (z is read only with `relu`; pass None without)."""
    g = _bn_rows(g)
    n, c = g.shape
    z = _bn_rows(z) if relu else None
    dz = torch.empty(n, c, dtype=torch.float32, device=g.device)
    _C.call("sng_row_dropout_bwd", g, _C.ptr(z), _C.ptr(g), n, c, max(z.stride(0), c) if relu else c, max(g.stride(0), c), int(row_offset),
            int(seed), int(call), float(p), int(relu), _C.ptr(dz), c)
    return dz


class RowDropout(torch.autograd.Function):
    """[relu +] counter-based dropout of a row block (row_dropout_fwd / row_dropout_bwd): saves z only, and only with relu -- the
    backward regenerates the mask.  `ops` supplies the two launch helpers (this module's, or the tests' CPU stand-ins)."""

    @staticmethod
    def forward(ctx, z, row_offset, seed, call, p, relu, ops):
        ctx.args, ctx.ops = (row_offset, seed, call, p, relu), ops
        ctx.save_for_backward(z if relu else None)
        return ops.row_dropout_fwd(z, row_offset, seed, call, p, relu)

    @staticmethod
    def backward(ctx, g):
        z, = ctx.saved_tensors
        return ctx.ops.row_dropout_bwd(z, g.contiguous(), *ctx.args), None, None, None, None, None, None


def rownorm(x, want_f32=True, want_f16=False, f16_ld=None, want_inv=False):
    """K0: F.normalize(x, p=2, dim=-1) (R: models/models.py:122).  Returns (xhat_f32, xhat_f16, inv_norm)."""
    _C.require_cuda(x)
    x = x.contiguous().float()
    n, d = x.shape
    xf = torch.empty_like(x) if want_f32 else None
    ldh = f16_ld or (d + 15) // 16 * 16
    xh = torch.empty(n, ldh, dtype=torch.float16, device=x.device) if want_f16 else None
    inv = torch.empty(n, dtype=torch.float32, device=x.device) if want_inv else None
    _C.call("sng_rownorm_f32", x, _C.ptr(x), n, d, d, _C.ptr(xf), d, _C.ptr(xh), ldh, _C.ptr(inv))
    return xf, xh, inv


def sddmm_dot(xhat, a, b):
    """s[e] = <xhat[a[e]], xhat[b[e]]> (R: SimGFAToolbox/dense.py:160-162)."""
    _C.require_cuda(xhat, a, b)
    xhat = xhat.contiguous()
    a = a.to(torch.int32).contiguous()
    b = b.to(torch.int32).contiguous()
    s = torch.empty(a.numel(), dtype=torch.float32, device=xhat.device)
    _C.call("sng_sddmm_dot", xhat, _C.ptr(xhat), xhat.size(0), xhat.size(1), xhat.size(1), _C.ptr(a), _C.ptr(b), a.numel(), _C.ptr(s))
    return s


class _NllLoss(torch.autograd.Function):
    @staticmethod
    def forward(ctx, logp, y):
        _C.require_cuda(logp, y)
        logp = logp.contiguous()
        y = y.contiguous().long()
        n, c = logp.shape
        out = torch.empty(2, dtype=torch.float32, device=logp.device)             # loss, count
        part = torch.empty(_C.PARTIALS, dtype=torch.float32, device=logp.device)
        _C.call("sng_nll_loss_fwd", logp, _C.ptr(logp), n, c, c, _C.ptr(y), _C.ptr(out), _C.ptr(out[1:]), _C.ptr(part))
        ctx.save_for_backward(y, out)
        ctx.shape = (n, c)
        return out[0]

    @staticmethod
    def backward(ctx, g):
        y, out = ctx.saved_tensors
        n, c = ctx.shape
        d = torch.empty(n, c, dtype=torch.float32, device=y.device)
        g = g.contiguous().float().reshape(1)
        _C.call("sng_nll_loss_bwd", y, n, c, c, _C.ptr(y), _C.ptr(g), _C.ptr(out[1:]), _C.ptr(d))
        return d, None


def nll_loss(logp, y, mask=None):
    """Mean negative log-likelihood of `logp` [N, C] (the models' log_softmax output) against labels `y` [N] -- what
    R: train.py:81 computes as F.nll_loss(out[mask], y[mask]).  `mask` (bool [N]) keeps the masked form in ONE pass: masked-out
    rows get the label -1 instead of being gathered away.  Fixed-order reductions: bit-reproducible, forward and backward."""
    if mask is not None:
        y = torch.where(mask, y, torch.full_like(y, -1))
    return _NllLoss.apply(logp, y)
