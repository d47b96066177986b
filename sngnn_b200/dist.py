"""Row sharding across GPUs (one process per GPU, torch.distributed; NCCL over NVLink on the B200 box).

The path shards by rows (SURVEY.md §8(e)):
  * similarity build: rank r owns query rows [lo_r, hi_r); the only exchanged data is x-hat (FP16 for the tensor
    cores + FP32 for the exact rescore), all-gathered once per build; outputs stay sharded.
  * aggregation forward: rank r owns target rows [lo_r, hi_r) of the CSR-by-target; h is all-gathered per layer.
The reference has no distributed code at all (SURVEY.md §2); nothing here replaces a reference file.

The collective plumbing below is backend-agnostic (works on CPU tensors with gloo, which is how tests/ cover it);
the compute callables default to the CUDA kernels and can be injected by the tests.
"""
import torch
import torch.distributed as dist

from . import functional as SF


def world():
    if dist.is_available() and dist.is_initialized():
        return dist.get_world_size(), dist.get_rank()
    return 1, 0


def rows_per_rank(n, world_size):
    return (n + world_size - 1) // world_size


def shard_bounds(n, world_size, rank):
    """Contiguous equal shards of ceil(n / world) rows; the last ranks may own fewer (possibly zero) rows."""
    r = rows_per_rank(n, world_size)
    return min(n, rank * r), min(n, (rank + 1) * r)


def all_gather_rows(local, n, out=None, pad=None):
    """All-gather row shards produced by `shard_bounds` into a [n, ld] tensor (every rank gets all rows).
    `local` holds this rank's rows; shards are padded to equal size for all_gather_into_tensor."""
    ws, rank = world()
    if ws == 1:
        return local
    r = rows_per_rank(n, ws)
    ld = local.size(1)
    if pad is None:
        pad = torch.zeros(r, ld, dtype=local.dtype, device=local.device)
    if out is None:
        out = torch.empty(ws * r, ld, dtype=local.dtype, device=local.device)
    pad[: local.size(0)].copy_(local)
    dist.all_gather_into_tensor(out, pad)
    return out[:n]


def half_operand(xf_all, ldh):
    """FP16 copy [n, ldh] (zero padded) of normalised FP32 rows [n, ld32]: the K1 tensor-core operand, converted locally."""
    xh = torch.zeros(xf_all.size(0), ldh, dtype=torch.float16, device=xf_all.device)
    w = min(ldh, xf_all.size(1))
    xh[:, :w] = xf_all[:, :w]
    return xh


def build_knn_sharded(x_local, n, top_k, thr=-1.0, remove_self=True, normalize=None, build=None):
    """Similarity-kNN of this rank's query rows against all n nodes.

    x_local: this rank's rows [hi-lo, d] of the feature matrix (shard_bounds(n, world, rank)).
    Returns (idx, sim, cnt) for the local rows (global column ids), exactly the rows [lo, hi) of the unsharded build."""
    ws, rank = world()
    lo, hi = shard_bounds(n, ws, rank)
    if x_local.size(0) != hi - lo:
        raise ValueError(f"rank {rank} must hold rows [{lo},{hi}) but got {x_local.size(0)} rows")
    if normalize is None or build is None:
        from . import simknn
        normalize = normalize or simknn.normalize_operands
        build = build or simknn.build_knn_normalized
    d = x_local.size(1)
    xf, xh = normalize(x_local)                       # K0 on the local shard only
    xf_all = all_gather_rows(xf, n)                   # ONE collective: FP32 x-hat (needed for the exact rescore anyway)
    # the tensor-core operand is the FP16 rounding of the same values, so it is converted locally instead of gathered:
    # bit-identical to what the owning rank's K0 emitted, and it saves the second all-gather (261 of 705 MB at pokec scale)
    xh_all = half_operand(xf_all, xh.size(1))
    if hi == lo:
        return None
    return build(xf_all, xh_all, d, top_k, thr, remove_self, lo, hi)


def edge_agg_forward_sharded(h_local, graph, top_k=None, thr=None, agg=None):
    """out_1 rows [lo, hi) from the all-gathered h, forward only (no autograd; see `edge_agg_sharded` for training)."""
    ws, rank = world()
    n = graph.n
    lo, hi = shard_bounds(n, ws, rank)
    h_all = all_gather_rows(h_local, n)
    shard = graph.row_slice(lo, hi)
    if agg is None:
        agg = SF.edge_topk_agg_rows
    return agg(h_all, shard, lo, top_k, thr)


# ------------------------------------------------------------------------------------------ training: sharded forward + backward
def _reduce_scatter_rows(full, n):
    """Sum `full` [ws*R, ld] (R = rows_per_rank) over ranks and return this rank's rows.  NCCL: reduce_scatter_tensor;
    backends without it (gloo on CPU, used by the tests): all_reduce + slice."""
    ws, rank = world()
    r = rows_per_rank(n, ws)
    lo, hi = shard_bounds(n, ws, rank)
    if dist.get_backend() == "nccl":
        out = torch.empty(r, full.size(1), dtype=full.dtype, device=full.device)
        dist.reduce_scatter_tensor(out, full.contiguous(), op=dist.ReduceOp.SUM)
        return out[: hi - lo]
    dist.all_reduce(full, op=dist.ReduceOp.SUM)
    return full[lo:hi]


class AllGatherRows(torch.autograd.Function):
    """h_all [n, C] = concatenation of every rank's row shard; backward = reduce-scatter (sum) of dL/dh_all -- the one
    exchange of the sharded backward (SURVEY.md §8(e)): a rank's targets gather from, and so send gradient to, any source row."""

    @staticmethod
    def forward(ctx, local, n):
        ctx.n = n
        return all_gather_rows(local.contiguous(), n)

    @staticmethod
    def backward(ctx, g_all):
        ws, _ = world()
        n = ctx.n
        if ws == 1:
            return g_all, None
        r = rows_per_rank(n, ws)
        full = g_all.new_zeros(ws * r, g_all.size(1))
        full[:n].copy_(g_all)
        return _reduce_scatter_rows(full, n).contiguous(), None


def edge_agg_sharded(h_local, graph, top_k=None, thr=None, agg=None):
    """Differentiable out_1 rows [lo, hi): all-gather h (autograd-aware), then K2 on the shard; its backward produces the
    shard's contribution to dL/dh of every node, which AllGatherRows.backward reduce-scatters.
    `agg(h_all, shard, row_offset, top_k, thr)` defaults to the CUDA kernels (functional.ShardedEdgeTopkAgg); the gloo tests
    inject a differentiable CPU oracle."""
    ws, rank = world()
    n = graph.n
    lo, hi = shard_bounds(n, ws, rank)
    h_all = AllGatherRows.apply(h_local, n)
    shard = graph.row_slice(lo, hi)
    if agg is None:
        agg = SF.ShardedEdgeTopkAgg.apply
    return agg(h_all, shard, lo, top_k, thr), shard


def pp_fuse_sharded(out1_local, w_weight, w_bias, beta, bias, shard, n, lo, fuse=None):
    """SNGNN++ fusion on a row shard: out rows [lo, hi) = beta * (A[lo:hi] @ W^T + b_w) + (1 - beta) * out_1 (+ bias), with
    the replicated parameter W^T [n, C] gathered over the shard's out-neighbours.  The parameter gradients this produces
    are PARTIAL (this rank's rows only), like every other parameter gradient of a sharded step: `allreduce_grads` sums them.
    `fuse` defaults to _ShardedPPFuse (K4 on the shard's by-source CSR; it completes dL/dw.weight on every rank itself); the
    gloo tests inject a differentiable dense CPU version."""
    if fuse is not None:
        return fuse(out1_local, w_weight, w_bias, beta, bias, shard, n, lo)
    return _ShardedPPFuse.apply(out1_local, w_weight, w_bias, beta, bias, shard, n, lo)


class _ShardedPPFuse(torch.autograd.Function):
    """Unfused SNGNN++ epilogue on a row shard (graphs whose in-lists differ from their out-lists): sng_pp_fuse_fwd over the
    shard's by-source CSR.  dL/dW^T rows [lo, hi) need g0 of ALL rows (all-gather of g0); the row blocks of the gradient
    are then all-gathered, so every rank ends up with the COMPLETE dL/dw.weight (no all-reduce of a zero-padded matrix)."""

    @staticmethod
    def forward(ctx, out1, w_weight, w_bias, beta, bias, shard, n, lo):
        out1 = SF._check_h(out1)
        operands = SF._structural_operands(w_weight, w_bias, beta, bias, out1.size(1))      # W^T [n, Cp] replicated
        out0, out = SF.pp_fuse_fwd(out1, *operands, shard.rowptr_out, shard.col_out)
        ctx.shard, ctx.c, ctx.n, ctx.has_bias = shard, w_weight.size(0), n, bias is not None
        ctx.save_for_backward(out0, out1, beta)
        return out

    @staticmethod
    def backward(ctx, g):
        out0, out1, beta = ctx.saved_tensors
        c = ctx.c
        g = g.contiguous()
        dbeta = SF.pp_beta_grad(out0, out1, g)
        g0 = g * beta
        dw = _complete_dw(g0, ctx.shard, ctx.n, c)
        dbias = g.sum(0)[:c] if ctx.has_bias else None
        return g - g0, dw, g0.sum(0)[:c], dbeta, dbias, None, None, None


def _gather_row_blocks_async(local, n):
    """Start the all-gather of row blocks without waiting for it: returns (work | None, result [n, ld], buffers the caller keeps
    alive until it has waited).  The collective runs on the backend's own stream; `work.wait()` makes the current stream
    wait for it.  (NCCL only; other backends gather at once.)"""
    ws, _ = world()
    local = local.contiguous()
    if ws == 1:
        return None, local, None
    if dist.get_backend() != "nccl":
        return None, all_gather_rows(local, n), None
    r = rows_per_rank(n, ws)
    ld = local.size(1)
    pad = local if local.size(0) == r else torch.zeros(r, ld, dtype=local.dtype, device=local.device)
    if pad is not local:
        pad[: local.size(0)].copy_(local)
    out = torch.empty(ws * r, ld, dtype=local.dtype, device=local.device)
    work = dist.all_gather_into_tensor(out, pad, async_op=True)
    return work, out[:n], (pad, out)


def _complete_dw(g0, shard, n, c, pending=None):
    """dL/dw.weight [C, N] (complete, identical on every rank) from this shard's g0 = beta * dL/dout rows: row t of dL/dW^T
    gathers g0 over the (shifted) sources of t's in-edges -- any row of g0, hence the all-gather.  `pending` = an all-gather of
    g0 the caller already started (`_gather_row_blocks_async`), so that it overlaps the caller's kernels."""
    if pending is None:
        g0_all = all_gather_rows(g0, n)
    else:
        work, g0_all, _keep = pending
        if work is not None:
            work.wait()
    if shard.n:
        dwt_local = SF.spmm(g0_all.contiguous(), shard.rowptr_in, shard.col_in_shift, shard.n)
    else:
        dwt_local = g0.new_zeros(0, g0.size(1))
    return SF._weight_grad(all_gather_rows(dwt_local, n), c)                     # row blocks of dL/dW^T [n, Cp]


class _ShardedFusedAgg(torch.autograd.Function):
    """SNGNN++ layer on a row shard of a SYMMETRIC graph: aggregation, structural term and beta blend in ONE pass over the
    shard's in-edges (sng_edge_fwd with the fused epilogue; R: models/models.py:124-136).  Backward: sng_edge_bwd in its
    row-shard form (the shard's contribution to dL/dh of every node, reduce-scattered by AllGatherRows, and its part of
    dL/dbeta, both from fixed-order sums), dL/dW^T as above."""

    @staticmethod
    def forward(ctx, h_all, w_weight, w_bias, beta, bias, shard, n, lo, top_k, thr):
        h_all = SF._check_h(h_all)
        fuse = SF._structural_operands(w_weight, w_bias, beta, bias, h_all.size(1))
        train = any(ctx.needs_input_grad)
        out, sel_src, sel_w, sel_q, sel_cnt, inv_norm, diff = SF._edge_fwd(h_all, shard, lo, int(top_k), thr, train, fuse, want_q=True)
        ctx.shard, ctx.c, ctx.n, ctx.lo, ctx.k, ctx.has_bias = shard, w_weight.size(0), n, lo, int(top_k), bias is not None
        ctx.save_for_backward(h_all, sel_src, sel_w, sel_q, sel_cnt, inv_norm, diff, beta)
        return out

    @staticmethod
    def backward(ctx, g):
        h_all, sel_src, sel_w, sel_q, sel_cnt, inv_norm, diff, beta = ctx.saved_tensors
        shard, c = ctx.shard, ctx.c
        g = g.contiguous()
        g0 = g * beta
        pending = _gather_row_blocks_async(g0, ctx.n)             # needed only for dL/dW^T below: overlaps the aggregation backward
        dh, _, dbeta = SF.edge_bwd(h_all, inv_norm, g, shard, ctx.k, sel_src, sel_w, sel_q, sel_cnt, beta, diff, row_offset=ctx.lo)
        dw = _complete_dw(g0, shard, ctx.n, c, pending)
        dbias = g.sum(0)[:c] if ctx.has_bias else None
        return dh, dw, g0.sum(0)[:c], dbeta, dbias, None, None, None, None, None


def _all_reduce_sums(sums):
    ws, _ = world()
    if ws > 1:
        dist.all_reduce(sums, op=dist.ReduceOp.SUM)
    return sums


def _update_running_stats(bn, sums, n):
    """running_mean / running_var (unbiased: N / (N - 1)) / num_batches_tracked, as nn.BatchNorm1d updates them in training,
    from the global FP64 sums (identical on every rank, so the buffers are too)."""
    bn.num_batches_tracked.add_(1)
    f = 1.0 / float(bn.num_batches_tracked) if bn.momentum is None else bn.momentum
    mean = sums[0] / n
    var = (sums[1] / n - mean * mean).clamp_min(0.0) * (n / (n - 1))
    bn.running_mean.mul_(1.0 - f).add_(mean.to(bn.running_mean.dtype), alpha=f)
    bn.running_var.mul_(1.0 - f).add_(var.to(bn.running_var.dtype), alpha=f)


class _ShardedBatchNorm(torch.autograd.Function):
    """y = bn(relu(z)) on a row shard with the batch statistics of all n rows (R: models/models.py:81-84).  Forward: the shard's
    FP64 sums, ONE all-reduce of the [2, C] sums, apply; backward: the same with (sum g, sum g ahat), which are also the complete
    dL/dbeta and dL/dgamma on every rank (the caller marks both parameters `_sng_grad_complete`).  Eval mode: the running
    statistics, no collective in the forward.  `ops` = the four launch helpers of functional.py (or the tests' CPU stand-ins)."""

    @staticmethod
    def forward(ctx, z, weight, bias, bn, n, ops):
        if bn.training:
            sums = _all_reduce_sums(ops.bn_fwd_stats(z))
            y, mean, rstd = ops.bn_fwd_apply(z, sums, n, bn.eps, weight, bias)
            _update_running_stats(bn, sums, n)
        else:
            mean, rstd = bn.running_mean.clone(), torch.rsqrt(bn.running_var + bn.eps)
            y, mean, rstd = ops.bn_fwd_apply(z, None, n, bn.eps, weight, bias, mean, rstd)
        ctx.n, ctx.training, ctx.ops = n, bn.training, ops
        ctx.save_for_backward(z, weight, mean, rstd)
        return y

    @staticmethod
    def backward(ctx, g):
        z, weight, mean, rstd = ctx.saved_tensors
        sums = _all_reduce_sums(ctx.ops.bn_bwd_stats(z, g, mean, rstd))
        dz = ctx.ops.bn_bwd_apply(z, g, sums if ctx.training else None, ctx.n, weight, mean, rstd)
        return dz, sums[1].to(weight.dtype), sums[0].to(weight.dtype), None, None, None


def _check_batch_norm(bn, n):
    if not (bn.affine and bn.track_running_stats):
        raise NotImplementedError("sharded_forward: BatchNorm needs affine=True and track_running_stats=True (what the models build)")
    if bn.training and n <= 1:
        raise ValueError(f"Expected more than 1 value per channel when training, got input size {torch.Size([n, bn.num_features])}")


def sharded_batch_norm(z, bn, n, ops=None):
    """bn(relu(z)) for this rank's rows z [hi - lo, C] of an n-row batch, `bn` an nn.BatchNorm1d replicated on every rank: in
    training the statistics span all n rows (one all-reduce each way) and the running buffers come out identical on every rank.
    `ops` defaults to functional's CUDA helpers (bn_fwd_stats / bn_fwd_apply / bn_bwd_stats / bn_bwd_apply)."""
    _check_batch_norm(bn, n)
    bn.weight._sng_grad_complete = True                   # the backward returns the global sums: allreduce_grads skips them
    bn.bias._sng_grad_complete = True
    return _ShardedBatchNorm.apply(z, bn.weight, bn.bias, bn, n, SF if ops is None else ops)


def allreduce_grads(params):
    """Sum the (partial, per-shard) parameter gradients over ranks: every parameter is replicated, every rank holds the
    gradient contribution of its own rows.  Structural weights whose gradient the sharded backward already assembled on
    every rank (row blocks all-gathered, see _complete_dw) are skipped."""
    ws, _ = world()
    if ws == 1:
        return
    for p in params:
        if p.grad is not None and not getattr(p, "_sng_grad_complete", False):
            dist.all_reduce(p.grad, op=dist.ReduceOp.SUM)


def sharded_forward(model, x_local, edge_index, n, agg=None, fuse=None, bn_ops=None):
    """Row-sharded forward of an SNGNN / SNGNN_Plus / SNGNN_Plus_Plus model (replicated parameters): this rank holds the
    feature rows [lo, hi) and returns the log-probabilities of those rows.  Mirrors _SNStack.forward / the conv forwards of
    models.py (R: models/models.py:76-86,116-137,233-242,322-329) with the aggregation and the ++ fusion replaced by their
    sharded forms.  denominator='selected' with candidates='edges' is not supported here.
    candidates='all_pairs' (either denominator): h is all-gathered, the rank builds the kNN lists of its own rows over every
    node (simknn.allpairs_topk_agg with rows = [lo, hi)) and aggregates them; the SNGNN++ structural term goes through
    pp_fuse_sharded.
    top_k <= 0: out_1 = 0 on the local rows (the reference runs no selection round), with zero gradients; SNGNN++ still adds
    its structural term through pp_fuse_sharded.
    bn=True: relu + BatchNorm of the hidden layers run as sharded_batch_norm, with the statistics of all n rows (training) or
    the running statistics (eval); `bn_ops` replaces its four CUDA helpers (the tests inject CPU stand-ins)."""
    import torch.nn.functional as F
    from . import graph as G, models as M, simknn
    convs = list(model.lins)
    for conv in convs:                                       # reject unsupported options before any collective or kernel
        if type(conv) is not M.SNConv and conv.candidates != "all_pairs" and conv.denominator != "candidates":
            raise NotImplementedError("sharded_forward: candidates='edges' with denominator='selected'")
    use_bn = getattr(model, "bn", False)
    if use_bn:
        for bn in model.bns:
            _check_batch_norm(bn, n)
    ws, rank = world()
    lo, hi = shard_bounds(n, ws, rank)
    x = x_local
    for i, conv in enumerate(convs):
        base = type(conv) is M.SNConv
        plus_plus = isinstance(conv, M.SNConv_plus_plus)
        all_pairs = not base and conv.candidates == "all_pairs"
        no_select = not base and conv.top_k <= 0
        g = G.prepare(edge_index, n, remove_self_loops=False if base else bool(conv.is_remove_self_loops))
        h = conv._hidden_norm(x)[0]                          # lin + bias in the library's kernel (its backward is the one-pass dW / db)
        injected = agg is not None or fuse is not None
        if plus_plus:
            conv.w.weight._sng_grad_complete = not injected      # the CUDA backward assembles the complete gradient itself
        if no_select:
            out = h * 0.0                                    # SNConv_plus._aggregate: zero out_1, zero (not missing) gradients
            if plus_plus:
                out = pp_fuse_sharded(out, conv.w.weight, conv.w.bias, conv.beta, conv.bias, g.row_slice(lo, hi), n, lo, fuse=fuse)
                out = out[:, :conv.lin.out_features]
            else:
                out = out[:, :conv.lin.out_features]
                if conv.bias is not None:
                    out = out + conv.bias
        elif plus_plus and not all_pairs and not injected and g.symmetric:
            h_all = AllGatherRows.apply(h, n)
            out = _ShardedFusedAgg.apply(h_all, conv.w.weight, conv.w.bias, conv.beta, conv.bias, g.row_slice(lo, hi), n, lo,
                                         conv.top_k, conv.thr)
            out = out[:, :conv.lin.out_features]
        else:
            if all_pairs:
                h_all = AllGatherRows.apply(h, n)
                out = simknn.allpairs_topk_agg(h_all, conv.top_k, conv.thr, bool(conv.is_remove_self_loops), conv.denominator,
                                               rows=(lo, hi))
                shard = g.row_slice(lo, hi) if plus_plus else None
            else:
                out, shard = edge_agg_sharded(h, g, None if base else conv.top_k, None if base else conv.thr, agg=agg)
            if plus_plus:
                out = pp_fuse_sharded(out, conv.w.weight, conv.w.bias, conv.beta, conv.bias, shard, n, lo, fuse=fuse)
                out = out[:, :conv.lin.out_features]
            else:
                out = out[:, :conv.lin.out_features]
                if conv.bias is not None:
                    out = out + conv.bias
        if i < len(convs) - 1:
            out = sharded_batch_norm(out, model.bns[i], n, bn_ops) if use_bn else F.relu(out)
            out = model.dropout(out)
        x = out
    return F.log_softmax(x, dim=1)
