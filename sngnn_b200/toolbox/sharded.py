"""Row-sharded forms of the Sim-GFA metrics that reduce over all pairs (SURVEY.md §8(e) "toolbox reductions"): every rank
holds the feature rows [lo, hi) of `dist.shard_bounds`, computes the FP64 class sums of its rows with `sng_class_sums_f64`,
and ONE all-reduce of the [K, d] sums (+ the [K] counts) gives every rank the closed forms <S_a, S_b> behind
R: SimGFAToolbox/dense.py:9-30 (node similarity) and :104-130 (class similarity).  The edge metrics shard by edges: each rank
scores its slice of the edge list against the all-gathered x-hat and the scalar mean is all-reduced.  The similarity
histogram shards by row tiles of its symmetric schedule over the all-gathered x-hat and all-reduces the integer counts.
Works with any torch.distributed backend (NCCL on the B200 box; the CPU tests inject the local kernels and use gloo)."""
import torch
import torch.distributed as dist

from .. import dist as sdist


def _allreduce(t):
    ws, _ = sdist.world()
    if ws > 1:
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
    return t


def _local_class_sums(x_local, y_local, num_classes, class_sums=None):
    if class_sums is None:
        from . import dense as D
        xhat = D._normalised(x_local)
        return D._class_sums(xhat, y_local, num_classes)
    return class_sums(x_local, y_local, num_classes)


def node_similarity_dense_large_parted_sharded(x_local, n, class_sums=None):
    """(None, (sum_all - N) / (N - 1) * N) of R: dense.py:9-30 from row shards: sum_all = <S, S>, S = sum of all unit rows."""
    s, _ = _local_class_sums(x_local, None, 1, class_sums)
    s = _allreduce(s.clone())
    total = (s[0] * s[0]).sum()
    return None, ((total - n) / (n - 1) * n).float()


def class_similarity_dense_large_sharded(x_local, y_local, num_classes, class_sums=None):
    """K x K matrix of mean cosine between classes (R: dense.py:104-130) from row shards."""
    s, cnt = _local_class_sums(x_local, y_local, num_classes, class_sums)
    s, cnt = _allreduce(s.clone()), _allreduce(cnt.clone())
    return ((s @ s.t()) / (cnt[:, None] * cnt[None, :])).float()


def linked_node_similarity_dense_sharded(x_local, edge_index, n, edge_cos=None):
    """Mean cosine over the edges (R: dense.py:33-62 / :152-155): x-hat all-gathered once, every rank scores the edge slice
    [rank * ceil(E / world), ...) and the (sum, count) pair is all-reduced.  Returns (local edge scores, global mean)."""
    ws, rank = sdist.world()
    if edge_cos is None:
        from . import dense as D
        from .. import functional as SF
        xhat_local = D._normalised(x_local)
        xhat = sdist.all_gather_rows(xhat_local, n)

        def edge_cos(xh, a, b):
            return SF.sddmm_dot(xh.contiguous(), a, b)
    else:
        xhat = sdist.all_gather_rows(torch.nn.functional.normalize(x_local.float(), dim=-1), n)
    e = edge_index.size(1)
    per = (e + ws - 1) // ws
    lo, hi = min(e, rank * per), min(e, (rank + 1) * per)
    ei = edge_index[:, lo:hi].to(xhat.device)
    s = edge_cos(xhat, ei[0], ei[1]) if hi > lo else xhat.new_zeros(0)
    acc = torch.stack([s.double().sum(), torch.tensor(float(hi - lo), dtype=torch.float64, device=s.device)])
    acc = _allreduce(acc)
    return s, (acc[0] / acc[1].clamp(min=1)).float()


def node_similarity_histogram_sharded(x_local, n, bins=200, range=(-1.0, 1.0), hist=None):
    """node_similarity_histogram of all n rows from row shards: x-hat all-gathered once (FP32), rank r scores a contiguous,
    equal share of the T = ceil(n / 128) row tiles of sng_simhist_f16's schedule (every row tile does the same work), and
    ONE all-reduce of the int64 counts.  Every rank returns (counts, edges), the counts equal bit for bit to the
    single-GPU call.  `hist(xhat, bins, lo, hi, tile_lo, tile_hi)` stands in for the kernel (CPU tests)."""
    from . import dense as D
    ws, rank = sdist.world()
    lo, hi = D._hist_range(bins, range)
    if hist is None:
        xhat = sdist.all_gather_rows(D._normalised(x_local), n)
        hist = D.simhist_tiles
    else:
        xhat = sdist.all_gather_rows(torch.nn.functional.normalize(x_local.float(), dim=-1), n)
    t = (n + D.TILE_ROWS - 1) // D.TILE_ROWS
    per = (t + ws - 1) // ws
    counts = hist(xhat, bins, lo, hi, min(t, rank * per), min(t, (rank + 1) * per))
    return _allreduce(counts), D._hist_edges(lo, hi, bins, counts.device)
