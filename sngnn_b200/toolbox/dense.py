"""Dense-feature similarity metrics (R: SimGFAToolbox/dense.py) on the GPU kernels.

  cosine at edges          -> K0 row-normalise + sng_sddmm_dot (never an N x N matrix; R builds one per node, dense.py:53-58)
  sums over all pairs      -> sng_class_sums_f64 closed form <S_a, S_b> (R materialises 1000-row blocks, dense.py:17-27,108-128)
  the N x N matrix itself  -> sng_gemm_nt_f16 on the tensor cores (tcgen05 / TMEM / TMA) with the FP16 split x-hat = hi + lo
                              ([hi|hi|lo] x [hi|lo|hi]^T = FP32 product to ~2^-22), only for the *_small functions that return it
  the distribution of the  -> sng_simhist_f16: the same split contraction with a binning epilogue, each unordered pair of
  N x N values                row tiles scored once, integer counts (nothing N x N is stored)
"""
import math

import torch

from .. import _C
from .. import functional as SF


def _dev(x):
    if not torch.cuda.is_available():
        raise RuntimeError("sngnn_b200.toolbox needs a CUDA device (there is no CPU path)")
    return x.device, torch.device("cuda", torch.cuda.current_device())


def _normalised(x):
    xf, _, _ = SF.rownorm(x.to(_dev(x)[1]).float())
    return xf


def _sort_by_source(edge_index):
    n = int(edge_index.max()) + 1
    return edge_index[:, (edge_index[0] * n + edge_index[1]).argsort(stable=True)]


def _class_sums(xhat, y=None, num_classes=1):
    n, d = xhat.shape
    sums = torch.zeros(num_classes, d, dtype=torch.float64, device=xhat.device)
    cnt = torch.zeros(num_classes, dtype=torch.float64, device=xhat.device)
    yy = None if y is None else y.to(xhat.device).to(torch.int32).contiguous()
    _C.call("sng_class_sums_f64", xhat, _C.ptr(xhat), _C.ptr(yy), n, d, d, num_classes, _C.ptr(sums), _C.ptr(cnt))
    return sums, cnt


def split_f16_operands(xhat):
    """A = [hi | hi | lo], B = [hi | lo | hi] (FP16, K' = 3 d padded to a multiple of 8) of the FP32 matrix xhat = hi + lo:
    one FP16 contraction A B^T over K' then equals xhat xhat^T up to the dropped lo.lo term (~2^-22 for unit rows)."""
    hi = xhat.half()
    lo = (xhat - hi.float()).half()
    n, d = xhat.shape
    kp = (3 * d + 7) // 8 * 8
    a = torch.zeros(n, kp, dtype=torch.float16, device=xhat.device)
    b = torch.zeros(n, kp, dtype=torch.float16, device=xhat.device)
    a[:, :d], a[:, d:2 * d], a[:, 2 * d:3 * d] = hi, hi, lo
    b[:, :d], b[:, d:2 * d], b[:, 2 * d:3 * d] = hi, lo, hi
    return a, b, 3 * d


def gemm_nt(a, b, k, row_scale=None, col_scale=None):
    """out [m, n] float32 = diag(row_scale) (a b^T) diag(col_scale) on the tensor cores (sng_gemm_nt_f16); a [m, lda], b [n, ldb] FP16."""
    _C.require_cuda(a, b, row_scale, col_scale)
    m, n = a.size(0), b.size(0)
    out = torch.empty(m, n, dtype=torch.float32, device=a.device)
    _C.call("sng_gemm_nt_f16", a, _C.ptr(a), a.size(1), _C.ptr(b), b.size(1), m, n, k, _C.ptr(row_scale), _C.ptr(col_scale), _C.ptr(out), n)
    return out


TILE_ROWS = 128        # rows per tile of sng_simhist_f16's schedule (include/sng.h)


def _hist_range(bins, range):
    lo, hi = float(range[0]), float(range[1])
    if isinstance(bins, bool) or not isinstance(bins, int) or bins < 1:
        raise ValueError(f"bins must be a positive int, got {bins!r}")
    if not (math.isfinite(lo) and math.isfinite(hi) and lo < hi):
        raise ValueError(f"range must be finite with lo < hi, got {range!r}")
    return lo, hi


def _hist_edges(lo, hi, bins, device):
    return torch.linspace(lo, hi, bins + 1, dtype=torch.float64, device=device)


def simhist_tiles(xhat, bins, lo, hi, tile_lo, tile_hi):
    """int64 [bins] counts of the ordered off-diagonal cosines scored by the row tiles [tile_lo, tile_hi) of sng_simhist_f16's
    symmetric schedule (128-row tiles; the counts of a split of [0, ceil(N / 128)) add up to the whole histogram)."""
    _C.require_cuda(xhat)
    a, b, k = split_f16_operands(xhat.contiguous())
    counts = torch.zeros(bins, dtype=torch.int64, device=xhat.device)
    _C.call("sng_simhist_f16", a, _C.ptr(a), a.size(1), _C.ptr(b), b.size(1), xhat.size(0), k, tile_lo, tile_hi, lo, hi, bins,
            _C.ptr(counts))
    return counts


def node_similarity_histogram(x, bins=200, range=(-1.0, 1.0)):
    """Histogram of the N (N - 1) off-diagonal cosines that node_similarity_dense_small returns, without the N x N matrix:
    (counts int64 [bins], edges float64 [bins + 1]) as numpy.histogram(values, bins, range) -- equal bins, the last one
    closed, values outside the range not counted.  Scores are the FP32 cosines of the split tensor-core contraction
    (error ~1e-5 or less, DESIGN.md §7), clamped to [-1, 1]; an all-zero row scores 0 with every row."""
    src, _ = _dev(x)
    lo, hi = _hist_range(bins, range)
    xhat = _normalised(x)
    t = (xhat.size(0) + TILE_ROWS - 1) // TILE_ROWS
    counts = simhist_tiles(xhat, bins, lo, hi, 0, t)
    return counts.to(src), _hist_edges(lo, hi, bins, src)


def cosine_similarity_dense_small(x):
    """R: dense.py:138-141 -- the full N x N cosine matrix."""
    src, dev = _dev(x)
    xhat = _normalised(x)
    a, b, k = split_f16_operands(xhat)
    return gemm_nt(a, b, k).to(src)


def node_similarity_dense_small(x):
    """R: dense.py:144-149 -- off-diagonal entries in row-major order, and their mean."""
    sim = cosine_similarity_dense_small(x)
    n = sim.size(0)
    off = sim[~torch.eye(n, dtype=torch.bool, device=sim.device)]
    return off, off.mean()


def node_similarity_dense_large_parted(x):
    """R: dense.py:9-30 -- (None, (sum_all - N) / (N - 1) * N), operator precedence of :28 reproduced."""
    src, _ = _dev(x)
    xhat = _normalised(x)
    s, _ = _class_sums(xhat)
    n = xhat.size(0)
    total = (s[0] * s[0]).sum()
    return None, ((total - n) / (n - 1) * n).float().to(src)


def _edge_cos(x, edge_index):
    src, dev = _dev(x)
    xhat = _normalised(x)
    ei = edge_index.to(dev)
    return SF.sddmm_dot(xhat, ei[0], ei[1]), src


def linked_node_similarity_dense_small(x, edge_index):
    """R: dense.py:152-155."""
    s, src = _edge_cos(x, edge_index)
    return s.reshape(-1, 1).to(src), s.mean().to(src)


def linked_node_similarity_dense_large(x, edge_index):
    """R: dense.py:33-62 -- edges sorted by (source, target); same values as the _small variant in that order."""
    return linked_node_similarity_dense_small(x, _sort_by_source(edge_index))


def _per_source_mean(s, src_ids, length):
    """scatter_mean of the edge scores by source id (R: SimGFAToolbox/dense.py:163, :86-97): sng_segment_mean, FP64 accumulation."""
    seg = src_ids.to(torch.int32).contiguous()
    out = torch.empty(length, dtype=torch.float32, device=s.device)
    wbytes = 12 * length + 256
    ws = torch.empty(wbytes, dtype=torch.uint8, device=s.device)
    _C.call("sng_segment_mean", s, _C.ptr(s.contiguous()), _C.ptr(seg), seg.numel(), length, _C.ptr(out), _C.ptr(ws), wbytes)
    return out


def neighborhood_similarity_dense_small(x, edge_index):
    """R: dense.py:158-164 -- scatter_mean over sources; output length = max source id + 1 (torch_scatter default)."""
    s, src = _edge_cos(x, edge_index)
    ids = edge_index[0].to(s.device)
    w = _per_source_mean(s, ids, int(ids.max()) + 1)
    return w.to(src), w.mean().to(src)


def neighborhood_similarity_dense_large(x, edge_index):
    """R: dense.py:65-101 -- per-node mean (isolated nodes count as 0), mean over ALL N nodes (:96)."""
    s, src = _edge_cos(x, edge_index)
    n = x.size(0)
    w = _per_source_mean(s, edge_index[0].to(s.device), n)
    return w.reshape(-1, 1).to(src), (w.sum() / n).to(src)


def class_similarity_dense_large(x, y):
    """R: dense.py:104-130 -- K x K matrix of mean cosine between classes (self pairs included on the diagonal)."""
    src, _ = _dev(x)
    k = len(torch.unique(y))
    xhat = _normalised(x)
    s, cnt = _class_sums(xhat, y, k)
    return ((s @ s.t()) / (cnt[:, None] * cnt[None, :])).float().to(src)


def class_similarity_dense_small(x, y):
    """R: dense.py:167-179."""
    m = class_similarity_dense_large(x, y)
    return m, m.mean()


def cosine_similarity(x):
    """R: utils/data_transform.py:83-86 -- x / ||x|| with NO eps (an all-zero row gives NaN, as in the reference)."""
    sim = cosine_similarity_dense_small(x)
    zero = (x.norm(dim=-1) == 0).to(sim.device)
    if zero.any():
        sim[zero, :] = float("nan")
        sim[:, zero] = float("nan")
    return sim


def edge_similarity_weight(x, edge_index):
    """R: utils/data_transform.py:89-91 -- cosine at the edges (SDDMM instead of an N x N matrix + gather)."""
    s, src = _edge_cos(x, edge_index)
    zero = (x.norm(dim=-1) == 0).to(s.device)
    if zero.any():
        ei = edge_index.to(s.device)
        s = torch.where(zero[ei[0]] | zero[ei[1]], torch.full_like(s, float("nan")), s)
    return s.to(src)
