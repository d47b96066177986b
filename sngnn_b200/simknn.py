"""All-pairs similarity-kNN builder (host side of K0 + K1, include/sng.h).

`build_knn` = "the reference selection rule on the complete graph" (SURVEY.md §0): for query node i the
candidates are all nodes j (minus i when remove_self), ranked by (cosine desc, j asc), at most top_k, cut at
the first cosine < thr -- i.e. R: models/models.py:145-156 applied to every pair, with the all-pairs cosine of
R: SimGFAToolbox/dense.py:17-27 computed on the tensor cores and never written to HBM.

Row sharding: `q_lo:q_hi` selects the query rows this call (this rank) owns; the database is always all of x.
"""
import torch

from . import _C
from . import functional as SF


def _pad_to(v, m):
    return (v + m - 1) // m * m


def normalize_operands(x):
    """K0: returns (xhat_f32 [N, ld32], xhat_f16 [N, ldh]) zero padded to ld32 = 4*ceil(d/4), ldh = 16*ceil(d/16)."""
    _C.require_cuda(x)
    x = x.contiguous().float()
    n, d = x.shape
    ld32, ldh = _pad_to(d, 4), _pad_to(d, 16)
    xf = torch.empty(n, ld32, dtype=torch.float32, device=x.device)
    xh = torch.empty(n, ldh, dtype=torch.float16, device=x.device)
    _C.call("sng_rownorm_f32", x, _C.ptr(x), n, d, d, _C.ptr(xf), ld32, _C.ptr(xh), ldh, None)
    return xf, xh


def list_width(n, top_k, remove_self):
    """Width of the lists a build returns: top_k up to SNG_KNN_MAX_TOPK (64), above it k_eff = min(top_k, n - remove_self),
    at least 1 (top_k = 2**40 asks for every neighbour with cosine >= thr)."""
    top_k = int(top_k)
    return top_k if top_k <= _C.KNN_MAX_TOPK else max(1, min(top_k, n - (1 if remove_self else 0)))


def build_knn_normalized(xf, xh, d, top_k, thr, remove_self=True, q_lo=0, q_hi=None, return_fallback=False):
    """K1 on already normalised operands (what a rank calls after the all-gather of x-hat).  return_fallback adds a device
    int32[2] = [rows that needed the exact scan, rows that needed the retry pass].
    The lists are list_width(n, top_k, remove_self) wide.  Up to SNG_KNN_MAX_TOPK (64) that is sng_simknn_build; wider lists
    take the wide build (sng_simknn_wide_count + _select), which reads the candidate total back to allocate the candidate
    buffer: one host synchronisation, so a wide build cannot be captured in a CUDA graph."""
    n = xf.size(0)
    q_hi = n if q_hi is None else q_hi
    nq = q_hi - q_lo
    if nq <= 0:
        raise ValueError("empty query range")
    if int(top_k) < 1:
        raise ValueError(f"top_k={top_k} must be >= 1")
    top_k = list_width(n, top_k, remove_self)
    if top_k > _C.KNN_MAX_TOPK:
        return _build_wide(xf, xh, d, top_k, thr, remove_self, q_lo, nq, return_fallback)
    dev = xf.device
    idx = torch.empty(nq, top_k, dtype=torch.int32, device=dev)
    sim = torch.empty(nq, top_k, dtype=torch.float32, device=dev)
    cnt = torch.empty(nq, dtype=torch.int32, device=dev)
    nfb = torch.zeros(2, dtype=torch.int32, device=dev)          # [rows that needed the exact scan, rows that needed the retry pass]
    wbytes = _C.lib().sng_simknn_workspace_bytes(nq, n, d, top_k)
    if wbytes == 0:
        raise RuntimeError(f"sng_simknn_workspace_bytes rejected nq={nq} n={n} d={d} top_k={top_k}: {_C.last_error()}")
    ws = torch.empty(wbytes, dtype=torch.uint8, device=dev)
    _C.require_cuda(xf, xh)
    _C.call("sng_simknn_build", xf, _C.ptr(xh[q_lo:]), _C.ptr(xh), xh.size(1), _C.ptr(xf[q_lo:]), _C.ptr(xf), xf.size(1),
            nq, q_lo, n, d, int(top_k), float(thr), int(bool(remove_self)),
            _C.ptr(idx), _C.ptr(sim), _C.ptr(cnt), _C.ptr(nfb), _C.ptr(nfb[1:]), _C.ptr(ws), wbytes)
    if return_fallback:
        return idx, sim, cnt, nfb
    return idx, sim, cnt


def _build_wide(xf, xh, d, k_eff, thr, remove_self, q_lo, nq, return_fallback):
    n = xf.size(0)
    if nq * k_eff >= 2 ** 31:
        raise ValueError(f"{nq} query rows x {k_eff} neighbours = {nq * k_eff} list entries: the lists are limited to < 2**31 "
                         "entries (int32 positions of the list transpose); use fewer rows per call or a smaller top_k")
    dev = xf.device
    _C.require_cuda(xf, xh)
    wbytes = _C.lib().sng_simknn_wide_workspace_bytes(nq, n, d, k_eff)
    if wbytes == 0:
        raise RuntimeError(f"sng_simknn_wide_workspace_bytes rejected nq={nq} n={n} d={d} top_k={k_eff}")
    ws = torch.empty(wbytes, dtype=torch.uint8, device=dev)
    offsets = torch.empty(nq + 1, dtype=torch.int64, device=dev)
    common = (_C.ptr(xh[q_lo:]), _C.ptr(xh), xh.size(1))
    _C.call("sng_simknn_wide_count", xf, *common, nq, q_lo, n, d, k_eff, float(thr), int(bool(remove_self)), _C.ptr(offsets),
            _C.ptr(ws), wbytes)
    total = int(offsets[nq])                                 # the wide build's one host synchronisation
    cand = torch.empty(max(total, 1), dtype=torch.int32, device=dev)
    idx = torch.empty(nq, k_eff, dtype=torch.int32, device=dev)
    sim = torch.empty(nq, k_eff, dtype=torch.float32, device=dev)
    cnt = torch.empty(nq, dtype=torch.int32, device=dev)
    nfb = torch.zeros(2, dtype=torch.int32, device=dev)      # [rows that needed the exact scan, 0: the wide build has no retry pass]
    _C.call("sng_simknn_wide_select", xf, *common, _C.ptr(xf[q_lo:]), _C.ptr(xf), xf.size(1), nq, q_lo, n, d, k_eff, float(thr),
            int(bool(remove_self)), _C.ptr(offsets), _C.ptr(cand), _C.ptr(idx), _C.ptr(sim), _C.ptr(cnt), _C.ptr(nfb), _C.ptr(ws), wbytes)
    if return_fallback:
        return idx, sim, cnt, nfb
    return idx, sim, cnt


def build_knn(x, top_k, thr=-1.0, remove_self=True, q_lo=0, q_hi=None, return_fallback=False):
    """idx [nq, k] int32 (-1 padded, rank order), sim [nq, k] float32, cnt [nq] int32; k = list_width(n, top_k, remove_self)."""
    xf, xh = normalize_operands(x)
    return build_knn_normalized(xf, xh, x.size(1), top_k, thr, remove_self, q_lo, q_hi, return_fallback)


def knn_to_csr(idx, cnt, sim=None):
    """CSR neighbour lists of fixed-width kNN lists (sng_knn_to_csr: exclusive scan + compaction on the device):
    rowptr int32 [nq+1], col int32 [nnz] (rank order within a row) and, with `sim`, val float32 [nnz]."""
    if not idx.is_cuda:                                      # host lists (tests of the host logic): same result with torch ops
        nq, k = idx.shape
        rowptr = torch.zeros(nq + 1, dtype=torch.int64)
        torch.cumsum(cnt.long().clamp(0, k), 0, out=rowptr[1:])
        keep = torch.arange(k)[None, :] < cnt[:, None]
        flat = keep.reshape(-1).nonzero().flatten()
        out = (rowptr.to(torch.int32), idx.reshape(-1)[flat].contiguous())
        return out + ((sim.reshape(-1)[flat].contiguous(),) if sim is not None else ())
    _C.require_cuda(idx, cnt, sim)
    idx, cnt = idx.contiguous(), cnt.contiguous()
    nq, k = idx.shape
    dev = idx.device
    rowptr = torch.empty(nq + 1, dtype=torch.int32, device=dev)
    col = torch.empty(nq * k, dtype=torch.int32, device=dev)
    val = torch.empty(nq * k, dtype=torch.float32, device=dev) if sim is not None else None
    wbytes = _C.lib().sng_knn_to_csr_workspace_bytes(nq)
    ws = torch.empty(wbytes, dtype=torch.uint8, device=dev)
    _C.call("sng_knn_to_csr", idx, _C.ptr(idx), _C.ptr(None if sim is None else sim.contiguous()), _C.ptr(cnt), nq, k, _C.ptr(rowptr), _C.ptr(col),
            _C.ptr(val), _C.ptr(ws), wbytes)
    nnz = int(rowptr[-1])
    return (rowptr, col[:nnz]) + ((val[:nnz],) if sim is not None else ())


def build_plan(nq, n, d, top_k):
    """The launch plan sng_simknn_build picks for this shape (sng_simknn_plan): dict with ew (epilogue warps per TMEM
    lane quarter), cand (slots per list), nsplit, seed_stride (0 = no seed pass), seed_q, stages, kblocks, lists."""
    import ctypes
    out = (ctypes.c_int32 * 8)()
    _C.check(_C.lib().sng_simknn_plan(nq, n, d, int(top_k), out), "sng_simknn_plan")
    return dict(zip(("ew", "cand", "nsplit", "seed_stride", "seed_q", "stages", "kblocks", "lists"), list(out)))


def seed_pass(xh_q, xh_all, d, seed_stride, force_ew=0):
    """Tensor-core seed pass only (tests / profiling): [nq, 16] group maxima over every seed_stride-th database row."""
    nq, n = xh_q.size(0), xh_all.size(0)
    seeds = torch.empty(nq, 16, dtype=torch.float32, device=xh_q.device)
    _C.call("sng_simknn_seed", xh_q, _C.ptr(xh_q), _C.ptr(xh_all), xh_all.size(1), nq, n, d, int(seed_stride), force_ew, _C.ptr(seeds))
    return seeds


def stage1_candidates(x, cand, thr_lo=-2.0, remove_self=True, force_ew=0, force_nsplit=0, seed_stride=0, seed_q=0):
    """Tensor-core stage only (tests / profiling): FP16-scored candidate lists [N, lists, cand] + per-list drop bounds.
    seed_stride > 0 runs the seed pass first and starts every row at its seed_q-th largest group maximum."""
    import ctypes
    xf, xh = normalize_operands(x)
    n, d = x.shape
    dev = x.device
    slots = 192                                              # lists * cand never exceeds this (kMaxCandTotal)
    ci = torch.empty(n * slots, dtype=torch.int32, device=dev)
    cv = torch.empty(n * slots, dtype=torch.float32, device=dev)
    cm = torch.empty(n * 64, dtype=torch.float32, device=dev)
    nl = ctypes.c_int(0)
    seeds = seed_pass(xh, xh, d, seed_stride, force_ew) if seed_stride > 0 else None
    _C.call("sng_simknn_stage1", xh, _C.ptr(xh), _C.ptr(xh), xh.size(1), n, 0, n, d, cand, float(thr_lo), int(remove_self),
            _C.ptr(ci), _C.ptr(cv), _C.ptr(cm), force_ew, force_nsplit, ctypes.byref(nl),
            _C.ptr(seeds), int(seed_q), int(seed_stride), None)
    s = nl.value
    return ci[: n * s * cand].reshape(n, s, cand), cv[: n * s * cand].reshape(n, s, cand), cm[: n * s].reshape(n, s), xf, xh


def allpairs_topk_agg(h, top_k, thr, remove_self, denominator="candidates", rows=None):
    """All-pairs candidate mode of SNConv_plus(_plus): kNN on the layer's own h (similarity is on lin(x),
    SURVEY.md D4), then the cosine-weighted mean.  `h` is the padded [N, Cp] hidden matrix.
    rows = (lo, hi): only query rows [lo, hi) (a row shard; `h` still holds every node, e.g. after an all-gather).  The build
    then runs on the same operands over those rows, so their lists and similarities equal the unsharded build's bit for bit;
    the output has hi - lo rows and its backward is their contribution to dL/dh of every node (zero for an empty range)."""
    n = h.size(0)
    lo, hi = (0, n) if rows is None else (int(rows[0]), int(rows[1]))
    if hi <= lo:                                          # empty shard: no build (it rejects empty ranges), zero contribution
        k = list_width(n, top_k, remove_self)
        idx = torch.empty(0, k, dtype=torch.int32, device=h.device)
        sim = torch.empty(0, k, dtype=torch.float32, device=h.device)
        cnt = torch.empty(0, dtype=torch.int32, device=h.device)
    else:
        xf, xh = normalize_operands(h.detach())
        idx, sim, cnt = build_knn_normalized(xf, xh, h.size(1), top_k, thr, remove_self, lo, hi)
    if denominator == "candidates":
        cand = float(n - 1 if remove_self else n)
        inv = torch.full((hi - lo,), 1.0 / max(cand, 1.0), dtype=torch.float32, device=h.device)
    else:
        inv = cnt.clamp(min=1).float().reciprocal()
    return SF.ListAgg.apply(h, idx, sim, cnt, inv, lo)
