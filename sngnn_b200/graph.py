"""One-time graph preparation for the edge-restricted path.

The reference re-does this work every forward in Python/PyG (R: models/models.py:117-127, :234-236, :323):
append N self loops, optionally drop every src==dst edge, and (for ++) build a COO adjacency with
sources shifted by min(src).  Here it is done once per (edge_index, flags), cached, and turned into the
int32 CSR arrays the kernels consume:

  * CSR by TARGET (`rowptr_in`, `col_in`): in-edges of every node in ORIGINAL EDGE-POSITION order -- the
    tie-break of the selection rule is "lowest position first" (SURVEY.md §3.3), so the order is part of
    the contract;  `inv_deg[i] = 1 / max(indeg(i), 1)` is the PyG aggr='mean' denominator.
  * CSR by SHIFTED SOURCE (`rowptr_out`, `col_out`): out-neighbours t of node (src - min src), for
    out_0 = A @ W^T (R: :124-130);  `col_in_shift = col_in - min(src)` serves its transpose in backward.
  * `tpos[p]` = position of by-target edge p in the by-source arrays: the transpose index that lets the backward of the
    aggregation run as two gather passes without float atomics (sng_edge_bwd).  `rowptr_tr` / `col_tr` name the by-source
    CSR that `tpos` points into: the same tensors as `rowptr_out` / `col_out` for a whole graph, the shard's own
    transpose for a row shard (`row_slice`).
  * `rows_long` / `rows_hub`: target rows with 32 < in-degree <= 1024 / > 1024 (the forward's degree dispatch), and
    `symmetric`: every in-list equals the out-list with min(src) == 0, which lets SNGNN++ gather W^T rows in the same pass.
The by-source arrays are always built: the deterministic backward of every model needs them.

CUDA `edge_index`: one call of `sng_graph_prepare` (stable radix sort by target / source, include/sng.h).  CPU tensors
(the host-logic and gloo tests): the same construction in torch, with a stable argsort.
"""
import weakref

import torch

_CACHE = {}
_CACHE_MAX = 8


class PreparedGraph:
    __slots__ = ("n", "num_edges", "rowptr_in", "col_in", "inv_deg", "src_shift", "rowptr_out", "col_out",
                 "col_in_shift", "_shards", "tpos", "rows_long", "rows_hub", "symmetric", "max_deg", "is_shard",
                 "chunk_tab", "lrows", "lrow_ptr", "chunk_tab_out", "lrows_out", "lrow_ptr_out", "rowptr_tr", "col_tr")

    @staticmethod
    def _chunk_tables(rowptr, lrows, n_chunks=None):
        """(chunk_tab [n_chunks, 4] = first edge position, edges, row, 0; lrow_ptr) of the rows `lrows` (ascending) of a CSR.
        `n_chunks` (the total, when the caller knows it) spares the host synchronisation of sizing the table."""
        dev = rowptr.device
        rp = rowptr.long()
        beg, deg = rp[lrows], rp[lrows + 1] - rp[lrows]
        nch = (deg + 31) // 32
        ptr = torch.zeros(lrows.numel() + 1, dtype=torch.int64, device=dev)
        torch.cumsum(nch, 0, out=ptr[1:])
        owner = torch.repeat_interleave(torch.arange(lrows.numel(), device=dev), nch, output_size=n_chunks)   # chunk -> its long row
        within = torch.arange(owner.numel(), device=dev) - ptr[owner]
        cbeg = beg[owner] + 32 * within
        clen = torch.minimum(deg[owner] - 32 * within, torch.full_like(within, 32))
        tab = torch.stack([cbeg, clen, lrows[owner], torch.zeros_like(cbeg)], 1).to(torch.int32).contiguous()
        return tab, ptr.to(torch.int32).contiguous()

    def build_chunks(self):
        """Degree dispatch tables of sng_edge_fwd / sng_edge_bwd: every row with more than 32 in-edges (out-edges for the
        by-source pass of the backward) is cut into chunks of <= 32 consecutive edges, so a hub is handled by many warps.
        Built once per graph."""
        self.chunk_tab = self.lrows = self.lrow_ptr = self.chunk_tab_out = self.lrows_out = self.lrow_ptr_out = None
        if self.rows_long is None:
            return
        lrows = torch.cat([self.rows_long, self.rows_hub]).long().sort().values
        self.chunk_tab, self.lrow_ptr = self._chunk_tables(self.rowptr_in, lrows)
        self.lrows = lrows.to(torch.int32).contiguous()
        if self.rowptr_tr is not None:
            rp = self.rowptr_tr.long()
            lr = ((rp[1:] - rp[:-1]) > 32).nonzero().flatten()                             # rows of the by-source CSR = source id - shift
            self.chunk_tab_out, self.lrow_ptr_out = self._chunk_tables(self.rowptr_tr, lr)
            self.lrows_out = (lr + self.src_shift).to(torch.int32).contiguous()               # true source ids

    def row_slice(self, lo, hi):
        """Row-sharded view (targets [lo, hi)) for multi-GPU aggregation: rowptr rebased to 0.  Cached per (lo, hi).

        The shard gets its own transpose index, so that its backward runs the same two gather passes as a whole graph's:
        `rowptr_tr` [n + 1] / `col_tr` = CSR by (source - src_shift) over ALL n source rows holding only the shard's
        in-edges, targets as shard-local ids; `tpos[p]` = position of shard by-target edge p in those arrays.  They are a
        stable compaction of the whole graph's by-source arrays (no sort), so every source row lists its shard edges in the
        whole graph's order, and the shard [0, n) has exactly the whole graph's transpose."""
        cache = getattr(self, "_shards", None)
        if cache is None:
            cache = self._shards = {}
        if (lo, hi) in cache:
            return cache[(lo, hi)]
        g = cache[(lo, hi)] = PreparedGraph()
        g.n = hi - lo
        b, e = int(self.rowptr_in[lo]), int(self.rowptr_in[hi])
        g.num_edges = e - b
        g.rowptr_in = (self.rowptr_in[lo:hi + 1] - b).contiguous()
        g.col_in = self.col_in[b:e].contiguous()
        g.inv_deg = self.inv_deg[lo:hi].contiguous()
        g.src_shift = self.src_shift
        g.col_in_shift = None if self.col_in_shift is None else self.col_in_shift[b:e].contiguous()
        g.rowptr_out = g.col_out = g.tpos = g.rowptr_tr = g.col_tr = None
        if self.tpos is not None:
            keep = (self.col_out >= lo) & (self.col_out < hi)                # by-source edges whose target is in the shard
            newpos = torch.zeros(keep.numel() + 1, dtype=torch.int64, device=keep.device)
            torch.cumsum(keep, 0, out=newpos[1:])                             # newpos[q] = kept edges before by-source position q
            g.rowptr_tr = newpos[self.rowptr_out.long()].to(torch.int32).contiguous()
            g.col_tr = (self.col_out[keep] - lo).to(torch.int32).contiguous()
            g.tpos = newpos[self.tpos[b:e].long()].to(torch.int32).contiguous()
        g.symmetric, g.max_deg, g.is_shard = False, self.max_deg, True
        g.rows_long = g.rows_hub = None
        if self.rows_long is not None:                       # shard-local degree lists
            for name in ("rows_long", "rows_hub"):
                r = getattr(self, name)
                setattr(g, name, (r[(r >= lo) & (r < hi)] - lo).contiguous())
        g.build_chunks()
        if self.rowptr_out is not None:                      # by-(shifted-)source CSR rows [lo, hi) for out_0 = A @ W^T
            bo, eo = int(self.rowptr_out[lo]), int(self.rowptr_out[hi])
            g.rowptr_out = (self.rowptr_out[lo:hi + 1] - bo).contiguous()
            g.col_out = self.col_out[bo:eo].contiguous()
        return g


def _csr_from_keys(keys, vals, n):
    """Stable sort of `vals` by `keys` (< n) -> (rowptr int32 [n+1], vals_sorted)."""
    perm = torch.argsort(keys, stable=True)
    counts = torch.bincount(keys, minlength=n)
    rowptr = torch.zeros(n + 1, dtype=torch.int64, device=keys.device)
    torch.cumsum(counts, 0, out=rowptr[1:])
    return rowptr.to(torch.int32), vals[perm], perm


def process_edges(edge_index, num_nodes, remove_self_loops):
    """R: models/models.py:117-120 -- loops appended at the END, then (optionally) every src==dst dropped."""
    loop = torch.arange(num_nodes, dtype=edge_index.dtype, device=edge_index.device)
    ei = torch.cat([edge_index, torch.stack([loop, loop])], dim=1)
    if remove_self_loops:
        ei = ei[:, ei[0] != ei[1]]
    return ei


def prepare(edge_index, num_nodes, remove_self_loops, processed=False):
    """Build (or fetch from cache) the PreparedGraph of `edge_index` [2,E] int64.

    remove_self_loops: False for base SNConv (R: :323), the `is_remove_self_loops` flag otherwise.
    The cache is keyed on the tensor object, its storage address and `_version`; writes that bypass the version counter
    (`edge_index.data[...] = ...`) are not seen -- call `clear_cache()` after such an edit.
    processed: `edge_index` already went through `process_edges` (used by tests)."""
    key = (edge_index.data_ptr(), tuple(edge_index.shape), edge_index._version, str(edge_index.device),
           int(num_nodes), bool(remove_self_loops), bool(processed))
    hit = _CACHE.get(key)
    if hit is not None and hit[0]() is edge_index:
        return hit[1]
    if edge_index.numel() and int(edge_index.max()) >= num_nodes:
        raise ValueError("edge_index refers to a node id >= num_nodes")
    if num_nodes >= 2 ** 31 or edge_index.size(1) + num_nodes >= 2 ** 31:
        raise ValueError("graph too large for int32 CSR")
    if edge_index.is_cuda and not processed:
        g = _prepare_cuda(edge_index, int(num_nodes), bool(remove_self_loops))
        if len(_CACHE) >= _CACHE_MAX:
            _CACHE.pop(next(iter(_CACHE)))
        _CACHE[key] = (weakref.ref(edge_index), g)
        return g
    ei = edge_index if processed else process_edges(edge_index, num_nodes, remove_self_loops)
    src, dst = ei[0], ei[1]
    g = PreparedGraph()
    g.n = int(num_nodes)
    g.num_edges = int(src.numel())
    g.rowptr_in, col_in, perm_in = _csr_from_keys(dst, src, g.n)
    g.col_in = col_in.to(torch.int32).contiguous()
    deg = (g.rowptr_in[1:] - g.rowptr_in[:-1])
    g.inv_deg = (1.0 / deg.to(torch.float32).clamp(min=1)).contiguous()
    g.is_shard = False
    g.src_shift = int(src.min()) if src.numel() else 0                # R: models/models.py:125
    g.rowptr_out, col_out, perm_out = _csr_from_keys(src - g.src_shift, dst, g.n)
    g.col_out = col_out.to(torch.int32).contiguous()
    g.col_in_shift = (g.col_in - g.src_shift).contiguous()
    inv_out = torch.empty_like(perm_out)
    inv_out[perm_out] = torch.arange(perm_out.numel(), device=perm_out.device)
    g.tpos = inv_out[perm_in].to(torch.int32).contiguous()
    g.rowptr_tr, g.col_tr = g.rowptr_out, g.col_out
    g.rows_long = ((deg > 32) & (deg <= 1024)).nonzero().flatten().to(torch.int32)
    g.rows_hub = (deg > 1024).nonzero().flatten().to(torch.int32)
    g.max_deg = int(deg.max()) if g.n else 0
    g.symmetric = bool(g.src_shift == 0 and torch.equal(g.rowptr_in, g.rowptr_out) and torch.equal(g.col_in, g.col_out))
    g.build_chunks()
    if len(_CACHE) >= _CACHE_MAX:
        _CACHE.pop(next(iter(_CACHE)))
    _CACHE[key] = (weakref.ref(edge_index), g)
    return g


def _prepare_cuda(edge_index, n, remove_self_loops):
    from . import _C
    lib = _C.lib()
    ei = edge_index.contiguous()
    if ei.dtype != torch.int64:
        ei = ei.long()
    e = ei.size(1)
    dev = ei.device
    cap = e + n
    g = PreparedGraph()
    g.n = n

    def i32(m):
        return torch.empty(m, dtype=torch.int32, device=dev)

    rowptr_in, col_in, rowptr_out, col_out, col_in_shift, tpos, long_rows = i32(n + 1), i32(cap), i32(n + 1), i32(cap), i32(cap), i32(cap), i32(n)
    g.inv_deg = torch.empty(n, dtype=torch.float32, device=dev)
    info = torch.zeros(8, dtype=torch.int32, device=dev)
    wbytes = lib.sng_graph_prepare_workspace_bytes(e, n)
    if wbytes == 0:
        raise ValueError("graph too large for int32 CSR")
    ws = torch.empty(wbytes, dtype=torch.uint8, device=dev)
    _C.call("sng_graph_prepare", ei, _C.ptr(ei), e, n, int(remove_self_loops), _C.ptr(rowptr_in), _C.ptr(col_in),
            _C.ptr(g.inv_deg), _C.ptr(rowptr_out), _C.ptr(col_out), _C.ptr(col_in_shift), _C.ptr(tpos), _C.ptr(long_rows), _C.ptr(info),
            _C.ptr(ws), wbytes)
    kept, shift, sym, n_long, n_hub, max_deg = (int(v) for v in info.tolist()[:6])   # one sync: the arrays are narrowed to the kept edges
    g.num_edges = kept
    g.rowptr_in, g.col_in = rowptr_in, col_in[:kept]
    g.src_shift = shift
    g.rowptr_out, g.col_out, g.col_in_shift, g.tpos = rowptr_out, col_out[:kept], col_in_shift[:kept], tpos[:kept]
    g.rowptr_tr, g.col_tr = g.rowptr_out, g.col_out
    g.rows_long = long_rows[:n_long].clone()
    g.rows_hub = long_rows[n - n_hub:].clone() if n_hub else long_rows[:0].clone()
    g.symmetric, g.max_deg, g.is_shard = sym != 0, max_deg, False
    g.build_chunks()
    return g


def clear_cache():
    _CACHE.clear()
