"""The transpose index of a row shard (PreparedGraph.row_slice): the by-source CSR over all source rows holding only the
shard's in-edges, and the shard's `tpos` into it, which let a shard's backward run the deterministic gather passes of
sng_edge_bwd.  Host logic on CPU graphs: ragged shards (a 1-row and an empty one included), sources shifted by
min(src) > 0, self loops kept and removed, source rows with more than 32 and more than 1024 out-edges."""
import pytest
import torch

N = 1500


def _graph(shift, remove_self_loops, seed=5):
    from sngnn_b200 import graph as G, synth
    ei = synth.make_graph(N, 8 * N, seed=seed)
    gen = torch.Generator().manual_seed(seed)
    extra = [torch.tensor([[shift], [0]])]
    for s, d in ((shift + 7, 1400), (shift + 40, 90)):                  # a hub source row and a long one
        t = torch.randperm(N, generator=gen)[:d]
        extra.append(torch.stack([torch.full_like(t, s), t]))
    ei = torch.cat([ei] + extra, 1)
    ei = ei[:, ei[0] >= shift]
    key = torch.unique(ei[0] * N + ei[1])
    g = G.prepare(torch.stack([key // N, key % N]), N, remove_self_loops)
    assert g.src_shift == shift
    return g


CASES = [(3, True), (0, True), (0, False)]                               # shift > 0 needs the self loops removed


@pytest.mark.parametrize("shift,rsl", CASES)
def test_whole_range_shard_has_the_whole_transpose(shift, rsl):
    g = _graph(shift, rsl)
    assert g.rowptr_tr is g.rowptr_out and g.col_tr is g.col_out
    s = g.row_slice(0, N)
    for name in ("tpos", "chunk_tab_out", "lrows_out", "lrow_ptr_out"):
        assert torch.equal(getattr(s, name), getattr(g, name)), name
    assert torch.equal(s.rowptr_tr, g.rowptr_out) and torch.equal(s.col_tr, g.col_out)


@pytest.mark.parametrize("shift,rsl", CASES)
def test_shard_transpose_is_the_restricted_whole_transpose(shift, rsl):
    g = _graph(shift, rsl)
    bounds = [0, 1, 1, 190, 191, N]                                      # 1-row, empty and ragged shards
    covered, hub_seen = 0, False
    for lo, hi in zip(bounds[:-1], bounds[1:]):
        s = g.row_slice(lo, hi)
        e = s.num_edges
        covered += e
        rp, col, tpos = s.rowptr_tr.long(), s.col_tr.long(), s.tpos.long()
        assert rp.numel() == N + 1 and int(rp[0]) == 0 and int(rp[-1]) == e == col.numel() == tpos.numel()
        assert torch.equal(torch.sort(tpos).values, torch.arange(e))     # a bijection onto the shard's edges
        # by-target edge p: local target row t_p, source col_in[p]
        t_p = torch.repeat_interleave(torch.arange(s.n), (s.rowptr_in[1:] - s.rowptr_in[:-1]).long())
        assert torch.equal(col[tpos], t_p)
        row_of = torch.searchsorted(rp, tpos, right=True) - 1            # by-source row holding position tpos[p]
        assert torch.equal(row_of, s.col_in.long() - shift)
        # per source row, the shard's edges keep the whole graph's order (stable compaction)
        b = int(g.rowptr_in[lo])
        assert torch.equal(torch.argsort(tpos), torch.argsort(g.tpos[b:b + e].long()))
        # by-source chunk tables: exactly the rows with more than 32 shard out-edges, cut into <= 32-edge chunks
        deg = rp[1:] - rp[:-1]
        long_rows = (deg > 32).nonzero().flatten()
        assert torch.equal(s.lrows_out.long(), long_rows + shift)
        tab, ptr = s.chunk_tab_out.long(), s.lrow_ptr_out.long()
        assert ptr.numel() == long_rows.numel() + 1 and int(ptr[-1]) == tab.size(0)
        for li, r in enumerate(long_rows.tolist()):
            ch = tab[int(ptr[li]):int(ptr[li + 1])]
            assert bool((ch[:, 1] <= 32).all() and (ch[:, 1] > 0).all())
            assert int(ch[0, 0]) == int(rp[r]) and int(ch[:, 1].sum()) == int(deg[r])
            assert torch.equal(ch[1:, 0], ch[:-1, 0] + ch[:-1, 1])
        hub_seen |= bool((deg > 1024).any())
    assert covered == g.num_edges and hub_seen                           # some shard keeps > 1024 of the hub's out-edges


def _edge_bwd_rc(n_total, n, row_offset, dwt):
    """sng_edge_bwd's argument checks (no launch: they fail before any device call) with placeholder pointers."""
    import ctypes
    from sngnn_b200 import _C
    p = ctypes.c_void_p(4096)
    c = 32
    return _C.lib().sng_edge_bwd(p, p, p, n_total, n, row_offset, c, c, c, p, p, p, p, p, 0, 100, 10, p, p, p, p,
                                 p, None, c, None, p, p, p, p, p if dwt else None, c, None, -1, None, None, 0, None, None)


def test_edge_bwd_rejects_bad_row_ranges_and_partial_dwt():
    from sngnn_b200 import _C
    assert _edge_bwd_rc(100, 40, 10, True) != 0 and "dwt" in _C.last_error()           # dL/dW^T of a partial shard
    assert _edge_bwd_rc(100, 40, 61, False) != 0 and "row_offset" in _C.last_error()   # row_offset + n > n_total
    assert _edge_bwd_rc(100, 40, -1, False) != 0 and "row_offset" in _C.last_error()
    assert _edge_bwd_rc(2 ** 31, 40, 0, False) != 0 and "out of range" in _C.last_error()
    assert _edge_bwd_rc(100, -1, 0, False) != 0
