"""The transpose of fixed-width neighbour lists (functional.list_transpose): the by-source index through which the all-pairs
backward (sng_list_bwd) runs the deterministic gather passes.  Host logic on CPU lists against a brute-force per-source
listing: -1 padding, empty rows, rows with fewer than k entries, a column that more than 1,024 rows select, lists of a
row shard (global columns, local rows).  And the one combination sharded_forward still rejects."""
import pytest
import torch


def _lists(nq, k, n_total, seed, hub=None):
    gen = torch.Generator().manual_seed(seed)
    idx = torch.randint(0, n_total, (nq, k), generator=gen, dtype=torch.int32)
    cnt = torch.randint(0, k + 1, (nq,), generator=gen, dtype=torch.int32)
    cnt[::7] = 0
    cnt[1::5] = k
    if hub is not None:
        idx[:, 0] = hub
    idx[torch.arange(k)[None, :] >= cnt[:, None]] = -1
    return idx, cnt


def _brute_force(idx, cnt, n_total):
    """Per source column j: the (row, rank) of every list entry holding j, in (row, rank) order."""
    per = [[] for _ in range(n_total)]
    for i in range(idx.size(0)):
        for t in range(int(cnt[i])):
            per[int(idx[i, t])].append((i, t))
    return per


@pytest.mark.parametrize("nq,k,n_total,hub", [(300, 10, 500, None), (2000, 4, 2100, 17), (50, 64, 3000, None),
                                                (1, 1, 10, None), (0, 10, 40, None)])
def test_list_transpose_matches_brute_force(nq, k, n_total, hub):
    from sngnn_b200 import functional as SF
    idx, cnt = _lists(nq, k, n_total, seed=nq + k, hub=hub)
    t = SF.list_transpose(idx, cnt, n_total)
    per = _brute_force(idx, cnt, n_total)
    assert t.rowptr_tr.dtype == torch.int32 and t.rowptr_tr.numel() == n_total + 1
    assert t.rowptr_tr.tolist() == [0] + list(torch.tensor([len(p) for p in per], dtype=torch.long).cumsum(0).tolist())
    nnz = int(t.rowptr_tr[-1])
    assert nnz == int(cnt.clamp(0, k).sum()) and t.col_tr.numel() >= nnz
    expect_sel_q = torch.full((nq, k), -1, dtype=torch.int32)
    for j in range(n_total):
        b = int(t.rowptr_tr[j])
        assert t.col_tr[b:b + len(per[j])].tolist() == [i for i, _ in per[j]], j
        for q, (i, s) in enumerate(per[j]):
            expect_sel_q[i, s] = b + q
    assert torch.equal(t.sel_q, expect_sel_q)
    if hub is not None:
        assert int(t.rowptr_tr[hub + 1] - t.rowptr_tr[hub]) > 1024


def test_list_transpose_of_a_shard_keeps_global_columns_and_local_rows():
    """Lists of rows [lo, hi) of a larger node set: sources are global ids, col_tr holds rows relative to lo, and the
    shard's transpose is the whole transpose restricted to its rows."""
    from sngnn_b200 import functional as SF
    n_total, k, lo, hi = 800, 6, 300, 520
    idx, cnt = _lists(n_total, k, n_total, seed=3)
    whole = SF.list_transpose(idx, cnt, n_total)
    part = SF.list_transpose(idx[lo:hi], cnt[lo:hi], n_total)
    for j in range(n_total):
        rows = whole.col_tr[int(whole.rowptr_tr[j]):int(whole.rowptr_tr[j + 1])]
        mine = rows[(rows >= lo) & (rows < hi)] - lo
        assert torch.equal(part.col_tr[int(part.rowptr_tr[j]):int(part.rowptr_tr[j + 1])], mine.to(torch.int32)), j
    sel = part.sel_q
    assert torch.equal(sel >= 0, torch.arange(k)[None, :] < cnt[lo:hi, None])
    assert torch.equal(part.col_tr[sel[sel >= 0].long()], torch.arange(hi - lo).repeat_interleave(cnt[lo:hi].long()).to(torch.int32))


def test_chunk_tables_of_a_list_transpose():
    """The staged source pass's tables over rowptr_tr: every source row with more than 32 entries cut into <= 32-entry
    chunks, rows ascending."""
    from sngnn_b200 import functional as SF
    n_total, k = 1500, 5
    idx, cnt = _lists(1400, k, n_total, seed=9, hub=11)
    cnt[:100] = cnt[:100].clamp(min=2)
    idx[:100, 0], idx[:100, 1] = 11, 40                                   # 40: a long row (100 entries)
    t = SF.list_transpose(idx, cnt, n_total, chunk_tables=True)
    deg = (t.rowptr_tr[1:] - t.rowptr_tr[:-1]).long()
    long_rows = (deg > 32).nonzero().flatten()
    assert 11 in long_rows.tolist() and 40 in long_rows.tolist()
    assert torch.equal(t.lrows.long(), long_rows)
    chunks = ((deg[long_rows] + 31) // 32).tolist()
    assert t.chunk_tab.size(0) == sum(chunks) and t.lrow_ptr.tolist() == [0] + torch.tensor(chunks).cumsum(0).tolist()
    for li, j in enumerate(long_rows.tolist()):
        rows = t.chunk_tab[int(t.lrow_ptr[li]):int(t.lrow_ptr[li + 1])]
        assert (rows[:, 2] == j).all() and int(rows[:, 1].sum()) == int(deg[j])
        assert rows[0, 0] == t.rowptr_tr[j] and (rows[1:, 0] - rows[:-1, 0] == 32).all()


def test_sharded_forward_rejects_edges_with_selected_denominator():
    import sngnn_b200.models as M
    from sngnn_b200 import dist as D
    n = 50
    model = M.SNGNN_Plus(8, 16, 3, n, 2, 4, 0.0, 1, 0.0, denominator="selected")
    ei = torch.stack([torch.arange(n), torch.arange(n).roll(1)])
    with pytest.raises(NotImplementedError, match="candidates='edges' with denominator='selected'"):
        D.sharded_forward(model, torch.randn(n, 8), ei, n)
