"""top_k > SNG_MAX_TOPK without a GPU: the argument checks of the per-edge entry points (sng_edge_fwd_wide /
sng_edge_bwd_wide), the one choice of form in functional.py, and row-sharded training at top_k > 64 with gloo (the CPU oracle
injected for the kernels), worlds 2 and 3, the last rank of world 3 without rows."""
import ctypes
import os
import socket

import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from conftest import ROOT

_P = ctypes.c_void_p
FAKE = _P(256)                         # never dereferenced: every call below fails its argument checks first


def _fwd(L, **kw):
    a = dict(h=FAKE, n_total=10, n=10, row_offset=0, c=4, ldh=4, rowptr=FAKE, col=FAKE, num_edges=40, chunk_tab=None, n_chunks=-1,
             lrows=None, lrow_ptr=None, n_lrows=0, rows_hub=None, n_hub=0, ws=None, wbytes=0, top_k=100, max_deg=30, thr=0.0,
             out=FAKE, ldo=4, flag=FAKE, train=1, inv_norm=FAKE, inv_ready=1, wt=None, ldw=4, b_w=None, beta=None, bias=None,
             diff=None, denominator=0, inv_denom=None)
    a.update(kw)
    return L.sng_edge_fwd_wide(*a.values(), None)


def _bwd(L, **kw):
    a = dict(h=FAKE, inv_norm=FAKE, g=FAKE, n_total=10, n=10, row_offset=0, c=4, ld=4, ldg=4, rowptr=FAKE, col=FAKE, tpos=FAKE,
             rowptr_out=FAKE, col_out=FAKE, shift=0, num_edges=40, flag=FAKE, inv_denom=None, beta=None, diff=None, lddiff=4,
             dbeta=None, coef=FAKE, dnt=FAKE, part=None, dh=FAKE, dwt=None, lddw=4, tab=None, n_chunks=-1, lrows=None,
             lrow_ptr=None, n_lrows=0, cpart=None)
    a.update(kw)
    return L.sng_edge_bwd_wide(*a.values(), None)


def test_wide_entry_points_validate_their_arguments():
    from sngnn_b200 import _C
    L = _C.lib()
    for kw, msg in ((dict(top_k=64), "top_k=64 must be > 64"), (dict(top_k=0), "top_k=0"), (dict(thr=-1.5), "thr"),
                    (dict(denominator=2), "denominator"), (dict(inv_denom=FAKE), "inv_denom"),
                    (dict(flag=None), "sel_flag"), (dict(flag=None, train=0, max_deg=200), "sel_flag"),
                    (dict(row_offset=5), "row_offset"), (dict(n=11), "row_offset"), (dict(max_deg=-1), "max_deg"),
                    (dict(c=516, ldh=516, ldo=516), "512"), (dict(inv_norm=None), "inv_norm"),
                    (dict(diff=FAKE), "diff"), (dict(n_hub=2), "hub")):
        assert _fwd(L, **kw) != 0, kw
        assert "sng_edge_fwd_wide" in _C.last_error() and msg in _C.last_error(), (kw, _C.last_error())
    # a cut with a row longer than the shared-memory stage needs the workspace for its keys
    assert L.sng_edge_fwd_wide_workspace_bytes(-1, 4, 10 ** 6, 8192) == 0
    assert L.sng_edge_fwd_wide_workspace_bytes(-1, 4, 10 ** 6, 8193) >= 4 * 10 ** 6
    assert L.sng_edge_fwd_wide_workspace_bytes(100, 32, 10, 10) == L.sng_edge_fwd_workspace_bytes(100, 32, 0)
    assert _fwd(L, max_deg=9000, num_edges=9000) == -4 and "workspace" in _C.last_error()
    for kw, msg in ((dict(flag=None), "sel_flag"), (dict(tpos=None), "tpos"), (dict(row_offset=3), "row_offset"),
                    (dict(dwt=FAKE, beta=FAKE, n=5), "dwt"), (dict(dbeta=FAKE), "dbeta"), (dict(coef=None), "null")):
        assert _bwd(L, **kw) != 0, kw
        assert "sng_edge_bwd_wide" in _C.last_error() and msg in _C.last_error(), (kw, _C.last_error())


def test_the_form_is_chosen_from_top_k_alone():
    from sngnn_b200 import _C, functional as SF
    assert _C.MAX_TOPK == 64
    assert [SF.per_edge_form(k) for k in (None, -1, 0, 1, 64, 65, 1000, 1 << 40)] == [False] * 5 + [True] * 3


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _graph(n, seed):
    """A random multigraph whose rows hold 40..150 in-edges (duplicates kept): top_k = 70 cuts most rows, 1000 none."""
    gen = torch.Generator().manual_seed(seed)
    dst = torch.repeat_interleave(torch.arange(n), torch.randint(40, 150, (n,), generator=gen))
    src = torch.randint(0, n, (dst.numel(),), generator=gen)
    perm = torch.randperm(dst.numel(), generator=gen)
    return torch.stack([src[perm], dst[perm]])


def _worker(rank, ws, port, kind, n, k, ret):
    import sys
    sys.path.insert(0, ROOT)
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=ws)
    import torch.nn.functional as F
    from sngnn_b200 import dist as D, synth
    import sngnn_b200.models as M
    from oracle import sn_ref
    fd, hid, ncls, thr = 10, 8, 3, -0.2
    x = synth.make_features(n, fd, "clustered", seed=1).double()
    ei = _graph(n, 5)
    y = synth.make_labels(n, ncls, seed=3)
    torch.manual_seed(7)
    if kind == "SNGNN_Plus":
        model = M.SNGNN_Plus(fd, hid, ncls, n, 2, k, thr, 1, 0.0)
    else:
        model = M.SNGNN_Plus_Plus(fd, hid, ncls, n, 2, k, thr, 0.5, 1, 0.0)
    model = model.double().train()
    lo, hi = D.shard_bounds(n, ws, rank)
    pe = sn_ref.process_edges(ei, n, True)

    def agg(h_all, shard, row_offset, top_k, th):
        return sn_ref.sn_aggregate(h_all, pe, top_k, th)[row_offset:row_offset + shard.n]

    def fuse(out1, w_w, w_b, beta, bias, shard, nn_, lo_):
        out0 = sn_ref.structural_term(pe, w_w, w_b, nn_)[lo_:lo_ + out1.size(0)]
        out0 = F.pad(out0, (0, out1.size(1) - out0.size(1)))
        out = beta * out0 + (1 - beta) * out1
        return out if bias is None else out + F.pad(bias, (0, out1.size(1) - bias.numel()))

    logp = D.sharded_forward(model, x[lo:hi].clone(), ei, n, agg=agg, fuse=fuse)
    (F.nll_loss(logp, y[lo:hi], reduction="sum") / n).backward()
    D.allreduce_grads(model.parameters())
    sd = {kk: v.detach().clone().requires_grad_(v.is_floating_point()) for kk, v in model.state_dict().items()}
    ref = sn_ref.stack_forward(kind, sn_ref.params_from_state_dict(sd, 2), x, ei, top_k=k, thr=thr, remove_self_loops=True)
    F.nll_loss(ref, y).backward()
    assert logp.size(0) == hi - lo
    assert torch.allclose(logp.detach(), ref.detach()[lo:hi], rtol=1e-9, atol=1e-11)
    for name, p in model.named_parameters():
        g_ref = sd[name].grad
        assert p.grad is not None and torch.allclose(p.grad, g_ref, rtol=1e-8, atol=1e-11), (kind, name, (p.grad - g_ref).abs().max())
    ret[rank] = True
    dist.barrier()
    dist.destroy_process_group()


def test_sharded_training_above_64_world2_and_world3():
    """sharded_forward at top_k = 70 (rows cut) and 1000 (none), gloo: rows and parameter gradients equal the unsharded oracle.
    World 3 over 4 nodes leaves the last rank without rows."""
    ctx = mp.get_context("spawn")
    for kind, ws, n, k in (("SNGNN_Plus_Plus", 2, 61, 70), ("SNGNN_Plus", 2, 40, 1000), ("SNGNN_Plus_Plus", 3, 4, 70)):
        ret = ctx.Manager().dict()
        port = _free_port()
        procs = [ctx.Process(target=_worker, args=(r, ws, port, kind, n, k, ret)) for r in range(ws)]
        for p in procs:
            p.start()
        for p in procs:
            p.join(180)
            if p.exitcode is None:
                p.terminate()
                p.join()
            assert p.exitcode == 0, f"{kind} world {ws}: worker exited with {p.exitcode}"
        assert dict(ret) == {r: True for r in range(ws)}
