"""The CPU oracle (oracle/sn_ref.py, oracle/toolbox_ref.py) against the golden vectors produced by the
reference's own unmodified code (oracle/make_golden.py).  CPU only."""
import pytest
import torch
import torch.nn.functional as F

from conftest import load_golden, golden_inputs, golden_state_dict, golden_grad
from oracle import sn_ref, toolbox_ref


def _run_oracle(g, run, x, ei, y):
    cfg = run["cfg"]
    sd = {k: v.clone().requires_grad_(v.is_floating_point() and "running" not in k) for k, v in golden_state_dict(g, run).items()}
    params = sn_ref.params_from_state_dict(sd, cfg["layers"])
    bns = None
    if cfg.get("bn"):
        bns = []
        for l in range(cfg["layers"] - 1):
            w, b = sd[f"bns.{l}.weight"], sd[f"bns.{l}.bias"]
            bns.append(lambda t, w=w, b=b: F.batch_norm(t, None, None, w, b, True, 0.1, 1e-5))
    out = sn_ref.stack_forward(run["kind"], params, x, ei, top_k=cfg.get("top_k"), thr=cfg.get("thr"),
                               remove_self_loops=bool(cfg.get("rsl", 0) == 1), bns=bns)
    mask = torch.arange(x.size(0)) % 2 == 0
    loss = F.nll_loss(out[mask], y[mask])
    loss.backward()
    return out.detach(), loss.detach(), {k: v.grad for k, v in sd.items() if v.requires_grad}


@pytest.mark.parametrize("fname", ["models_tiny.pt", "models_small.pt", "models_chameleon.pt"])
def test_models_match_reference(fname):
    g = load_golden(fname)
    x, ei, y = golden_inputs(g)
    for run in g["runs"]:
        out, loss, grads = _run_oracle(g, run, x, ei, y)
        tag = f"{fname} {run['kind']} {run['cfg']}"
        torch.testing.assert_close(out, run["logp"], rtol=1e-5, atol=1e-6, msg=lambda m: f"{tag}: {m}")
        torch.testing.assert_close(loss, run["loss"], rtol=1e-5, atol=1e-6)
        for k, gref in run["grads"].items():
            got, ref, _ = golden_grad(grads[k], gref)
            torch.testing.assert_close(got, ref, rtol=1e-4, atol=1e-6, msg=lambda m: f"{tag} grad {k}: {m}")


def test_edge_select_matches_iterated_scatter_max():
    """edge_rank == the k-round argmax/knock-out loop (naive per-target restatement of R models.py:145-154)."""
    torch.manual_seed(0)
    E, N = 500, 40
    dst = torch.randint(0, N - 3, (E,))
    s = torch.randn(E).clamp(-1, 1)
    s[::7] = s[3]                      # ties
    for k, thr in ((1, 0.0), (3, -0.5), (50, 0.2)):
        sel = torch.zeros(E, dtype=torch.bool)
        for i in range(N):
            pos = (dst == i).nonzero().flatten().tolist()
            pos.sort(key=lambda p: (-s[p].item(), p))
            for p in pos[:k]:
                if s[p] < thr:
                    break
                sel[p] = True
        assert torch.equal(sel, sn_ref.edge_select(s, dst, k, thr))


def test_toolbox_matches_reference():
    g = load_golden("toolbox.pt")
    x, ei, y = g["x"], g["edge_index"].long(), g["y"]
    T = toolbox_ref
    close = lambda a, b, **kw: torch.testing.assert_close(torch.as_tensor(a).float(), torch.as_tensor(b).float(),
                                                          rtol=kw.get("rtol", 1e-4), atol=kw.get("atol", 1e-5))
    close(T.node_similarity_dense_large_parted(g["x1200"])[1], g["node_large_parted"], rtol=1e-3)
    close(T.class_similarity_dense_large(g["x1200"], g["y1200"]), g["class_large_1200"])
    for name, fn, args in (("linked_large", T.linked_node_similarity_dense_large, (x, ei)),
                           ("nbr_large", T.neighborhood_similarity_dense_large, (x, ei)),
                           ("node_small", T.node_similarity_dense_small, (x,)),
                           ("linked_small", T.linked_node_similarity_dense_small, (x, ei)),
                           ("nbr_small", T.neighborhood_similarity_dense_small, (x, ei)),
                           ("class_small", T.class_similarity_dense_small, (x, y))):
        got, ref = fn(*args), g[name]
        assert got[0].shape == ref[0].shape, name
        close(got[0], ref[0])
        close(got[1], ref[1])
    close(T.class_similarity_dense_large(x, y), g["class_large"])
    from scipy import sparse as sp
    import numpy as np
    adj = sp.csc_matrix((np.ones(ei.size(1)), (ei[0].numpy(), ei[1].numpy())), shape=(x.size(0), x.size(0)))
    for name, fn, args in (("sp_node", T.node_similarity_sparse, (adj,)),
                           ("sp_linked", T.linked_node_similarity_sparse, (adj, ei)),
                           ("sp_nbr", T.neighborhood_similarity_sparse, (adj, ei))):
        got, ref = fn(*args), g[name]
        assert got[0].shape == ref[0].shape, name
        close(got[0], ref[0])
        close(got[1], ref[1])
    close(T.class_similarity_sparse(adj, y), g["sp_class"])
    close(T.edge_similarity_weight(g["esw_x"], ei), g["esw"])


def test_allpairs_oracle_is_reference_rule_on_complete_graph():
    """simknn_allpairs == edge_select on the complete graph (SURVEY.md §0 definition of all-pairs mode)."""
    torch.manual_seed(1)
    N, d = 70, 8
    x = torch.randn(N, d)
    x[5] = x[9]; x[11] = 0
    n = sn_ref.rownorm(x)
    for remove_self in (True, False):
        src = torch.arange(N).repeat(N)                 # sorted by target, then source ascending
        dst = torch.arange(N).repeat_interleave(N)
        if remove_self:
            keep = src != dst
            src, dst = src[keep], dst[keep]
        s = (n[dst] @ n.t())[torch.arange(dst.numel()), src]      # same mm values the all-pairs oracle sees
        for k, thr in ((3, 0.0), (5, 0.3), (80, -1.0)):
            sel = sn_ref.edge_select(s, dst, k, thr)
            idx, sim, cnt = sn_ref.simknn_allpairs(x, k, thr, remove_self, block=32)
            for i in range(N):
                got = set(idx[i, :cnt[i]].tolist())
                want = set(src[sel & (dst == i)].tolist())
                assert got == want, (i, k, thr, remove_self)
