"""The C-ABI library loads without a GPU and exports exactly what include/sng.h declares; host-side logic
(graph preparation, argument validation) runs on CPU.  No compute kernels are launched here."""
import ctypes
import os
import re

import pytest
import torch

from conftest import ROOT


def _header_functions():
    src = open(os.path.join(ROOT, "include", "sng.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(sng_[a-z0-9_]+)\s*\(", src)))


def test_library_exports_every_declared_symbol():
    from sngnn_b200 import _C
    lib = _C.lib()
    names = _header_functions()
    assert len(names) >= 12
    for n in names:
        assert hasattr(lib, n), f"{n} declared in include/sng.h but not exported by libsng.so"
    assert sorted(_C.SIGNATURES) == names, "sngnn_b200/_C.py SIGNATURES out of sync with include/sng.h"
    assert lib.sng_version() >= 100


@pytest.mark.skipif(torch.cuda.is_available(), reason="checks the no-GPU error path")
def test_no_gpu_is_a_loud_error_not_a_fallback():
    from sngnn_b200 import _C, functional as SF, graph as G
    a, b, c = ctypes.c_int(), ctypes.c_int(), ctypes.c_int()
    rc = _C.lib().sng_device_info(ctypes.byref(a), ctypes.byref(b), ctypes.byref(c))
    assert rc == -3 and "device" in _C.last_error().lower()
    g = G.prepare(torch.tensor([[0, 1], [1, 0]]), 2, True)
    with pytest.raises(RuntimeError, match="no CPU path"):
        SF.edge_topk_agg(torch.randn(2, 4), g, 1, 0.0)


def test_argument_validation_without_device():
    from sngnn_b200 import _C
    L = _C.lib()
    assert L.sng_rownorm_f32(None, 4, 4, 4, None, 4, None, 4, None, None) == -1
    assert "sng_rownorm_f32" in _C.last_error()
    assert L.sng_simknn_workspace_bytes(0, 10, 4, 1) == 0
    assert L.sng_simknn_workspace_bytes(1000, 1000, 65, 10) > 1000 * 32 * 8


def test_graph_prepare_matches_reference_edge_processing():
    from sngnn_b200 import graph as G, synth
    from oracle import sn_ref
    n = 50
    ei = synth.make_graph(n, 300, seed=9, hub_offset=2.0)
    ei = torch.cat([ei, torch.tensor([[3, 3], [3, 7]])], dim=1)        # an original self loop and a duplicate-able edge
    for rsl in (True, False):
        g = G.prepare(ei, n, rsl)
        pe = sn_ref.process_edges(ei, n, rsl)
        assert torch.equal(G.process_edges(ei, n, rsl), pe)
        # CSR by target keeps original positions
        for i in range(n):
            want = pe[0][pe[1] == i]
            got = g.col_in[g.rowptr_in[i]:g.rowptr_in[i + 1]].long()
            assert torch.equal(got, want)
        deg = torch.bincount(pe[1], minlength=n).clamp(min=1).float()
        assert torch.allclose(g.inv_deg, 1 / deg)
        m = int(pe[0].min())
        assert g.src_shift == m
        for i in range(n):
            want = sorted(pe[1][pe[0] - m == i].tolist())
            got = sorted(g.col_out[g.rowptr_out[i]:g.rowptr_out[i + 1]].tolist())
            assert got == want
        assert G.prepare(ei, n, rsl) is g                                 # cache hit
    sl = g.row_slice(10, 30)
    assert sl.n == 20 and int(sl.rowptr_in[0]) == 0 and sl.col_in.numel() == int(g.rowptr_in[30] - g.rowptr_in[10])


def test_module_surface_matches_reference_signatures():
    import inspect
    import sngnn_b200.models as M
    sig = lambda f: [p for p in inspect.signature(f).parameters if p != "self"]
    assert sig(M.SNGNN.__init__) == ["in_channels", "hidden_channels", "out_channels", "num_layers", "bn"]
    assert sig(M.SNGNN_Plus.__init__)[:10] == ["in_channels", "hidden_channels", "out_channels", "num_nodes", "num_layers", "top_k",
                                               "thr", "is_remove_self_loops", "droput_rate", "bn"]
    assert sig(M.SNGNN_Plus_Plus.__init__)[:11] == ["in_channels", "hidden_channels", "out_channels", "num_nodes", "num_layers",
                                                    "top_k", "thr", "init_beta", "is_remove_self_loops", "droput_rate", "bn"]
    assert sig(M.SNConv_plus_plus.__init__)[:9] == ["in_channels", "out_channels", "num_nodes", "top_k", "thr", "init_beta",
                                                    "is_remove_self_loops", "bias", "aggr"]
    m = M.SNGNN_Plus_Plus(8, 4, 3, 20, 2, init_beta=0.25)
    assert float(m.lins[0].beta) == 0.25 and m.lins[0].w.weight.shape == (4, 20)
    assert sorted(k for k in m.state_dict()) == sorted(
        [f"lins.{l}.{n}" for l in (0, 1) for n in ("beta", "lin.weight", "lin.bias", "w.weight", "w.bias")])


def test_simknn_plan_is_host_logic():
    """sng_simknn_plan needs no GPU: the launch plan of the build for the named shapes (DESIGN.md §5)."""
    from sngnn_b200 import simknn
    p = simknn.build_plan(1632803, 1632803, 65, 10)                      # pokec: split mode, seeded 1/32 with the 5th of 16 group maxima
    assert (p["ew"], p["kblocks"], p["nsplit"], p["seed_stride"], p["seed_q"], p["cand"]) == (4, 2, 1, 32, 5, 32), p
    assert p["stages"] % p["kblocks"] == 0
    p = simknn.build_plan(204101, 1632803, 65, 10)                       # one rank of an 8-GPU build: same plan
    assert (p["ew"], p["nsplit"], p["seed_stride"]) == (4, 1, 32), p
    p = simknn.build_plan(169343, 169343, 128, 10)                       # arxiv-year shape: 662 tiles -> 1/16 sample
    assert (p["ew"], p["nsplit"], p["seed_stride"], p["seed_q"]) == (4, 1, 16, 6), p
    p = simknn.build_plan(21168, 169343, 128, 10)                        # one rank of 8 on it: column splits, still seeded
    assert p["nsplit"] == 3 and p["seed_stride"] == 16, p
    p = simknn.build_plan(2923922, 2923922, 269, 10)                     # snap-patents: K = 272 -> two 256-column stages
    assert (p["ew"], p["kblocks"], p["seed_stride"]) == (2, 5, 32), p
    p = simknn.build_plan(2277, 2277, 2325, 10)                          # Chameleon's raw features: streamed query block, one epilogue warp per quarter
    assert p["ew"] == 1 and p["kblocks"] == 37, p
    p = simknn.build_plan(100000, 100000, 512, 50)                       # sweep corner: A alone is 128 KB -> thinner margin, 2 stages
    assert p["ew"] == 1 and 64 <= p["cand"] <= 72 and p["stages"] >= 2 and p["seed_q"] <= 12, p      # margin >= 14 before a third ring stage
    p = simknn.build_plan(2277, 2277, 2325 // 8, 10)                     # tiny database: column-split, unseeded
    assert p["nsplit"] > 1 and p["seed_stride"] == 0, p
    import pytest
    with pytest.raises(RuntimeError):
        simknn.build_plan(1000, 1000, 65, 1000)                          # top_k out of range -> loud error


def test_structural_weight_lives_in_transposed_storage():
    """w.weight keeps the reference's name / shape [C, N] but is stored as W^T [N, C] row-major, so the kernels read the
    parameter itself: no cached transpose that an in-place edit (`w.data.mul_(2)`, which bypasses the version counter)
    could leave stale.  The layout must survive load_state_dict, deepcopy and the optimizer state."""
    import copy
    import sngnn_b200.models as M
    from sngnn_b200 import functional as SF
    m = M.SNGNN_Plus_Plus(8, 4, 3, 20, 2, init_beta=0.25)
    w = m.lins[0].w.weight
    assert w.shape == (4, 20) and w.stride() == (1, 4) and w.t().is_contiguous()
    wt = SF._padded_wt(w, 4)
    assert wt.data_ptr() == w.data_ptr()                                  # a view of the parameter, not a copy
    w.data.mul_(2)                                                        # no version bump: a cached copy would now be stale
    assert torch.equal(SF._padded_wt(w, 4), w.detach().t())
    m.load_state_dict({k: v.clone().contiguous() for k, v in m.state_dict().items()})
    assert m.lins[0].w.weight.stride() == (1, 4) and copy.deepcopy(m).lins[0].w.weight.stride() == (1, 4)
    opt = torch.optim.Adam(m.parameters())
    for p in m.parameters():
        p.grad = torch.ones_like(p)
    opt.step()
    assert opt.state[m.lins[0].w.weight]["exp_avg"].stride() == (1, 4)
    w3 = m.lins[1].w.weight                                               # C = 3: padded copy, zero tail
    wt3 = SF._padded_wt(w3, 4)
    assert wt3.shape == (20, 4) and torch.equal(wt3[:, :3], w3.detach().t()) and wt3[:, 3].abs().sum() == 0


def test_top_k_zero_follows_the_reference():
    """R: models/models.py:250 -- `for i in range(self.top_k)` runs no round for top_k <= 0: every weight stays 0."""
    import sngnn_b200.models as M
    conv = M.SNConv_plus(6, 4, 10, top_k=0, thr=0.0)
    h = torch.randn(10, 4, requires_grad=True)
    out = conv._aggregate(h, None)
    assert out.shape == (10, 4) and out.abs().sum() == 0
    out.sum().backward()
    assert h.grad is not None and h.grad.abs().sum() == 0


def test_knn_to_csr_host_logic():
    from sngnn_b200 import simknn
    idx = torch.tensor([[4, 2, -1], [-1, -1, -1], [0, 1, 3]], dtype=torch.int32)
    cnt = torch.tensor([2, 0, 3], dtype=torch.int32)
    sim = torch.arange(9.0).reshape(3, 3)
    rowptr, col, val = simknn.knn_to_csr(idx, cnt, sim)
    assert rowptr.tolist() == [0, 2, 2, 5] and col.tolist() == [4, 2, 0, 1, 3] and val.tolist() == [0.0, 1.0, 6.0, 7.0, 8.0]
    assert len(simknn.knn_to_csr(idx, cnt)) == 2
