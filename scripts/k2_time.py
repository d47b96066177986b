"""Times the edge-path kernels alone on the pokec-shaped graph (C = 32): fused / unfused forward (train + inference),
deterministic backward, scatter backward.  python scripts/k2_time.py [shape] [C] [k]"""
import sys, os, json
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from sngnn_b200 import synth, graph as G, functional as SF

shape = sys.argv[1] if len(sys.argv) > 1 else "pokec"
C = int(sys.argv[2]) if len(sys.argv) > 2 else 32
k = int(sys.argv[3]) if len(sys.argv) > 3 else 10
dev = "cuda"
N, Fd, E, _ = synth.SHAPES[shape]
ei = synth.make_graph(N, E, seed=1, device=dev, symmetric=True)
g = G.prepare(ei, N, True)
Ep = g.num_edges
torch.manual_seed(0)
h = torch.randn(N, C, device=dev)
gg = torch.randn(N, C, device=dev)
wt = torch.randn(N, C, device=dev)
bw = torch.randn(C, device=dev); beta = torch.full((1,), 0.5, device=dev)
fuse = (wt, bw, beta, None)


def timed(fn, steps=10, warm=3):
    for _ in range(warm): fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(steps): fn()
    b.record(); torch.cuda.synchronize()
    return a.elapsed_time(b) / steps


res = {"shape": shape, "N": N, "edges": Ep, "C": C, "k": k, "symmetric": g.symmetric, "n_long": int(g.rows_long.numel()),
       "n_hub": int(g.rows_hub.numel()), "max_deg": g.max_deg}
hbm = 6499.0
b_plain = Ep * (4 * C + 4) + N * (8 * C + 8)
res["fwd_infer_ms"] = timed(lambda: SF._edge_fwd(h, g, 0, k, 0.0, False))
res["fwd_train_ms"] = timed(lambda: SF._edge_fwd(h, g, 0, k, 0.0, True, want_q=True))
res["fwd_fused_infer_ms"] = timed(lambda: SF._edge_fwd(h, g, 0, k, 0.0, False, fuse))
res["fwd_fused_train_ms"] = timed(lambda: SF._edge_fwd(h, g, 0, k, 0.0, True, fuse, want_q=True))
res["fwd_infer_frac_hbm"] = b_plain / res["fwd_infer_ms"] / 1e6 / hbm
res["fwd_train_frac_hbm"] = (b_plain + 8 * N * k) / res["fwd_train_ms"] / 1e6 / hbm
res["fwd_fused_infer_frac_hbm"] = (b_plain + Ep * 4 * C) / res["fwd_fused_infer_ms"] / 1e6 / hbm
tab, g.chunk_tab = g.chunk_tab, None
res["fwd_general_kernel_infer_ms"] = timed(lambda: SF._edge_fwd(h, g, 0, k, 0.0, False))
g.chunk_tab = tab
out, ss, sw, sq, sc, inv, diff = SF._edge_fwd(h, g, 0, k, 0.0, True, fuse, want_q=True)
nsel = int(sc.sum())
res["selected_edges"] = nsel


def bwd(fused):
    SF.edge_bwd(h, inv, gg, g, k, ss, sw, sq, sc, beta if fused else None, diff if fused else None)


res["bwd_det_ms"] = timed(lambda: bwd(False))
res["bwd_det_fused_ms"] = timed(lambda: bwd(True))
b_bwd = nsel * (3 * 4 * C + 16) + 5 * N * 4 * C
res["bwd_det_frac_hbm"] = b_bwd / res["bwd_det_ms"] / 1e6 / hbm
res["bwd_scatter_ms"] = timed(lambda: SF.edge_agg_bwd_scatter(h, inv, gg, g.rowptr_in, g.col_in, N, 0, k, ss, sw, sc, g.inv_deg))
res["spmm_ms"] = timed(lambda: SF.spmm(gg, g.rowptr_in, g.col_in_shift, N))
print(json.dumps(res))
