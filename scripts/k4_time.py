"""K3 / K4 / full SNGNN++ forward-backward timing on the pokec-shaped graph."""
import sys, os, json
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from sngnn_b200 import synth, graph as G, functional as SF
C = int(sys.argv[1]) if len(sys.argv) > 1 else 32
N, Fd, E, _ = synth.SHAPES["pokec"]
dev = "cuda"
ei = synth.make_graph(N, E, seed=1, device=dev, symmetric=True)
g = G.prepare(ei, N, True)
torch.manual_seed(0)
x = torch.randn(N, C, device=dev)
def timed(f, reps=10):
    for _ in range(3): f()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps): f()
    b.record(); torch.cuda.synchronize()
    return a.elapsed_time(b) / reps
ms_spmm = timed(lambda: SF.spmm(x, g.rowptr_in, g.col_in_shift, N))
w = torch.randn(C, N, device=dev); bw = torch.zeros(C, device=dev); beta = torch.full((1,), 0.5, device=dev)
ms_pp = timed(lambda: SF.PPFuse.apply(x, w, bw, beta, None, g))
print(json.dumps(dict(C=C, spmm_ms=round(ms_spmm, 3), ppfuse_ms=round(ms_pp, 3))))
