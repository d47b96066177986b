"""A/B timing of the edge kernels at the pokec shape: python scripts/edge_ab.py [lib path] [C].  Run it once per library,
alternating, and compare the JSON lines."""
import sys, os, json
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from sngnn_b200 import _C
if len(sys.argv) > 1 and sys.argv[1] != "-":
    _C._LIB_PATH = os.path.abspath(sys.argv[1])
C = int(sys.argv[2]) if len(sys.argv) > 2 else 32
from sngnn_b200 import synth, graph as G, functional as SF
dev = "cuda"
N, Fd, E, _ = synth.SHAPES["pokec"]
ei = synth.make_graph(N, E, seed=1, device=dev, symmetric=True)
g = G.prepare(ei, N, True)
torch.manual_seed(0)
h = torch.randn(N, C, device=dev); gg = torch.randn(N, C, device=dev)
fuse = (torch.randn(N, C, device=dev), torch.randn(C, device=dev), torch.full((1,), 0.5, device=dev), None)


def timed(fn, steps=10, warm=3):
    for _ in range(warm): fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(steps): fn()
    b.record(); torch.cuda.synchronize()
    return round(a.elapsed_time(b) / steps, 4)


res = {"lib": os.path.basename(_C._LIB_PATH), "C": C}
res["fwd_infer"] = timed(lambda: SF._edge_fwd(h, g, 0, 10, 0.0, False))
res["fwd_train"] = timed(lambda: SF._edge_fwd(h, g, 0, 10, 0.0, True, want_q=True))
res["fwd_fused_infer"] = timed(lambda: SF._edge_fwd(h, g, 0, 10, 0.0, False, fuse))
res["fwd_fused_train"] = timed(lambda: SF._edge_fwd(h, g, 0, 10, 0.0, True, fuse, want_q=True))
out, ss, sw, sq, sc, inv, diff = SF._edge_fwd(h, g, 0, 10, 0.0, True, fuse, want_q=True)
res["bwd_plain"] = timed(lambda: SF.edge_bwd(h, inv, gg, g, 10, ss, sw, sq, sc, None, None))
res["bwd_fused"] = timed(lambda: SF.edge_bwd(h, inv, gg, g, 10, ss, sw, sq, sc, fuse[2], diff))
print(json.dumps(res))
