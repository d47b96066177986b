"""top_k > 64 on the edge path (the per-edge form) at the pokec shape, against the paths it sits between.

For C = 32 and C = 4, clustered features (so that thr = 0.5 matters), top_k = 100, 1,000 and max_deg (no row cut), alternating
in one process (CUDA-event medians per call, training forms):
  * the per-edge form: cut + aggregation forward (sng_edge_fwd_wide), the same with the fused SNGNN++ epilogue, the backward
    (sng_edge_bwd_wide), and one SNGNN++ layer step (fused forward + backward through autograd);
  * the select-every-edge kernels of the base SNConv (top_k <= 0: the same gathers, no selection -- the floor to approach);
  * the selection-list path at top_k = 10 (sng_edge_fwd_denom + sng_edge_bwd_denom);
  * a plain torch forward: sddmm_dot scores, per-row ranks from two stable sorts, index_add.
Bytes follow DESIGN.md §6: forward E'(4C+4) + N(8C+8), plus E_cut(4C+4) for the cut's second gather of the cut rows and E'
flag bytes; backward E'(12C+16) + 5N 4C + E'.  Shares of HBM use 7.7 TB/s.  h (209 MB at C = 32) is larger than the L2.

    python scripts/wide_k_time.py [--reps 10] [--rounds 5] [--out FILE]

Prints one JSON object with the card's name and power limit."""
import argparse
import json
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from sngnn_b200 import functional as SF, graph as G, synth  # noqa: E402
from scripts.shard_bwd_time import card, time_alternating  # noqa: E402

HBM = 7.7e12


def torch_forward(h, xhat, src, dst, deg, k, thr):
    """out_1 by a torch composition: scores, ranks by (score desc, position asc) inside each row, index_add."""
    s = SF.sddmm_dot(xhat, dst, src)
    o1 = torch.argsort(s, descending=True, stable=True)
    order = o1[torch.argsort(dst[o1], stable=True)]
    rank = torch.empty_like(order)
    start = torch.cumsum(deg, 0) - deg
    rank[order] = torch.arange(order.numel(), device=h.device) - start[dst[order]]
    w = torch.where((rank < k) & (s >= thr), s, torch.zeros_like(s))
    out = torch.zeros_like(h).index_add_(0, dst, w[:, None] * h[src])
    return out / deg.clamp(min=1)[:, None]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("wide_k_time.py needs a CUDA device")
    n, _, e, _ = synth.SHAPES["pokec"]
    dev = "cuda"
    ei = synth.make_graph(n, e, device=dev, symmetric=True)
    g = G.prepare(ei, n, True)
    del ei
    deg = (g.rowptr_in[1:] - g.rowptr_in[:-1]).long()
    dst = torch.repeat_interleave(torch.arange(n, device=dev), deg).to(torch.int32)
    src = g.col_in
    ep = g.num_edges
    res = {"card": card(), "shape": {"nodes": n, "edges": ep, "max_deg": g.max_deg}, "runs": []}
    thr = 0.5
    for c in (32, 4):
        h = synth.make_features(n, c, "clustered", seed=5, device=dev)
        gg = torch.randn(n, c, device=dev)
        xhat = SF.rownorm(h)[0]
        wt = (torch.randn(n, c, device=dev) * 0.1).requires_grad_(True)
        wb, beta = torch.randn(c, device=dev).requires_grad_(True), torch.full((1,), 0.5, device=dev).requires_grad_(True)
        fuse = SF._structural_operands(wt.t(), wb, beta, None, c)
        hg = h.clone().requires_grad_(True)
        _, ss, sw, sq, sc, inv10, _ = SF._edge_fwd(h, g, 0, 10, thr, True, want_q=True)
        inv0 = SF._edge_fwd(h, g, 0, 0, None, True)[5]
        for k in (100, 1000, g.max_deg):
            kk = min(k, g.max_deg)
            cut = deg > kk
            n_cut, e_cut = int(cut.sum()), int(deg[cut].sum())
            _, flags, inv, _ = SF._edge_fwd_wide(h, g, 0, k, thr, True)
            nsel = int(flags[:ep].sum())
            fns = {
                "wide_fwd": lambda: SF._edge_fwd_wide(h, g, 0, k, thr, True),
                "wide_fwd_fused": lambda: SF._edge_fwd_wide(h, g, 0, k, thr, True, fuse),
                "wide_bwd": lambda: SF.edge_bwd_wide(h, inv, gg, g, flags),
                "wide_layer_step": lambda: SF.EdgeWideAgg.apply(hg, g, 0, k, thr, wt.t(), wb, beta, None).backward(gg),
                "all_edges_fwd": lambda: SF._edge_fwd(h, g, 0, 0, None, True),
                "all_edges_bwd": lambda: SF.edge_bwd(h, inv0, gg, g, 0, None, None, None, None),
                "lists_k10_fwd": lambda: SF._edge_fwd(h, g, 0, 10, thr, True, want_q=True),
                "lists_k10_bwd": lambda: SF.edge_bwd(h, inv10, gg, g, 10, ss, sw, sq, sc),
                "torch_fwd": lambda: torch_forward(h, xhat, src, dst, deg, kk, thr),
            }
            t = time_alternating(fns, args.reps, args.rounds)
            hg.grad = wt.grad = wb.grad = beta.grad = None
            fwd_bytes = ep * (4 * c + 4) + n * (8 * c + 8) + e_cut * (4 * c + 4) + ep
            bwd_bytes = ep * (12 * c + 16) + 5 * n * 4 * c + ep
            row = dict(c=c, top_k=k, thr=thr, rows_cut=n_cut, edges_in_cut_rows=e_cut, selected=nsel,
                       **{f"{kk_}_ms": v for kk_, v in t.items()},
                       fwd_gb=fwd_bytes / 1e9, bwd_gb=bwd_bytes / 1e9,
                       fwd_hbm_share=fwd_bytes / HBM / (t["wide_fwd"] * 1e-3), bwd_hbm_share=bwd_bytes / HBM / (t["wide_bwd"] * 1e-3),
                       flag_mb=ep / 1e6, lists_would_be_gb=n * min(k, g.max_deg) * 12 / 1e9)              # sel_src, sel_w, sel_q
            res["runs"].append(row)
            print(json.dumps(row), file=sys.stderr, flush=True)
            del flags, inv, fns
        del h, gg, xhat, wt, hg, fuse, ss, sw, sq, sc
        torch.cuda.empty_cache()
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
