"""Aggregation backward of one rank's row shard at the pokec shape, emulated on one GPU.

For C = 32 / top_k = 10 and C = 4 / top_k = 10 and 1, 2, 4, 8 shards, rank 0's shard [0, ceil(N / S)) is timed, alternating in
the same process:
  * shard form:   sng_edge_bwd with row_offset through the shard's transpose index (functional.edge_bwd, no float atomics);
  * scatter form: sng_edge_agg_bwd with its two zero-filled [N, C] accumulators and the norm_bwd_finish pass
                  (functional.edge_agg_bwd_scatter, FP32 atomics), the sharded backward before the shard form existed.
With --ref-lib (a libsng.so built from the commit before sng_edge_bwd took n_total / row_offset), the unsharded
sng_edge_bwd of this build and of that one also run alternately on the whole graph, plain and fused, and their outputs are
compared with torch.equal.

    python scripts/shard_bwd_time.py [--ref-lib PATH] [--reps 20] [--rounds 5] [--out FILE]

Prints one JSON object (card name and power limit included).  Times are CUDA-event medians per call; h (209 MB at C = 32)
is larger than the L2, so the gathers come from HBM."""
import argparse
import ctypes
import json
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from sngnn_b200 import _C, dist as D, functional as SF, graph as G, synth  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return {"device": torch.cuda.get_device_name(0), "nvidia_smi": q[0] if q else "unavailable"}


def time_alternating(fns, reps, rounds):
    """{name: median ms per call}: every round runs each function `reps` times between two events, in turn."""
    for f in fns.values():
        f()
    torch.cuda.synchronize()
    per = {k: [] for k in fns}
    for _ in range(rounds):
        for name, f in fns.items():
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            for _ in range(reps):
                f()
            b.record()
            b.synchronize()
            per[name].append(a.elapsed_time(b) / reps)
    return {k: sorted(v)[len(v) // 2] for k, v in per.items()}


def ref_edge_bwd(lib, h, inv_norm, g, graph, k, ss, sw, sq, sc, beta=None, diff=None):
    """functional.edge_bwd on the whole graph through the previous ABI (sng_edge_bwd without n_total / row_offset)."""
    n, cp = h.shape
    dev = h.device
    fused = beta is not None
    coef = torch.empty(max(graph.num_edges, 1) * 2, dtype=torch.float32, device=dev)
    dnt, dh = torch.empty_like(h), torch.empty_like(h)
    dbeta = dwt = part = None
    if fused:
        dbeta = torch.empty(1, dtype=torch.float32, device=dev)
        part = torch.empty(_C.PARTIALS, dtype=torch.float32, device=dev)
        dwt = torch.empty(n, cp, dtype=torch.float32, device=dev)
    tab = graph.chunk_tab_out if cp <= 32 else None
    n_chunks = -1 if tab is None else int(tab.size(0))
    cpart = None
    if n_chunks > 0:
        cg = 4
        while cg < cp:
            cg *= 2
        cpart = torch.empty(n_chunks * 3 * cg, dtype=torch.float32, device=dev)
    P = _C.ptr
    rc = lib.sng_edge_bwd(P(h), P(inv_norm), P(g), n, cp, cp, cp, P(graph.rowptr_in), P(graph.col_in), P(graph.tpos),
                          P(graph.rowptr_out), P(graph.col_out), graph.src_shift, graph.num_edges, k, P(ss), P(sw), P(sq), P(sc),
                          P(beta), P(diff if fused else None), cp, P(dbeta), P(coef), P(dnt), P(part), P(dh), P(dwt), cp,
                          P(tab), n_chunks, P(graph.lrows_out if tab is not None else None),
                          P(graph.lrow_ptr_out if tab is not None else None), 0 if tab is None else int(graph.lrows_out.numel()),
                          P(cpart), _C.stream(h))
    if rc != 0:
        raise RuntimeError(f"reference sng_edge_bwd failed (rc={rc}): {lib.sng_last_error().decode()}")
    return dh, dwt, dbeta


def load_ref(path):
    lib = ctypes.CDLL(os.path.abspath(path))
    args = _C.SIGNATURES["sng_edge_bwd"][1]
    lib.sng_edge_bwd.restype, lib.sng_edge_bwd.argtypes = ctypes.c_int, args[:4] + args[6:]      # no n / row_offset after n_total
    lib.sng_last_error.restype = ctypes.c_char_p
    return lib


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--ref-lib", default=None)
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("shard_bwd_time.py needs a CUDA device")
    n, _, e, _ = synth.SHAPES["pokec"]
    dev = "cuda"
    ei = synth.make_graph(n, e, device=dev, symmetric=True)
    g = G.prepare(ei, n, True)
    del ei
    res = {"card": card(), "shape": {"nodes": n, "edges": g.num_edges, "symmetric": g.symmetric}, "shards": [], "unsharded": []}
    ref = load_ref(args.ref_lib) if args.ref_lib else None
    thr = 0.0
    for c, k in ((32, 10), (4, 10)):
        torch.manual_seed(3)
        h = torch.randn(n, c, device=dev)
        gg = torch.randn(n, c, device=dev)
        for s in (1, 2, 4, 8):
            lo, hi = D.shard_bounds(n, s, 0)
            sh = g.row_slice(lo, hi)
            _, ss, sw, sq, sc, inv, _ = SF._edge_fwd(h, sh, lo, k, thr, True, want_q=True)
            gs = gg[lo:hi].contiguous()
            fns = {"shard_form": lambda: SF.edge_bwd(h, inv, gs, sh, k, ss, sw, sq, sc, row_offset=lo),
                   "scatter_form": lambda: SF.edge_agg_bwd_scatter(h, inv, gs, sh.rowptr_in, sh.col_in, sh.n, lo, k, ss, sw, sc, sh.inv_deg)}
            t = time_alternating(fns, args.reps, args.rounds)
            a, b = fns["shard_form"]()[0], fns["scatter_form"]()
            rel = float((a - b).abs().max() / b.abs().max())
            res["shards"].append({"c": c, "top_k": k, "shards": s, "rows": [lo, hi], "edges": sh.num_edges,
                                  "shard_form_ms": t["shard_form"], "scatter_form_ms": t["scatter_form"],
                                  "ratio_shard_over_scatter": t["shard_form"] / t["scatter_form"], "max_rel_diff": rel})
            print(json.dumps(res["shards"][-1]), file=sys.stderr, flush=True)
            del ss, sw, sq, sc, inv, fns
        if ref is not None:
            fuse = (torch.randn(n, c, device=dev) * 0.1, torch.randn(c, device=dev), torch.full((1,), 0.5, device=dev), None)
            for fused in (False, True):
                _, ss, sw, sq, sc, inv, diff = SF._edge_fwd(h, g, 0, k, thr, True, fuse if fused else None, want_q=True)
                beta = fuse[2] if fused else None
                fns = {"this_build": lambda: SF.edge_bwd(h, inv, gg, g, k, ss, sw, sq, sc, beta, diff),
                       "parent_build": lambda: ref_edge_bwd(ref, h, inv, gg, g, k, ss, sw, sq, sc, beta, diff)}
                t = time_alternating(fns, args.reps, args.rounds)
                new, old = fns["this_build"](), fns["parent_build"]()
                equal = all((x is None and y is None) or torch.equal(x, y) for x, y in zip(new, old))
                res["unsharded"].append({"c": c, "top_k": k, "fused": fused, "this_build_ms": t["this_build"],
                                         "parent_build_ms": t["parent_build"], "bit_identical": equal})
                print(json.dumps(res["unsharded"][-1]), file=sys.stderr, flush=True)
                del ss, sw, sq, sc, inv, diff, fns
        del h, gg
        torch.cuda.empty_cache()
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
