"""denominator='selected' on the edge path at the pokec shape: timing against the Python path it replaces and against the
default mode, and (with --ref-lib) the default mode against the previous build, bit for bit.

For C = 32 and C = 4, top_k = 10, thr = 0, alternating in one process (CUDA-event medians per call):
  * SNGNN++ layer, forward and forward + backward (autograd): the previous 'selected' path (EdgeAgg in candidates mode,
    a rescale by deg / max(cnt, 1), then K4 sng_pp_fuse_fwd / _bwd) against the fused single pass with the mode in the kernel;
  * kernels: sng_edge_fwd_denom (training form, plain and fused) and sng_edge_bwd_denom, 'selected' against 'candidates'.
With --ref-lib (a libsng.so built from the commit before sng_edge_fwd_denom existed), functional._edge_fwd / edge_bwd in the
default mode run through both libraries on the same seeded inputs, plain and fused, and every output is compared with
torch.equal.

    python scripts/selected_time.py [--ref-lib PATH] [--reps 20] [--rounds 7] [--out FILE]

Prints one JSON object (card name and power limit included).  h (209 MB at C = 32) is larger than the L2."""
import argparse
import ctypes
import json
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from sngnn_b200 import _C, functional as SF, graph as G, synth  # noqa: E402
from scripts.shard_bwd_time import card, time_alternating  # noqa: E402


class ParentLib:
    """The previous libsng.so behind the current call sites: the *_denom entry points map to sng_edge_fwd / sng_edge_bwd,
    which they extend, in the default mode (denominator 0, no inv_denom)."""

    def __init__(self, path):
        self.lib = ctypes.CDLL(os.path.abspath(path))
        for name, (res, args) in _C.SIGNATURES.items():
            if not name.endswith("_denom"):
                f = getattr(self.lib, name)
                f.restype, f.argtypes = res, args

    def __getattr__(self, name):
        return getattr(self.lib, name)

    def sng_edge_fwd_denom(self, *a):
        *args, denominator, inv_denom, stream = a
        assert denominator == 0 and inv_denom is None
        return self.lib.sng_edge_fwd(*args, stream)

    def sng_edge_bwd_denom(self, *a):
        *args, inv_denom, stream = a
        assert inv_denom is None
        return self.lib.sng_edge_bwd(*args, stream)


def default_mode_outputs(h, gg, g, k, fuse):
    """(forward outputs, backward outputs) of _edge_fwd / edge_bwd in the default mode, training form."""
    fwd = SF._edge_fwd(h, g, 0, k, 0.0, True, fuse, want_q=True)
    out, ss, sw, sq, sc, inv, diff = fwd
    bwd = SF.edge_bwd(h, inv, gg, g, k, ss, sw, sq, sc, fuse[2] if fuse else None, diff)
    return [t for t in fwd if t is not None], [t for t in bwd if t is not None]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--ref-lib", default=None)
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=7)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("selected_time.py needs a CUDA device")
    n, _, e, _ = synth.SHAPES["pokec"]
    dev = "cuda"
    ei = synth.make_graph(n, e, device=dev, symmetric=True)
    g = G.prepare(ei, n, True)
    del ei
    res = {"card": card(), "shape": {"nodes": n, "edges": g.num_edges, "symmetric": g.symmetric}, "layer": [], "kernels": [],
           "parent_parity": []}
    k, thr = 10, 0.0
    for c in (32, 4):
        torch.manual_seed(3)
        h = torch.randn(n, c, device=dev)
        gg = torch.randn(n, c, device=dev)
        wt = (torch.randn(n, c, device=dev) * 0.1).requires_grad_(True)
        wb, beta = torch.randn(c, device=dev).requires_grad_(True), torch.full((1,), 0.5, device=dev).requires_grad_(True)
        st = (wt.t(), wb, beta, None)
        hg = h.clone().requires_grad_(True)

        def old_layer():           # the previous SNConv_plus_plus path for denominator='selected'
            out1, (_, _, sc) = SF.edge_topk_agg(hg, g, k, thr, return_selection=True)
            return SF.PPFuse.apply(out1 * (sc.clamp(min=1).float() * g.inv_deg).reciprocal()[:, None], *st, g)

        def new_layer():
            return SF.edge_topk_agg(hg, g, k, thr, structural=st, denominator="selected")

        def step(f):
            return lambda: f().backward(gg)

        t = time_alternating({"old_fwd": old_layer, "new_fwd": new_layer, "old_step": step(old_layer), "new_step": step(new_layer)},
                             args.reps, args.rounds)
        o, nw = old_layer().detach(), new_layer().detach()
        res["layer"].append(dict(c=c, top_k=k, **{f"{kk}_ms": v for kk, v in t.items()},
                                 max_rel_diff=float((o - nw).abs().max() / o.abs().max())))
        print(json.dumps(res["layer"][-1]), file=sys.stderr, flush=True)
        hg.grad = wt.grad = wb.grad = beta.grad = None

        fuse = SF._structural_operands(wt.t(), wb, beta, None, c)
        for fused in (False, True):
            fu = fuse if fused else None
            inv_d = torch.empty(n, device=dev)
            _, ss, sw, sq, sc, inv, diff = SF._edge_fwd(h, g, 0, k, thr, True, fu, want_q=True)
            _, ss2, sw2, sq2, sc2, _, diff2 = SF._edge_fwd(h, g, 0, k, thr, True, fu, want_q=True, denominator="selected", inv_denom=inv_d)
            b = fuse[2] if fused else None
            fns = {"fwd_candidates": lambda: SF._edge_fwd(h, g, 0, k, thr, True, fu, want_q=True),
                   "fwd_selected": lambda: SF._edge_fwd(h, g, 0, k, thr, True, fu, want_q=True, denominator="selected", inv_denom=inv_d),
                   "bwd_candidates": lambda: SF.edge_bwd(h, inv, gg, g, k, ss, sw, sq, sc, b, diff),
                   "bwd_selected": lambda: SF.edge_bwd(h, inv, gg, g, k, ss2, sw2, sq2, sc2, b, diff2, inv_denom=inv_d)}
            t = time_alternating(fns, args.reps, args.rounds)
            res["kernels"].append(dict(c=c, top_k=k, fused=fused, **{f"{kk}_ms": v for kk, v in t.items()}))
            print(json.dumps(res["kernels"][-1]), file=sys.stderr, flush=True)
            del ss, sw, sq, sc, diff, ss2, sw2, sq2, sc2, diff2, fns

        if args.ref_lib:
            for fused in (False, True):
                fu = fuse if fused else None
                new = default_mode_outputs(h, gg, g, k, fu)
                this_lib, _C._lib = _C._lib, ParentLib(args.ref_lib)
                try:
                    old = default_mode_outputs(h, gg, g, k, fu)
                finally:
                    _C._lib = this_lib
                equal = [torch.equal(a, b) for a, b in zip(new[0] + new[1], old[0] + old[1])]
                res["parent_parity"].append(dict(c=c, top_k=k, fused=fused, tensors=len(equal), bit_identical=all(equal)))
                print(json.dumps(res["parent_parity"][-1]), file=sys.stderr, flush=True)
        del h, gg, wt, hg, fuse
        torch.cuda.empty_cache()
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
