"""The models at top_k <= SNG_MAX_TOPK through this build and through a previous libsng.so, bit for bit.

SNGNN_Plus and SNGNN_Plus_Plus (symmetric graph: the fused pass; asymmetric: aggregation + K4) at top_k = 1, 10 and 64, both
denominators, hidden widths 32 and 128: one training forward + backward per library on the same seeded inputs and parameters,
and every output and parameter gradient compared with torch.equal.

    python scripts/lib_parity.py --ref-lib PATH [--candidates all_pairs] [--out FILE]

With --candidates all_pairs the models select among all nodes, and simknn.build_knn's lists at the same top_k are compared
too.

Prints one JSON object; exits non-zero when any tensor differs."""
import argparse
import copy
import ctypes
import json
import os
import sys

import torch
import torch.nn.functional as F

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import sngnn_b200.models as M  # noqa: E402
from sngnn_b200 import _C, graph as G, synth  # noqa: E402


def load(path):
    """A previous libsng.so with the signatures of the entry points it exports."""
    lib = ctypes.CDLL(os.path.abspath(path))
    for name, (res, args) in _C.SIGNATURES.items():
        if hasattr(lib, name):
            f = getattr(lib, name)
            f.restype, f.argtypes = res, args
    return lib


def step(model, data, y):
    model.zero_grad()
    out = model(data)
    F.nll_loss(out, y).backward()
    return [out.detach()] + [p.grad.clone() for p in model.parameters()]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--ref-lib", required=True)
    ap.add_argument("--candidates", default="edges", choices=("edges", "all_pairs"))
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("lib_parity.py needs a CUDA device")
    ref_lib = load(args.ref_lib)
    n, fd, ncls = 20000, 48, 5
    x = synth.make_features(n, fd, "clustered", seed=1).cuda()
    y = synth.make_labels(n, ncls, seed=3).cuda()
    rows, ok = [], True
    if args.candidates == "all_pairs":
        from sngnn_b200 import simknn
        for k in (1, 10, 64):
            new = simknn.build_knn(x, k, 0.2, True)
            this, _C._lib = _C._lib, ref_lib
            try:
                old = simknn.build_knn(x, k, 0.2, True)
            finally:
                _C._lib = this
            same = all(torch.equal(a, b) for a, b in zip(new, old))
            ok &= same
            rows.append(dict(build_knn=True, top_k=k, bit_identical=same))
            print(json.dumps(rows[-1]), file=sys.stderr, flush=True)
    for symmetric in (True, False):
        ei = synth.make_graph(n, 300000, seed=2, symmetric=symmetric, hub_offset=3.0).cuda()
        data = synth.GraphData(x, ei)
        G.clear_cache()
        for kind in ("SNGNN_Plus", "SNGNN_Plus_Plus"):
            for hid in (32, 128):
                for k in (1, 10, 64):
                    for den in ("candidates", "selected"):
                        torch.manual_seed(0)
                        cls = M.SNGNN_Plus if kind == "SNGNN_Plus" else M.SNGNN_Plus_Plus
                        extra = (0.5,) if kind == "SNGNN_Plus_Plus" else ()
                        model = cls(fd, hid, ncls, n, 2, k, 0.2, *extra, 1, 0.0, denominator=den,
                                    candidates=args.candidates).cuda().train()
                        other = copy.deepcopy(model)
                        new = step(model, data, y)
                        this, _C._lib = _C._lib, ref_lib
                        try:
                            old = step(other, data, y)
                        finally:
                            _C._lib = this
                        same = all(torch.equal(a, b) for a, b in zip(new, old))
                        ok &= same
                        rows.append(dict(kind=kind, symmetric=symmetric, hidden=hid, top_k=k, denominator=den, tensors=len(new),
                                         bit_identical=same))
                        print(json.dumps(rows[-1]), file=sys.stderr, flush=True)
    line = json.dumps({"cases": len(rows), "all_bit_identical": ok, "rows": rows})
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")
    sys.exit(0 if ok else 1)


if __name__ == "__main__":
    main()
