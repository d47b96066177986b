"""Timing of the wide all-pairs build (top_k > 64: sng_simknn_wide_count + sng_simknn_wide_select) and of ListAgg at k = 100.

For each shape (N, d = 65, the bench's clustered z-scored features) and each (k, thr): the whole build, its count call (seed
pass + count sweep + scan) and its select call (emit sweep + rescore / sort + exact scan), the rows that took the exact scan,
and the candidate total.  Then K1 at k = 64 on the same operands, a blocked torch baseline (row-block FP32 mm + topk; N = 100 k
only), and ListAgg forward / backward at k = 100, C = 32.  A case whose build takes longer than --budget seconds ends its
shape's larger cases ("not measured").  Prints one JSON object with the card's name and power limit.

    python scripts/allpairs_wide_k_time.py [--shapes 100k,400k,pokec] [--out FILE]"""
import argparse
import json
import os
import subprocess
import sys
import time

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from sngnn_b200 import _C, functional as SF, simknn, synth  # noqa: E402

SHAPES = {"100k": 100000, "400k": 400000, "pokec": 1632803}
CASES = [(100, -1.0), (100, 0.9), (256, -1.0), (256, 0.9), (1000, -1.0), (1000, 0.9)]
D = 65


def ev_time(fn):
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    r = fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b), r


def wide_build(xf, xh, k, thr):
    """simknn._build_wide with the two calls timed apart (the read-back of the total sits between them)."""
    n = xf.size(0)
    wbytes = _C.lib().sng_simknn_wide_workspace_bytes(n, n, D, k)
    ws = torch.empty(wbytes, dtype=torch.uint8, device="cuda")
    off = torch.empty(n + 1, dtype=torch.int64, device="cuda")
    common = (_C.ptr(xh), _C.ptr(xh), xh.size(1))
    t_count, _ = ev_time(lambda: _C.call("sng_simknn_wide_count", xf, *common, n, 0, n, D, k, float(thr), 1, _C.ptr(off), _C.ptr(ws), wbytes))
    total = int(off[n])
    cand = torch.empty(max(total, 1), dtype=torch.int32, device="cuda")
    idx = torch.empty(n, k, dtype=torch.int32, device="cuda")
    sim = torch.empty(n, k, dtype=torch.float32, device="cuda")
    cnt = torch.empty(n, dtype=torch.int32, device="cuda")
    nex = torch.zeros(1, dtype=torch.int32, device="cuda")
    t_sel, _ = ev_time(lambda: _C.call("sng_simknn_wide_select", xf, *common, _C.ptr(xf), _C.ptr(xf), xf.size(1), n, 0, n, D, k, float(thr), 1,
                                       _C.ptr(off), _C.ptr(cand), _C.ptr(idx), _C.ptr(sim), _C.ptr(cnt), _C.ptr(nex), _C.ptr(ws), wbytes))
    return dict(count_ms=t_count, select_ms=t_sel, total_ms=t_count + t_sel, candidates=total, exact_rows=int(nex[0]),
                mean_cnt=float(cnt.float().mean())), (idx, sim, cnt)


def torch_blocked(xf, k, block=4096):
    n = xf.size(0)
    x = xf[:, :D]
    for lo in range(0, n, block):
        s = x[lo:lo + block] @ x.t()
        s[torch.arange(s.size(0)), torch.arange(lo, lo + s.size(0))] = float("-inf")
        torch.topk(s, k, dim=1)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--shapes", default=",".join(SHAPES))
    ap.add_argument("--budget", type=float, default=60.0)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("allpairs_wide_k_time.py needs a CUDA device")
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True, text=True).stdout.strip()
    res = {"device": torch.cuda.get_device_name(0), "nvidia_smi": smi, "shapes": {}}
    for name in args.shapes.split(","):
        n = SHAPES[name]
        x = synth.make_features(n, D, "clustered", seed=0, device="cuda", zscore=True)
        xf, xh = simknn.normalize_operands(x)
        del x
        rows = {}
        simknn.build_knn_normalized(xf, xh, D, 64, 0.0, True)                     # warm-up (module load, attributes)
        rows["k1_k64_thr-1_ms"], _ = ev_time(lambda: simknn.build_knn_normalized(xf, xh, D, 64, -1.0, True))
        wide_build(xf, xh, 100, 0.9)                                               # warm-up of the wide kernels
        over = False
        for k, thr in CASES:
            key = f"k{k}_thr{thr}"
            if over:
                rows[key] = "not measured"
                continue
            t0 = time.time()
            r, out = wide_build(xf, xh, k, thr)
            rows[key] = r
            print(name, key, json.dumps(r), file=sys.stderr, flush=True)
            if k == 100 and thr == -1.0:
                c = 32
                h = torch.randn(n, c, device="cuda")
                idx, sim, cnt = out
                inv = 1.0 / cnt.clamp(min=1).float()
                hd = h.clone().requires_grad_(True)
                SF.ListAgg.apply(hd, idx, sim, cnt, inv, 0).sum().backward()       # warm-up
                t_f, o = ev_time(lambda: SF.ListAgg.apply(hd, idx, sim, cnt, inv, 0))
                t_b, _ = ev_time(lambda: o.sum().backward())
                rows["listagg_k100_c32"] = dict(forward_ms=t_f, backward_ms=t_b)
            del out
            if time.time() - t0 > args.budget:
                over = True
        if name == "100k":
            torch_blocked(xf, 100, 4096)
            rows["torch_blocked_k100_ms"], _ = ev_time(lambda: torch_blocked(xf, 100))
        res["shapes"][name] = rows
        del xf, xh
        torch.cuda.empty_cache()
    line = json.dumps(res)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
