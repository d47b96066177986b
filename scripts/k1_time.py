"""A/B timing of K1 (the similarity-kNN build) between this build of libsng.so and a previous one, on the bench's inputs.

For each shape the FP32 / FP16 operands are built once (bench.py's seeded features), then the two libraries alternate
`--rounds` times.  Per library and round: the main pass alone (sng_simknn_stage1, launched as bench.py launches it: the
build's plan, its seeds, a zeroed sweep phase) and the whole sng_simknn_build, each as the mean of `--reps` calls between CUDA
events.  Prints medians and spreads (max - min over the rounds) per library, the card and its power limit, and whether the two
builds' idx / sim / cnt are equal (torch.equal: the final lists are exact and sim comes from the deterministic FP32 dot, so any
difference is a bug).  Shapes: pokec, arxiv-year and N = 4 M d = 64 run the small-K (EW = 4) kernel, N = 1 M d = 256 the
two-stage one (EW = 2) as a control.

    python scripts/k1_time.py --ref-lib PATH [--rounds 5] [--reps 2] [--shapes pokec,arxiv,n4m_d64,n1m_d256] [--out FILE]
"""
import argparse
import ctypes
import json
import os
import statistics
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from sngnn_b200 import _C, simknn, synth  # noqa: E402
from scripts.lib_parity import load  # noqa: E402

# name: (n, d, top_k, features, zscore) -- the bench's headline shape and three of its `configs`
SHAPES = {"pokec": (1632803, 65, 10, "clustered", True),
          "arxiv": (169343, 128, 10, "clustered", False),
          "n4m_d64": (4000000, 64, 5, "clustered", False),
          "n1m_d256": (1000000, 256, 20, "clustered", False)}
THR = 0.0                                                    # bench.py's default


class using:
    """Route the library's entry points (simknn.*, _C.call) through `lib` inside the block."""
    def __init__(self, lib):
        self.lib = lib

    def __enter__(self):
        self.saved, _C._lib = _C._lib, self.lib

    def __exit__(self, *exc):
        _C._lib = self.saved


def timed(fn, reps):
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / reps


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError) as exc:
        q = f"nvidia-smi unavailable: {exc}"
    return {"device": torch.cuda.get_device_name(0), "nvidia_smi": q}


def run_shape(name, libs, rounds, reps):
    n, d, k, features, zscore = SHAPES[name]
    x = synth.make_features(n, d, features, seed=0, device="cuda", zscore=zscore)
    with using(libs["new"]):
        xf, xh = simknn.normalize_operands(x)
    del x
    ldh = xh.size(1)
    plan = {}
    for tag, lib in libs.items():
        with using(lib):
            plan[tag] = simknn.build_plan(n, n, d, k)
    ci = torch.empty(n * 192, dtype=torch.int32, device="cuda")      # lists * cand <= 192 slots per row
    cv = torch.empty(n * 192, dtype=torch.float32, device="cuda")
    cm = torch.empty(n * 64, dtype=torch.float32, device="cuda")
    sweep_phase = torch.zeros(8, dtype=torch.int32, device="cuda")
    thr_lo = THR - 1.01 * (2.0 ** -10 + 1.2e-4)
    outs, seeds = {}, {}

    def build(tag):
        with using(libs[tag]):
            outs[tag] = simknn.build_knn_normalized(xf, xh, d, k, THR, True, return_fallback=True)

    def main_pass(tag):
        pl, ns = plan[tag], ctypes.c_int(0)
        with using(libs[tag]):
            sweep_phase.zero_()
            _C.call("sng_simknn_stage1", xh, _C.ptr(xh), _C.ptr(xh), ldh, n, 0, n, d, pl["cand"], thr_lo, 1, _C.ptr(ci), _C.ptr(cv),
                    _C.ptr(cm), pl["ew"], pl["nsplit"], ctypes.byref(ns), _C.ptr(seeds.get(tag)), pl["seed_q"], pl["seed_stride"],
                    _C.ptr(sweep_phase))

    for tag, lib in libs.items():                            # warm-up: modules, function attributes, allocator
        with using(lib):
            if plan[tag]["seed_stride"] > 0:
                seeds[tag] = simknn.seed_pass(xh, xh, d, plan[tag]["seed_stride"], plan[tag]["ew"])
        build(tag)
        main_pass(tag)
    ms = {tag: {"main_pass": [], "build": []} for tag in libs}
    for r in range(rounds):
        order = list(libs) if r % 2 == 0 else list(libs)[::-1]
        for tag in order:
            ms[tag]["main_pass"].append(timed(lambda: main_pass(tag), reps))
            ms[tag]["build"].append(timed(lambda: build(tag), reps))
    equal = {f: torch.equal(a, b) for f, a, b in zip(("idx", "sim", "cnt"), outs["new"][:3], outs["ref"][:3])}
    summary = {tag: {what: {"median_ms": statistics.median(v), "spread_ms": max(v) - min(v), "ms": v} for what, v in m.items()}
               for tag, m in ms.items()}
    res = {"shape": name, "n": n, "d": d, "top_k": k, "plan": plan["new"], "plans_equal": plan["new"] == plan["ref"], **summary,
           "main_pass_ratio": summary["new"]["main_pass"]["median_ms"] / summary["ref"]["main_pass"]["median_ms"],
           "build_ratio": summary["new"]["build"]["median_ms"] / summary["ref"]["build"]["median_ms"],
           "outputs_equal": equal, "fallback_retry": {t: [int(v) for v in o[3].tolist()] for t, o in outs.items()}}
    del xf, xh, ci, cv, cm, outs, seeds
    torch.cuda.empty_cache()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--ref-lib", required=True)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--reps", type=int, default=2)
    ap.add_argument("--shapes", default=",".join(SHAPES))
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("k1_time.py needs a CUDA device")
    if args.rounds < 1 or args.reps < 1:
        ap.error("--rounds and --reps must be at least 1")
    libs = {"new": _C.lib(), "ref": load(args.ref_lib)}
    head = {"gpu": gpu_info(), "ref_lib": os.path.abspath(args.ref_lib), "rounds": args.rounds, "reps": args.reps}
    print(json.dumps(head), flush=True)
    rows, ok = [], True
    for name in args.shapes.split(","):
        res = run_shape(name, libs, args.rounds, args.reps)
        ok &= all(res["outputs_equal"].values())
        rows.append(res)
        print(json.dumps({k: v for k, v in res.items() if k not in ("new", "ref")} |
                         {t: {w: round(res[t][w]["median_ms"], 3) for w in res[t]} for t in ("new", "ref")} |
                         {"spread": {t: {w: round(res[t][w]["spread_ms"], 3) for w in res[t]} for t in ("new", "ref")}}), flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump({**head, "shapes": rows, "all_outputs_equal": ok}, f, indent=1)
    sys.exit(0 if ok else 1)


if __name__ == "__main__":
    main()
