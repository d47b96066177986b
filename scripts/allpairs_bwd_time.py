"""Backward of the all-pairs list aggregation: the list transpose, the gather form against the scatter form, and one
all-pairs SNGNN_Plus training step.

  * transpose:    functional.list_transpose of one rank's lists (sng_list_transpose + the chunk tables of the staged source
                  pass, which read two counts back: one host synchronisation);
  * gather form:  functional.list_bwd = that transpose + sng_list_bwd (no float atomics);
  * scatter form: functional.edge_agg_bwd_scatter = sng_edge_agg_bwd (FP32 atomics, two zero-filled [N, C] accumulators).
Lists come from the K1 build (sng_simknn_build, top_k = 10) on clustered features of width C = 32 at the arxiv-year shape
(N = 169,343) and the pokec shape (N = 1,632,803); the C = 4 rows reuse the pokec C = 32 lists with fresh h and g (the list
structure, not the feature width, decides the transpose).  For 1, 2, 4, 8 shards, rank 0's rows [0, ceil(N / S)) are timed,
the functions alternating in the same process.  The training step (zero_grad, forward, loss, backward, Adam) runs at the
arxiv-year shape with SNGNN_Plus(hidden 32, 2 layers, candidates='all_pairs', top_k = 10); under torchrun it runs
row-sharded (dist.sharded_forward) on every rank and rank 0 reports.

    python scripts/allpairs_bwd_time.py [--reps 10] [--rounds 5] [--steps 10] [--out FILE]
    torchrun --nproc_per_node 8 scripts/allpairs_bwd_time.py --step-only

Prints one JSON object (card name and power limit included).  Times are CUDA-event medians per call."""
import argparse
import json
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from sngnn_b200 import dist as D, functional as SF, simknn, synth  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return {"device": torch.cuda.get_device_name(), "nvidia_smi": q[0] if q else "unavailable"}


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


def backward_rows(name, n, c, k, lists, reps, rounds):
    idx, sim, cnt = lists
    torch.manual_seed(5)
    h = torch.randn(n, c, device="cuda")
    gg = torch.randn(n, c, device="cuda")
    _, _, inv_norm = SF.rownorm(h, want_f32=False, want_inv=True)
    out = []
    for s in (1, 2, 4, 8):
        lo, hi = D.shard_bounds(n, s, 0)
        si, ss, sc = idx[lo:hi].contiguous(), sim[lo:hi].contiguous(), cnt[lo:hi].contiguous()
        inv = torch.full((hi - lo,), 1.0 / (n - 1), device="cuda")
        g = gg[lo:hi].contiguous()
        fns = {"transpose": lambda: SF.list_transpose(si, sc, n, chunk_tables=c <= 32),
               "gather_form": lambda: SF.list_bwd(h, inv_norm, g, si, ss, sc, inv, lo),
               "scatter_form": lambda: SF.edge_agg_bwd_scatter(h, inv_norm, g, None, None, hi - lo, lo, k, si, ss, sc, inv)}
        t = time_alternating(fns, reps, rounds)
        a, b = fns["gather_form"](), fns["scatter_form"]()
        tr = fns["transpose"]()
        deg = (tr.rowptr_tr[1:] - tr.rowptr_tr[:-1])
        row = {"shape": name, "c": c, "top_k": k, "shards": s, "rows": [lo, hi], "entries": int(tr.rowptr_tr[-1]),
               "max_selected_by": int(deg.max()), "transpose_ms": t["transpose"], "gather_form_ms": t["gather_form"],
               "gather_passes_ms": t["gather_form"] - t["transpose"], "scatter_form_ms": t["scatter_form"],
               "max_rel_diff": float((a - b).abs().max() / b.abs().max())}
        print(json.dumps(row), file=sys.stderr, flush=True)
        out.append(row)
    return out


def training_step(steps):
    """Median ms of one SNGNN_Plus all-pairs training step at the arxiv-year shape (row-sharded under torchrun)."""
    import sngnn_b200.models as M
    n, fd, e, ncls = synth.SHAPES["arxiv-year"]
    ws, rank = D.world()
    dev = torch.device("cuda", torch.cuda.current_device())
    x = synth.make_features(n, fd, "clustered", seed=1, device=dev)
    ei = synth.make_graph(n, e, seed=2, device=dev)
    y = synth.make_labels(n, ncls, seed=3, device=dev)
    torch.manual_seed(7)
    model = M.SNGNN_Plus(fd, 32, ncls, n, 2, 10, 0.0, 1, 0.5, candidates="all_pairs").to(dev).train()
    opt = torch.optim.Adam(model.parameters(), lr=0.01)
    lo, hi = D.shard_bounds(n, ws, rank)
    data = synth.GraphData(x, ei)

    def step():
        opt.zero_grad(set_to_none=True)
        if ws == 1:
            loss = SF.nll_loss(model(data), y)
        else:
            loss = SF.nll_loss(D.sharded_forward(model, x[lo:hi].contiguous(), ei, n), y[lo:hi]) * ((hi - lo) / n)
        loss.backward()
        D.allreduce_grads(model.parameters())
        opt.step()

    for _ in range(2):
        step()
    torch.cuda.synchronize()
    ts = []
    for _ in range(steps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        step()
        b.record()
        b.synchronize()
        ts.append(a.elapsed_time(b))
    return {"shape": "arxiv-year", "model": "SNGNN_Plus(hidden 32, 2 layers, all_pairs, top_k 10)", "gpus": ws,
            "step_ms": sorted(ts)[len(ts) // 2]}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--step-only", action="store_true")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("allpairs_bwd_time.py needs a CUDA device")
    if "RANK" in os.environ:
        import torch.distributed as dist
        torch.cuda.set_device(int(os.environ["LOCAL_RANK"]))
        dist.init_process_group("nccl")
    res = {"card": card()}
    if not args.step_only:
        res["backward"] = []
        for name in ("arxiv-year", "pokec"):
            n = synth.SHAPES[name][0]
            x = synth.make_features(n, 32, "clustered", seed=4, device="cuda")
            lists = simknn.build_knn(x, 10, -1.0, True)
            del x
            res["backward"] += backward_rows(name, n, 32, 10, lists, args.reps, args.rounds)
            if name == "pokec":
                res["backward"] += backward_rows(name, n, 4, 10, lists, args.reps, args.rounds)
            del lists
            torch.cuda.empty_cache()
    res["training_step"] = training_step(args.steps)
    ws, rank = D.world()
    if rank == 0:
        line = json.dumps(res)
        print(line)
        if args.out:
            os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
            with open(args.out, "w") as f:
                f.write(line + "\n")
    if ws > 1:
        import torch.distributed as dist
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
