"""Similarity histogram (toolbox node_similarity_histogram, kernel sng_simhist_f16) on the GPU.

  * kernel: N = 100 k, 400 k and 1,632,803 (pokec) at d = 65, 128, 256, iid ('normal') and clustered features of
    synth.make_features, and N = 50 k at d = 2,325 (the Chameleon raw width); 200 bins over [-1, 1].  Per workload: the
    median time of the kernel call (operands prepared once), ordered pairs per second N (N - 1) / t, and the share of the
    sustained dense FP16 peak the project quotes (1,355.6 TFLOP/s) reached by N^2 K' FLOP (the symmetric schedule scores
    N^2 / 2 pairs at 2 K' FLOP each), with K' both padded (K blocks of 64, what the tensor cores run) and algorithmic (3d).
  * baselines at N = 50 k, d = 65: the N x N route on the same card (node_similarity_dense_small + torch.histc), and the
    reference's CPU pattern (1000-row torch.mm blocks against all rows + histogram) on a slab of rows, extrapolated to N.
  * --world W: the sharded call (all-gather + kernel + all-reduce) at the pokec shape, d = 65, on W ranks over NCCL.

    python scripts/simhist_time.py [--reps 3] [--slab 2000] [--world 2 4 8] [--rank-timeout S] [--out FILE]

Prints one JSON object (card name and power limit included).  Times are CUDA-event medians per call."""
import argparse
import json
import os
import socket
import subprocess
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from sngnn_b200 import synth  # noqa: E402
from sngnn_b200.toolbox import dense as D  # noqa: E402

PEAK_TFLOPS = 1355.6             # sustained dense FP16 rate of the B200 the project quotes (DESIGN.md §4)
POKEC_N = 1632803


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return {"device": torch.cuda.get_device_name(0), "nvidia_smi": q[0] if q else "unavailable"}


def median_ms(fn, reps, warmup=1):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        ts.append(a.elapsed_time(b))
    return sorted(ts)[len(ts) // 2]


def kernel(n, d, kind, reps):
    xhat = D._normalised(synth.make_features(n, d, kind, seed=d, device="cuda"))
    a, b, k = D.split_f16_operands(xhat)
    del xhat
    t = (n + D.TILE_ROWS - 1) // D.TILE_ROWS
    counts = torch.zeros(200, dtype=torch.int64, device="cuda")
    from sngnn_b200 import _C

    def run():
        counts.zero_()
        _C.call("sng_simhist_f16", a, _C.ptr(a), a.size(1), _C.ptr(b), b.size(1), n, k, 0, t, -1.0, 1.0, 200, _C.ptr(counts))

    ms = median_ms(run, reps)
    assert int(counts.sum()) == n * (n - 1)
    kpad = -(-k // 64) * 64
    return {"N": n, "d": d, "features": kind, "ms": round(ms, 3), "pairs_per_s": float(f"{n * (n - 1) / (ms * 1e-3):.4g}"),
            "K_padded": kpad, "K_alg": k, "peak_share_padded_K": round(n * n * kpad / (ms * 1e-3) / (PEAK_TFLOPS * 1e12), 4),
            "peak_share_alg_K": round(n * n * k / (ms * 1e-3) / (PEAK_TFLOPS * 1e12), 4)}


def baselines(n, d, reps, slab):
    x = synth.make_features(n, d, "clustered", seed=d)
    xg = x.cuda()
    new_ms = median_ms(lambda: D.node_similarity_histogram(xg, 200), reps)

    def dense():
        vals = D.node_similarity_dense_small(xg)[0]
        return torch.histc(vals, 200, -1.0, 1.0)

    dense_ms = median_ms(dense, reps)
    torch.cuda.empty_cache()
    xn = torch.nn.functional.normalize(x, dim=-1)            # the reference's CPU pattern, on `slab` rows
    t0 = time.perf_counter()
    h = torch.zeros(200)
    for r0 in range(0, slab, 1000):
        h += torch.histc(xn[r0:r0 + 1000] @ xn.t(), 200, -1.0, 1.0)
    cpu_s = time.perf_counter() - t0
    return {"N": n, "d": d, "node_similarity_histogram_ms": round(new_ms, 3),
            "dense_small_plus_histc_ms": round(dense_ms, 3), "speedup_vs_dense": round(dense_ms / new_ms, 2),
            "cpu_reference_pattern_s_extrapolated": round(cpu_s * n / slab, 2),
            "cpu_reference_pattern_note": f"measured on {slab} rows x {n} in {cpu_s:.3f} s, scaled by N / {slab} (extrapolated)",
            "host_cores": os.cpu_count(), "torch_threads": torch.get_num_threads()}


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _rank_worker(rank, ws, port, reps, ret):
    import torch.distributed as dist
    from sngnn_b200 import dist as SD
    from sngnn_b200.toolbox.sharded import node_similarity_histogram_sharded
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=ws, device_id=dev)
    n = POKEC_N
    lo, hi = SD.shard_bounds(n, ws, rank)
    x = synth.make_features(n, 65, "normal", seed=65, device=dev)[lo:hi].contiguous()
    ms = median_ms(lambda: node_similarity_histogram_sharded(x, n, 200), reps)
    t = torch.tensor([ms], device=dev)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    if rank == 0:
        ret[ws] = round(float(t), 3)
    dist.barrier()
    dist.destroy_process_group()


def multi_gpu(worlds, reps, timeout):
    gpus = torch.cuda.device_count()
    out = {}
    for ws in worlds:
        if ws > gpus:
            out[ws] = f"not measured ({gpus} GPU(s) on this box)"
            continue
        import torch.multiprocessing as mp
        ctx = mp.get_context("spawn")
        ret = ctx.Manager().dict()
        port = _free_port()
        procs = [ctx.Process(target=_rank_worker, args=(r, ws, port, reps, ret)) for r in range(ws)]
        for p in procs:
            p.start()
        deadline = time.monotonic() + timeout
        for p in procs:                       # a rank that raised leaves the others waiting in a collective: bound the wait
            p.join(max(0.0, deadline - time.monotonic()))
        for p in procs:
            if p.is_alive():
                p.terminate()
                p.join(30)
                if p.is_alive():
                    p.kill()
                    p.join()
        out[ws] = ret.get(ws, "failed (exit codes %s)" % [p.exitcode for p in procs])
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--slab", type=int, default=2000, help="rows of the CPU reference-pattern slab")
    ap.add_argument("--world", type=int, nargs="*", default=[2, 4, 8])
    ap.add_argument("--rank-timeout", type=float, default=600.0)
    ap.add_argument("--out")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("simhist_time.py measures on a CUDA device; there is none")
    res = {"card": card(), "bins": 200, "range": [-1.0, 1.0], "peak_tflops_quoted": PEAK_TFLOPS, "kernel": []}
    for n in (100000, 400000, POKEC_N):
        for d in (65, 128, 256):
            for kind in ("normal", "clustered"):
                res["kernel"].append(kernel(n, d, kind, args.reps))
                torch.cuda.empty_cache()
    res["kernel"].append(kernel(50000, 2325, "clustered", args.reps))
    torch.cuda.empty_cache()
    res["baselines"] = baselines(50000, 65, args.reps, args.slab)
    res["sharded_pokec_d65_ms"] = multi_gpu(args.world, args.reps, args.rank_timeout)
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
