"""ReLU + BatchNorm of a row-sharded training step at the pokec shape (N = 1,632,803), on one GPU.

  * kernels: the library's forward (sng_bn_fwd_stats + sng_bn_fwd_apply) and backward (sng_bn_bwd_stats + sng_bn_bwd_apply)
    against torch's F.relu + F.batch_norm(training=True) forward and autograd backward on the same tensors, at C = 32 and 128,
    alternating in this process, with the max differences of y, dz, dgamma, dbeta and the share of the measured HBM copy peak
    (6,499 GB/s) that the algorithmic bytes reach: forward 3 * 4NC (z read twice, y written), backward 5 * 4NC (z and g read
    twice, dz written).  z is 209 MB at C = 32, larger than the L2, so every pass comes from HBM.
  * step: a world-1 dist.sharded_forward training step (forward + nll loss + backward) of SNGNN_Plus_Plus (hidden 32,
    2 layers, top_k 10) on the pokec-shaped graph with bn=True against bn=False, alternating; with --world W (2 <= W <=
    the GPUs present) the same step on W ranks over NCCL, one process per GPU.

    python scripts/shard_bn_time.py [--reps 20] [--rounds 5] [--steps 5] [--world 2 4 8] [--rank-timeout S] [--out FILE]

Prints one JSON object (card name and power limit included).  Times are CUDA-event medians per call."""
import argparse
import json
import os
import socket
import subprocess
import sys
import time

import torch
import torch.nn.functional as F

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from sngnn_b200 import dist as D, functional as SF, synth  # noqa: E402

HBM_COPY_GBS = 6499.0            # measured device-to-device copy rate of the B200 the project quotes (DESIGN.md)
EPS = 1e-5


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


def kernels(n, c, reps, rounds):
    gen = torch.Generator(device="cuda").manual_seed(c)
    z = torch.randn(n, c, device="cuda", generator=gen) + 0.3
    g = torch.randn(n, c, device="cuda", generator=gen)
    gamma = torch.rand(c, device="cuda", generator=gen) + 0.5
    beta = torch.randn(c, device="cuda", generator=gen)
    state = {}

    def ours_fwd():
        sums = SF.bn_fwd_stats(z)
        state["y"], state["mean"], state["rstd"] = SF.bn_fwd_apply(z, sums, n, EPS, gamma, beta)

    def ours_bwd():
        state["bsums"] = SF.bn_bwd_stats(z, g, state["mean"], state["rstd"])
        state["dz"] = SF.bn_bwd_apply(z, g, state["bsums"], n, gamma, state["mean"], state["rstd"])

    zt, wt, bt = z.clone().requires_grad_(True), gamma.clone().requires_grad_(True), beta.clone().requires_grad_(True)

    def torch_fwd():
        state["ty"] = F.batch_norm(F.relu(zt), None, None, wt, bt, True, 0.1, EPS)

    def torch_bwd():
        state["tgrads"] = torch.autograd.grad(state["ty"], (zt, wt, bt), g, retain_graph=True)

    ours_fwd(); torch_fwd()
    t = time_alternating({"ours_fwd": ours_fwd, "torch_fwd": torch_fwd, "ours_bwd": ours_bwd, "torch_bwd": torch_bwd}, reps, rounds)
    dz_t, dw_t, db_t = state["tgrads"]
    diff = {"y": float((state["y"] - state["ty"]).abs().max()), "dz": float((state["dz"] - dz_t).abs().max()),
            "dgamma": float((state["bsums"][1].float() - dw_t).abs().max()), "dbeta": float((state["bsums"][0].float() - db_t).abs().max())}
    fwd_bytes, bwd_bytes = 3 * 4 * n * c, 5 * 4 * n * c
    res = {"C": c, "ms": {k: round(v, 4) for k, v in t.items()}, "max_abs_diff_vs_torch": diff,
           "bytes": {"fwd": fwd_bytes, "bwd": bwd_bytes},
           "floor_ms": {"fwd": round(fwd_bytes / HBM_COPY_GBS / 1e6, 4), "bwd": round(bwd_bytes / HBM_COPY_GBS / 1e6, 4)}}
    res["share_of_copy_peak"] = {"fwd": round(res["floor_ms"]["fwd"] / t["ours_fwd"], 3), "bwd": round(res["floor_ms"]["bwd"] / t["ours_bwd"], 3)}
    res["torch_share_of_copy_peak"] = {"fwd": round(res["floor_ms"]["fwd"] / t["torch_fwd"], 3),
                                       "bwd": round(res["floor_ms"]["bwd"] / t["torch_bwd"], 3)}
    return res


def make_step(dev, lo, hi, bn):
    import sngnn_b200.models as M
    N, Fd, E, C = synth.SHAPES["pokec"]
    x = synth.make_features(N, Fd, "clustered", seed=0, device=dev, zscore=True)
    ei = synth.make_graph(N, E, seed=1, device=dev, symmetric=True)
    y = synth.make_labels(N, C, seed=2, device=dev)
    torch.manual_seed(2)
    model = M.SNGNN_Plus_Plus(Fd, 32, C, N, 2, 10, 0.0, 0.5, 1, 0.0, bn=bn).to(dev).train()
    x_loc, y_loc = x[lo:hi].contiguous(), y[lo:hi]

    def step():
        model.zero_grad()
        (SF.nll_loss(D.sharded_forward(model, x_loc, ei, N), y_loc) * ((hi - lo) / N)).backward()
        D.allreduce_grads(model.parameters())
    return step


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _rank_worker(rank, ws, port, steps, ret):
    import torch.distributed as dist
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=ws, device_id=dev)
    lo, hi = D.shard_bounds(synth.SHAPES["pokec"][0], ws, rank)
    fns = {f"bn={bn}": make_step(dev, lo, hi, bn) for bn in (True, False)}
    for f in fns.values():
        f()
    per = {k: [] for k in fns}
    for _ in range(steps):
        for name, f in fns.items():
            dist.barrier()
            torch.cuda.synchronize()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            f()
            b.record()
            b.synchronize()
            t = torch.tensor([a.elapsed_time(b)], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)                 # a step lasts as long as its slowest rank
            per[name].append(float(t))
    if rank == 0:
        ret[ws] = {k: round(sorted(v)[len(v) // 2], 3) for k, v in per.items()}
    dist.barrier()
    dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--world", type=int, nargs="*", default=[2, 4, 8])
    ap.add_argument("--rank-timeout", type=float, default=600.0, help="seconds to wait for the ranks of one world size")
    ap.add_argument("--out")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("shard_bn_time.py measures on a CUDA device; there is none")
    n = synth.SHAPES["pokec"][0]
    res = {"card": card(), "N": n, "kernels": [kernels(n, c, args.reps, args.rounds) for c in (32, 128)]}
    torch.cuda.empty_cache()
    fns = {f"bn={bn}": make_step("cuda", 0, n, bn) for bn in (True, False)}
    step_ms = time_alternating(fns, 1, args.steps)
    res["step_world1_ms"] = {k: round(v, 3) for k, v in step_ms.items()}
    res["step_world1_bn_overhead_ms"] = round(step_ms["bn=True"] - step_ms["bn=False"], 3)
    del fns
    torch.cuda.empty_cache()
    gpus = torch.cuda.device_count()
    multi = {}
    for ws in args.world:
        if ws > gpus:
            multi[ws] = f"not measured ({gpus} GPU(s) on this box)"
            continue
        import torch.multiprocessing as mp
        ctx = mp.get_context("spawn")
        ret = ctx.Manager().dict()
        port = _free_port()
        procs = [ctx.Process(target=_rank_worker, args=(r, ws, port, args.steps, ret)) for r in range(ws)]
        for p in procs:
            p.start()
        deadline = time.monotonic() + args.rank_timeout
        for p in procs:                       # a rank that raised leaves the others waiting in a collective: bound the wait
            p.join(max(0.0, deadline - time.monotonic()))
        for p in procs:
            if p.is_alive():
                p.terminate()
                p.join(30)
                if p.is_alive():
                    p.kill()
                    p.join()
        multi[ws] = ret.get(ws, "failed (exit codes %s)" % [p.exitcode for p in procs])
    res["step_multi_gpu_ms"] = multi
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
