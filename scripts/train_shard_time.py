"""Counter-based row dropout and the row-sharded trainer at the pokec shape (N = 1,632,803), on the GPUs present.

  * kernels: sng_row_dropout_fwd (relu fused) and sng_row_dropout_bwd against torch's F.relu + F.dropout forward and its autograd
    backward on the same tensors, at C = 32 and 128, alternating in this process.  Byte floors: forward 8NC (z read, y written),
    backward 12NC (z and g read, dz written), over a device-to-device copy measured in the same run (the share of the copy peak).
    z is 209 MB at C = 32, larger than the 126 MB L2, so every pass comes from HBM.
  * epochs: `python -m sngnn_b200.train --dataset pokec --model SNGNN_Plus_Plus` (hidden 32, 2 layers, top_k 10, dropout 0.5) on
    one GPU without torchrun, and under torchrun at world 1 and at every GPU count given (default: 2, 4, 8 up to the GPUs present);
    the median epoch time after the first two epochs, from the trainer's own running-mean log.

    python scripts/train_shard_time.py [--reps 20] [--rounds 5] [--epochs 8] [--world 1 2 4 8] [--timeout S] [--out FILE]

Prints one JSON object (card name and power limit included); counts that were not run are recorded as "not measured"."""
import argparse
import json
import os
import re
import signal
import subprocess
import sys

import torch
import torch.nn.functional as F

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from sngnn_b200 import functional as SF  # noqa: E402

N = 1632803
P = 0.5


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    return {"device": torch.cuda.get_device_name(0), "nvidia_smi": q[0] if q else "unavailable", "gpus": torch.cuda.device_count()}


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


def copy_rate_gbs(reps, rounds):
    src = torch.empty(1 << 30, dtype=torch.uint8, device="cuda")
    dst = torch.empty_like(src)
    ms = time_alternating({"copy": lambda: dst.copy_(src)}, reps, rounds)["copy"]
    return 2 * src.numel() / (ms * 1e-3) / 1e9                      # read + write


def kernels(c, reps, rounds, copy_gbs):
    gen = torch.Generator(device="cuda").manual_seed(c)
    z = torch.randn(N, c, device="cuda", generator=gen)
    g = torch.randn(N, c, device="cuda", generator=gen)
    zt = z.clone().requires_grad_(True)
    yt = F.dropout(F.relu(zt), P, True)
    fns = {
        "ours_fwd": lambda: SF.row_dropout_fwd(z, 0, 7, 0, P, True),
        "ours_bwd": lambda: SF.row_dropout_bwd(z, g, 0, 7, 0, P, True),
        "torch_fwd": lambda: F.dropout(F.relu(z), P, True),
        "torch_bwd": lambda: torch.autograd.grad(yt, zt, g, retain_graph=True),
    }
    ms = time_alternating(fns, reps, rounds)
    floors = {"fwd": 8 * N * c, "bwd": 12 * N * c}
    out = {"C": c, "ms": {k: round(v, 4) for k, v in ms.items()}, "floor_bytes": floors}
    for d in ("fwd", "bwd"):
        gbs = floors[d] / (ms["ours_" + d] * 1e-3) / 1e9
        out[f"ours_{d}_GBs"] = round(gbs, 1)
        out[f"ours_{d}_share_of_copy_peak"] = round(gbs / copy_gbs, 3)
        out[f"speedup_{d}_vs_torch"] = round(ms["torch_" + d] / ms["ours_" + d], 2)
    return out


TRAIN_ARGS = ("--dataset pokec --model SNGNN_Plus_Plus --num_layers 2 --hidden_channels 32 --top_k 10 --thr 0.0 --init_beta 0.5 "
              "--dropout 0.5 --patience 1000 --log-every 1").split()


def epoch_ms(cmd, env, timeout):
    """Median epoch time (ms) after the first two epochs, from the running means of the `Time(s)` log lines; None on failure."""
    p = subprocess.Popen(cmd, env=env, cwd=ROOT, start_new_session=True, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    try:
        out, _ = p.communicate(timeout=timeout)
    except subprocess.TimeoutExpired:
        out = None
    finally:
        for sig in (signal.SIGTERM, signal.SIGKILL):                 # leave no rank behind
            try:
                os.killpg(p.pid, sig)
            except ProcessLookupError:
                break
            try:
                p.wait(20)
            except subprocess.TimeoutExpired:
                pass
    if out is None or p.returncode != 0:
        return None, (out or "timeout")[-2000:]
    means = [float(m) for m in re.findall(r"Time\(s\): ([0-9.]+)", out)]
    per = [means[0]] + [(k + 1) * means[k] - k * means[k - 1] for k in range(1, len(means))]
    steady = sorted(per[2:]) or per
    return round(1e3 * steady[len(steady) // 2], 1), out.strip().splitlines()[-1]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--epochs", type=int, default=8)
    ap.add_argument("--world", type=int, nargs="*", default=None)
    ap.add_argument("--timeout", type=float, default=900.0)
    ap.add_argument("--out", type=str, default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("train_shard_time.py measures on a CUDA device; none is present")
    res = {"card": card(), "N": N, "p": P}
    copy_gbs = copy_rate_gbs(a.reps, a.rounds)
    res["copy_GBs"] = round(copy_gbs, 1)
    res["kernels"] = [kernels(c, a.reps, a.rounds, copy_gbs) for c in (32, 128)]
    torch.cuda.empty_cache()
    ngpu = torch.cuda.device_count()
    worlds = a.world if a.world is not None else [1] + [w for w in (2, 4, 8) if w <= ngpu]
    args = TRAIN_ARGS + ["--epochs", str(a.epochs)]
    env = {k: v for k, v in os.environ.items() if k not in ("WORLD_SIZE", "RANK", "LOCAL_RANK", "MASTER_ADDR", "MASTER_PORT")}
    env["PYTHONPATH"] = ROOT + os.pathsep + env.get("PYTHONPATH", "")
    epochs = {}
    ms, last = epoch_ms([sys.executable, "-m", "sngnn_b200.train"] + args, env, a.timeout)
    epochs["single_gpu"] = {"epoch_ms": ms if ms is not None else "not measured", "last_line": last}
    for w in (1, 2, 4, 8):
        if w not in worlds or w > ngpu:
            epochs[f"torchrun_{w}"] = "not measured"
            continue
        cmd = [sys.executable, "-m", "torch.distributed.run", "--standalone", f"--nproc-per-node={w}", "-m", "sngnn_b200.train"] + args
        ms, last = epoch_ms(cmd, env, a.timeout)
        epochs[f"torchrun_{w}"] = {"epoch_ms": ms if ms is not None else "not measured", "last_line": last}
    res["epochs"] = epochs
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
