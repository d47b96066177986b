#!/usr/bin/env python
"""Headline benchmark of the similarity-navigated aggregation hot path (BASELINE.json).

    python bench.py --gpus N --steps K --warmup W            # ours (torchrun launches N>1)
    python bench.py --impl reference --gpus N --steps K ...  # the reference's CPU path (oracle port), rank 0 only
    python bench.py ... --dump-outputs DIR                   # + the last timed step's neighbour lists, sampled rows, as .npy

One step = one all-pairs similarity-kNN build (K0 normalise -> [all-gather of x-hat at N>1] -> K1 tensor-core
stage + FP32 rescore + exact fallback) of the pokec-shaped synthetic feature matrix (1,632,803 x 65, top_k=10),
query rows sharded across ranks (strong scaling: the graph is fixed, SURVEY.md §8(e)).
`value` = ordered pairs / s = N*N / max-over-ranks device time, inputs resident in HBM.
`e2e`   = the same through the public API from pinned HOST features to HOST neighbour lists (copies timed by their own events).
Also in the line (same run, separately timed, not part of `value`):
  `configs`      the other BASELINE.json configurations -- build Gpairs/s + roofline fraction + index parity on sampled rows for
                 the arxiv-year / snap-patents shapes, three corners of the sweep grid and the headline shape with iid-normal
                 features; model epochs (GPU ms, oracle CPU ms, logits / gradient parity) for the Chameleon and arxiv shapes
  `epoch_ms` ... the SNGNN++ epoch on the pokec-shaped graph (row-sharded at N>1, with `parity_epoch` = sharded vs unsharded)
  `agg`          the fused aggregation kernels alone (GB/s against the HBM roofline) + their parity on sampled rows
`roofline` is for the tensor-core kernel of the headline build.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

METRIC = "simknn_build_gpairs_per_s"
UNIT = "Gpairs/s"


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="pokec", help="shape name from sngnn_b200.synth.SHAPES")
    ap.add_argument("--top_k", type=int, default=10)
    ap.add_argument("--thr", type=float, default=0.0)
    ap.add_argument("--features", default="clustered", choices=["clustered", "normal"])
    ap.add_argument("--skip-epoch", action="store_true", help="only the kNN build (used under ncu)")
    ap.add_argument("--skip-cpu", action="store_true")
    ap.add_argument("--skip-configs", action="store_true", help="only the headline shape")
    ap.add_argument("--cpu-rows", type=int, default=2048, help="query-row slab of the CPU baseline sample")
    ap.add_argument("--parity-rows", type=int, default=4096, help="sampled query rows of the headline parity gate")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the neighbour lists of the last timed step of the headline build "
                                                          "(a fixed sample of query rows) to DIR/{rows,idx,sim,cnt}.npy")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    return args


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm=d["hbm_gbs"], tf_burst=d["bf16_tflops"], tf_sust=d["bf16_tflops_sustained"], src="measured")
    return dict(hbm=6650.0, tf_burst=1590.0, tf_sust=1400.0, src="fallback")


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "200",
                                          "-i", str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.proc.terminate()
        sm = sorted(int(float(r[1])) for r in self.rows if len(r) >= 8 and r[1].replace(".", "").isdigit())
        mx = [int(float(r[2])) for r in self.rows if len(r) >= 8 and r[2].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[i] for r in self.rows if len(r) >= 8 for i in range(4) if r[4 + i].lower().startswith("active")})
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons,
                "samples": len(sm)}


# ------------------------------------------------------------------------------------------- reference arm
def cpu_knn_sample(x, rows, top_k, thr, block=1000):
    """The reference's CPU path for this metric: blocked x-hat @ x-hat^T in 1000-row blocks
    (R: SimGFAToolbox/dense.py:17-27) + the selection rule, as restated in oracle/sn_ref.py."""
    from oracle import sn_ref
    t0 = time.perf_counter()
    sn_ref.simknn_allpairs(x, top_k, thr, True, 0, rows, block=block)
    return time.perf_counter() - t0


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from sngnn_b200 import synth
    torch.set_num_threads(os.cpu_count() or 1)       # torchrun pins OMP_NUM_THREADS=1; the reference arm uses every host core
    N, Fd, E, C = synth.SHAPES[args.workload]
    x = synth.make_features(N, Fd, args.features, seed=0, zscore=(args.workload == "pokec"))
    rows = min(args.cpu_rows // 4 if args.cpu_rows >= 2048 else args.cpu_rows, N)      # bounded sample per step
    for _ in range(args.warmup):
        cpu_knn_sample(x, min(rows, 256), args.top_k, args.thr)
    ts = [cpu_knn_sample(x, rows, args.top_k, args.thr) for _ in range(args.steps)]
    t = sum(ts) / len(ts)
    val = rows * N / t / 1e9
    sample = f"{rows} query rows x all {N} columns per step (blocked torch.mm + stable sort, float32)"
    line = {"impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": t * 1e3, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": {"workload": f"{args.workload}-shape all-pairs kNN build N={N} d={Fd} top_k={args.top_k} thr={args.thr}",
                       "features": args.features, "sample": sample},
            "cpu_baseline": {"value": val, "unit": UNIT, "cores": torch.get_num_threads(), "kind": "port", "sample": sample},
            "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    emit(line)


# ------------------------------------------------------------------------------------------------- our arm
def ev():
    return torch.cuda.Event(enable_timing=True)


def timed(fn, steps, warmup, sync_all=None):
    for _ in range(warmup):
        fn()
    if sync_all:
        sync_all()
    torch.cuda.synchronize()
    a, b = ev(), ev()
    a.record()
    for _ in range(steps):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / steps          # ms per call


class Ctx:
    """Process-wide bench state: ranks, device, collectives."""

    def __init__(self):
        import torch.distributed as dist
        self.dist = dist
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.rank = int(os.environ.get("RANK", "0"))
        self.local = int(os.environ.get("LOCAL_RANK", "0"))
        torch.cuda.set_device(self.local)
        self.dev = torch.device("cuda", self.local)
        if self.world > 1:
            dist.init_process_group("nccl", device_id=self.dev)

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()

    def max_over_ranks(self, *vals):
        t = torch.tensor(list(vals), device=self.dev, dtype=torch.float64)
        if self.world > 1:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return [float(v) for v in t]

    def bounds(self, n):
        r = (n + self.world - 1) // self.world
        return r, min(n, self.rank * r), min(n, (self.rank + 1) * r)


def sample_rows(n, world, count, seed=7):
    """Query rows of a parity gate: the first rows, the last (partial) 256-row tile, both ends of every rank's shard, and a
    uniform sample of the rest -- about `count` distinct rows in all (not 'the first 256')."""
    r = (n + world - 1) // world
    fixed = list(range(min(8, n))) + list(range(max(0, n - 200), n))
    for k in range(world):
        lo, hi = min(n, k * r), min(n, (k + 1) * r)
        fixed += [v for v in (lo, lo + 1, hi - 2, hi - 1) if 0 <= v < n]
    g = torch.Generator().manual_seed(seed)
    rest = torch.randint(0, n, (max(count - len(set(fixed)), 0),), generator=g).tolist()
    return torch.tensor(sorted(set(fixed + rest)), dtype=torch.long)


def rows_of_shards(cx, rows, lo, hi, *shards):
    """Global query rows `rows` of tensors whose rows [lo, hi) this rank holds: every rank contributes the rows of its
    shard and every rank receives all of them (integers padded with -2, floats with -inf, combined by MAX)."""
    mine = (rows >= lo) & (rows < hi)
    sel = (rows[mine] - lo).to(cx.dev)
    out = []
    for t in shards:
        fill = float("-inf") if t.is_floating_point() else -2
        got = torch.full((rows.numel(),) + tuple(t.shape[1:]), fill, dtype=t.dtype, device=cx.dev)
        got[mine.to(cx.dev)] = t[sel]
        if cx.world > 1:
            cx.dist.all_reduce(got, op=cx.dist.ReduceOp.MAX)
        out.append(got)
    return out


def knn_parity(cx, x, idx, cnt, lo, hi, k, thr, count, n_fallback, n_retry):
    """Index parity of a (sharded) build on sampled rows: every rank contributes the sampled rows of its shard, rank 0
    compares with the FP64 oracle (exact / in-band (FP64 gap < 1e-6) / out-of-band, which must be 0)."""
    n = x.size(0)
    rows = sample_rows(n, cx.world, count)
    got_i, got_c = rows_of_shards(cx, rows, lo, hi, idx, cnt)
    fb = torch.tensor([n_fallback, n_retry], device=cx.dev, dtype=torch.int64)
    if cx.world > 1:
        cx.dist.all_reduce(fb, op=cx.dist.ReduceOp.SUM)
    if cx.rank != 0:
        return None
    from oracle import sn_ref
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from parity import compare_lists
    torch.set_num_threads(os.cpu_count() or 1)
    xc = x.cpu()
    n64 = sn_ref.rownorm(xc.double())
    iref, _, cref = sn_ref.simknn_rows(xc, rows, k, thr, True, block=max(16, min(256, (1 << 28) // n)), normalized=n64)
    res = compare_lists(got_i, got_c, iref, cref, lambda r, j: (n64[rows[r]] * n64[j]).sum(-1), thr)
    res.update(rows_checked=int(rows.numel()), rows_span=[int(rows.min()), int(rows.max())], shards_covered=cx.world,
               fallback_rows=int(fb[0]), retry_rows=int(fb[1]))
    return res


DUMP_BYTES = 48 << 20


def dump_outputs(cx, out_dir, n, lo, hi, idx, sim, cnt):
    """The neighbour lists one build step returns (idx -1 padded, sim 0 padded, cnt), on a fixed sample of query rows that
    depends only on n, so that runs on any number of GPUs and two builds of the library can be compared file for file:
    rows / idx / cnt as float64 (exact integers), sim as float32, at most DUMP_BYTES in all."""
    import numpy as np
    k = idx.size(1)
    rows = sample_rows(n, 1, min(n, 1 << 18, DUMP_BYTES // (12 * k + 16)), seed=13)
    got_i, got_s, got_c = rows_of_shards(cx, rows, lo, hi, idx, sim, cnt)
    if cx.rank != 0:
        return
    os.makedirs(out_dir, exist_ok=True)
    for name, t, dt in (("rows", rows, np.float64), ("idx", got_i, np.float64), ("sim", got_s, np.float32), ("cnt", got_c, np.float64)):
        np.save(os.path.join(out_dir, name + ".npy"), t.cpu().numpy().astype(dt))


def build_case(cx, pk, n, d, k, thr, features, steps, warmup, parity_rows, zscore=False, e2e=False, kernel_alone=False, cpu_rows=0,
               phases=True, dump_dir=None):
    """One all-pairs similarity-kNN build configuration: timing (max over ranks), optional end-to-end timing from pinned host
    memory, the tensor-core main pass alone (roofline), index parity on sampled rows."""
    import ctypes
    from sngnn_b200 import _C, simknn, synth
    dev, world = cx.dev, cx.world
    x = synth.make_features(n, d, features, seed=0, device=dev, zscore=zscore)
    R, lo, hi = cx.bounds(n)
    nq = hi - lo
    ld32, ldh = simknn._pad_to(d, 4), simknn._pad_to(d, 16)
    xf_all = xh_all = xf_pad = None
    if world > 1:
        xf_all = torch.zeros(world * R, ld32, dtype=torch.float32, device=dev)
        xh_all = torch.zeros(world * R, ldh, dtype=torch.float16, device=dev)
        xf_pad = torch.zeros(R, ld32, dtype=torch.float32, device=dev)

    def normalise_and_gather(x_shard):
        xf, xh = simknn.normalize_operands(x_shard)
        if world == 1:
            return xf, xh
        xf_pad[:nq].copy_(xf)
        cx.dist.all_gather_into_tensor(xf_all, xf_pad)       # NCCL over NVLink; FP32 x-hat is the only exchanged data
        xh_all[:, :ld32].copy_(xf_all)                         # the FP16 tensor-core operand is converted locally (bit-identical to K0's)
        return xf_all[:n], xh_all[:n]

    out = {}

    def step_resident():
        xf, xh = normalise_and_gather(x[lo:hi])
        out["r"] = simknn.build_knn_normalized(xf, xh, d, k, thr, True, lo, hi, return_fallback=True)

    cx.barrier()
    ms = timed(step_resident, steps, warmup, cx.barrier)
    if dump_dir:
        dump_outputs(cx, dump_dir, n, lo, hi, *out["r"][:3])
    res = {"n": n, "d": d, "top_k": k, "thr": thr, "features": features, "steps": steps, "warmup": warmup}
    ms_e2e = None
    if e2e:
        # end-to-end: pinned host features -> device -> ... -> host neighbour lists; the copies are timed by their own events
        x_host = x[lo:hi].cpu().pin_memory()
        idx_host = torch.empty(nq, k, dtype=torch.int32).pin_memory()
        sim_host = torch.empty(nq, k, dtype=torch.float32).pin_memory()
        cnt_host = torch.empty(nq, dtype=torch.int32).pin_memory()
        x_stage = torch.empty_like(x[lo:hi])
        evs = []

        def step_e2e():
            e0, e1, e2, e3 = ev(), ev(), ev(), ev()
            e0.record()
            x_stage.copy_(x_host, non_blocking=True)
            e1.record()
            xf, xh = normalise_and_gather(x_stage)
            idx, sim, cnt = simknn.build_knn_normalized(xf, xh, d, k, thr, True, lo, hi)
            e2.record()
            idx_host.copy_(idx, non_blocking=True)
            sim_host.copy_(sim, non_blocking=True)
            cnt_host.copy_(cnt, non_blocking=True)
            e3.record()
            evs.append((e0, e1, e2, e3))

        ms_e2e = timed(step_e2e, steps, max(1, warmup - 2), cx.barrier)
        last = evs[-steps:]
        res["e2e_copy_ms"] = {"h2d": sum(a.elapsed_time(b) for a, b, _, _ in last) / len(last),
                              "d2h": sum(c.elapsed_time(e) for _, _, c, e in last) / len(last)}
        res["h2d_bytes"] = x_host.numel() * 4
        res["d2h_bytes"] = idx_host.numel() * 4 + sim_host.numel() * 4 + cnt_host.numel() * 4
        del x_host, idx_host, sim_host, cnt_host, x_stage, evs
    ph = {}

    def phase_a():
        ph["ops"] = normalise_and_gather(x[lo:hi])

    def phase_b():
        xf_, xh_ = ph["ops"]
        simknn.build_knn_normalized(xf_, xh_, d, k, thr, True, lo, hi)

    ms_gather = timed(phase_a, 2 if phases else 1, 1 if phases else 0, cx.barrier)
    ms_build = timed(phase_b, 2, 1, cx.barrier) if phases else 0.0
    ms, ms_gather, ms_build = cx.max_over_ranks(ms, ms_gather, ms_build)
    if ms_e2e is not None:
        ms_e2e = cx.max_over_ranks(ms_e2e)[0]
    idx, sim, cnt, nfb = out["r"]
    plan = simknn.build_plan(nq, n, d, k)
    res.update(ms_per_step=ms, gpairs_per_s=float(n) * float(n) / (ms * 1e-3) / 1e9, ms_e2e=ms_e2e, plan=plan,
               phase_ms={"normalise_and_allgather": ms_gather, "build_call": ms_build})
    # ---- the dominant kernel alone: tensor-core main pass on this rank's rows, launched exactly as the build launches it
    xf, xh = ph["ops"]
    ew, cand = plan["ew"], plan["cand"]
    ci = torch.empty(nq * 192, dtype=torch.int32, device=dev)      # lists * cand <= 192 slots per row
    cv = torch.empty(nq * 192, dtype=torch.float32, device=dev)
    cm = torch.empty(nq * 64, dtype=torch.float32, device=dev)
    ns = ctypes.c_int(0)
    thr_lo = thr - 1.01 * (2.0 ** -10 + 1.2e-4)
    seeds, ms_seed = None, 0.0
    if plan["seed_stride"] > 0:
        seeds = simknn.seed_pass(xh[lo:hi], xh, d, plan["seed_stride"], ew)
        if kernel_alone:
            ms_seed = timed(lambda: simknn.seed_pass(xh[lo:hi], xh, d, plan["seed_stride"], ew), 2, 1)
    sweep_phase = torch.zeros(8, dtype=torch.int32, device=dev)

    def stage1_only():
        sweep_phase.zero_()
        _C.call("sng_simknn_stage1", xh, _C.ptr(xh[lo:]), _C.ptr(xh), ldh, nq, lo, n, d, cand, thr_lo, 1, _C.ptr(ci), _C.ptr(cv),
                _C.ptr(cm), ew, plan["nsplit"], ctypes.byref(ns), _C.ptr(seeds), plan["seed_q"], plan["seed_stride"], _C.ptr(sweep_phase))

    ms_k1 = timed(stage1_only, 2 if phases else 1, 1)
    flops = 2.0 * nq * n * d
    achieved_tf = flops / (ms_k1 * 1e-3) / 1e12
    res["roofline"] = {"bound": "tensor", "kernel": "simknn_stage1_kernel<%d,false> (main pass)" % ew, "achieved": achieved_tf,
                       "peak": pk["tf_sust"], "unit": "TFLOP/s", "frac": achieved_tf / pk["tf_sust"], "frac_of_burst_peak": achieved_tf / pk["tf_burst"],
                       "kernel_ms": ms_k1,
                       "algorithmic_flops_per_launch": flops, "share_of_step": ms_k1 / ms, "seed_pass_ms": ms_seed}
    del ci, cv, cm, seeds
    res["parity"] = knn_parity(cx, x, idx, cnt, lo, hi, k, thr, parity_rows, int(nfb[0]), int(nfb[1]))
    if cpu_rows and cx.rank == 0 and world == 1:
        torch.set_num_threads(os.cpu_count() or 1)
        xc = x.cpu()
        cpu_knn_sample(xc, 128, k, thr)
        tc = cpu_knn_sample(xc, min(cpu_rows, n), k, thr)
        res["cpu"] = {"value": min(cpu_rows, n) * n / tc / 1e9, "unit": UNIT, "cores": torch.get_num_threads(), "kind": "port",
                      "sample": f"{min(cpu_rows, n)} query rows x all {n} columns, blocked torch.mm (1000-row blocks) + stable sort, float32, {tc:.1f} s"}
    del x, out, ph, xf, xh, idx, sim, cnt
    torch.cuda.empty_cache()
    return res


def oracle_epoch(kind, sd, layers, x, ei, y, k, thr, rsl, lr=0.01, wd=5e-4):
    """The reference's epoch on the host cores (R: train.py:136-138 = train step + 2 evaluation forwards) through the
    oracle restatement of models.py; returns seconds per epoch."""
    import torch.nn.functional as F
    from oracle import sn_ref
    torch.set_num_threads(os.cpu_count() or 1)
    params = {kk: v.detach().cpu().clone().contiguous().requires_grad_(v.is_floating_point()) for kk, v in sd.items()}
    opt = torch.optim.Adam([p for p in params.values() if p.requires_grad], lr=lr, weight_decay=wd)
    t0 = time.perf_counter()
    opt.zero_grad()
    out = sn_ref.stack_forward(kind, sn_ref.params_from_state_dict(params, layers), x, ei, top_k=k, thr=thr, remove_self_loops=rsl)
    F.nll_loss(out, y).backward()
    opt.step()
    with torch.no_grad():
        for _ in range(2):
            sn_ref.stack_forward(kind, sn_ref.params_from_state_dict(params, layers), x, ei, top_k=k, thr=thr, remove_self_loops=rsl)
    return time.perf_counter() - t0


def model_parity(kind, sd, layers, x, ei, y, k, thr, rsl, lists, logits, grads):
    """The two halves of the parity contract for one train step of a model (SURVEY.md §8(d)):
    (a) every layer's selection lists against the reference rule evaluated in FP64 on the layer's input (exact / in band --
        the FP64 scores involved within 1e-6 -- / out of band, which must be 0);
    (b) with the selection GIVEN, logits and every parameter gradient against the oracle within 1e-5.
    On tie-dense inputs (a 5-class output layer puts 10^5 cosines within 1e-5 of 1) two correct FP32 implementations
    legitimately choose different k-th neighbours, so a single end-to-end 1e-5 comparison would test luck, not correctness."""
    import torch.nn.functional as F
    from oracle import sn_ref
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from parity import compare_lists
    torch.set_num_threads(os.cpu_count() or 1)
    N = x.size(0)
    forced = [(a.cpu().long(), b.cpu().long()) for a, b in lists]
    params = {kk: v.detach().cpu().clone().contiguous().requires_grad_(v.is_floating_point()) for kk, v in sd.items()}
    inputs = []
    out = sn_ref.stack_forward(kind, sn_ref.params_from_state_dict(params, layers), x, ei, top_k=k, thr=thr, remove_self_loops=rsl,
                               forced=forced, layer_inputs=inputs)
    F.nll_loss(out, y).backward()
    lerr = float((logits - out.detach()).abs().max() / (out.detach().abs().max() + 1e-12))
    gerr = max(float((grads[kk] - p.grad).abs().max() / (p.grad.abs().max() + 1e-12)) for kk, p in params.items() if p.grad is not None)
    pe = sn_ref.process_edges(ei, N, rsl)
    sel = []
    for l, xin in enumerate(inputs):
        h64 = F.linear(xin.double(), params[f"lins.{l}.lin.weight"].detach().double(), params[f"lins.{l}.lin.bias"].detach().double())
        n64 = F.normalize(h64, dim=-1, eps=1e-12)
        s64 = (n64[pe[1]] * n64[pe[0]]).sum(-1)
        rank = sn_ref.edge_rank(s64, pe[1])
        m = (rank < k) & (s64 >= thr)
        iref = torch.full((N, k), -1, dtype=torch.long)
        iref[pe[1][m], rank[m]] = pe[0][m]
        cref = torch.zeros(N, dtype=torch.long).index_add(0, pe[1][m], torch.ones(int(m.sum()), dtype=torch.long))
        r = compare_lists(forced[l][0], forced[l][1], iref, cref, lambda rr, jj: (n64[rr] * n64[jj]).sum(-1), thr)
        sel.append({"layer": l, "exact": r["exact"], "in_band": r["in_band"], "out_of_band": r["out_of_band"]})
    ok = lerr < 1e-5 and gerr < 1e-5 and all(v["out_of_band"] == 0 for v in sel)
    return {"selection_vs_fp64_rule": sel, "given_selection": {"max_rel_logit_err": lerr, "max_rel_grad_err": gerr, "tolerance": 1e-5},
            "ok": bool(ok), "against": "oracle (CPU restatement of R models.py), first train step"}


def model_case(cx, name, kind, layers, hid, k, thr, beta, feature_kind):
    """One model configuration on ONE GPU: GPU epoch ms, the oracle's CPU epoch, selection / logits / gradient parity of a train step."""
    import torch.nn.functional as F
    from sngnn_b200 import synth
    import sngnn_b200.models as M
    import sngnn_b200.functional as SF
    dev = cx.dev
    N, Fd, E, C = synth.SHAPES[name]
    x = synth.make_features(N, Fd, feature_kind, seed=0)
    ei = synth.make_graph(N, E, seed=1, symmetric=True)
    y = synth.make_labels(N, C, seed=2)
    torch.manual_seed(2)
    if kind == "SNGNN_Plus_Plus":
        model = M.SNGNN_Plus_Plus(Fd, hid, C, N, layers, k, thr, beta, 1, 0.0)
    else:
        model = M.SNGNN_Plus(Fd, hid, C, N, layers, k, thr, 1, 0.0)
    sd0 = {kk: v.detach().clone() for kk, v in model.state_dict().items()}
    model = model.to(dev)
    data = synth.GraphData(x, ei).to(dev)
    yd = y.to(dev)
    opt = torch.optim.Adam(model.parameters(), lr=0.01, weight_decay=5e-4, fused=True)
    model.train()
    SF.record_selection = []
    out = model(data)
    lists, SF.record_selection = SF.record_selection, None
    F.nll_loss(out, yd).backward()
    logits = out.detach().cpu()
    grads = {kk: p.grad.detach().cpu().clone() for kk, p in model.named_parameters()}

    def epoch():
        model.train()
        opt.zero_grad()
        SF.nll_loss(model(data), yd).backward()
        opt.step()
        model.eval()
        with torch.no_grad():
            model(data)
            model(data)

    ep_ms = timed(epoch, 5, 2)
    cpu_s = oracle_epoch(kind, sd0, layers, x, ei, y, k, thr, True) if cx.world == 1 else float("nan")   # host baseline: N = 1 only
    parity = model_parity(kind, sd0, layers, x, ei, y, k, thr, True, lists, logits, grads)
    del model, data
    torch.cuda.empty_cache()
    return {"model": kind, "shape": name, "nodes": N, "features": Fd, "edges": E, "layers": layers, "hidden": hid, "top_k": k, "thr": thr,
            "epoch_ms_gpu": ep_ms, "epoch_ms_cpu_oracle": None if cpu_s != cpu_s else cpu_s * 1e3, "cpu_cores": torch.get_num_threads(), "parity": parity}


def agg_parity(g, h, out, sel_src, sel_cnt, k, thr, fuse, out_fused, count=4096):
    """The fused aggregation kernels on sampled target rows of the pokec-shaped graph against the FP64 oracle restricted to
    the in-edges of those rows (selection lists exact or in band, outputs within 1e-5)."""
    from oracle import sn_ref
    n = g.n
    rows = sample_rows(n, 1, count, seed=11)
    deg = (g.rowptr_in[1:] - g.rowptr_in[:-1]).cpu()
    rows = torch.unique(torch.cat([rows, deg.topk(4).indices.long()]))          # + the four largest hubs
    h64, rp, col = h.double().cpu(), g.rowptr_in.cpu(), g.col_in.cpu()
    ref, lists = sn_ref.sn_aggregate_rows(h64, rp, col, rows, k, thr)
    got = out[rows.to(out.device)].double().cpu()
    err = float((got - ref).abs().max() / (ref.abs().max() + 1e-12))
    n64 = torch.nn.functional.normalize(h64, dim=-1, eps=1e-12)
    exact = in_band = bad = 0
    ss, sc = sel_src.cpu(), sel_cnt.cpu()
    for r, want in zip(rows.tolist(), lists):
        have = ss[r, : int(sc[r])].tolist()
        if have == want:
            exact += 1
            continue
        m = min(len(have), len(want))
        sa = (n64[r] * n64[torch.tensor(have, dtype=torch.long)]).sum(-1) if have else torch.zeros(0, dtype=torch.float64)
        sb = (n64[r] * n64[torch.tensor(want, dtype=torch.long)]).sum(-1) if want else torch.zeros(0, dtype=torch.float64)
        ok = (m == 0 or float((sa[:m] - sb[:m]).abs().max()) < 1e-6) and all(abs(float(v) - thr) < 1e-6 for v in list(sa[m:]) + list(sb[m:]))
        in_band += ok
        bad += not ok
    res = {"rows_checked": int(rows.numel()), "max_degree_checked": int(deg[rows].max()), "exact": exact, "in_band": in_band,
           "out_of_band": bad, "max_rel_out_err": err}
    if fuse is not None:
        wt, bw, beta, _ = fuse
        ref_f, _ = sn_ref.sn_aggregate_rows(h64, rp, col, rows, k, thr, wt.double().cpu(), bw.double().cpu(), float(beta))
        gotf = out_fused[rows.to(out_fused.device)].double().cpu()
        res["max_rel_fused_out_err"] = float((gotf - ref_f).abs().max() / (ref_f.abs().max() + 1e-12))
    res["ok"] = bool(bad == 0 and err < 1e-5 and res.get("max_rel_fused_out_err", 0.0) < 1e-5)
    return res


def run_ours(args):
    from sngnn_b200 import _C, synth
    import sngnn_b200.models as M
    import sngnn_b200.functional as SF
    from sngnn_b200 import graph as G
    import torch.nn.functional as F

    cx = Ctx()
    world, rank, dev = cx.world, cx.rank, cx.dev
    _C.lib()                                     # fail loudly if libsng.so is missing
    pk = peaks()
    N, Fd, E, C = synth.SHAPES[args.workload]
    k, thr = args.top_k, args.thr

    sampler = ClockSampler(cx.local)
    if rank == 0:
        sampler.start()
    head = build_case(cx, pk, N, Fd, k, thr, args.features, args.steps, args.warmup, args.parity_rows, zscore=(args.workload == "pokec"),
                      e2e=True, kernel_alone=True, cpu_rows=0 if args.skip_cpu else args.cpu_rows, dump_dir=args.dump_outputs)
    clocks = sampler.stop() if rank == 0 else None

    # ---- the other BASELINE.json configurations (build) --------------------------------------------------------
    configs = {}
    if not args.skip_configs:
        cases = [("arxiv-year_shape", dict(n=169343, d=128, k=10, features="clustered")),
                 ("snap-patents_shape", dict(n=2923922, d=269, k=10, features="clustered")),
                 ("sweep_N4M_d64_k5", dict(n=4000000, d=64, k=5, features="clustered")),
                 ("sweep_N1M_d256_k20", dict(n=1000000, d=256, k=20, features="clustered")),
                 # the clustered generator at d = 512 puts the ~390 members of a cluster within 4e-3 of each other -- inside the FP16
                 # scoring error -- so two thirds of the rows fail the first proof and go through the retry pass (192 slots per row)
                 ("sweep_N400k_d512_k50", dict(n=400000, d=512, k=50, features="clustered")),
                 ("sweep_N400k_d512_k50_iid_normal", dict(n=400000, d=512, k=50, features="normal")),
                 (f"{args.workload}_shape_iid_normal", dict(n=N, d=Fd, k=k, features="normal"))]
        for name, c in cases:
            try:
                r = build_case(cx, pk, c["n"], c["d"], c["k"], thr, c["features"], 2, 1, 512, zscore=name.startswith("pokec"), phases=False)
                configs[name] = {"n": r["n"], "d": r["d"], "top_k": r["top_k"], "features": r["features"], "n_gpus": world,
                                 "ms_per_step": r["ms_per_step"], "gpairs_per_s": r["gpairs_per_s"],
                                 "main_pass_frac_of_tensor_peak": r["roofline"]["frac"], "main_pass_ms": r["roofline"]["kernel_ms"],
                                 # the denominator is the SUSTAINED library-GEMM rate under this pod's power cap (a kernel that runs for
                                 # seconds); a value above 1 means this kernel sustains more than that GEMM does -- the burst figure bounds both
                                 "main_pass_frac_of_burst_peak": r["roofline"]["frac_of_burst_peak"],
                                 "phase_ms": r["phase_ms"], "plan": r["plan"], "parity": r["parity"]}
            except Exception as exc:                       # a failing side configuration must not cost the headline line
                configs[name] = {"error": f"{type(exc).__name__}: {exc}"[:300]}
                torch.cuda.empty_cache()

    # ---- SNGNN++ epoch (row-sharded at N>1) + aggregation kernels alone on the pokec-shaped graph ----------------
    extras = {}
    if not args.skip_epoch:
        from sngnn_b200 import dist as D
        torch.cuda.empty_cache()
        x = synth.make_features(N, Fd, args.features, seed=0, device=dev, zscore=(args.workload == "pokec"))
        ei = synth.make_graph(N, E, seed=1, device=dev, symmetric=True)
        y = synth.make_labels(N, C, seed=2, device=dev)
        R, lo, hi = cx.bounds(N)
        prep = []
        for _ in range(3):                                    # first call pays cudaMalloc of the sort workspace; report the warm one
            G.clear_cache()
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            g = G.prepare(ei, N, True)
            torch.cuda.synchronize()
            prep.append((time.perf_counter() - t0) * 1e3)
        prep_ms = min(prep)
        Ep = g.num_edges
        hid = 32
        torch.manual_seed(2)
        model = M.SNGNN_Plus_Plus(Fd, hid, C, N, 2, k, thr, 0.5, 1, 0.0 if world > 1 else 0.5).to(dev)
        opt = torch.optim.Adam(model.parameters(), lr=0.01, weight_decay=5e-4, fused=True)      # one launch instead of ~30 foreach kernels
        data = synth.GraphData(x, ei)
        x_loc, y_loc = x[lo:hi].contiguous(), y[lo:hi]

        def forward():                                        # world > 1: row-sharded forward (replicated parameters)
            if world == 1:
                return model(data)
            return D.sharded_forward(model, x_loc, ei, N)

        def loss_of(out):                                     # R: train.py:81, through the library's one-pass nll kernels
            return SF.nll_loss(out, y) if world == 1 else SF.nll_loss(out, y_loc) * ((hi - lo) / N)

        def train_step():                                     # fwd + loss + bwd + Adam (SURVEY.md §8(d)(iii))
            model.train()
            opt.zero_grad()
            loss_of(forward()).backward()
            D.allreduce_grads(model.parameters())
            opt.step()

        def epoch():                                          # R: train.py:136-138 = train step + val + test forwards
            train_step()
            model.eval()
            with torch.no_grad():
                forward()
                forward()

        def fwd_only():
            model.eval()
            with torch.no_grad():
                forward()

        # parity of the sharded step against the unsharded CUDA model (same parameters), before any optimizer step
        parity_epoch = None
        if world > 1:
            model.train()
            model.zero_grad()
            lp = forward()
            loss_of(lp).backward()
            D.allreduce_grads(model.parameters())
            sh_grads = {kk: p.grad.detach().clone() for kk, p in model.named_parameters()}
            model.zero_grad()
            if rank == 0:
                ref = model(data)
                F.nll_loss(ref, y).backward()
                lerr = float((lp.detach() - ref.detach()[lo:hi]).abs().max() / (ref.detach().abs().max() + 1e-12))
                gerr = max(float((sh_grads[kk] - p.grad).abs().max() / (p.grad.abs().max() + 1e-12)) for kk, p in model.named_parameters())
                parity_epoch = {"max_rel_logit_err": lerr, "max_rel_grad_err": gerr, "rows": [lo, hi], "tolerance": 1e-5,
                                "ok": bool(lerr < 1e-5 and gerr < 2e-5),
                                "against": "unsharded CUDA model on rank 0, same parameters (sharded backward = scatter form, FP32 atomics)"}
                model.zero_grad()
                del ref
            cx.barrier()
        ep_ms = timed(epoch, 5, 3, cx.barrier)
        fw_ms = timed(fwd_only, 5, 1, cx.barrier)
        ts_ms = timed(train_step, 5, 1, cx.barrier)
        ep_ms, fw_ms, ts_ms = cx.max_over_ranks(ep_ms, fw_ms, ts_ms)
        extras = {"epoch_ms": ep_ms, "forward_ms": fw_ms, "train_step_ms": ts_ms, "graph_prep_ms": prep_ms, "graph_prep_first_call_ms": prep[0],
                  "epoch_config": f"SNGNN_Plus_Plus 2 layers hidden {hid} top_k={k} thr={thr} init_beta=0.5 on {args.workload}-shape graph "
                                  f"({Ep} edges after loop processing, symmetric={g.symmetric}); epoch = fwd+loss+bwd+Adam + 2 eval forwards (R train.py:136-138)" +
                                  (f"; rows sharded over {world} ranks: all-gather of h per layer, reduce-scatter of dL/dh, row blocks of dL/dW^T all-gathered, "
                                   "all-reduce of the small parameter gradients" if world > 1 else ""),
                  "parity_epoch": parity_epoch}
        del model, opt
        torch.cuda.empty_cache()
        # fused aggregation kernels alone (whole graph on this rank's device), C = 32
        torch.manual_seed(3)
        h = torch.randn(N, hid, device=dev)
        gg = torch.randn(N, hid, device=dev)
        fuse = (torch.randn(N, hid, device=dev) * 0.1, torch.randn(hid, device=dev), torch.full((1,), 0.5, device=dev), None)
        k2_inf = timed(lambda: SF._edge_fwd(h, g, 0, k, thr, False), 10, 3)
        k2_trn = timed(lambda: SF._edge_fwd(h, g, 0, k, thr, True, want_q=True), 10, 3)
        k2_fus = timed(lambda: SF._edge_fwd(h, g, 0, k, thr, False, fuse), 10, 3)
        out1, ss, sw, sq, sc, inv_norm, _ = SF._edge_fwd(h, g, 0, k, thr, True, want_q=True)
        outf, _, _, _, _, _, diff = SF._edge_fwd(h, g, 0, k, thr, True, fuse, want_q=True)

        def k2_bwd(fused):
            SF.edge_bwd(h, inv_norm, gg, g, k, ss, sw, sq, sc, fuse[2] if fused else None, diff if fused else None)

        k2b_ms = timed(lambda: k2_bwd(False), 10, 3)
        k2bf_ms = timed(lambda: k2_bwd(True), 10, 3)
        nsel = int(sc.sum())
        bytes_fwd = Ep * (4 * hid + 4) + N * (8 * hid + 8)                       # SURVEY.md §8(d), inference form (no saved lists)
        bytes_trn = bytes_fwd + 8 * N * k
        bytes_fus = bytes_fwd + Ep * 4 * hid
        bytes_bwd = nsel * (3 * 4 * hid + 16) + 5 * N * 4 * hid

        def gbs(b, ms_):
            return b / (ms_ * 1e-3) / 1e9

        extras["agg"] = {"channels": hid, "selected_edges": nsel, "peak_gbs": pk["hbm"],
                         "fwd_ms": k2_inf, "fwd_gbs": gbs(bytes_fwd, k2_inf), "fwd_frac_hbm": gbs(bytes_fwd, k2_inf) / pk["hbm"],
                         "fwd_train_ms": k2_trn, "fwd_train_frac_hbm": gbs(bytes_trn, k2_trn) / pk["hbm"],
                         "fwd_fused_ms": k2_fus, "fwd_fused_gbs": gbs(bytes_fus, k2_fus), "fwd_fused_frac_hbm": gbs(bytes_fus, k2_fus) / pk["hbm"],
                         "bwd_ms": k2b_ms, "bwd_gbs": gbs(bytes_bwd, k2b_ms), "bwd_frac_hbm": gbs(bytes_bwd, k2b_ms) / pk["hbm"],
                         "bwd_fused_ms": k2bf_ms,
                         "algorithmic_bytes": {"fwd": bytes_fwd, "fwd_train": bytes_trn, "fwd_fused": bytes_fus, "bwd": bytes_bwd},
                         "kernels": ["row_inv_norm_kernel", "edge_fwd_staged_kernel (rows <= 32 edges)", "edge_fwd_staged_kernel (32-edge chunks of long rows)",
                                     "edge_fwd_merge_kernel", "edge_bwd_target_kernel", "edge_bwd_source_kernel"],
                         "backward": "deterministic: two gather passes through the transpose index, no float atomics"}
        if rank == 0:
            extras["agg"]["parity"] = agg_parity(g, h, out1, ss, sc, k, thr, fuse, outf)
        del h, gg, fuse, out1, outf, x, ei, y, g
        G.clear_cache()
        torch.cuda.empty_cache()
        # the two small model configurations of BASELINE.json (one GPU, with the oracle's CPU epoch beside them)
        if rank == 0 and not args.skip_cpu and not args.skip_configs:
            for name, kw in (("chameleon", dict(kind="SNGNN_Plus_Plus", layers=1, hid=32, k=10, thr=0.9, beta=0.0, feature_kind="binary")),
                             ("arxiv-year", dict(kind="SNGNN_Plus", layers=2, hid=32, k=10, thr=0.0, beta=0.0, feature_kind="clustered"))):
                try:
                    configs[f"model_{kw['kind']}_{name}_shape"] = model_case(cx, name, **kw)
                except Exception as exc:
                    configs[f"model_{kw['kind']}_{name}_shape"] = {"error": f"{type(exc).__name__}: {exc}"[:300]}
        cx.barrier()

    if rank == 0:
        ms, ms_e2e = head["ms_per_step"], head["ms_e2e"]
        pairs = float(N) * float(N)
        plan = head["plan"]
        ldh, ld32 = (Fd + 15) // 16 * 16, (Fd + 3) // 4 * 4
        traffic = None
        tp = os.path.join(ROOT, "profiles", "traffic.json")
        if os.path.exists(tp):
            traffic = json.load(open(tp)).get(f"stage1:{args.workload}:{world}")
        roofline = dict(head["roofline"], traffic=traffic, peak_source=pk["src"] + " (sustained bf16/fp16 dense)", plan=plan,
                        phase_ms_rank0=head["phase_ms"])
        line = {"metric": METRIC, "value": pairs / (ms * 1e-3) / 1e9, "unit": UNIT, "n_gpus": world, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
                "dtype": "f16 tensor-core scores + f32 exact rescore", "data": "synthetic",
                "config": {"workload": f"{args.workload}-shape all-pairs similarity-kNN build: N={N} d={Fd} top_k={k} thr={thr} remove_self=1, "
                                       f"query rows sharded over {world} GPU(s)",
                           "features": args.features, "l2": "inputs larger than L2 (x-hat f16 %.0f MB, f32 %.0f MB)" % (N * ldh * 2 / 1e6, N * ld32 * 4 / 1e6),
                           "parallelism": f"row-shard x{world}" + (" + one NCCL all-gather of FP32 x-hat (FP16 operand converted locally)" if world > 1 else "")},
                "e2e": {"value": pairs / (ms_e2e * 1e-3) / 1e9, "unit": UNIT, "h2d_bytes_per_step": head["h2d_bytes"],
                        "d2h_bytes_per_step": head["d2h_bytes"], "ms_per_step": ms_e2e, "copy_ms_rank0": head["e2e_copy_ms"]},
                "gpu_launches": (16 + (1 if plan["seed_stride"] > 0 else 0)) * args.steps,
                "kernels_per_step": ["rownorm_kernel"] + (["simknn_stage1_kernel<seed>"] if plan["seed_stride"] > 0 else []) +
                                    ["simknn_stage1_kernel", "simknn_rescore_kernel", "simknn_retry_rounds_kernel", "simknn_retry_gather_kernel", "simknn_stage1_kernel (retry)",
                                     "simknn_rescore_kernel (retry)", "4 x (simknn_fb_scan_kernel, simknn_fb_merge_kernel)", "simknn_fb_stream_kernel"],
                "roofline": roofline, "cpu_baseline": head.get("cpu"), "clocks": clocks, "parity": head["parity"], "configs": configs}
        line.update(extras)
        emit(line)
    if world > 1:
        cx.dist.barrier()
        cx.dist.destroy_process_group()


_RESULT_FD = None


def emit(line):
    """The ONE JSON line of the contract, on the real stdout (see main)."""
    data = (json.dumps(line) + "\n").encode()
    if _RESULT_FD is None:
        sys.stdout.write(data.decode()); sys.stdout.flush()
    else:
        os.write(_RESULT_FD, data)


def main():
    global _RESULT_FD
    # Libraries print to file descriptor 1 behind Python's back (NCCL announces its version there when a communicator is
    # created): keep the real stdout for the result line only and send everything else to stderr.
    sys.stdout.flush()
    _RESULT_FD = os.dup(1)
    os.dup2(2, 1)
    args = parse()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
