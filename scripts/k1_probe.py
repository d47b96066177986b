"""Timing probe of the tensor-core stage (sng_simknn_stage1) over a grid of shapes / data / thresholds."""
import ctypes, sys, os, json
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from sngnn_b200 import _C, simknn, synth

dev = "cuda"
def run(n, d, kind, thr_lo, mb, ns, cand=16, reps=3, nq=None, seed_stride=0, seed_q=0):
    x = synth.make_features(n, d, kind, seed=0, device=dev)
    xf, xh = simknn.normalize_operands(x)
    nq = nq or n
    ci = torch.empty(nq * 512, dtype=torch.int32, device=dev)
    cv = torch.empty(nq * 512, dtype=torch.float32, device=dev)
    cm = torch.empty(nq * 64, dtype=torch.float32, device=dev)
    nsv = ctypes.c_int(0)
    seeds = None
    if seed_stride > 0:
        def g():
            return simknn.seed_pass(xh[:nq], xh, d, seed_stride, mb)
        seeds = g(); torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(reps): g()
        b.record(); torch.cuda.synchronize()
        print(json.dumps(dict(seed_pass_ms=round(a.elapsed_time(b) / reps, 3), stride=seed_stride)), flush=True)
    phase = torch.zeros(8, dtype=torch.int32, device=dev)
    def f():
        phase.zero_()
        _C.check(_C.lib().sng_simknn_stage1(_C.ptr(xh), _C.ptr(xh), xh.size(1), nq, 0, n, d, cand, thr_lo, 1, _C.ptr(ci), _C.ptr(cv), _C.ptr(cm), mb, ns, ctypes.byref(nsv), _C.ptr(seeds), seed_q, seed_stride, _C.ptr(phase), _C.stream()), "s1")
    f(); torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps): f()
    b.record(); torch.cuda.synchronize()
    ms = a.elapsed_time(b) / reps
    print(json.dumps(dict(n=n, nq=nq, d=d, kind=kind, thr_lo=thr_lo, ew=mb, lists=nsv.value, cand=cand, seed=(seed_stride, seed_q), ms=round(ms, 3),
                          gpairs=round(nq * n / ms / 1e6, 1), tflops=round(2 * nq * n * d / ms / 1e9, 1))), flush=True)

if __name__ == "__main__":
    cfgs = eval(sys.argv[1]) if len(sys.argv) > 1 else [
        (262144, 65, "normal", 2.0, 4, 1), (262144, 65, "normal", -2.0, 4, 1), (262144, 65, "clustered", -2.0, 4, 1),
        (262144, 65, "normal", 2.0, 2, 1), (262144, 128, "normal", 2.0, 4, 1), (262144, 128, "normal", -2.0, 4, 1),
        (262144, 256, "normal", 2.0, 2, 1), (262144, 256, "normal", -2.0, 2, 1),
        (262144, 512, "normal", 2.0, 1, 1), (262144, 512, "normal", -2.0, 1, 1), (262144, 512, "normal", -2.0, 2, 1)]
    for c in cfgs:
        run(*c)
