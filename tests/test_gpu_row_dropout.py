"""GPU side of the counter-based row dropout (sng_row_dropout_fwd / _bwd): the kernels bit for bit against the numpy oracle, shard
invariance, repeatability and the mask statistics at the pokec shape; world-1 sharded_forward with dist.RowDropout against an
FP64 reference under the oracle's masks; and the trainer under torchrun -- world 1 against the single-GPU trainer, and (with
>= 2 GPUs) 2 ranks against 1 with dropout on."""
import json
import os
import signal
import subprocess
import sys

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from conftest import ROOT
from oracle import dropout_ref as R

pytestmark = pytest.mark.gpu
DEV = "cuda"
BIG_OFFSET = 2**33 // 4 + 3                       # e = row_offset * c >= 2^33 for every c >= 4: the high counter word is in use


def _operands(n, c, ld, shift, seed):
    g = torch.Generator().manual_seed(seed)
    buf = torch.randn(n, ld + shift, generator=g)
    buf[::7, shift] = 0.0                                               # exact zeros: relu's backward passes none of them
    buf[:, shift + c:] = float("nan")                                   # columns beyond c must never be read
    z = buf.to(DEV)[:, shift:shift + c]
    gy = torch.randn(n, c, generator=g).to(DEV)
    return z, gy


@pytest.mark.parametrize("c", [1, 3, 4, 32, 130, 512])
@pytest.mark.parametrize("layout", ["contiguous", "strided", "misaligned"])
@pytest.mark.parametrize("row_offset", [0, BIG_OFFSET])
def test_kernels_match_the_oracle_bit_for_bit(c, layout, row_offset):
    from sngnn_b200 import functional as SF
    n = 257
    ld, shift = {"contiguous": (c, 0), "strided": (c + 4, 0), "misaligned": (c + 3, 1)}[layout]
    z, gy = _operands(n, c, ld, shift, c + row_offset % 97)
    assert z.stride(0) == ld + shift
    zn, gn = z.cpu().numpy(), gy.cpu().numpy()
    seed, call = 0x0123456789ABCDEF, 2**33 + 11
    for p in (0.0, 0.1, 0.5, 0.9, 1.0):
        for relu in (False, True):
            y = SF.row_dropout_fwd(z, row_offset, seed, call, p, relu)
            dz = SF.row_dropout_bwd(z if relu else None, gy, row_offset, seed, call, p, relu)
            assert np.array_equal(y.cpu().numpy(), R.forward(zn, row_offset, seed, call, p, relu)), (p, relu)
            assert np.array_equal(dz.cpu().numpy(), R.backward(zn, gn, row_offset, seed, call, p, relu)), (p, relu)


@pytest.mark.parametrize("c", [3, 32])
def test_shard_invariance_and_repeatability(c):
    from sngnn_b200 import functional as SF
    n, seed, call, p = 100003, 42, 9, 0.5
    z, gy = _operands(n, c, c, 0, 5)
    y = SF.row_dropout_fwd(z, 0, seed, call, p, True)
    dz = SF.row_dropout_bwd(z, gy, 0, seed, call, p, True)
    bounds = [(0, 33334), (33334, 33334), (33334, 66668), (66668, n)]
    ys = [SF.row_dropout_fwd(z[lo:hi], lo, seed, call, p, True) for lo, hi in bounds]
    dzs = [SF.row_dropout_bwd(z[lo:hi], gy[lo:hi], lo, seed, call, p, True) for lo, hi in bounds]
    assert torch.equal(torch.cat(ys), y) and torch.equal(torch.cat(dzs), dz)
    assert torch.equal(SF.row_dropout_fwd(z, 0, seed, call, p, True), y)
    assert torch.equal(SF.row_dropout_bwd(z, gy, 0, seed, call, p, True), dz)


@pytest.mark.parametrize("p", [0.1, 0.5, 0.9])
def test_mask_statistics_at_the_pokec_shape(p):
    """Keep rate within 6 sigma of 1 - p; rows i and lo + i (lo = the second shard's first row at world 2) agree as independent
    masks do, (1 - p)^2 + p^2 -- not 1, as generators seeded alike on every rank would make them."""
    from sngnn_b200 import functional as SF
    n, c = 1632803, 32
    keep = SF.row_dropout_fwd(torch.ones(n, c, device=DEV), 0, 1234, 0, p, False) != 0
    m = keep.numel()
    rate = keep.double().mean().item()
    assert abs(rate - (1 - p)) < 6 * (p * (1 - p) / m) ** 0.5, rate
    lo = (n + 1) // 2
    agree = (keep[:n - lo] == keep[lo:]).double().mean().item()
    q = (1 - p) ** 2 + p ** 2
    assert abs(agree - q) < 6 * (q * (1 - q) / ((n - lo) * c)) ** 0.5, (agree, q)


@pytest.mark.parametrize("kind,bn", [("SNGNN", False), ("SNGNN_Plus", False), ("SNGNN_Plus_Plus", False), ("SNGNN_Plus", True),
                                     ("SNGNN_Plus_Plus", True)])
def test_sharded_forward_world1_with_row_dropout_matches_fp64(kind, bn):
    """world 1 (no process group), training, p = 0.5: logits and every gradient against the unsharded FP64 forward / backward
    under the oracle's masks (the tolerances of test_gpu_shard_bn.py)."""
    from sngnn_b200 import dist as D
    from test_dist_gloo_dropout import CALL0, SEED, _model, _problem, _reference
    n, k, layers = 2000, 3, 3
    x, ei, y = _problem(n)
    model = _model(kind, n, bn, k=k, layers=layers).float()
    if bn:
        for b in model.bns:
            b.weight.data.uniform_(0.5, 1.5)
            b.bias.data.uniform_(-0.5, 0.5)
    sd = {kk: v.detach().double().clone().requires_grad_("running" not in kk) for kk, v in model.state_dict().items() if v.is_floating_point()}
    model = model.to(DEV).train()
    rd = D.RowDropout(SEED)
    rd.calls = CALL0
    logp = D.sharded_forward(model, x.float().to(DEV), ei.to(DEV), n, dropout=rd)
    F.nll_loss(logp, y.to(DEV)).backward()
    assert rd.calls == CALL0 + layers - 1
    ref = _reference(kind, sd, x, ei, k, layers, bn)
    F.nll_loss(ref, y).backward()
    torch.testing.assert_close(logp.detach().cpu().double(), ref.detach(), rtol=1e-5, atol=2e-6)
    for name, p in model.named_parameters():
        g_ref = sd[name].grad
        tol = 1e-4 if name.endswith("beta") else 2e-5
        err = float((p.grad.cpu().double() - g_ref).abs().max() / (g_ref.abs().max() + 1e-30))
        assert err < tol, (name, err)


# ------------------------------------------------------------------------------------------------ the trainer under torchrun
_RANK_SCRIPT = r'''
import hashlib, json, os, sys
sys.path.insert(0, {root!r})
from sngnn_b200 import train as T
seen = {{}}
inner = T.train_sharded
def spy(model, *a, **k):
    r = inner(model, *a, **k)
    seen["params"] = hashlib.sha256(b"".join(p.detach().cpu().contiguous().numpy().tobytes() for p in model.parameters())).hexdigest()
    return r
T.train_sharded = spy
final, hist = T.main(sys.argv[2:], log=lambda *_: None)
with open(os.path.join(sys.argv[1], "rank%s.json" % os.environ["RANK"]), "w") as f:
    json.dump(dict(final=final, hist=hist, params=seen["params"]), f)
'''

ARGS = "--dataset small --num_layers 2 --hidden_channels 32 --top_k 4 --thr 0.0 --init_beta 0.3 --patience 100 --log-every 1".split()


def _launch(cmd, env, timeout=600):
    """Run `cmd` in its own process group; on timeout (or any error) terminate whatever of it is still running."""
    p = subprocess.Popen(cmd, env=env, cwd=ROOT, start_new_session=True, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    try:
        out, _ = p.communicate(timeout=timeout)
    except subprocess.TimeoutExpired:
        out = None
    finally:
        for sig in (signal.SIGTERM, signal.SIGKILL):
            try:
                os.killpg(p.pid, sig)
            except ProcessLookupError:
                break
            try:
                p.wait(20)
            except subprocess.TimeoutExpired:
                pass
    assert out is not None, f"{cmd} did not finish within {timeout} s"
    assert p.returncode == 0, out[-6000:]
    return out


def _run_ranks(tmp_path, ws, args, torchrun=True):
    script = tmp_path / "rank.py"
    script.write_text(_RANK_SCRIPT.format(root=ROOT))
    out = tmp_path / f"out{ws}"
    out.mkdir()
    env = {k: v for k, v in os.environ.items() if k not in ("WORLD_SIZE", "RANK", "LOCAL_RANK", "MASTER_ADDR", "MASTER_PORT")}
    if torchrun:
        cmd = [sys.executable, "-m", "torch.distributed.run", "--standalone", f"--nproc-per-node={ws}", str(script), str(out)] + args
    else:
        from test_dist_gloo_bn import _free_port
        env.update(WORLD_SIZE="1", RANK="0", LOCAL_RANK="0", LOCAL_WORLD_SIZE="1", MASTER_ADDR="127.0.0.1", MASTER_PORT=str(_free_port()))
        cmd = [sys.executable, str(script), str(out)] + args
    _launch(cmd, env)
    return [json.loads((out / f"rank{r}.json").read_text()) for r in range(ws)]


@pytest.mark.parametrize("model", ["SNGNN_Plus", "SNGNN_Plus_Plus"])
def test_torchrun_world1_matches_the_single_gpu_trainer(tmp_path, model):
    """WORLD_SIZE=1 in the environment: the sharded trainer, dropout 0, against `python -m sngnn_b200.train` without torchrun over
    four epochs (the tolerances of test_train.py)."""
    from sngnn_b200 import train as T
    args = ARGS + ["--model", model, "--dropout", "0", "--epochs", "4"]
    lines = []
    final1, hist1 = T.main(args, log=lines.append)
    assert not any("world_size" in l for l in lines)
    got, = _run_ranks(tmp_path, 1, args, torchrun=False)
    assert len(got["hist"]) == len(hist1) == 4
    for ep, (a, b) in enumerate(zip(got["hist"], hist1)):
        for j in (0, 2, 4):
            assert a[j] == pytest.approx(b[j], rel=2e-4, abs=2e-5), (ep, j, a, b)
        for j in (1, 3, 5):
            assert a[j] == pytest.approx(b[j], abs=0.01), (ep, j, a, b)


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_torchrun_two_ranks_follow_one_with_dropout(tmp_path):
    """torchrun --nproc-per-node 2 against 1, dropout 0.5: epoch 0's training loss within 1e-6, the first 3 epochs' losses within
    1e-4; after training the parameters are bit-identical on both ranks."""
    args = ARGS + ["--model", "SNGNN_Plus_Plus", "--dropout", "0.5", "--epochs", "3"]
    one, = _run_ranks(tmp_path, 1, args)
    two = _run_ranks(tmp_path, 2, args)
    assert two[0]["params"] == two[1]["params"] and two[0]["hist"] == two[1]["hist"]
    assert two[0]["hist"][0][0] == pytest.approx(one["hist"][0][0], rel=1e-6)
    for a, b in zip(two[0]["hist"], one["hist"]):
        for j in (0, 2, 4):
            assert a[j] == pytest.approx(b[j], rel=1e-4), (a, b)
