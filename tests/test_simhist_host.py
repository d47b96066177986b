"""Host side of the similarity histogram (no GPU): the FP64 reference against numpy.histogram, the C ABI's argument checks,
and the row-tile sharding of node_similarity_histogram_sharded over gloo with an FP64 stand-in of the kernel's schedule."""
import ctypes
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from conftest import ROOT


def _tiles_ref(xhat, bins, lo, hi, tile_lo, tile_hi):
    """FP64 stand-in of sng_simhist_f16 on row tiles [tile_lo, tile_hi): tile I scores (I, (I + s) mod T), s = 0 .. T // 2
    (s = T / 2 only for I < T / 2 when T is even); the diagonal tile counts i < j, every counted score twice."""
    from oracle import simhist_ref
    x = xhat.double()
    n = x.size(0)
    t = (n + 127) // 128
    counts = torch.zeros(bins, dtype=torch.int64)
    for i in range(tile_lo, tile_hi):
        for s in range(t // 2 + (1 if (t % 2 or i < t // 2) else 0)):
            j = (i + s) % t
            a, b = x[i * 128:(i + 1) * 128], x[j * 128:(j + 1) * 128]
            sc = a @ b.t()
            if s == 0:
                sc = sc[torch.triu(torch.ones_like(sc, dtype=torch.bool), diagonal=1)]
            counts += 2 * simhist_ref.histogram_with_slack(sc, bins, (lo, hi), 0.0)[0]
    return counts


@pytest.mark.parametrize("bins,rng", [(1, (-1.0, 1.0)), (7, (-1.0, 1.0)), (200, (-1.0, 1.0)), (50, (0.0, 1.0)), (13, (-0.3, 0.45))])
def test_reference_matches_numpy_histogram(bins, rng):
    from oracle import simhist_ref
    from sngnn_b200 import synth
    x = synth.make_features(300, 9, "clustered", seed=7)
    counts, slack = simhist_ref.node_similarity_histogram_ref(x, bins, rng, 1e-6, block=64)
    xn = torch.nn.functional.normalize(x.double(), dim=-1)
    s = (xn @ xn.t()).clamp(-1, 1)
    vals = s[~torch.eye(300, dtype=torch.bool)].numpy()
    ref, _ = np.histogram(vals, bins, rng)
    assert counts.sum() <= 300 * 299
    assert (counts.numpy() - ref).__abs__().max() <= slack.max() and (slack >= 0).all()
    if rng == (-1.0, 1.0):
        assert int(counts.sum()) == 300 * 299


def test_reference_exact_values_and_closed_last_bin():
    from oracle import simhist_ref
    s = torch.tensor([-1.0, -0.5, 0.0, 0.0, 0.5, 1.0, 1.0 + 1e-12, 1.5], dtype=torch.float64)
    c, sl = simhist_ref.histogram_with_slack(s, 2, (-1.0, 1.0), 0.0)
    assert c.tolist() == [2, 6] and sl.tolist() == [0, 0]
    c, _ = simhist_ref.histogram_with_slack(s, 4, (-0.5, 0.5), 0.0)
    assert c.tolist() == [1, 0, 2, 1]                       # -1 and 1 fall outside; 0.5 is the closed last bin
    _, sl = simhist_ref.histogram_with_slack(torch.tensor([0.2500001], dtype=torch.float64), 4, (-0.5, 0.5), 1e-6)
    assert sl.tolist() == [0, 0, 1, 1]                       # 0.25 is the edge between bins 2 and 3


def test_schedule_stand_in_covers_every_pair_once():
    for n in (1, 2, 127, 128, 129, 257, 384, 520):
        x = torch.randn(n, 3, dtype=torch.float64)
        xh = torch.nn.functional.normalize(x, dim=-1)
        t = (n + 127) // 128
        assert int(_tiles_ref(xh, 1, -1.0, 1.0, 0, t).sum()) == n * (n - 1)


def test_abi_rejects_bad_arguments_without_a_device():
    from sngnn_b200 import _C
    L = _C.lib()
    p, c = ctypes.c_void_p(4096), ctypes.c_void_p(8192)

    def call(n=300, k=24, lda=24, tlo=0, thi=3, lo=-1.0, hi=1.0, bins=200, a=p, counts=c):
        return L.sng_simhist_f16(a, lda, p, lda, n, k, tlo, thi, lo, hi, bins, counts, None)

    for kw, msg in ((dict(bins=0), "bins"), (dict(bins=4097), "bins"), (dict(lo=1.0, hi=-1.0), "range"),
                    (dict(lo=float("nan")), "range"), (dict(hi=float("inf")), "range"), (dict(lda=20), "multiples of 8"),
                    (dict(k=32, lda=24), "lda"), (dict(a=ctypes.c_void_p(4100)), "aligned"), (dict(n=0), "sizes"),
                    (dict(n=1 << 31), "sizes"), (dict(thi=4), "tile range"), (dict(tlo=2, thi=1), "tile range"),
                    (dict(counts=None), "sizes")):
        assert call(**kw) == -1, kw
        assert "sng_simhist_f16" in _C.last_error() and msg in _C.last_error(), (kw, _C.last_error())
    assert call(tlo=2, thi=2) == 0                          # an empty tile range adds nothing and launches nothing


def test_python_surface_rejects_bad_arguments():
    from sngnn_b200.toolbox import dense as D
    for bins, rng in ((0, (-1, 1)), (2.5, (-1, 1)), (True, (-1, 1)), (10, (1, -1)), (10, (0, float("nan")))):
        with pytest.raises(ValueError):
            D._hist_range(bins, rng)


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    return port


def _worker(rank, ws, port, n, bins, rng, ret):
    import sys
    sys.path.insert(0, ROOT)
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=ws)
    from sngnn_b200 import dist as D, synth
    from sngnn_b200.toolbox import sharded as TS
    from oracle import simhist_ref
    x = synth.make_features(n, 11, "clustered", seed=5)
    lo, hi = D.shard_bounds(n, ws, rank)
    counts, edges = TS.node_similarity_histogram_sharded(x[lo:hi], n, bins, rng, hist=_tiles_ref)
    ref, _ = simhist_ref.node_similarity_histogram_ref(x, bins, rng, 0.0)
    gathered = [torch.zeros_like(counts) for _ in range(ws)]
    dist.all_gather(gathered, counts)
    ret[rank] = (counts.dtype == torch.int64 and all(torch.equal(g, counts) for g in gathered) and torch.equal(counts, ref)
                 and edges.shape == (bins + 1,) and float(edges[0]) == rng[0] and float(edges[-1]) == rng[1])
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.parametrize("ws,n,bins,rng", [(2, 300, 200, (-1.0, 1.0)), (3, 200, 7, (0.0, 1.0)), (3, 257, 40, (-0.5, 0.9))])
def test_sharded_histogram_gloo_matches_unsharded_oracle(ws, n, bins, rng):
    """World 3 at n = 200 (two row tiles) leaves the last rank without tiles; it still joins the all-reduce."""
    ctx = mp.get_context("spawn")
    ret = ctx.Manager().dict()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, ws, port, n, bins, rng, ret)) for r in range(ws)]
    for p in procs:
        p.start()
    for p in procs:
        p.join(180)
        assert p.exitcode == 0, f"worker exited with {p.exitcode}"
    assert dict(ret) == {r: True for r in range(ws)}
