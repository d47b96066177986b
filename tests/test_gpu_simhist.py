"""Similarity histogram on the B200 (sng_simhist_f16 / toolbox node_similarity_histogram): exact scores, random features
against the FP64 reference within its per-bin slack, agreement with the N x N route, determinism over tile splits, scale
and the 2-GPU sharded form."""
import os
import socket

import pytest
import torch

from conftest import ROOT

pytestmark = pytest.mark.gpu


def delta(d):
    """Per-pair bound |score - FP64 cosine| for unit rows at feature width d (DESIGN.md §7): 1e-6 for the FP32 normalisation
    and the dropped lo.lo term, plus one truncated FP32 accumulator add (< 2^-23) per 16-element MMA step of K' = 3d."""
    return 1e-6 + 2.0 ** -23 * -(-3 * d // 16)


def _ref(x, bins, rng, dl):
    from oracle import simhist_ref
    return simhist_ref.node_similarity_histogram_ref(x.cuda(), bins, rng, dl, block=2048)


def _hist(x, bins, rng):
    from sngnn_b200.toolbox import node_similarity_histogram
    return node_similarity_histogram(x.cuda(), bins, rng)[0]


def _axis_rows(n, d=8, seed=0):
    """Rows e_k, -e_k, duplicates and zero rows: every cosine is exactly -1, 0 or 1."""
    g = torch.Generator().manual_seed(seed)
    x = torch.zeros(n, d)
    k = torch.randint(0, d, (n,), generator=g)
    sign = torch.where(torch.rand(n, generator=g) < 0.5, -1.0, 1.0)
    x[torch.arange(n), k] = sign
    x[torch.rand(n, generator=g) < 0.1] = 0.0
    return x


def test_exact_scores_equal_the_reference_exactly():
    for n in (1, 2, 127, 128, 129, 257, 384):
        x = _axis_rows(n, seed=n)
        for bins in (1, 2, 200):
            for rng in ((-1.0, 1.0), (0.0, 1.0), (-0.5, 0.5)):
                got = _hist(x, bins, rng)
                ref, _ = _ref(x, bins, rng, 0.0)
                assert torch.equal(got, ref), (n, bins, rng, got.nonzero().flatten().tolist(), ref.nonzero().flatten().tolist())
        assert int(_hist(x, 200, (-1.0, 1.0)).sum()) == n * (n - 1)


@pytest.mark.parametrize("kind,n,d", [("normal", 20000, 16), ("clustered", 20000, 65), ("normal", 12000, 128),
                                      ("clustered", 8000, 300), ("binary", 2277, 2325), ("clustered", 2277, 2325)])
def test_random_features_within_slack_of_fp64(kind, n, d):
    from sngnn_b200 import synth
    x = synth.make_features(n, d, kind, seed=d)
    dl = delta(d)
    for bins, rng in ((7, (-1.0, 1.0)), (200, (-1.0, 1.0)), (1000, (-1.0, 1.0)), (200, (0.85, 0.95)), (1000, (-0.2, 0.6))):
        got = _hist(x, bins, rng)
        ref, slack = _ref(x, bins, rng, dl)
        diff = (got - ref).abs()
        assert (diff <= slack).all(), (kind, n, d, bins, rng, int((diff - slack).max()))
        if rng == (-1.0, 1.0):
            assert int(got.sum()) == int(ref.sum()) == n * (n - 1)
        else:
            assert abs(int(got.sum()) - int(ref.sum())) <= int(slack[0] + slack[-1])


def test_agrees_with_binning_of_the_dense_matrix():
    import sngnn_b200.toolbox as T
    from oracle import simhist_ref
    from sngnn_b200 import synth
    x = synth.make_features(3000, 65, "clustered", seed=11)
    vals = T.node_similarity_dense_small(x.cuda())[0]
    for bins, rng in ((200, (-1.0, 1.0)), (50, (0.5, 1.0))):
        got, edges = T.node_similarity_histogram(x.cuda(), bins, rng)
        ref, slack = simhist_ref.histogram_with_slack(vals, bins, rng, delta(65))
        assert ((got - ref).abs() <= slack).all()
        assert got.device == x.cuda().device and got.dtype == torch.int64 and edges.dtype == torch.float64
        torch.testing.assert_close(edges.cpu(), torch.linspace(rng[0], rng[1], bins + 1, dtype=torch.float64))
    counts, edges = T.node_similarity_histogram(x, 200)                    # host input -> host output
    assert not counts.is_cuda and not edges.is_cuda


def test_deterministic_over_runs_and_tile_splits():
    from sngnn_b200.toolbox import dense as D
    from sngnn_b200 import synth
    x = synth.make_features(5000, 65, "clustered", seed=3)
    xhat = D._normalised(x)
    t = (5000 + 127) // 128
    whole = D.simhist_tiles(xhat, 200, -1.0, 1.0, 0, t)
    assert torch.equal(whole, D.simhist_tiles(xhat, 200, -1.0, 1.0, 0, t))
    for cuts in ((0, 17, t), (0, 5, 5, t), (0, 1, 20, 39, t), (0, 0, 13, 26, t)):
        parts = sum(D.simhist_tiles(xhat, 200, -1.0, 1.0, a, b) for a, b in zip(cuts[:-1], cuts[1:]))
        assert torch.equal(parts, whole), cuts
    assert int(whole.sum()) == 5000 * 4999


def test_scale():
    from sngnn_b200.toolbox import dense as D, node_similarity_histogram
    from oracle import simhist_ref
    from sngnn_b200 import synth
    n = 200000
    counts, _ = node_similarity_histogram(synth.make_features(n, 65, "normal", seed=1, device="cuda"), 200)
    assert int(counts.sum()) == n * (n - 1)
    n = 50000
    xhat = D._normalised(synth.make_features(n, 65, "clustered", seed=2, device="cuda"))
    got = D.simhist_tiles(xhat, 200, -1.0, 1.0, 0, (n + 127) // 128)
    a, b, k = D.split_f16_operands(xhat)
    ref = torch.zeros_like(got)
    slack = torch.zeros_like(got)
    for r0 in range(0, n, 5000):                                           # the N x N matrix of the same operands, by row blocks
        m = D.gemm_nt(a[r0:r0 + 5000], b, k)
        r = torch.arange(m.size(0), device=m.device)
        m[r, r0 + r] = float("nan")                                        # the diagonal is not counted
        c, s = simhist_ref.histogram_with_slack(m[~m.isnan()], 200, (-1.0, 1.0), delta(65))
        ref += c
        slack += s
    assert ((got - ref).abs() <= slack).all()
    assert int(got.sum()) == int(ref.sum()) == n * (n - 1)


def test_argument_errors_raise():
    from sngnn_b200.toolbox import dense as D, node_similarity_histogram
    x = torch.randn(300, 5, device="cuda")
    with pytest.raises(ValueError):
        node_similarity_histogram(x, 0)
    with pytest.raises(ValueError):
        node_similarity_histogram(x, 10, (1.0, -1.0))
    with pytest.raises(RuntimeError, match="bins"):
        node_similarity_histogram(x, 5000)
    with pytest.raises(RuntimeError, match="tile range"):
        D.simhist_tiles(D._normalised(x), 10, -1.0, 1.0, 0, 4)
    with pytest.raises(RuntimeError, match="CUDA tensors"):
        D.simhist_tiles(torch.randn(10, 4), 10, -1.0, 1.0, 0, 1)


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _worker(rank, ws, port, ret):
    import sys
    sys.path.insert(0, ROOT)
    import torch.distributed as dist
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=ws, device_id=dev)
    from sngnn_b200 import dist as D, synth
    from sngnn_b200.toolbox import node_similarity_histogram
    from sngnn_b200.toolbox.sharded import node_similarity_histogram_sharded
    n = 30001
    x = synth.make_features(n, 65, "clustered", seed=4).to(dev)
    lo, hi = D.shard_bounds(n, ws, rank)
    counts, _ = node_similarity_histogram_sharded(x[lo:hi].contiguous(), n, 200)
    ret[rank] = torch.equal(counts, node_similarity_histogram(x, 200)[0])
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_two_rank_nccl_equals_single_gpu():
    import torch.multiprocessing as mp
    ctx = mp.get_context("spawn")
    ret = ctx.Manager().dict()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, 2, port, ret)) for r in range(2)]
    for p in procs:
        p.start()
    for p in procs:
        p.join(300)
        assert p.exitcode == 0, f"worker exited with {p.exitcode}"
    assert dict(ret) == {0: True, 1: True}
