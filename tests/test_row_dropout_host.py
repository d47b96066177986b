"""Host side of the counter-based row dropout: the numpy oracle (oracle/dropout_ref.py) -- Philox4x32-10 known answers, keep
rate, shard invariance, p in {0, 1}, the high counter word -- and the argument validation of sng_row_dropout_fwd / _bwd, which
rejects bad arguments before touching a device (an empty shard returns 0 without a launch)."""
import ctypes

import numpy as np
import pytest

from oracle import dropout_ref as R


def test_philox_known_answers():
    for ctr, key, want in R.KAT:
        assert tuple(int(w) for w in R.philox4x32_10(*ctr, *key)) == want


@pytest.mark.parametrize("p", [0.1, 0.5, 0.9])
def test_keep_fraction(p):
    n, c = 4000, 32
    keep = R.keep_mask(n, c, 123, seed=99, call=3, p=p)
    sigma = np.sqrt(p * (1 - p) / keep.size)
    assert abs(keep.mean() - (1 - p)) < 6 * sigma
    assert abs(keep[:, :8].mean() - (1 - p)) < 6 * np.sqrt(p * (1 - p) / (n * 8))     # no channel is favoured


@pytest.mark.parametrize("c", [1, 3, 4, 130])
def test_shards_concatenate_to_the_whole(c):
    n, seed, call, p = 101, 2**40 + 5, 7, 0.5
    whole = R.keep_mask(n, c, 0, seed, call, p)
    bounds = [(0, 34), (34, 34), (34, 68), (68, 101)]
    assert np.array_equal(np.concatenate([R.keep_mask(hi - lo, c, lo, seed, call, p) for lo, hi in bounds]), whole)
    assert not np.array_equal(R.keep_mask(n, c, 0, seed, call + 1, p), whole)       # the call index changes the masks
    assert not np.array_equal(R.keep_mask(n, c, 0, seed + 1, call, p), whole)
    z = np.random.default_rng(0).standard_normal((n, c)).astype(np.float32)
    for relu in (False, True):
        y = R.forward(z, 0, seed, call, p, relu)
        assert np.array_equal(np.concatenate([R.forward(z[lo:hi], lo, seed, call, p, relu) for lo, hi in bounds]), y)


def test_p_zero_and_one():
    z = np.random.default_rng(1).standard_normal((50, 6)).astype(np.float32)
    g = np.random.default_rng(2).standard_normal((50, 6)).astype(np.float32)
    assert R.keep_mask(50, 6, 0, 1, 0, 0.0).all() and not R.keep_mask(50, 6, 0, 1, 0, 1.0).any()
    assert np.array_equal(R.forward(z, 0, 1, 0, 0.0, False), z)
    assert np.array_equal(R.forward(z, 0, 1, 0, 0.0, True), np.maximum(z, 0))
    assert np.array_equal(R.backward(z, g, 0, 1, 0, 0.0, True), np.where(z > 0, g, 0))
    for dt in (np.float32, np.float64):                                  # a select, not inf * 0: exact zeros, no NaN
        y = R.forward(z.astype(dt), 0, 1, 0, 1.0, False)
        assert y.dtype == dt and np.array_equal(y, np.zeros_like(y)) and not np.signbit(y).any()
        assert np.array_equal(R.backward(None, g.astype(dt), 0, 1, 0, 1.0, False), np.zeros_like(g, dtype=dt))
    assert R.threshold(0.5) == 2**23 and R.threshold(1.0) == 2**24 and R.scale32(0.5) == np.float32(2.0)


def test_high_counter_word():
    """Rows far enough out that e >> 2 >= 2^32: the mask follows the 64-bit group index, not its low word."""
    c, seed, call, p = 32, 17, 2, 0.5
    row_offset = (2**34 + 12345) * 4 // c                                # e = row_offset * c >= 2^36
    keep = R.keep_mask(3, c, row_offset, seed, call, p)
    e = row_offset * c + 1 * c + 5                                       # element (1, 5)
    q = e >> 2
    w = R.philox4x32_10(q & 0xFFFFFFFF, q >> 32, call, 0, seed, 0)[e & 3]
    assert q >> 32 > 0 and keep[1, 5] == (int(w) >> 8 >= R.threshold(p))
    low = (row_offset * c) % 2**32 // c                                 # the same low group word without the high word
    assert not np.array_equal(R.keep_mask(3, c, low, seed, call, p), keep)


def test_abi_argument_validation_without_device():
    from sngnn_b200 import _C
    L = _C.lib()
    buf = ctypes.c_void_p(16)                                            # never dereferenced: every call below is rejected first
    fwd = lambda n=8, c=4, ldz=4, ro=0, p=0.5, y=buf, ldy=4, z=buf: L.sng_row_dropout_fwd(z, n, c, ldz, ro, 1, 0, p, 1, y, ldy, None)
    bwd = lambda n=8, c=4, ldz=4, ldg=4, ro=0, p=0.5, relu=1, z=buf, g=buf, dz=buf, lddz=4: L.sng_row_dropout_bwd(
        z, g, n, c, ldz, ldg, ro, 1, 0, p, relu, dz, lddz, None)
    cases = [(dict(p=-0.1), "p"), (dict(p=1.5), "p"), (dict(p=float("nan")), "p"), (dict(c=0), "bad arguments"), (dict(n=-1), "bad arguments"),
             (dict(ro=-1), "bad arguments"), (dict(ldz=3), "leading"), (dict(ro=2**61, c=4), "overflows"), (dict(z=None), "NULL")]
    for kw, what in cases + [(dict(ldy=3), "leading"), (dict(y=None), "NULL")]:
        assert fwd(**kw) == -1 and what in _C.last_error(), (kw, _C.last_error())
    for kw, what in cases + [(dict(ldg=3), "leading"), (dict(lddz=2), "leading"), (dict(g=None, relu=0), "NULL"), (dict(dz=None), "NULL")]:
        assert bwd(**kw) == -1 and what in _C.last_error(), (kw, _C.last_error())
    assert fwd(n=0, z=None, y=None) == 0                                 # an empty shard: nothing to launch
    assert bwd(n=0, z=None, g=None, dz=None) == 0
