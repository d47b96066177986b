"""Edge cases of K1's small-K (SPLIT, EW = 4) mode -- two MMA issuers taking alternate tiles, each tile two N = 128 halves
in four 128-column accumulator stages -- through the checks of test_gpu_simknn.py: sweeps of 1, 2 and an odd number of tiles,
column splits of unequal odd length, the seed-pass column groups, and a seeded build whose rows go through the retry pass."""
import pytest

import test_gpu_simknn as base

pytestmark = pytest.mark.gpu


@pytest.fixture
def debug_env():
    from sngnn_b200 import _C
    _C.lib().sng_set_debug_env(1)
    yield
    _C.lib().sng_set_debug_env(0)


# n = 200 / 500 / 1250: 1, 2 and 5 tiles per sweep (one issuer idle, each issuer once, issuer 0 one tile ahead);
# n = 2700 in 3 splits: 11 tiles as 3 + 4 + 4; n = 1750 in 2 splits: 7 tiles as 3 + 4.  d = 64: one K block, d = 65: two.
@pytest.mark.parametrize("n,d,ew,ns", [(200, 65, 4, 1), (500, 65, 4, 1), (1250, 65, 4, 1), (200, 64, 4, 1), (500, 64, 4, 1), (1250, 64, 4, 1),
                                       (2700, 65, 4, 3), (1750, 64, 4, 2)])
def test_split_stage1_candidates_contain_true_topk(n, d, ew, ns):
    base.test_stage1_candidates_contain_true_topk(n, d, ew, ns)


# samples of 6 tiles (2600 / 2) and 3 tiles (2500 / 4): every (tile parity, 32-column chunk) group, odd sweeps
@pytest.mark.parametrize("n,d,stride,ew", [(2600, 65, 2, 4), (2500, 64, 4, 4)])
def test_split_seed_pass_group_maxima(n, d, stride, ew):
    base.test_seed_pass_group_maxima(n, d, stride, ew)


# q = 1: the seeded threshold is far too aggressive, so many rows go through the retry pass, whose grid is sized for the
# maximum (idle CTA pairs leave at once)
@pytest.mark.parametrize("n,d,k,thr,rs,kind,stride,q", [(20000, 65, 10, -1.0, True, "clustered", 2, 1), (20000, 64, 10, -1.0, True, "normal", 2, 1)])
def test_split_seeded_build_through_retry_matches_oracle(n, d, k, thr, rs, kind, stride, q, monkeypatch, debug_env):
    base.test_seeded_build_matches_oracle(n, d, k, thr, rs, kind, stride, q, monkeypatch, debug_env)
