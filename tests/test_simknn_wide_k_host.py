"""The wide all-pairs build without a GPU: argument checks of sng_simknn_wide_count / _select and the Python-side rejection
of lists with 2^31 or more entries, which happens before any kernel runs."""
import ctypes

import pytest
import torch

_P = ctypes.c_void_p
FAKE = _P(256)                         # never dereferenced: every call below fails its argument checks first


def _count(L, **kw):
    a = dict(xq=FAKE, xall=FAKE, ldh=80, nq=100, q_offset=0, n=1000, d=65, top_k=100, thr=0.0, rs=1, offsets=FAKE, ws=FAKE,
             wbytes=1 << 40)
    a.update(kw)
    return L.sng_simknn_wide_count(*a.values(), None)


def _select(L, **kw):
    a = dict(xq=FAKE, xall=FAKE, ldh=80, xq32=FAKE, xall32=FAKE, ld32=68, nq=100, q_offset=0, n=1000, d=65, top_k=100, thr=0.0,
             rs=1, offsets=FAKE, cand=FAKE, idx=FAKE, sim=FAKE, cnt=FAKE, n_exact=None, ws=FAKE, wbytes=1 << 40)
    a.update(kw)
    return L.sng_simknn_wide_select(*a.values(), None)


def test_wide_entry_points_validate_their_arguments():
    from sngnn_b200 import _C
    L = _C.lib()
    common = ((dict(xq=None), "null operand"), (dict(top_k=0), "top_k=0"), (dict(n=1, nq=1, rs=1), "no candidate column"),
              (dict(q_offset=950), "beyond"), (dict(ldh=72), "ldb"), (dict(d=5000, ldh=5008), "not supported"),
              (dict(nq=50000, n=50000, top_k=2 ** 40), "2^31"), (dict(ws=None), "workspace"), (dict(wbytes=16), "workspace too small"))
    for fn, call in (("sng_simknn_wide_count", _count), ("sng_simknn_wide_select", _select)):
        for kw, msg in common + ((dict(offsets=None), "null"),):
            assert call(L, **kw) != 0, (fn, kw)
            assert fn in _C.last_error() and msg in _C.last_error(), (fn, kw, _C.last_error())
    for kw in (dict(ld32=66), dict(xq32=None), dict(cand=None), dict(idx=None)):
        assert _select(L, **kw) != 0 and "sng_simknn_wide_select" in _C.last_error(), kw
    assert L.sng_simknn_wide_workspace_bytes(0, 10, 8, 100) == 0
    assert L.sng_simknn_wide_workspace_bytes(50000, 50000, 8, 2 ** 40) == 0
    assert L.sng_simknn_wide_workspace_bytes(100, 1000, 65, 100) > 0


def test_list_entry_limit_is_rejected_before_any_kernel():
    from sngnn_b200 import simknn
    n, d = 50000, 4
    xf = torch.zeros(n, d)                                    # host tensors: nothing may reach the library
    xh = torch.zeros(n, 16, dtype=torch.float16)
    with pytest.raises(ValueError, match="2\\*\\*31"):
        simknn.build_knn_normalized(xf, xh, d, 2 ** 40, 0.5, True)
    with pytest.raises(ValueError, match="2\\*\\*31"):
        simknn.build_knn_normalized(xf, xh, d, 46000, 0.5, True)
    assert simknn.list_width(n, 2 ** 40, True) == n - 1 and simknn.list_width(n, 2 ** 40, False) == n
    assert simknn.list_width(10, 50, True) == 50            # up to 64 the width is top_k itself, as before
    assert simknn.list_width(10, 100, True) == 9


def test_list_transpose_and_backward_accept_any_width():
    from sngnn_b200 import _C
    L = _C.lib()
    assert L.sng_list_transpose_workspace_bytes(1000, 1000, 5000) > 0
    assert L.sng_list_transpose_workspace_bytes(1 << 20, 1 << 12, 5000) == 0         # 2^32 entries
