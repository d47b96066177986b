"""FP64 reference of the node-pair similarity histogram (sngnn_b200.toolbox.node_similarity_histogram).

TEST INFRASTRUCTURE ONLY (same import rule as `oracle/toolbox_ref.py`).

The values are those node_similarity_dense_small returns (R: SimGFAToolbox/dense.py:144-149): the N (N - 1) off-diagonal
cosines of the eps-normalised rows, binned with numpy.histogram's rule.  Besides the counts it returns a per-bin slack
("in band" of DESIGN.md §2 applied to bins): a kernel whose scores are within delta of the FP64 cosines can only differ
from these counts, bin by bin, by pairs that lie within delta of an edge that decides their count.
"""
import builtins

import torch
import torch.nn.functional as F


def histogram_with_slack(s, bins, range, delta):
    """(counts, slack) int64 [bins] of the values s (any shape, float64): clamped to [-1, 1], bin = floor((s - lo) * bins /
    (hi - lo)), s == hi in the last bin, values outside [lo, hi] not counted.  slack[b] = number of values within `delta`
    (strictly) of an edge of bin b whose side decides the count: interior edges, and lo / hi unless they are -1 / 1 (the
    clamp keeps a value there whatever its rounding)."""
    lo, hi = float(range[0]), float(range[1])
    s = s.reshape(-1).double().clamp(-1.0, 1.0)
    t = (s - lo) * (bins / (hi - lo))
    keep = (s >= lo) & (s <= hi)
    b = t.floor().clamp(0, bins - 1).long()
    counts = torch.bincount(b[keep], minlength=bins)
    slack = torch.zeros(bins, dtype=torch.int64, device=s.device)
    if delta > 0:
        e = t.round()                                       # nearest edge index
        near = ((t - e).abs() * ((hi - lo) / bins) < delta) & (e >= 0) & (e <= bins)
        near &= ~((e == 0) & (lo <= -1.0)) & ~((e == bins) & (hi >= 1.0))
        ei = e[near].long()
        slack += torch.bincount((ei - 1)[ei >= 1], minlength=bins)[:bins]          # the bin below the edge
        slack += torch.bincount(ei[ei < bins], minlength=bins)[:bins]              # the bin above it
    return counts, slack


def node_similarity_histogram_ref(x, bins, range, delta, block=1024):
    """FP64 (counts, slack) of the N (N - 1) off-diagonal cosines of the eps-normalised rows of x, blocked over rows (runs on
    x's device).  A kernel whose scores are within delta of these cosines gives |counts_kernel - counts| <= slack per bin."""
    n = F.normalize(x.double(), p=2.0, dim=-1)
    N = n.size(0)
    counts = torch.zeros(bins, dtype=torch.int64, device=n.device)
    slack = torch.zeros_like(counts)
    for r0 in builtins.range(0, N, block):             # `range` is the histogram range here, as in numpy.histogram
        r1 = min(N, r0 + block)
        s = n[r0:r1] @ n.t()
        off = torch.ones_like(s, dtype=torch.bool)
        r = torch.arange(r1 - r0, device=n.device)
        off[r, r0 + r] = False
        c, sl = histogram_with_slack(s[off], bins, range, delta)
        counts += c
        slack += sl
    return counts, slack
