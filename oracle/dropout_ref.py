"""numpy oracle of the counter-based row dropout (include/sng.h: sng_row_dropout_fwd / sng_row_dropout_bwd).

Philox4x32-10 (Salmon et al., "Parallel random numbers: as easy as 1, 2, 3", SC 2011; the Random123 multipliers and Weyl
constants) keyed by (seed lo, seed hi); element e = (row_offset + i) c + j of a layer of logical width c takes word e & 3 of
the block at counter (e >> 2 lo, e >> 2 hi, call lo, call hi) and is kept iff (w >> 8) >= round(p 2^24).  The forward and
backward below follow the kernels' select form in FP32 (bit-exact targets) and in FP64 (references for the sharded tests).
"""
import numpy as np

M0, M1 = np.uint64(0xD2511F53), np.uint64(0xCD9E8D57)
W0, W1 = 0x9E3779B9, 0xBB67AE85
_MASK32 = np.uint64(0xFFFFFFFF)

# Random123 known-answer vectors (kat_vectors: philox4x32 10): (counter, key) -> output
KAT = [
    ((0, 0, 0, 0), (0, 0), (0x6627e8d5, 0xe169c58d, 0xbc57ac4c, 0x9b00dbd8)),
    ((0xffffffff,) * 4, (0xffffffff,) * 2, (0x408f276d, 0x41c83b0e, 0xa20bc7c6, 0x6d5451fd)),
    ((0x243f6a88, 0x85a308d3, 0x13198a2e, 0x03707344), (0xa4093822, 0x299f31d0), (0xd16cfe09, 0x94fdcceb, 0x5001e420, 0x24126ea1)),
]


def philox4x32_10(c0, c1, c2, c3, k0, k1):
    """Philox4x32-10 on arrays of 32-bit counter words (broadcast); returns the four output words as uint64 arrays < 2^32."""
    c0, c1, c2, c3 = (np.asarray(v, dtype=np.uint64) & _MASK32 for v in (c0, c1, c2, c3))
    k0, k1 = int(k0) & 0xFFFFFFFF, int(k1) & 0xFFFFFFFF
    for _ in range(10):
        p0, p1 = M0 * c0, M1 * c2                     # < 2^64: exact in uint64
        hi0, lo0, hi1, lo1 = p0 >> np.uint64(32), p0 & _MASK32, p1 >> np.uint64(32), p1 & _MASK32
        c0, c1, c2, c3 = hi1 ^ c1 ^ np.uint64(k0), lo1, hi0 ^ c3 ^ np.uint64(k1), lo0
        k0, k1 = (k0 + W0) & 0xFFFFFFFF, (k1 + W1) & 0xFFFFFFFF
    return c0, c1, c2, c3


def threshold(p):
    """t = round(p 2^24) of the FP32 p the kernel receives (ties away from zero, as floor(x + 0.5))."""
    return int(np.floor(float(np.float32(p)) * 16777216.0 + 0.5))


def scale32(p):
    """s = 1.0f / (1.0f - p) in FP32 (inf at p = 1, where every element is dropped)."""
    with np.errstate(divide="ignore"):
        return np.float32(1.0) / (np.float32(1.0) - np.float32(p))


def keep_mask(n, c, row_offset, seed, call, p):
    """bool [n, c]: the keep bits of rows [row_offset, row_offset + n) of a width-c layer."""
    e = (np.uint64(row_offset) + np.arange(n, dtype=np.uint64))[:, None] * np.uint64(c) + np.arange(c, dtype=np.uint64)[None, :]
    q = e >> np.uint64(2)
    seed, call = int(seed), int(call)
    w = philox4x32_10(q & _MASK32, q >> np.uint64(32), call & 0xFFFFFFFF, call >> 32, seed & 0xFFFFFFFF, seed >> 32)
    sel = (e & np.uint64(3)).astype(np.int64)
    word = np.choose(sel, w)
    return (word >> np.uint64(8)) >= np.uint64(threshold(p))


def forward(z, row_offset, seed, call, p, relu):
    """FP32: exactly the kernel's y; FP64 input: the same select in FP64 with s = 1 / (1 - p)."""
    z = np.asarray(z)
    keep = keep_mask(z.shape[0], z.shape[1], row_offset, seed, call, p)
    a = np.maximum(z, 0) if relu else z
    s = scale32(p) if z.dtype == np.float32 else (1.0 / (1.0 - float(np.float32(p))) if p < 1 else np.inf)
    with np.errstate(over="ignore", invalid="ignore"):
        return np.where(keep, a * s, np.zeros((), z.dtype)).astype(z.dtype)


def backward(z, g, row_offset, seed, call, p, relu):
    g = np.asarray(g)
    keep = keep_mask(g.shape[0], g.shape[1], row_offset, seed, call, p)
    if relu:
        keep = keep & (np.asarray(z) > 0)
    s = scale32(p) if g.dtype == np.float32 else (1.0 / (1.0 - float(np.float32(p))) if p < 1 else np.inf)
    with np.errstate(over="ignore", invalid="ignore"):
        return np.where(keep, g * s, np.zeros((), g.dtype)).astype(g.dtype)
