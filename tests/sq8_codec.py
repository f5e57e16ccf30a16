"""Host restatement of the SQ8 row codec (include/zvdb_b200.h, ZVDB_STORAGE_SQ8), for the tests.

train and encode are single IEEE float32 operations, which numpy reproduces exactly. The decode is one fused multiply-add,
fmaf((float)c, s, o), which numpy does not have: here it is computed exactly in float64 (c * s is exact there: 8 bits
times 24), the sum is rounded to odd (TwoSum error term, then the neighbour with an odd last bit when inexact), and the
result rounded once to float32. Rounding to odd with at least two extra bits and then to nearest gives the correctly
rounded sum, i.e. the bits of fmaf. tests/test_gpu_sq8_storage.py checks it against the C library's fmaf.
"""
import numpy as np


def _ordered(x):
    """float32 -> the order-preserving uint32 map of the kernels (-0 below +0)."""
    u = np.ascontiguousarray(x, np.float32).view(np.uint32)
    return u ^ np.where(u >> 31 != 0, np.uint32(0xFFFFFFFF), np.uint32(0x80000000))


def _from_ordered(o):
    o = np.asarray(o, np.uint32)
    return np.where(o >> 31 != 0, o ^ np.uint32(0x80000000), ~o).astype(np.uint32).view(np.float32)


def train(X, row_floats=None):
    """(scale, offset) float32 of the stored rows X [n, dim]: offset = min, scale = (max - min) / 255 per dimension;
    zero for padding up to row_floats when it is given."""
    X = np.ascontiguousarray(X, np.float32)
    o = _ordered(X)
    lo, hi = _from_ordered(o.min(axis=0)), _from_ordered(o.max(axis=0))
    scale = (hi - lo) / np.float32(255.0)
    offset = lo.copy()
    if row_floats is not None and row_floats > X.shape[1]:
        pad = np.zeros(row_floats - X.shape[1], np.float32)
        scale, offset = np.concatenate([scale, pad]), np.concatenate([offset, pad])
    return scale.astype(np.float32), offset.astype(np.float32)


def encode(X, scale, offset):
    """uint8 codes: clamp(rint((x - o) / s), 0, 255), 0 where s == 0."""
    X = np.asarray(X, np.float32)
    d = X.shape[-1]
    s, o = np.asarray(scale, np.float32)[:d], np.asarray(offset, np.float32)[:d]
    with np.errstate(divide="ignore", invalid="ignore", over="ignore"):
        v = np.rint((X - o) / np.where(s == 0, np.float32(1), s))
    c = np.clip(v, 0, 255)
    c = np.where(s == 0, 0, c)
    return c.astype(np.uint8)


def decode(C, scale, offset):
    """float32 rows fmaf((float)c, s, o), bit-exact."""
    C = np.asarray(C, np.uint8)
    d = C.shape[-1]
    s, o = np.asarray(scale, np.float32)[:d].astype(np.float64), np.asarray(offset, np.float32)[:d].astype(np.float64)
    p = C.astype(np.float64) * s                 # exact
    t = p + o
    bp = t - o                                   # TwoSum: t + err == p + o exactly
    err = (p - bp) + (o - (t - bp))
    even = (t.view(np.uint64) & np.uint64(1)) == 0
    fix = (err != 0) & even
    t = np.where(fix, np.nextafter(t, np.where(err > 0, np.inf, -np.inf)), t)
    return t.astype(np.float32)


def sq8_rows(X, codebook=None):
    """The rows an SQ8 traversal sees: decode(encode(X)) with the given codebook, or one trained on X."""
    scale, offset = codebook if codebook is not None else train(X)
    return decode(encode(X, scale, offset), scale, offset)
