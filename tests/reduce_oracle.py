"""numpy restatement of the field reductions (stencil_b200.reduce, sb_reduce) -- the reference the reduction tests
compare against, in float64 and in np.longdouble."""
from typing import Sequence

import numpy as np

from oracle.np_oracle import Vec, box

FOUR_PI = 4.0 * np.pi  # AcReal(4.0) * M_PI as a double, astaroth/reductions.cuh:47-50

REDUCE_OPERANDS = {"VALUE": 1, "DIFF": 2, "VECTOR": 3, "EXP": 1, "ALFVEN": 4}


def reduce_terms(kind: str, arrays: Sequence[np.ndarray], pos: Vec, ext: Vec, dtype=np.float64):
    """Per-cell value f and square g of a reduction over a box, in `dtype` (np.float64 or np.longdouble).  The filters of
    astaroth/reductions.cuh:18-52: dvalue / dsquared (VALUE), dlength_vec / dsquared_vec (VECTOR), exp and
    dexp_squared (EXP), dlength_alf / dsquared_alf (ALFVEN), and the difference of two fields (DIFF).  Every operation
    is rounded to `dtype` in the order written here: ((a*a + b*b) + c*c)."""
    n = REDUCE_OPERANDS[kind]
    assert len(arrays) == n, (kind, len(arrays))
    a, b, c, d = (list(box(x, pos, ext).astype(dtype) for x in arrays) + [None] * 3)[:4]
    if kind == "VALUE":
        return a, a * a
    if kind == "DIFF":
        t = a - b
        return t, t * t
    if kind == "EXP":
        e = np.exp(a)
        return e, e * e
    s = (a * a + b * b) + c * c
    if kind == "VECTOR":
        return np.sqrt(s), s
    den = dtype(FOUR_PI) * np.exp(d)
    return np.sqrt(s) / np.sqrt(den), s / den


def reduce_box(kind: str, arrays: Sequence[np.ndarray], pos: Vec, ext: Vec, dtype=np.float64) -> dict:
    """min f, max f, sum f, sum g (and the cell count) over the box [pos, pos + ext) of whole allocations.  An empty box
    gives +inf, -inf, 0, 0; a NaN anywhere in the box makes all four NaN."""
    f, g = reduce_terms(kind, arrays, pos, ext, dtype)
    if f.size == 0:
        return dict(min=dtype(np.inf), max=dtype(-np.inf), sum=dtype(0), sum2=dtype(0), count=0)
    return dict(min=f.min(), max=f.max(), sum=f.sum(dtype=dtype), sum2=g.sum(dtype=dtype), count=int(f.size))
