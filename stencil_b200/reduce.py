"""Deterministic field reductions: min, max, sum and rms of a value per cell (sb_reduce, stencil_b200/csrc/reduce.cu).

The kinds are the filters of the reference's astaroth extract (astaroth/reductions.cuh:18-52); each RTYPE_* of
astaroth/user_defines.h:161-169 is one field of one pass:

    RTYPE_MAX, RTYPE_MIN, RTYPE_SUM          VALUE  .max / .min / .sum
    RTYPE_RMS                                VALUE  .rms
    RTYPE_RMS_EXP                            EXP    .rms
    RTYPE_ALFVEN_MAX / _MIN / _RMS           ALFVEN .max / .min / .rms   (operands uux, uuy, uuz, lnrho)
    length of a vector field (acReduceVec)   VECTOR .max / .min / .rms

Values and sums are FP64 for FP32 fields too.  Results are deterministic: the device combine has a fixed order, and the
host combines per-subdomain results in a fixed order (`combine`), so equal inputs give equal bits on every call.
"""
from __future__ import annotations

import ctypes as C
import math
from typing import Dict, Iterable, NamedTuple, Sequence, Tuple

from ._lib import Pitched, ReduceResult, StencilError, check, i3, lib, stream_ptr

VALUE, DIFF, VECTOR, EXP, ALFVEN = 0, 1, 2, 3, 4
NUM_OPERANDS = {VALUE: 1, DIFF: 2, VECTOR: 3, EXP: 1, ALFVEN: 4}

# one reduction before combining: (min f, max f, sum f, sum g, cells)
Partial = Tuple[float, float, float, float, int]
EMPTY: Partial = (math.inf, -math.inf, 0.0, 0.0, 0)


class Stats(NamedTuple):
    min: float
    max: float
    sum: float
    sum2: float  # sum of the squares g (for DIFF: the squared L2 norm of the difference)
    rms: float  # sqrt(sum2 / count); NaN for an empty region
    count: int


def _nan_min(m: float, f: float) -> float:
    return f if (f < m or f != f) else m


def _nan_max(m: float, f: float) -> float:
    return f if (f > m or f != f) else m


def combine(parts: Iterable[Partial]) -> Stats:
    """Combine partial results in the order given.  NaN in any part makes min, max and the sums NaN, like the kernel."""
    mn, mx, s, s2, n = EMPTY
    for p in parts:
        mn, mx = _nan_min(mn, float(p[0])), _nan_max(mx, float(p[1]))
        s += float(p[2])
        s2 += float(p[3])
        n += int(p[4])
    return Stats(mn, mx, s, s2, math.sqrt(s2 / n) if n else math.nan, n)


def combine_ranks(local: Dict[tuple, Partial], order: Sequence[tuple], world_size: int) -> Stats:
    """Collective over the ranks of torch.distributed when world_size > 1: every rank passes the partials of the subdomains
    it owns (keyed by global subdomain index), and every rank returns the combine of all of them in `order` -- the same
    bits on every rank, whichever rank owns which subdomain."""
    merged = dict(local)
    if world_size > 1:
        from .dist import all_gather_object

        for part in all_gather_object(local):
            merged.update(part)
    missing = [tuple(i) for i in order if tuple(i) not in merged]
    if missing:
        raise ValueError(f"no partial result for subdomains {missing}")
    return combine(merged[tuple(i)] for i in order)


class Workspace:
    """Device memory of one reduction at a time on one GPU (sb_reduce_workspace_bytes), zeroed once at creation."""

    def __init__(self, device: int):
        self.device = int(device)
        self.nbytes = int(check(lib().sb_reduce_workspace_bytes(self.device)))
        p = C.c_void_p()
        check(lib().sb_malloc(C.byref(p), self.nbytes, self.device))
        self.ptr = int(p.value)
        check(lib().sb_memset(C.c_void_p(self.ptr), 0, self.nbytes, self.device, None))
        check(lib().sb_device_sync(self.device))

    def launch(self, kind: int, operands: Sequence[Pitched], dtype_size: int, acc_origin, lo, hi, stream=None) -> None:
        """Enqueue one sb_reduce over [lo, hi) (global coordinates) on `stream`; `result` reads it back."""
        n = NUM_OPERANDS.get(kind)  # an unknown kind is rejected by the library
        if n is not None and len(operands) != n:
            raise StencilError(f"reduction kind {kind} takes {n} operands, got {len(operands)}")
        ops = (Pitched * max(1, len(operands)))(*operands)
        check(lib().sb_reduce(int(kind), ops, int(dtype_size), i3(acc_origin), i3(lo), i3(hi), C.c_void_p(self.ptr), stream_ptr(stream)))

    def result(self, stream=None) -> Tuple[float, float, float, float]:
        """(min, max, sum, sum2) of the last launch on `stream`; waits for it."""
        r = ReduceResult()
        check(lib().sb_memcpy(C.byref(r), C.c_void_p(self.ptr), C.sizeof(r), self.device, stream_ptr(stream)))
        check(lib().sb_stream_sync(self.device, stream_ptr(stream)))
        return (r.min, r.max, r.sum, r.sum2)

    def free(self) -> None:
        if self.ptr:
            lib().sb_free(C.c_void_p(self.ptr), self.device)
            self.ptr = 0

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


def cells(lo, hi) -> int:
    return math.prod(max(0, int(hi[a]) - int(lo[a])) for a in range(3))


def reduce_box(kind: int, operands: Sequence[Pitched], dtype_size: int, acc_origin, lo, hi, workspace: Workspace, stream=None) -> Stats:
    """One reduction over the box [lo, hi) (global coordinates; acc_origin = global coordinate of allocation element
    (0,0,0)) of raw device allocations, waited for on `stream`."""
    workspace.launch(kind, operands, dtype_size, acc_origin, lo, hi, stream)
    return combine([workspace.result(stream) + (cells(lo, hi),)])
