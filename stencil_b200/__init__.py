"""stencil_b200 -- B200-native halo exchange + jacobi hot path behind the cwpearson/stencil API.

The compute lives in hand-written sm_100a CUDA (stencil_b200/csrc) behind a C ABI
(include/stencil_b200.h); this package is the Python host mirror of the reference's domain API.
"""
from ._lib import LIB_PATH, StencilError, lib  # noqa: F401
from .domain import (  # noqa: F401
    ALL_DIRS,
    CopyPlan,
    DataHandle,
    DistributedDomain,
    LocalDomain,
    Method,
    Partition,
    PlacementStrategy,
    Radius,
    box_copy,
    fill,
    get_neighbor,
    halo_extent,
    halo_pos,
    jacobi3d,
    prime_factors,
    raw_size,
)
from .reduce import ALFVEN, DIFF, EXP, VALUE, VECTOR, Stats, Workspace, reduce_box  # noqa: F401

__all__ = [n for n in dir() if not n.startswith("_")]
