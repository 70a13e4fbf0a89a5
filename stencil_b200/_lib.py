"""ctypes binding of the C ABI (include/stencil_b200.h -> stencil_b200/libstencil_b200.so).

There is no CPU fallback: if the shared library is missing or a CUDA call fails, the call raises.
"""
from __future__ import annotations

import ctypes as C
import os
from typing import Sequence

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("SB_LIB_PATH") or os.path.join(_HERE, "libstencil_b200.so")


class StencilError(RuntimeError):
    pass


class Pitched(C.Structure):
    """sb_pitched: the cudaPitchedPtr the reference passes around (ptr, pitch bytes, rows per plane)."""

    _fields_ = [("ptr", C.c_void_p), ("pitch", C.c_int64), ("ysize", C.c_int64)]


class BoxCopy(C.Structure):
    """sb_box_copy"""

    _fields_ = [
        ("dst", Pitched),
        ("dst_pos", C.c_int64 * 3),
        ("src", Pitched),
        ("src_pos", C.c_int64 * 3),
        ("extent", C.c_int64 * 3),
        ("elem_size", C.c_int64),
    ]


I3 = C.c_int64 * 3
I27 = C.c_int64 * 27

class AstarothParams(C.Structure):
    """sb_astaroth_params: the uniforms solve<> reads through DCONST (astaroth/user_kernels.h:389-427)."""

    _fields_ = [(n, C.c_double) for n in ("inv_dsx", "inv_dsy", "inv_dsz", "dt", "cs2_sound", "gamma", "cp_sound", "lnrho0", "lnT0", "mu0", "nu_visc", "zeta", "eta")]


class HaloPush(C.Structure):
    """sb_halo_push: the six face neighbours' output allocations (-x, +x, -y, +y, -z, +z)."""

    _fields_ = [("nbr", Pitched * 6), ("nbr_zsize", C.c_int64 * 6), ("x_dense", C.c_int64 * 2), ("x_recv", C.c_void_p * 2)]


FUSED_MAX_GROUPS = 4096  # SB_FUSED_MAX_GROUPS


class StepSync(C.Structure):
    """sb_step_sync: per-face mailbox rows of the in-kernel handshake of sb_jacobi3d_fused_sync."""

    _fields_ = [("wait_rows", C.c_void_p * 6), ("signal_rows", C.c_void_p * 6), ("wait_value", C.c_uint32), ("signal_value", C.c_uint32)]


class ReduceResult(C.Structure):
    """sb_reduce_result: min f, max f, sum f, sum g of one reduction (see stencil_b200.reduce)."""

    _fields_ = [(n, C.c_double) for n in ("min", "max", "sum", "sum2")]


# every symbol include/stencil_b200.h declares: (restype, argtypes)
_SIGS = {
    "sb_last_error": (C.c_char_p, []),
    "sb_version": (C.c_int, []),
    "sb_launch_count": (C.c_uint64, []),
    "sb_halo_pos": (C.c_int, [I3, I3, I27, C.c_int, I3]),
    "sb_halo_extent": (C.c_int, [I3, I3, I27, I3]),
    "sb_raw_size": (C.c_int, [I3, I27, I3]),
    "sb_prime_factors": (C.c_int, [C.c_int64, C.POINTER(C.c_int64), C.c_int]),
    "sb_rank_partition": (C.c_int, [I3, C.c_int64, I3, I3, I3]),
    "sb_node_partition": (C.c_int, [I3, I27, C.c_int64, C.c_int64, I3, I3, I3, I3]),
    "sb_subdomain_size": (C.c_int, [I3, I3, I3, I3]),
    "sb_subdomain_origin": (C.c_int, [I3, I3, I3, I3]),
    "sb_interior": (C.c_int, [I3, I3, I27, I3, I3]),
    "sb_exterior": (C.c_int, [I3, I3, I27, C.POINTER(C.c_int64), C.POINTER(C.c_int64)]),
    "sb_pack": (C.c_int, [C.c_void_p, Pitched, I3, I3, C.c_int64, C.c_void_p]),
    "sb_unpack": (C.c_int, [Pitched, C.c_void_p, I3, I3, C.c_int64, C.c_void_p]),
    "sb_translate": (C.c_int, [Pitched, I3, Pitched, I3, I3, C.c_int64, C.c_void_p]),
    "sb_copy_plan_create": (C.c_int, [C.POINTER(C.c_void_p), C.c_int, C.POINTER(BoxCopy), C.c_int64]),
    "sb_copy_plan_launch": (C.c_int, [C.c_void_p, C.c_void_p]),
    "sb_copy_plan_bytes": (C.c_int64, [C.c_void_p]),
    "sb_copy_plan_num_tiles": (C.c_int64, [C.c_void_p]),
    "sb_copy_plan_num_tma_segments": (C.c_int64, [C.c_void_p]),
    "sb_copy_plan_destroy": (C.c_int, [C.c_void_p]),
    "sb_signal": (C.c_int, [C.POINTER(C.c_void_p), C.c_int, C.c_uint32, C.c_int, C.c_void_p]),
    "sb_wait": (C.c_int, [C.c_void_p, C.c_int, C.c_uint32, C.c_int, C.c_void_p]),
    "sb_jacobi3d": (C.c_int, [Pitched, Pitched, C.c_int, I3, I3, I3, I3, I3, C.c_void_p]),
    "sb_jacobi3d_regions": (C.c_int, [Pitched, Pitched, C.c_int, I3, C.c_int, C.POINTER(C.c_int64), C.POINTER(C.c_int64), I3, I3, C.c_void_p]),
    "sb_astaroth_substep": (C.c_int, [C.c_int, C.POINTER(C.c_void_p), C.POINTER(C.c_void_p), C.c_int, I3, I3, I3, C.POINTER(AstarothParams), C.c_int, C.c_void_p]),
    "sb_jacobi3d_fused": (C.c_int, [Pitched, Pitched, C.c_int, I3, I3, I3, I3, I3, C.POINTER(HaloPush), C.c_void_p]),
    "sb_jacobi3d_fused_sync": (C.c_int, [Pitched, Pitched, C.c_int, I3, I3, I3, I3, I3, C.POINTER(HaloPush), C.POINTER(StepSync), C.c_void_p]),
    "sb_fill": (C.c_int, [Pitched, C.c_int, I3, I3, I3, C.c_double, C.c_void_p]),
    "sb_sqdiff": (C.c_int, [Pitched, Pitched, C.c_int, I3, I3, I3, C.c_void_p, C.c_void_p]),
    "sb_reduce_workspace_bytes": (C.c_int64, [C.c_int]),
    "sb_reduce": (C.c_int, [C.c_int, C.POINTER(Pitched), C.c_int, I3, I3, I3, C.c_void_p, C.c_void_p]),
    "sb_device_count": (C.c_int, [C.POINTER(C.c_int)]),
    "sb_malloc": (C.c_int, [C.POINTER(C.c_void_p), C.c_size_t, C.c_int]),
    "sb_free": (C.c_int, [C.c_void_p, C.c_int]),
    "sb_memset": (C.c_int, [C.c_void_p, C.c_int, C.c_size_t, C.c_int, C.c_void_p]),
    "sb_memcpy": (C.c_int, [C.c_void_p, C.c_void_p, C.c_size_t, C.c_int, C.c_void_p]),
    "sb_stream_sync": (C.c_int, [C.c_int, C.c_void_p]),
    "sb_device_sync": (C.c_int, [C.c_int]),
    "sb_enable_peer": (C.c_int, [C.c_int, C.c_int, C.POINTER(C.c_int)]),
    "sb_ipc_export": (C.c_int, [C.c_void_p, C.c_void_p]),
    "sb_ipc_import": (C.c_int, [C.c_void_p, C.c_int, C.POINTER(C.c_void_p)]),
    "sb_ipc_close": (C.c_int, [C.c_void_p, C.c_int]),
}

_lib = None


def lib() -> C.CDLL:
    """Load the shared library (once).  Raises StencilError if it has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise StencilError(
                f"{LIB_PATH} not found: build it with `make` (or `python -c 'import __graft_entry__ as g; g.build()'`); "
                "stencil_b200 has no CPU fallback"
            )
        L = C.CDLL(LIB_PATH)
        for name, (res, args) in _SIGS.items():
            fn = getattr(L, name)  # AttributeError if the header and the library drifted apart
            fn.restype = res
            fn.argtypes = args
        _lib = L
    return _lib


def check(rc: int) -> int:
    if rc < 0:
        raise StencilError(f"stencil_b200 error {rc}: {lib().sb_last_error().decode()}")
    return rc


def i3(v: Sequence[int]) -> I3:
    return I3(int(v[0]), int(v[1]), int(v[2]))


def o3():
    return I3(0, 0, 0)


def t3(a) -> tuple:
    return (int(a[0]), int(a[1]), int(a[2]))


def stream_ptr(stream) -> C.c_void_p:
    """Accept None (default stream), an int handle, or a torch.cuda.Stream."""
    if stream is None:
        return C.c_void_p(0)
    if isinstance(stream, int):
        return C.c_void_p(stream)
    return C.c_void_p(stream.cuda_stream)
