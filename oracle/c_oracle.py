"""ctypes front-end of oracle/stencil_oracle.c -- CPU oracle (TEST INFRASTRUCTURE, see oracle/__init__.py)."""
from __future__ import annotations

import ctypes as C
import os
import subprocess
from typing import Sequence, Tuple

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_SO = os.path.join(_HERE, "_build", "liboracle.so")


class Vec(C.Structure):
    _fields_ = [("x", C.c_int64), ("y", C.c_int64), ("z", C.c_int64)]

    @staticmethod
    def of(v: Sequence[int]) -> "Vec":
        return Vec(int(v[0]), int(v[1]), int(v[2]))


class Copy(C.Structure):
    _fields_ = [
        ("dst", C.c_void_p),
        ("src", C.c_void_p),
        ("draw", Vec),
        ("dpos", Vec),
        ("sraw", Vec),
        ("spos", Vec),
        ("ext", Vec),
        ("es", C.c_int64),
    ]


class AcParams(C.Structure):
    """so_ac_params: the uniforms solve<> reads (astaroth/user_kernels.h:389-427)."""

    _fields_ = [(n, C.c_double) for n in ("inv_dsx", "inv_dsy", "inv_dsz", "dt", "cs2_sound", "gamma", "cp_sound", "lnrho0", "lnT0", "mu0", "nu_visc", "zeta", "eta")]


def astaroth_conf_params(dt: float = 1e-8) -> AcParams:
    """The values the reference driver ends up with: astaroth/astaroth.conf:10-67 for what the file sets,
    the *_DEFAULT_VALUE statics (astaroth/user_kernels.h:30-35, 329, 367) for what it leaves out (NaN-filled
    config entries are skipped by acDeviceLoadScalarUniform, astaroth/kernels.cu:96-100), dt from
    astaroth/astaroth.cu:578."""
    ds = 0.04908738521
    return AcParams(1.0 / ds, 1.0 / ds, 1.0 / ds, dt, 1.0, 0.5, 1.0, 1.3, 1.2, 1.4, 5e-3, 0.01, 5e-3)


def build(force: bool = False) -> str:
    """Compile the C oracle with gcc (present in this image and on the GPU box)."""
    srcs = [os.path.join(_HERE, f) for f in ("stencil_oracle.c", "astaroth_oracle.c")]
    stale = (not os.path.exists(_SO)) or os.path.getmtime(_SO) < max(os.path.getmtime(s) for s in srcs)
    if force or stale:
        march = "x86-64-v3"
        try:
            with open("/proc/cpuinfo") as f:
                if " avx2 " not in f.read():
                    march = "x86-64"
        except OSError:
            pass
        subprocess.check_call(["make", "-C", _HERE, "-s", "-B", f"MARCH={march}"])
    return _SO


_lib = None


def lib() -> C.CDLL:
    global _lib
    if _lib is None:
        build()
        L = C.CDLL(_SO)
        L.so_num_threads.restype = C.c_int
        L.so_set_num_threads.argtypes = [C.c_int]
        L.so_translate.argtypes = [C.c_void_p, Vec, Vec, C.c_void_p, Vec, Vec, Vec, C.c_int64]
        L.so_pack.argtypes = [C.c_void_p, C.c_void_p, Vec, Vec, Vec, C.c_int64]
        L.so_unpack.argtypes = [C.c_void_p, Vec, Vec, C.c_void_p, Vec, C.c_int64]
        L.so_translate_many.argtypes = [C.POINTER(Copy), C.c_int64]
        for suf, ct in (("f32", C.c_float), ("f64", C.c_double)):
            getattr(L, "so_jacobi_" + suf).argtypes = [C.c_void_p, C.c_void_p, Vec, Vec, Vec, Vec, Vec, Vec]
            getattr(L, "so_fill_" + suf).argtypes = [C.c_void_p, Vec, Vec, Vec, ct]
            getattr(L, "so_sqdiff_" + suf).argtypes = [C.c_void_p, C.c_void_p, Vec, Vec, Vec]
            getattr(L, "so_sqdiff_" + suf).restype = C.c_double
        for suf in ("f32", "f64", "f80"):
            getattr(L, "so_astaroth_substep_" + suf).argtypes = [
                C.c_int, C.POINTER(C.c_void_p), C.POINTER(C.c_void_p), C.c_int64, C.c_int64,
                C.POINTER(C.c_int64), C.POINTER(C.c_int64), C.POINTER(AcParams),
            ]  # fmt: skip
        _lib = L
    return _lib


def _raw(a: np.ndarray) -> Vec:
    assert a.ndim == 3 and a.flags.c_contiguous
    return Vec(a.shape[2], a.shape[1], a.shape[0])


def _suffix(a: np.ndarray) -> str:
    return {np.dtype(np.float32): "f32", np.dtype(np.float64): "f64"}[a.dtype]


def num_threads() -> int:
    return lib().so_num_threads()


def set_num_threads(n: int) -> None:
    lib().so_set_num_threads(n)


def translate(dst: np.ndarray, dpos, src: np.ndarray, spos, ext) -> None:
    assert dst.dtype.itemsize == src.dtype.itemsize
    lib().so_translate(dst.ctypes.data, _raw(dst), Vec.of(dpos), src.ctypes.data, _raw(src), Vec.of(spos), Vec.of(ext), src.dtype.itemsize)


def pack(src: np.ndarray, pos, ext) -> np.ndarray:
    out = np.empty(ext[0] * ext[1] * ext[2], dtype=src.dtype)
    lib().so_pack(out.ctypes.data, src.ctypes.data, _raw(src), Vec.of(pos), Vec.of(ext), src.dtype.itemsize)
    return out


def unpack(dst: np.ndarray, buf: np.ndarray, pos, ext) -> None:
    assert buf.flags.c_contiguous
    lib().so_unpack(dst.ctypes.data, _raw(dst), Vec.of(pos), buf.ctypes.data, Vec.of(ext), dst.dtype.itemsize)


def make_copies(items) -> Tuple[C.Array, int]:
    """items: iterable of (dst_arr, dpos, src_arr, spos, ext) -> a ctypes array for translate_many."""
    items = list(items)
    arr = (Copy * len(items))()
    for i, (d, dpos, s, spos, ext) in enumerate(items):
        arr[i] = Copy(d.ctypes.data, s.ctypes.data, _raw(d), Vec.of(dpos), _raw(s), Vec.of(spos), Vec.of(ext), s.dtype.itemsize)
    return arr, len(items)


def translate_many(copies, n: int) -> None:
    lib().so_translate_many(copies, n)


def jacobi_region(dst: np.ndarray, src: np.ndarray, acc_origin, lo, hi, clo, chi) -> None:
    assert dst.shape == src.shape and dst.dtype == src.dtype
    getattr(lib(), "so_jacobi_" + _suffix(src))(
        dst.ctypes.data, src.ctypes.data, _raw(src), Vec.of(acc_origin), Vec.of(lo), Vec.of(hi), Vec.of(clo), Vec.of(chi)
    )


def fill(dst: np.ndarray, pos, ext, v: float) -> None:
    getattr(lib(), "so_fill_" + _suffix(dst))(dst.ctypes.data, _raw(dst), Vec.of(pos), Vec.of(ext), v)


def sqdiff(a: np.ndarray, b: np.ndarray, pos, ext) -> float:
    return getattr(lib(), "so_sqdiff_" + _suffix(a))(a.ctypes.data, b.ctypes.data, _raw(a), Vec.of(pos), Vec.of(ext))


def longdouble_is_extended() -> bool:
    """True where np.longdouble is the x87 80-bit format (64-bit mantissa), i.e. the `f80` oracle is a real reference."""
    return np.finfo(np.longdouble).nmant >= 63


def astaroth_substep(step: int, fin, fout, lo, hi, params: "AcParams") -> None:
    """solve<step> on the memory-offset box [lo, hi) (astaroth/kernels.cu:62-87).  fin / fout: 8 arrays
    (lnrho, uux, uuy, uuz, ax, ay, az, entropy) of identical (mz, my, mx) shape and dtype (float32, float64, or
    longdouble for the extended-precision reference); fout is updated in place."""
    a0 = fin[0]
    assert len(fin) == 8 and len(fout) == 8
    for a in list(fin) + list(fout):
        assert a.shape == a0.shape and a.dtype == a0.dtype and a.flags.c_contiguous
    mz, my, mx = a0.shape
    pin = (C.c_void_p * 8)(*[a.ctypes.data for a in fin])
    pout = (C.c_void_p * 8)(*[a.ctypes.data for a in fout])
    clo, chi = (C.c_int64 * 3)(*lo), (C.c_int64 * 3)(*hi)
    if a0.dtype == np.longdouble:
        assert longdouble_is_extended(), "np.longdouble is not the 80-bit format the f80 oracle is compiled for"
        suf = "f80"
    else:
        suf = _suffix(a0)
    getattr(lib(), "so_astaroth_substep_" + suf)(step, pin, pout, mx, my, clo, chi, C.byref(params))
