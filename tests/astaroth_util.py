"""Shared pieces of the astaroth parity tests (CPU and GPU sides)."""
import os

import numpy as np

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "astaroth_solve_ref.npz")
DS = 0.04908738521

# Error bound of the CUDA kernels, in units of the dtype's epsilon, relative to max(1, max|f|) of each field: see
# tolerance().  Every kernel variant measured within 5.5 of the extended-precision oracle on a B200 (DESIGN.md 2.3).
K_ULP = 32

# The uniforms of solve<> in AstarothParams / AcParams field order, after inv_dsx, inv_dsy, inv_dsz, dt.
PARAM_NAMES = ("cs2_sound", "gamma", "cp_sound", "lnrho0", "lnT0", "mu0", "nu_visc", "zeta", "eta")
# astaroth.conf (stencil_b200.astaroth.conf_params): equal spacings, nu == eta, cs2 == cp == 1, so a kernel that mixes
# those up still matches.
CONF = dict(inv_ds=(1.0 / DS,) * 3, cs2_sound=1.0, gamma=0.5, cp_sound=1.0, lnrho0=1.3, lnT0=1.2, mu0=1.4, nu_visc=5e-3, zeta=0.01, eta=5e-3)
# every value distinct and none equal to 1: swapping two parameters, or dividing where the code should multiply,
# changes the result
DISTINCT = dict(inv_ds=(1.0 / 0.049, 1.0 / 0.053, 1.0 / 0.046), cs2_sound=0.7, gamma=0.6, cp_sound=1.6, lnrho0=1.3, lnT0=1.2, mu0=1.4,
                nu_visc=4e-3, zeta=0.013, eta=6e-3)  # fmt: skip
PARAM_SETS = {"conf": CONF, "distinct": DISTINCT}
# dt = 1e-3 moves lnrho and A by < 1 % per substep, so a check at that dt mostly sees the rounding of `in`; at DT_RATE the
# first substep moves every field by more than 10 % of its max (asserted where it is used), so the rates are what is checked
DT_RATE = 0.05


BOXES = [
    # raw size (x,y,z), lo, hi
    ((38, 34, 30), (3, 3, 3), (35, 31, 27)),  # the whole compute region, partial tiles in x and y
    ((70, 26, 41), (3, 3, 3), (67, 23, 38)),
    ((40, 40, 40), (6, 6, 6), (34, 34, 34)),  # an interior region
    ((40, 40, 40), (3, 3, 3), (6, 37, 37)),  # x-face exterior slab (thin -> cell kernel under AUTO)
    ((40, 40, 40), (6, 34, 3), (34, 37, 37)),  # y-face slab
    ((40, 40, 40), (6, 6, 34), (34, 34, 37)),  # z-face slab
    ((23, 22, 21), (5, 4, 3), (16, 17, 18)),  # odd row length: no TMA
]


def param_values(pset: dict, dt: float) -> tuple:
    """The 13 doubles of AstarothParams / AcParams (same field order) for a parameter set and dt."""
    return (*pset["inv_ds"], dt, *(pset[n] for n in PARAM_NAMES))


def make_fields(shape_xyz, seed: int, dtype=np.float64, smooth: float = 1.0, noise: float = 0.25):
    """16 arrays (in[8], out[8]) of raw size shape_xyz (x, y, z): seeded noise + a smooth component, all O(1)."""
    mx, my, mz = shape_xyz
    rng = np.random.default_rng(seed)
    a = rng.uniform(-1.0, 1.0, size=(16, mz, my, mx))
    Z, Y, X = np.meshgrid(np.arange(mz) * DS, np.arange(my) * DS, np.arange(mx) * DS, indexing="ij")
    for f in range(16):
        a[f] = noise * a[f] + smooth * np.sin((1 + f % 3) * X + 0.3 * f) * np.cos((1 + f % 2) * Y) * np.sin(2 * Z + f)
    return [np.ascontiguousarray(a[f].astype(dtype)) for f in range(16)]


def box_slice(lo, hi):
    """[lo, hi) in (x, y, z) as an index of a [z, y, x] array."""
    return (slice(lo[2], hi[2]), slice(lo[1], hi[1]), slice(lo[0], hi[0]))


def reference_substeps(fin, fout, lo, hi, params) -> list:
    """The extended-precision oracle (`f80`) chained over solve<0>, <1>, <2> into one `out`, as the driver does, on the
    given (float32 or float64) inputs widened exactly.  Returns, per substep, the 8 fields of `out` on the box."""
    from oracle import c_oracle as co

    wide_in = [a.astype(np.longdouble) for a in fin]
    cur = [a.astype(np.longdouble) for a in fout]
    res = []
    for step in range(3):
        co.astaroth_substep(step, wide_in, cur, lo, hi, params)
        res.append([c[box_slice(lo, hi)].copy() for c in cur])
    return res


def err_over_eps(got, want, dtype) -> np.ndarray:
    """Per field: max|got - want| / max(1, max|want|), in units of finfo(dtype).eps.  got / want: the 8 fields on the box."""
    eps = float(np.finfo(dtype).eps)
    out = []
    for a, b in zip(got, want):
        b = b.astype(np.longdouble)
        err = np.abs(a.astype(np.longdouble) - b).max()
        out.append(float(err / max(np.longdouble(1), np.abs(b).max())) / eps)
    return np.array(out)


def tolerance(dtype) -> float:
    """Relative to max(1, max|f|) of the compared field: K_ULP units of the dtype's epsilon (FP64 7.1e-15, FP32 3.8e-6).
    The CUDA kernels contract a*b+c into FMAs, hoist 1/cp and 1/mu0, and fold exp(lnT0 + arg); the FP32 / FP64 oracles
    (-ffp-contract=off) do not.  Either side lands a few ulp of the field from the extended-precision result, far below
    what a wrong coefficient, a swapped parameter or a wrong neighbour moves (tests/test_oracle_astaroth.py)."""
    return K_ULP * float(np.finfo(dtype).eps)
