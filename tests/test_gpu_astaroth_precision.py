"""The astaroth solve<step> kernels (stencil_b200/csrc/astaroth.cu) against the extended-precision oracle, at a bound of
K_ULP units of the dtype's epsilon (astaroth_util.tolerance).

Every variant (AUTO, CELL, TILE, TEAM, TEAM_TMA, TEAM3_TMA) and both dtypes, over
  * two parameter sets: astaroth.conf, and one with every value distinct (catches nu / eta, one spacing for three axes,
    cp multiplied instead of divided, which the conf values cannot tell apart);
  * dt = 1e-3 and a rate-dominated dt (every field moves by more than 10 % in one substep);
  * whole regions, interior regions, every face slab, corners, boxes narrower than a tile in x and y, boxes one or two
    planes deep, z chunks that do not divide the depth;
  * inputs 8 bytes past a 16-byte boundary (how LocalDomain places FP64 radius-3 allocations), fields with different
    16-byte phases, odd row lengths, FP32: the TMA-fed kernels run where they apply and are rejected where they do not;
and two checks that need no tolerance: dt = 0 leaves `out` equal to `in` on the box and untouched outside it, and NaN in
every input cell outside the stencil footprint never reaches the result.

Each test records the worst err / eps per field as the junit property `err_over_eps` (pytest --junitxml)."""
import numpy as np
import pytest

import stencil_b200 as sb
from astaroth_util import BOXES, DISTINCT, DT_RATE, K_ULP, PARAM_SETS, box_slice, err_over_eps, make_fields, param_values, reference_substeps
from gpu_util import DevArray
from oracle import c_oracle as co
from stencil_b200 import astaroth as ac

pytestmark = pytest.mark.gpu
needs_f80 = pytest.mark.skipif(not co.longdouble_is_extended(), reason="np.longdouble is not the 80-bit extended format: no reference")

VARIANTS = [ac.AUTO, ac.CELL, ac.TILE, ac.TEAM, ac.TEAM_TMA, ac.TEAM3_TMA]
VNAMES = {ac.AUTO: "auto", ac.CELL: "cell", ac.TILE: "tile", ac.TEAM: "team", ac.TEAM_TMA: "team_tma", ac.TEAM3_TMA: "team3_tma"}
DTYPES = [np.float64, np.float32]
DTS = {"dt1e-3": 1e-3, "dtrate": DT_RATE}


def tma_rejects(variant, dtype, mx, shifts=None) -> bool:
    """The TMA-fed kernels need FP64, a row of a multiple of 16 bytes and one 16-byte phase for all 8 inputs; asked for
    explicitly where that does not hold, the call is rejected (TEAM falls back to the cp.async-fed ring instead)."""
    if variant not in (ac.TEAM_TMA, ac.TEAM3_TMA):
        return False
    return np.dtype(dtype) != np.float64 or mx % 2 != 0 or len(set(shifts or [0])) > 1


def params(pset: dict, dt: float):
    v = param_values(pset, dt)
    return ac.AstarothParams(*v), co.AcParams(*v)


def upload(a: np.ndarray, shift: int):
    """`a` in device memory `shift` elements past the start of a (256-byte aligned) allocation: (DevArray, pointer)."""
    buf = np.zeros(a.size + shift, a.dtype)
    buf[shift:] = a.ravel()
    d = DevArray(buf)
    return d, d.ptr + shift * a.itemsize


def run_substeps(fin, fout, lo, hi, gp, variant, shifts=None):
    """solve<0>, <1>, <2> into one `out` on the GPU, inputs uploaded once (input f `shifts[f]` elements past an aligned
    allocation).  Returns the 8 `out` arrays after each substep."""
    shifts = shifts or [0] * 8
    ins = [upload(a, s) for a, s in zip(fin, shifts)]
    outs = [upload(a, 0) for a in fout]
    mz, my, mx = fin[0].shape
    try:
        res = []
        for step in range(3):
            ac.substep(step, [p for _, p in ins], [p for _, p in outs], fin[0].dtype.itemsize, (mx, my, mz), lo, hi, gp, variant)
            res.append([d.get().reshape(fin[0].shape) for d, _ in outs])
        return res
    finally:
        for d, _ in ins + outs:
            d.free()


_REF = {}


def reference(raw, lo, hi, dtype, pset_name, dt, seed, poison=False):
    """(fin, fout, per-substep f80 reference on the box), computed once per case: the variants of a case are
    parametrized innermost, so they run back to back and a few cached cases suffice."""
    key = (raw, lo, hi, np.dtype(dtype).str, pset_name, dt, seed, poison)
    if key not in _REF:
        if len(_REF) >= 4:
            _REF.clear()
        f = make_fields(raw, seed=seed, dtype=dtype)
        fin, fout = f[:8], f[8:]
        if poison:
            fin, fout = poisoned(fin, fout, lo, hi)
        _REF[key] = (fin, fout, reference_substeps(fin, fout, lo, hi, params(PARAM_SETS[pset_name], dt)[1]))
    return _REF[key]


def poisoned(fin, fout, lo, hi):
    """NaN in every input cell outside the stencil footprint [lo - 3, hi + 3) and in every `out` cell outside [lo, hi)."""
    foot = box_slice([v - 3 for v in lo], [v + 3 for v in hi])
    pin, pout = [], []
    for a in fin:
        p = np.full_like(a, np.nan)
        p[foot] = a[foot]
        pin.append(p)
    for a in fout:
        p = np.full_like(a, np.nan)
        p[box_slice(lo, hi)] = a[box_slice(lo, hi)]
        pout.append(p)
    return pin, pout


def check_against_reference(got, fout, ref, lo, hi, dtype, record_property, what):
    """Every substep within K_ULP eps of the reference on the box, every cell outside the box untouched."""
    inside = box_slice(lo, hi)
    worst = np.zeros(8)
    for step in range(3):
        box = [a[inside] for a in got[step]]
        for f, a in enumerate(box):
            assert np.isfinite(a).all(), (what, step, ac.FIELDS[f], "non-finite output")
        r = err_over_eps(box, ref[step], dtype)
        worst = np.maximum(worst, r)
        assert (r <= K_ULP).all(), (what, step, {ac.FIELDS[f]: round(float(r[f]), 2) for f in range(8)})
    record_property("err_over_eps", {ac.FIELDS[f]: round(float(worst[f]), 3) for f in range(8)})
    outside = np.ones(fout[0].shape, dtype=bool)
    outside[inside] = False
    for a, b in zip(got[2], fout):
        assert np.array_equal(a[outside], b[outside], equal_nan=True), (what, "wrote outside the box")


def assert_rate_dominated(fin, ref, lo, hi):
    """The first substep moves every field by at least 10 % of its max on the box: the check sees the rates."""
    inside = box_slice(lo, hi)
    for f in range(8):
        a = fin[f][inside].astype(np.longdouble)
        assert np.abs(ref[0][f] - a).max() >= 0.1 * np.abs(a).max(), ("dt is not rate-dominated", ac.FIELDS[f])


def run_case(raw, lo, hi, dtype, variant, pset_name, dt, record_property, seed=7, shifts=None, poison=False):
    fin, fout, ref = reference(raw, lo, hi, dtype, pset_name, dt, seed, poison)
    gp = params(PARAM_SETS[pset_name], dt)[0]
    if tma_rejects(variant, dtype, raw[0], shifts):
        with pytest.raises(sb.StencilError):
            run_substeps(fin, fout, lo, hi, gp, variant, shifts)
        return
    got = run_substeps(fin, fout, lo, hi, gp, variant, shifts)
    check_against_reference(got, fout, ref, lo, hi, dtype, record_property, (raw, lo, hi, pset_name, dt))


def box_id(b):
    return "{}-{}-{}".format(*["x".join(map(str, v)) for v in b])


@needs_f80
@pytest.mark.parametrize("variant", VARIANTS, ids=[VNAMES[v] for v in VARIANTS])
@pytest.mark.parametrize("box", BOXES, ids=[box_id(b) for b in BOXES])
@pytest.mark.parametrize("dt", list(DTS.values()), ids=list(DTS))
@pytest.mark.parametrize("pset", list(PARAM_SETS))
@pytest.mark.parametrize("dtype", DTYPES, ids=["f64", "f32"])
def test_substeps_within_bound(dtype, variant, pset, dt, box, record_property):
    if dt == DT_RATE:
        fin, _, ref = reference(*box, dtype, pset, dt, 7)
        assert_rate_dominated(fin, ref, box[1], box[2])
    run_case(*box, dtype, variant, pset, dt, record_property)


def edge_boxes():
    m = 40
    boxes = [
        ((m, m, m), (m - 6, 3, 3), (m - 3, m - 3, m - 3)),  # +x face slab
        ((m, m, m), (6, 3, 3), (m - 6, 6, m - 3)),  # low-y slab
        ((m, m, m), (6, 6, 3), (m - 6, m - 6, 6)),  # low-z slab
    ]
    for cz in (3, m - 6):  # the eight 3x3x3 corners
        for cy in (3, m - 6):
            for cx in (3, m - 6):
                boxes.append(((m, m, m), (cx, cy, cz), (cx + 3, cy + 3, cz + 3)))
    # narrower than, equal to and wider than one tile in x (TX = 16, 32); even raw rows so that TMA applies
    for ex in (1, 15, 16, 17, 31, 32, 33):
        mx = ex + 6 + (ex % 2)
        boxes.append(((mx, 20, 16), (3, 3, 3), (3 + ex, 12, 13)))
    # either side of every TY (8 FP32 tile and team, 10 three teams, 12 two teams, 14 and 16 FP64 tile)
    for ey in range(7, 18):
        boxes.append(((28, ey + 8, 14), (4, 4, 3), (24, 4 + ey, 11)))
    return boxes


EDGE_BOXES = edge_boxes()


@needs_f80
@pytest.mark.parametrize("variant", VARIANTS, ids=[VNAMES[v] for v in VARIANTS])
@pytest.mark.parametrize("box", EDGE_BOXES, ids=[box_id(b) for b in EDGE_BOXES])
@pytest.mark.parametrize("dtype", DTYPES, ids=["f64", "f32"])
def test_edge_boxes_within_bound(dtype, variant, box, record_property):
    """Faces, corners and partial tiles; distinct parameters at the rate-dominated dt (the 10 % criterion is asserted
    on the larger boxes of test_substeps_within_bound: a corner's few cells need not meet it)."""
    run_case(*box, dtype, variant, "distinct", DT_RATE, record_property)


@needs_f80
@pytest.mark.parametrize("variant", VARIANTS, ids=[VNAMES[v] for v in VARIANTS])
@pytest.mark.parametrize("depth,zchunk", [(1, 1), (2, 1), (2, 0), (7, 3), (11, 4)])
@pytest.mark.parametrize("dtype", DTYPES, ids=["f64", "f32"])
def test_shallow_boxes_and_zchunks(dtype, variant, depth, zchunk, monkeypatch, record_property):
    """Boxes one or two planes deep, and z chunks (SB_AC_ZCHUNK; 0 = automatic) that do not divide the depth: the ring
    warm-up at every chunk start and the last, shorter chunk."""
    monkeypatch.setenv("SB_AC_ZCHUNK", str(zchunk))
    raw = (40, 36, depth + 8)
    run_case(raw, (3, 3, 4), (37, 33, 4 + depth), dtype, variant, "distinct", DT_RATE, record_property)


@needs_f80
@pytest.mark.parametrize("variant", [ac.AUTO, ac.TEAM, ac.TEAM_TMA, ac.TEAM3_TMA], ids=lambda v: VNAMES[v])
@pytest.mark.parametrize("layout", ["all+8", "mixed", "mixed-odd"])
def test_input_alignment(variant, layout, record_property):
    """FP64 inputs 8 bytes past a 16-byte boundary run on the TMA-fed kernels (the tensor map's base is shifted);
    inputs of different 16-byte phases, or odd rows, are rejected by them and served by the cp.async-fed team kernel."""
    shifts = {"all+8": [1] * 8, "mixed": [0, 1] * 4, "mixed-odd": [1, 1, 0, 1, 0, 0, 1, 0]}[layout]
    raw = (41, 30, 26) if layout == "mixed-odd" else (42, 30, 26)
    run_case(raw, (3, 3, 3), (raw[0] - 3, 27, 23), np.float64, variant, "distinct", DT_RATE, record_property, shifts=shifts)


ZERO_BOXES = [
    ((38, 34, 30), (3, 3, 3), (35, 31, 27)),
    ((40, 40, 40), (34, 3, 3), (37, 37, 37)),
    ((40, 28, 24), (5, 4, 6), (22, 13, 8)),
    ((23, 22, 21), (5, 4, 3), (16, 17, 18)),
]


@pytest.mark.parametrize("variant", VARIANTS, ids=[VNAMES[v] for v in VARIANTS])
@pytest.mark.parametrize("box", ZERO_BOXES, ids=[box_id(b) for b in ZERO_BOXES])
@pytest.mark.parametrize("dtype", DTYPES, ids=["f64", "f32"])
def test_dt_zero_is_identity(dtype, variant, box):
    """dt = 0 and out = in on the box: every substep must leave the box equal to `in` bit for bit (a NaN or infinity in
    any rate makes 0 * rate NaN) and the NaN sentinel outside it untouched (a write to a wrong cell replaces it)."""
    raw, lo, hi = box
    f = make_fields(raw, seed=5, dtype=dtype)
    fin = f[:8]
    inside = box_slice(lo, hi)
    fout = []
    for a in fin:
        o = np.full_like(a, np.nan)
        o[inside] = a[inside]
        fout.append(o)
    gp = params(DISTINCT, 0.0)[0]
    if tma_rejects(variant, dtype, raw[0]):
        with pytest.raises(sb.StencilError):
            run_substeps(fin, fout, lo, hi, gp, variant)
        return
    got = run_substeps(fin, fout, lo, hi, gp, variant)
    for step in range(3):
        for f in range(8):
            assert np.array_equal(got[step][f], fout[f], equal_nan=True), (step, ac.FIELDS[f])


POISON_BOXES = [
    ((38, 34, 30), (3, 3, 3), (35, 31, 27)),
    ((40, 40, 40), (6, 6, 6), (34, 34, 34)),
    ((40, 40, 40), (8, 9, 7), (25, 22, 10)),
    ((40, 40, 40), (34, 3, 3), (37, 37, 37)),
    ((46, 40, 40), (9, 20, 20), (10, 27, 29)),
    ((23, 22, 21), (5, 4, 3), (16, 17, 18)),
]


@needs_f80
@pytest.mark.parametrize("variant", VARIANTS, ids=[VNAMES[v] for v in VARIANTS])
@pytest.mark.parametrize("box", POISON_BOXES, ids=[box_id(b) for b in POISON_BOXES])
@pytest.mark.parametrize("dtype", DTYPES, ids=["f64", "f32"])
def test_nan_outside_footprint(dtype, variant, box, record_property):
    """Every input cell outside [lo - 3, hi + 3) is NaN (and every `out` cell outside the box): a read past the stencil,
    from a partial tile, a wrong ring slot or a wrong plane, makes an output NaN."""
    run_case(*box, dtype, variant, "distinct", DT_RATE, record_property, poison=True)


@pytest.mark.parametrize("dtype", DTYPES, ids=["f64", "f32"])
def test_benchmark_size_substep(dtype, record_property):
    """One substep on the 256^3 compute region of the benchmark with the default variant (its grid and z-chunk choice)
    against the same-precision oracle at twice the bound (both sides round)."""
    m = 256 + 6
    rng = np.random.default_rng(17)
    fin = [rng.uniform(-0.5, 0.5, (m, m, m)).astype(dtype) for _ in range(8)]
    fout = [rng.uniform(-0.5, 0.5, (m, m, m)).astype(dtype) for _ in range(8)]
    lo, hi = (3, 3, 3), (m - 3, m - 3, m - 3)
    gp, op = params(PARAM_SETS["conf"], 1e-3)
    din = [DevArray(a) for a in fin]
    dout = [DevArray(a) for a in fout]
    try:
        ac.substep(1, [d.ptr for d in din], [d.ptr for d in dout], np.dtype(dtype).itemsize, (m, m, m), lo, hi, gp, ac.AUTO)
        got = [d.get() for d in dout]
    finally:
        for d in din + dout:
            d.free()
    co.astaroth_substep(1, fin, fout, lo, hi, op)
    inside = box_slice(lo, hi)
    r = err_over_eps([a[inside] for a in got], [b[inside] for b in fout], dtype)
    record_property("err_over_eps", {ac.FIELDS[f]: round(float(r[f]), 3) for f in range(8)})
    assert (r <= 2 * K_ULP).all(), r
