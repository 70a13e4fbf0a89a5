"""GPU checks of the field reductions (sb_reduce, stencil_b200/csrc/reduce.cu) against the numpy oracle
(tests/reduce_oracle.py): min and max exact (VALUE, DIFF, VECTOR) or within 4 ulp (EXP, ALFVEN), sums within
1e-12 of the sum of |terms| of the extended-precision oracle, for every kind, both dtypes, the allocation layouts the
library makes and thin / odd / edge boxes; ghost cells, NaN, empty boxes, determinism, errors; DistributedDomain.reduce,
Astaroth.diagnostics and Jacobi3D.residual."""
import ctypes as C
import math
import struct

import numpy as np
import pytest

import stencil_b200 as sb
from oracle import np_oracle as no
import reduce_oracle as ro
from stencil_b200 import reduce as R
from stencil_b200._lib import Pitched, check, lib

pytestmark = pytest.mark.gpu

KINDS = {"VALUE": R.VALUE, "DIFF": R.DIFF, "VECTOR": R.VECTOR, "EXP": R.EXP, "ALFVEN": R.ALFVEN}
EXACT = ("VALUE", "DIFF", "VECTOR")


class Alloc:
    """A [z, y, x] allocation in device memory starting `lead` bytes into its cudaMalloc block."""

    def __init__(self, host: np.ndarray, lead: int = 0):
        self.shape, self.dtype, self.lead = host.shape, host.dtype, lead
        p = C.c_void_p()
        check(lib().sb_malloc(C.byref(p), host.nbytes + 32, 0))
        self.base = int(p.value)
        self.ptr = self.base + lead
        self.put(host)

    def put(self, host: np.ndarray) -> None:
        host = np.ascontiguousarray(host, dtype=self.dtype)
        check(lib().sb_memcpy(C.c_void_p(self.ptr), host.ctypes.data, host.nbytes, 0, None))
        check(lib().sb_device_sync(0))

    def pitched(self) -> Pitched:
        return Pitched(self.ptr, self.shape[2] * self.dtype.itemsize, self.shape[1])

    def __del__(self):
        lib().sb_free(C.c_void_p(self.base), 0)


# layout name -> (dtype, radius, compute size, leads of the operands); the leads follow LocalDomain.lead_bytes
LAYOUTS = {
    "f64_r1": (np.float64, 1, (70, 9, 6), (8, 8, 8, 8)),  # 576-byte rows: every row 16-byte aligned at the first compute cell
    "f64_r3": (np.float64, 3, (66, 7, 5), (8, 8, 8, 8)),
    "f64_mixed": (np.float64, 1, (70, 9, 6), (8, 0, 8, 0)),  # operands in different 16-byte phases: scalar rows
    "f32_r1_alt": (np.float32, 1, (68, 9, 6), (0, 0, 0, 0)),  # 280-byte rows: phases alternate between 0 and 8
    "f32_mixed": (np.float32, 1, (68, 9, 6), (0, 4, 8, 12)),
}


def boxes(r, n):
    """(name, lo, hi) in allocation coordinates (acc_origin = 0)."""
    hi = tuple(r + n[a] for a in range(3))
    raw = tuple(n[a] + 2 * r for a in range(3))
    return [
        ("compute", (r, r, r), hi),
        ("cell", (r + 3, r + 2, r + 1), (r + 4, r + 3, r + 2)),
        ("row", (r, r + 1, r + 2), (hi[0], r + 2, r + 3)),
        ("plane", (r, r, r + 1), (hi[0], hi[1], r + 2)),
        ("x1", (r, r, r), (r + 1, hi[1], hi[2])),
        ("x2", (hi[0] - 2, r, r), (hi[0], hi[1], hi[2])),
        ("x3", (r + 5, r, r), (r + 8, hi[1], hi[2])),
        ("odd", (r + 1, r + 1, r), (r + 1 + 37, hi[1], r + 3)),  # 37 cells from an odd start: head, vectors and tail
        ("wide_odd", (r + 3, r, r), (hi[0] - 2, hi[1], hi[2])),
        ("last_row", (0, raw[1] - 1, raw[2] - 1), raw),  # ends at the last byte of the allocation
    ]


def run(kind, allocs, lo, hi, ws, acc=(0, 0, 0), stream=None):
    return R.reduce_box(KINDS[kind], [a.pitched() for a in allocs], allocs[0].dtype.itemsize, acc, lo, hi, ws, stream)


def assert_matches(kind, got, arrays, lo, hi):
    ext = tuple(hi[a] - lo[a] for a in range(3))
    want = ro.reduce_box(kind, arrays, lo, ext)
    wantl = ro.reduce_box(kind, arrays, lo, ext, dtype=np.longdouble)
    f, g = ro.reduce_terms(kind, arrays, lo, ext)
    assert got.count == want["count"]
    for k in ("min", "max"):
        w = float(want[k])
        if kind in EXACT:
            assert getattr(got, k) == w, (k, getattr(got, k), w)
        else:
            assert abs(getattr(got, k) - w) <= 4 * np.spacing(abs(w)), (k, getattr(got, k), w)
    assert abs(got.sum - float(wantl["sum"])) <= 1e-12 * float(np.abs(f).sum()), (got.sum, wantl["sum"])
    assert abs(got.sum2 - float(wantl["sum2"])) <= 1e-12 * float(np.abs(g).sum()), (got.sum2, wantl["sum2"])


@pytest.fixture(scope="module")
def ws():
    w = R.Workspace(0)
    yield w
    w.free()


def make_arrays(layout, seed, ghost=None):
    dtype, r, n, leads = LAYOUTS[layout]
    raw = tuple(n[a] + 2 * r for a in range(3))
    rng = np.random.default_rng(seed)
    hosts = [rng.uniform(-2.0, 2.0, raw[::-1]).astype(dtype) for _ in range(4)]
    if ghost is not None:
        for h in hosts:
            inner = no.box(h, (r, r, r), n).copy()
            h[...] = ghost
            no.box(h, (r, r, r), n)[...] = inner
    return hosts, [Alloc(h, leads[i]) for i, h in enumerate(hosts)], r, n


@pytest.mark.parametrize("layout", list(LAYOUTS))
@pytest.mark.parametrize("kind", list(KINDS))
def test_boxes_match_oracle(kind, layout, ws):
    hosts, allocs, r, n = make_arrays(layout, seed=5)
    k = ro.REDUCE_OPERANDS[kind]
    for name, lo, hi in boxes(r, n):
        got = run(kind, allocs[:k], lo, hi, ws)
        assert_matches(kind, got, hosts[:k], lo, hi)


@pytest.mark.parametrize("layout", ["f64_r1", "f64_r3", "f32_r1_alt", "f32_mixed"])
@pytest.mark.parametrize("kind", list(KINDS))
def test_ghost_cells_change_nothing(kind, layout, ws):
    k = ro.REDUCE_OPERANDS[kind]
    res = []
    for ghost in (0.0, np.nan, 1e300 if LAYOUTS[layout][0] == np.float64 else 3e38):
        hosts, allocs, r, n = make_arrays(layout, seed=9, ghost=ghost)
        lo, hi = (r, r, r), tuple(r + n[a] for a in range(3))
        got = run(kind, allocs[:k], lo, hi, ws)
        assert_matches(kind, got, hosts[:k], lo, hi)
        res.append(tuple(struct.pack("<d", v) for v in got[:4]))
    assert res[0] == res[1] == res[2]


@pytest.mark.parametrize("layout", ["f64_r1", "f32_r1_alt"])
@pytest.mark.parametrize("kind", list(KINDS))
def test_nan_inside_the_box_shows(kind, layout, ws):
    k = ro.REDUCE_OPERANDS[kind]
    for where in ((0, 0, 0), (7, 3, 2), (-1, -1, -1)):  # offsets into the compute region; -1 = its last cell
        hosts, allocs, r, n = make_arrays(layout, seed=3)
        lo, hi = (r, r, r), tuple(r + n[a] for a in range(3))
        x, y, z = [r + (where[a] if where[a] >= 0 else n[a] + where[a]) for a in range(3)]
        hosts[k - 1][z, y, x] = np.nan
        allocs[k - 1].put(hosts[k - 1])
        got = run(kind, allocs[:k], lo, hi, ws)
        assert all(math.isnan(v) for v in (got.min, got.max, got.sum, got.sum2)), (where, got)


def test_empty_box_gives_identities(ws):
    hosts, allocs, r, n = make_arrays("f64_r1", seed=1)
    for lo, hi in (((1, 1, 1), (1, 5, 5)), ((1, 1, 1), (5, 1, 5)), ((1, 1, 1), (5, 5, 1)), ((0, 0, 0), (0, 0, 0))):
        got = run("VALUE", allocs[:1], lo, hi, ws)
        assert (got.min, got.max, got.sum, got.sum2, got.count) == (math.inf, -math.inf, 0.0, 0.0, 0)
    # and the workspace is ready for the next launch
    lo, hi = (1, 1, 1), (71, 10, 7)
    assert_matches("VALUE", run("VALUE", allocs[:1], lo, hi, ws), hosts[:1], lo, hi)


def test_repeated_and_concurrent_calls_are_bit_identical():
    import torch

    rng = np.random.default_rng(2)
    raw = (130, 130, 130)
    a = Alloc(rng.standard_normal(raw[::-1]), 8)
    b = Alloc(rng.standard_normal(raw[::-1]) * 1e3 + 7.0, 8)
    lo, hi = (1, 1, 1), (129, 129, 129)
    w1, w2 = R.Workspace(0), R.Workspace(0)
    solo_a = run("VALUE", [a], lo, hi, w1)
    solo_b = run("DIFF", [b, a], lo, hi, w2)
    for _ in range(3):
        assert run("VALUE", [a], lo, hi, w1) == solo_a
    s1, s2 = torch.cuda.Stream(), torch.cuda.Stream()
    for _ in range(5):
        w1.launch(R.VALUE, [a.pitched()], 8, (0, 0, 0), lo, hi, s1)
        w2.launch(R.DIFF, [b.pitched(), a.pitched()], 8, (0, 0, 0), lo, hi, s2)
        w1.launch(R.VALUE, [a.pitched()], 8, (0, 0, 0), lo, hi, s1)
    ra, rb = w1.result(s1), w2.result(s2)
    bits = lambda t: [struct.pack("<d", v) for v in t]  # noqa: E731
    assert bits(ra) == bits(solo_a[:4]) and bits(rb) == bits(solo_b[:4])
    w1.free()
    w2.free()


def test_invalid_arguments_raise(ws):
    hosts, allocs, r, n = make_arrays("f64_r1", seed=1)
    L = lib()
    p = allocs[0].pitched()
    acc, lo, hi = (0, 0, 0), (1, 1, 1), (5, 5, 5)
    with pytest.raises(sb.StencilError, match="kind"):
        ws.launch(9, [p], 8, acc, lo, hi)
    with pytest.raises(sb.StencilError, match="dtype_size"):
        ws.launch(R.VALUE, [p], 2, acc, lo, hi)
    with pytest.raises(sb.StencilError, match="operands"):
        ws.launch(R.DIFF, [p], 8, acc, lo, hi)
    with pytest.raises(sb.StencilError, match="differ"):
        ws.launch(R.DIFF, [p, Pitched(allocs[1].ptr, p.pitch + 8, p.ysize)], 8, acc, lo, hi)
    with pytest.raises(sb.StencilError, match="null"):
        ws.launch(R.DIFF, [p, Pitched(None, p.pitch, p.ysize)], 8, acc, lo, hi)
    with pytest.raises(sb.StencilError, match="past the row"):
        ws.launch(R.VALUE, [p], 8, acc, lo, (73, 5, 5))
    with pytest.raises(sb.StencilError, match="past the"):
        ws.launch(R.VALUE, [p], 8, acc, lo, (5, 12, 5))
    with pytest.raises(sb.StencilError, match="outside"):
        ws.launch(R.VALUE, [p], 8, (2, 0, 0), lo, hi)
    with pytest.raises(sb.StencilError, match="hi < lo"):
        ws.launch(R.VALUE, [p], 8, acc, (5, 5, 5), (4, 6, 6))
    with pytest.raises(sb.StencilError, match="aligned"):
        ws.launch(R.VALUE, [Pitched(allocs[0].ptr + 4, p.pitch, p.ysize)], 8, acc, lo, hi)
    ops = (Pitched * 1)(p)
    with pytest.raises(sb.StencilError, match="null"):
        check(L.sb_reduce(R.VALUE, ops, 8, sb._lib.i3(acc), sb._lib.i3(lo), sb._lib.i3(hi), None, None))
    # nothing above launched or disturbed the workspace
    lo, hi = (1, 1, 1), (71, 10, 7)
    assert_matches("VALUE", run("VALUE", allocs[:1], lo, hi, ws), hosts[:1], lo, hi)


def test_512_cubed_fp64_value(ws):
    """The benchmark's allocation: 514^3 doubles, 8 bytes into the block (LocalDomain.lead_bytes)."""
    import torch

    raw = 514
    t = torch.empty(raw**3 + 2, dtype=torch.float64, device="cuda:0")
    g = torch.Generator(device="cuda:0")
    g.manual_seed(4)
    t.normal_(generator=g)
    torch.cuda.synchronize()
    ptr = t.data_ptr() + 8
    assert ptr % 16 == 8
    p = Pitched(ptr, raw * 8, raw)
    got = R.reduce_box(R.VALUE, [p], 8, (-1, -1, -1), (0, 0, 0), (512, 512, 512), ws)
    host = t[1 : 1 + raw**3].cpu().numpy().reshape(raw, raw, raw)[1:513, 1:513, 1:513]
    assert got.count == 512**3
    assert got.min == float(host.min()) and got.max == float(host.max())
    s = sum(np.sum(host[z], dtype=np.longdouble) for z in range(512))
    s2 = sum(np.sum(host[z] * host[z], dtype=np.longdouble) for z in range(512))
    abs_sum = float(sum(np.abs(host[z]).sum() for z in range(512)))
    assert abs(got.sum - float(s)) <= 1e-12 * abs_sum
    assert abs(got.sum2 - float(s2)) <= 1e-12 * float(s2)


# ------------------------------------------------------------------------------------------ DistributedDomain
def global_field(size, seed, dtype):
    return np.random.default_rng(seed).uniform(-3.0, 3.0, size[::-1]).astype(dtype)


def scatter(dd, h, glob, which="curr"):
    for d in dd.domains():
        o, sz = d.origin(), d.size()
        host = np.full(tuple(reversed(d.raw_size())), np.nan, dtype=glob.dtype)  # NaN ghosts: must not be read
        rm = tuple(d.radius().dir(tuple(-1 if b == a else 0 for b in range(3))) for a in range(3))
        no.box(host, rm, sz)[...] = no.box(glob, o, sz)
        d.quantity_from_host(h.id, host, which)


@pytest.mark.parametrize("dtype", [np.float64, np.float32])
def test_distributed_reduce_on_1_2_4_8_subdomains(dtype):
    size = (60, 44, 36)
    glob = [global_field(size, s, dtype) for s in (1, 2, 3)]
    glob_next = global_field(size, 4, dtype)
    full = ((0, 0, 0), size)
    cases = [
        ("VALUE", lambda hs: [hs[0]], [glob[0]]),
        ("EXP", lambda hs: [hs[0]], [glob[0]]),
        ("VECTOR", lambda hs: hs, glob),
        ("DIFF", lambda hs: [(hs[0], "curr"), (hs[0], "next")], [glob[0], glob_next]),
    ]
    seen = {}
    for ndom in (1, 2, 4, 8):
        dd = sb.DistributedDomain(*size)
        dd.set_gpus([0] * ndom)
        dd.set_radius(sb.Radius.constant(2))
        hs = [dd.add_data(dtype, f"q{i}") for i in range(3)]
        dd.realize()
        try:
            assert len(dd.domains()) == ndom
            for h, gl in zip(hs, glob):
                scatter(dd, h, gl)
            scatter(dd, hs[0], glob_next, "next")
            for kind, ops, arrays in cases:
                got = dd.reduce(KINDS[kind], ops(hs))
                assert_matches(kind, got, arrays, *full)
                if kind in seen:
                    assert (got.min, got.max, got.count) == seen[kind]
                seen[kind] = (got.min, got.max, got.count)
                assert dd.reduce(KINDS[kind], ops(hs)) == got  # repeatable to the bit
        finally:
            dd.close()


def test_astaroth_diagnostics_after_two_iterations():
    from astaroth_util import make_fields

    from stencil_b200 import astaroth as ac

    size = (32, 24, 28)
    dd = sb.DistributedDomain(*size)
    dd.set_gpus([0, 0])
    dd.set_radius(3)
    handles = [dd.add_data(np.float64, name) for name in ac.FIELDS]
    dd.realize()
    try:
        glob = make_fields(size, seed=5, dtype=np.float64)
        for q, h in enumerate(handles):
            scatter(dd, h, glob[q])
            scatter(dd, h, glob[8 + q], "next")
        sim = ac.Astaroth(dd, handles, ac.conf_params(dt=1e-3))
        for _ in range(2):
            sim.step()
        diag = sim.diagnostics()
        # the fields after two iterations, gathered on the host
        fields = [np.zeros(size[::-1]) for _ in range(8)]
        for d in dd.domains():
            for q in range(8):
                no.box(fields[q], d.origin(), d.size())[...] = d.interior_to_host(q)
        full = ((0, 0, 0), size)
        assert set(diag) == {"uu", *ac.FIELDS}
        assert_matches("VECTOR", diag["uu"], fields[1:4], *full)
        for q, name in enumerate(ac.FIELDS):
            assert_matches("VALUE", diag[name], [fields[q]], *full)
            assert diag[name].rms == math.sqrt(diag[name].sum2 / diag[name].count)
    finally:
        dd.close()


@pytest.mark.parametrize("schedule", ["step", "step_fused"])
def test_jacobi_residual_matches_oracle(schedule):
    from stencil_b200.jacobi import Jacobi3D, jacobi_radius

    n = 48
    dd = sb.DistributedDomain(n, n, n)
    dd.set_gpus([0, 0, 0, 0])
    dd.set_radius(jacobi_radius())
    h = dd.add_data(np.float64, "d")
    dd.realize()
    try:
        jac = Jacobi3D(dd, h)
        jac.init(0.5)
        for _ in range(3):
            getattr(jac, schedule)()
        got = jac.residual()
        s = 0.0
        for d in dd.domains():
            sz = d.size()
            r = no.residual_l2(d.quantity_to_host(0, "curr"), d.quantity_to_host(0, "next"), (1, 1, 1), sz)
            s += r * r
        want = math.sqrt(s)
        assert want > 0 and abs(got - want) <= 1e-12 * want, (got, want)
    finally:
        jac.close()
        dd.close()


def test_two_ranks_match_one_process():
    """torchrun, one rank per GPU: tests/mp_reduce_check.py."""
    import os
    import subprocess
    import sys

    import torch

    if torch.cuda.device_count() < 2:
        pytest.skip("needs >= 2 GPUs")
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr", "127.0.0.1",
           "--master-port", "29541", os.path.join(root, "tests", "mp_reduce_check.py")]
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    assert out.returncode == 0 and "mp_reduce_check OK" in out.stdout, out.stdout[-2000:] + out.stderr[-4000:]
