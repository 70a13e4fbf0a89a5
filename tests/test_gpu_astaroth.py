"""GPU parity of the astaroth solve<step> kernels (stencil_b200/csrc/astaroth.cu) against the CPU oracle
(oracle/astaroth_oracle.c), against golden vectors produced by the REFERENCE's own kernels on a B200
(tests/golden/astaroth_solve_ref.npz), and through DistributedDomain (interior || exchange -> exterior, 3 substeps,
swap) against the oracle's single-address-space exchange.  Floating point: tolerances in astaroth_util.tolerance."""
import os

import numpy as np
import pytest

import stencil_b200 as sb
from astaroth_util import BOXES, GOLDEN, make_fields, tolerance
from gpu_util import DevArray
from oracle import c_oracle as co
from oracle import geometry as g
from oracle import np_oracle as no
from stencil_b200 import astaroth as ac

pytestmark = pytest.mark.gpu


def tma_applies(dtype, raw) -> bool:
    """The TMA-fed team kernel needs FP64 and rows that are a multiple of 16 bytes (an even number of doubles)."""
    return np.dtype(dtype) == np.float64 and raw[0] % 2 == 0


def run_gpu(step, fin, fout, lo, hi, params, variant):
    """fin / fout: lists of 8 host arrays; returns the 8 updated `out` arrays."""
    if variant in (ac.TEAM_TMA, ac.TEAM3_TMA) and not tma_applies(fin[0].dtype, fin[0].shape[::-1]):
        pytest.skip("TMA-fed kernel: FP64 with an even row length only")
    din = [DevArray(a) for a in fin]
    dout = [DevArray(a) for a in fout]
    mz, my, mx = fin[0].shape
    ac.substep(step, [d.ptr for d in din], [d.ptr for d in dout], fin[0].dtype.itemsize, (mx, my, mz), lo, hi, params, variant)
    res = [d.get() for d in dout]
    for d in din + dout:
        d.free()
    return res


def assert_close(got, want, dtype, what):
    tol = tolerance(dtype)
    for f, (a, b) in enumerate(zip(got, want)):
        scale = max(1.0, float(np.abs(b).max()))
        err = float(np.abs(a.astype(np.float64) - b.astype(np.float64)).max())
        assert err <= tol * scale, (what, ac.FIELDS[f], err, scale)


@pytest.mark.parametrize("dtype", [np.float64, np.float32])
@pytest.mark.parametrize("variant", [ac.AUTO, ac.CELL, ac.TILE, ac.TEAM, ac.TEAM_TMA, ac.TEAM3_TMA])
@pytest.mark.parametrize("box", BOXES, ids=[f"{b[0]}-{b[1]}-{b[2]}" for b in BOXES])
def test_substeps_match_oracle(dtype, variant, box):
    raw, lo, hi = box
    fields = make_fields(raw, seed=7, dtype=dtype)
    fin, fout = fields[:8], fields[8:]
    params = ac.conf_params(dt=1e-3)
    op = co.astaroth_conf_params(1e-3)
    cur_gpu = [a.copy() for a in fout]
    cur_cpu = [a.copy() for a in fout]
    for step in range(3):  # like the driver: three substeps into the same `out`, no swap in between
        cur_gpu = run_gpu(step, fin, cur_gpu, lo, hi, params, variant)
        co.astaroth_substep(step, fin, cur_cpu, lo, hi, op)
        assert_close(cur_gpu, cur_cpu, dtype, f"step {step}")
    # nothing outside the box was touched
    for a, b in zip(cur_gpu, fout):
        m = np.ones(a.shape, dtype=bool)
        m[lo[2] : hi[2], lo[1] : hi[1], lo[0] : hi[0]] = False
        assert np.array_equal(a[m], b[m])


@pytest.mark.parametrize("variant", [ac.CELL, ac.TILE, ac.TEAM, ac.TEAM_TMA, ac.TEAM3_TMA])
@pytest.mark.parametrize("shape", [0, 1])
def test_tile_shapes_and_zchunks(variant, shape, monkeypatch):
    """Both tile shapes per precision (SB_AC_SHAPE) and a forced short z chunk (ring warm-up at every chunk start)."""
    monkeypatch.setenv("SB_AC_SHAPE", str(shape))
    monkeypatch.setenv("SB_AC_ZCHUNK", "5")
    for dtype in (np.float64, np.float32):
        if variant in (ac.TEAM_TMA, ac.TEAM3_TMA) and dtype == np.float32:
            continue
        raw, lo, hi = (50, 45, 29), (3, 3, 3), (47, 42, 26)
        fields = make_fields(raw, seed=11, dtype=dtype)
        fin, fout = fields[:8], fields[8:]
        got = run_gpu(2, fin, fout, lo, hi, ac.conf_params(dt=1e-3), variant)
        want = [a.copy() for a in fout]
        co.astaroth_substep(2, fin, want, lo, hi, co.astaroth_conf_params(1e-3))
        assert_close(got, want, dtype, f"shape {shape}")


@pytest.mark.skipif(not os.path.exists(GOLDEN), reason="golden vectors not generated yet (oracle/ref/make_astaroth_golden.py)")
@pytest.mark.parametrize("variant", [ac.CELL, ac.TILE, ac.TEAM, ac.TEAM_TMA, ac.TEAM3_TMA])
def test_matches_reference_kernel_golden(variant):
    """The reference's own solve<0,1,2> (astaroth/kernels.cu, compiled unmodified for sm_100a) produced these."""
    z = np.load(GOLDEN)
    n, dt = int(z["n"]), float(z["dt"])
    inputs, outputs = z["inputs"], z["outputs"]
    m = n + 6
    fin = [np.ascontiguousarray(inputs[f]) for f in range(8)]
    cur = [np.ascontiguousarray(inputs[8 + f]) for f in range(8)]
    for step in range(3):
        cur = run_gpu(step, fin, cur, (3, 3, 3), (m - 3, m - 3, m - 3), ac.conf_params(dt=dt), variant)
        got = [a[3:-3, 3:-3, 3:-3] for a in cur]
        assert_close(got, [outputs[step, f] for f in range(8)], np.float64, f"golden step {step}")


@pytest.mark.parametrize("dtype", [np.float64, np.float32])
@pytest.mark.parametrize("ndom", [1, 2])
@pytest.mark.parametrize("overlap", [True, False])
@pytest.mark.parametrize("variant", [ac.AUTO, ac.TEAM])
def test_iteration_through_distributed_domain(dtype, ndom, overlap, variant):
    """astaroth/astaroth.cu:551-640: per substep interior || exchange -> exterior; swap after the third.  Two
    iterations on 24x20x28 split over `ndom` subdomains, against oracle exchange + oracle solve."""
    import torch

    size = (24, 20, 28)
    ng = torch.cuda.device_count()
    dd = sb.DistributedDomain(*size)
    dd.set_gpus([i % ng for i in range(ndom)])
    dd.set_radius(3)
    handles = [dd.add_data(dtype, name) for name in ac.FIELDS]
    dd.realize()
    ro = g.Radius.constant(3)
    od = no.Domains(size, ro, [dtype] * 8, n_subdomains=ndom)
    nxt = {i: [np.zeros_like(a) for a in od.arrays[i]] for i in od.indices}
    try:
        # same initial state on both sides: seeded fields over the GLOBAL compute region, scattered to the subdomains
        glob = make_fields(size, seed=3, dtype=dtype)
        for di, d in enumerate(dd.domains()):
            i = dd.domain_idx_[di]
            o, sz = od.origins[i], od.sizes[i]
            for q in range(8):
                for which, src in (("curr", glob[q]), ("next", glob[8 + q])):
                    host = np.zeros(tuple(reversed(d.raw_size())), dtype=dtype)
                    no.box(host, (3, 3, 3), sz)[...] = src[o[2] : o[2] + sz[2], o[1] : o[1] + sz[1], o[0] : o[0] + sz[0]]
                    d.quantity_from_host(q, host, which)
                    if which == "curr":
                        od.arrays[i][q][...] = host
                    else:
                        nxt[i][q][...] = host
        params = ac.conf_params(dt=1e-3)
        op = co.astaroth_conf_params(1e-3)
        # (LocalDomain places FP64 r=3 allocations 8 bytes into their block: the TMA-fed kernel's shifted tensor base)
        sim = ac.Astaroth(dd, handles, params, overlap=overlap, variant=variant)
        for it in range(2):
            sim.step()
            for sub in range(3):
                od.exchange()
                for i in od.indices:
                    sz = od.sizes[i]
                    co.astaroth_substep(sub, od.arrays[i], nxt[i], (3, 3, 3), (3 + sz[0], 3 + sz[1], 3 + sz[2]), op)
            for i in od.indices:
                od.arrays[i], nxt[i] = nxt[i], od.arrays[i]
        for di, d in enumerate(dd.domains()):
            i = dd.domain_idx_[di]
            sz = od.sizes[i]
            got = [no.box(d.quantity_to_host(q), (3, 3, 3), sz) for q in range(8)]
            want = [no.box(od.arrays[i][q], (3, 3, 3), sz) for q in range(8)]
            assert_close(got, want, dtype, f"domain {i}")
    finally:
        dd.close()
