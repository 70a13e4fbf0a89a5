"""CPU checks of the reductions: the C ABI result struct, the host combine (identities, NaN, rms, fixed order), the numpy
oracle's filters against formulas written out cell by cell, and the cross-rank combine over `gloo` (every rank gets the
same bits whichever rank owns which subdomain)."""
import math
import os
import socket
import struct
import subprocess
import sys

import numpy as np
import pytest
import reduce_oracle as ro
import torch.multiprocessing as mp

from stencil_b200 import reduce as R

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def bits(x: float) -> bytes:
    return struct.pack("<d", x)


def test_result_struct_matches_the_header(tmp_path):
    import ctypes as C

    from stencil_b200._lib import ReduceResult

    src = tmp_path / "probe.c"
    src.write_text(
        '#include <stdio.h>\n#include <stddef.h>\n#include "stencil_b200.h"\n'
        'int main(void) { printf("%zu %zu %zu\\n", sizeof(sb_reduce_result), offsetof(sb_reduce_result, sum2), sizeof(sb_reduce_kind)); '
        "return SB_REDUCE_VALUE != 0 || SB_REDUCE_DIFF != 1 || SB_REDUCE_VECTOR != 2 || SB_REDUCE_EXP != 3 || SB_REDUCE_ALFVEN != 4; }\n"
    )
    exe = tmp_path / "probe"
    subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), str(src), "-o", str(exe)])
    size, off, kind_size = [int(v) for v in subprocess.check_output([str(exe)]).split()]
    assert size == C.sizeof(ReduceResult) == 32
    assert off == ReduceResult.sum2.offset
    assert kind_size == C.sizeof(C.c_int)
    assert (R.VALUE, R.DIFF, R.VECTOR, R.EXP, R.ALFVEN) == (0, 1, 2, 3, 4)


def test_combine_identities_and_rms():
    s = R.combine([])
    assert (s.min, s.max, s.sum, s.sum2, s.count) == (math.inf, -math.inf, 0.0, 0.0, 0) and math.isnan(s.rms)
    s = R.combine([R.EMPTY, (1.0, 3.0, 4.0, 10.0, 2), R.EMPTY, (-2.0, 0.5, -1.5, 4.25, 2)])
    assert (s.min, s.max, s.sum, s.sum2, s.count) == (-2.0, 3.0, 2.5, 14.25, 4)
    assert s.rms == math.sqrt(14.25 / 4)


@pytest.mark.parametrize("where", [0, 1, 2])
def test_combine_propagates_nan(where):
    parts = [(1.0, 2.0, 3.0, 4.0, 1), (0.0, 5.0, 1.0, 1.0, 1), (-1.0, 1.0, 0.0, 2.0, 1)]
    nan = float("nan")
    parts[where] = (nan, nan, nan, nan, 1)
    s = R.combine(parts)
    assert all(math.isnan(v) for v in (s.min, s.max, s.sum, s.sum2, s.rms)) and s.count == 3


def test_combine_order_is_the_order_given():
    parts = [(0.0, 0.0, 1e16, 0.0, 1), (0.0, 0.0, 1.0, 0.0, 1), (0.0, 0.0, -1e16, 0.0, 1), (0.0, 0.0, 1.0, 0.0, 1)]
    assert R.combine(parts).sum == 1.0  # (((1e16 + 1) - 1e16) + 1): the first 1 is lost
    assert R.combine([parts[i] for i in (0, 2, 1, 3)]).sum == 2.0


def _cells(kind, arrays, pos, ext):
    """The filters written out per cell with Python floats (IEEE double): the hand restatement the oracle must match."""
    out = []
    for z in range(pos[2], pos[2] + ext[2]):
        for y in range(pos[1], pos[1] + ext[1]):
            for x in range(pos[0], pos[0] + ext[0]):
                v = [float(a[z, y, x]) for a in arrays]
                if kind == "VALUE":
                    f, g = v[0], v[0] * v[0]
                elif kind == "DIFF":
                    f = v[0] - v[1]
                    g = f * f
                elif kind == "EXP":
                    f = math.exp(v[0])
                    g = f * f
                else:
                    s = (v[0] * v[0] + v[1] * v[1]) + v[2] * v[2]
                    if kind == "VECTOR":
                        f, g = math.sqrt(s), s
                    else:
                        den = 4.0 * math.pi * math.exp(v[3])
                        f, g = math.sqrt(s) / math.sqrt(den), s / den
                out.append((f, g))
    return out


@pytest.mark.parametrize("kind", ["VALUE", "DIFF", "VECTOR", "EXP", "ALFVEN"])
@pytest.mark.parametrize("dtype", [np.float32, np.float64])
def test_oracle_filters_vs_formulas(kind, dtype):
    rng = np.random.default_rng(7)
    arrays = [rng.uniform(-2, 2, (5, 6, 7)).astype(dtype) for _ in range(ro.REDUCE_OPERANDS[kind])]
    pos, ext = (1, 2, 0), (5, 3, 4)
    want = _cells(kind, arrays, pos, ext)
    f, g = ro.reduce_terms(kind, arrays, pos, ext)
    tol = 0 if kind in ("VALUE", "DIFF", "VECTOR") else 4  # numpy's exp may differ from libm's by an ulp
    wf = np.array([w[0] for w in want])
    wg = np.array([w[1] for w in want])
    assert np.all(np.abs(f.ravel() - wf) <= tol * np.spacing(np.abs(wf)))
    assert np.all(np.abs(g.ravel() - wg) <= tol * np.spacing(np.abs(wg)))
    r = ro.reduce_box(kind, arrays, pos, ext)
    assert r["min"] == f.min() and r["max"] == f.max() and r["count"] == len(want)
    # the extended-precision variant agrees to within the FP64 rounding of the terms
    rl = ro.reduce_box(kind, arrays, pos, ext, dtype=np.longdouble)
    for k in ("min", "max", "sum", "sum2"):
        scale = np.sum(np.abs(f if k != "sum2" else g))
        assert abs(float(rl[k]) - float(r[k])) <= 1e-14 * max(scale, 1.0), (k, rl[k], r[k])


def test_oracle_empty_box_and_nan():
    a = np.zeros((4, 4, 4))
    r = ro.reduce_box("VALUE", [a], (1, 1, 1), (0, 2, 2))
    assert (r["min"], r["max"], r["sum"], r["sum2"], r["count"]) == (np.inf, -np.inf, 0.0, 0.0, 0)
    a[2, 2, 2] = np.nan
    r = ro.reduce_box("VALUE", [a], (1, 1, 1), (2, 2, 2))
    assert all(np.isnan(r[k]) for k in ("min", "max", "sum", "sum2"))


# ------------------------------------------------------------------------------------------ cross-rank combine (gloo)
def _partial_table(n_sub: int):
    """Partials whose sums change with the order they are added in (+-1e16 between small values)."""
    rng = np.random.default_rng(11)
    out = []
    for k in range(n_sub):
        s = (1e16, float(rng.uniform(1, 2)), -1e16, float(rng.uniform(1, 2)))[k % 4]
        out.append((float(rng.uniform(-5, 0)), float(rng.uniform(0, 5)), s, abs(s) * 3.0 + 0.1, int(rng.integers(1, 1000))))
    return out


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _worker(rank, world, port, size, per_rank, reverse, out_q):
    try:
        sys.path.insert(0, ROOT)
        import torch.distributed as td

        os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world), LOCAL_RANK=str(rank))
        td.init_process_group("gloo", rank=rank, world_size=world)
        import stencil_b200 as sb
        from stencil_b200 import reduce as R

        dd = sb.DistributedDomain(*size)
        dd.set_gpus([0] * per_rank)
        dd.set_radius(sb.Radius.constant(1))
        dd.add_data(np.float64)
        dd.do_placement()  # partition + ownership, no GPU
        order = dd.partition_.indices()
        owner = dd._owner
        if reverse:  # the same partition with the ranks' shares swapped around
            owner = {idx: (world - 1 - r, s) for idx, (r, s) in owner.items()}
        table = _partial_table(len(order))
        local = {idx: table[k] for k, idx in enumerate(order) if owner[idx][0] == rank}
        assert len(local) == per_rank
        s = R.combine_ranks(local, order, world)
        td.destroy_process_group()
        out_q.put((rank, tuple(bits(v) for v in (s.min, s.max, s.sum, s.sum2, s.rms)) + (s.count,)))
    except Exception:  # pragma: no cover
        import traceback

        out_q.put((rank, "FAIL: " + traceback.format_exc()))


@pytest.mark.parametrize("world,per_rank,size", [(2, 1, (16, 12, 10)), (2, 4, (32, 32, 32)), (4, 1, (16, 16, 16)), (4, 2, (32, 16, 16))])
def test_combine_across_ranks_over_gloo(world, per_rank, size):
    import stencil_b200 as sb

    part = sb.Partition(size, sb.Radius.constant(1), 1, world * per_rank)
    order = part.indices()
    table = _partial_table(len(order))
    s = R.combine(table)
    want = tuple(bits(v) for v in (s.min, s.max, s.sum, s.sum2, s.rms)) + (s.count,)
    # the test has power: with three or more subdomains another order of the same partials gives other bits
    assert len(table) < 3 or R.combine(table[::-1]).sum != s.sum or R.combine(table[1:] + table[:1]).sum != s.sum
    ctx = mp.get_context("spawn")
    for reverse in (False, True):
        q = ctx.Queue()
        port = _free_port()
        procs = [ctx.Process(target=_worker, args=(r, world, port, size, per_rank, reverse, q)) for r in range(world)]
        for p in procs:
            p.start()
        results = dict(q.get(timeout=180) for _ in range(world))
        for p in procs:
            p.join(timeout=60)
        assert all(results[r] == want for r in range(world)), (reverse, results)
