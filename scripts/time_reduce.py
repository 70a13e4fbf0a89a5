"""Time the field reductions (sb_reduce) on one GPU and write DIR/time_reduce.json + DIR/time_reduce.txt.

    python scripts/time_reduce.py --out DIR [--reps 50]

Cases: 512^3 FP64 VALUE (radius-1 layout, first compute cell 16-byte aligned), 512^3 FP32 VALUE (radius 1: rows
alternate between two 16-byte phases), 512^3 FP64 DIFF, 256^3 FP64 VECTOR (radius 3), Astaroth.diagnostics() at 256^3
FP64 (9 reductions, 11 field reads), the existing sb_sqdiff against DIFF at 512^3, and torch on the same compute-region
view (aminmax + sum + sum(x*x)) as what a user would write without this library.  Every input is larger than the
126 MB L2.  Bytes = operands x element size x cells (each operand read once); GB/s over CUDA-event time per launch.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import stencil_b200 as sb  # noqa: E402
from stencil_b200 import reduce as R  # noqa: E402
from stencil_b200._lib import Pitched, check, i3, lib, stream_ptr  # noqa: E402

DATASHEET_GBS = 7700.0  # HGX B200 data sheet, one GPU
MEASURED_COPY_GBS = 6480.5  # copy rate measured for this project on a B200 (README.md, profiles/)


def peak():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "MEASURED_PEAKS.json hbm_gbs"
    except (OSError, KeyError, ValueError):
        return DATASHEET_GBS, "data sheet 7.7 TB/s (no MEASURED_PEAKS.json)"


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()  # fmt: skip
    except (OSError, subprocess.SubprocessError):
        out = ""
    return out or torch.cuda.get_device_name(0) + " (power limit not readable)"


def field(raw, dtype, lead_bytes, seed):
    """A device allocation of raw (x, y, z) elements starting lead_bytes into its block, filled with N(0, 1) on the GPU."""
    n = raw[0] * raw[1] * raw[2]
    es = np.dtype(dtype).itemsize
    t = torch.empty(n + 16 // es, dtype=torch.float64 if es == 8 else torch.float32, device="cuda:0")
    g = torch.Generator(device="cuda:0")
    g.manual_seed(seed)
    t.normal_(generator=g)
    off = lead_bytes // es
    view = t[off : off + n].view(raw[2], raw[1], raw[0])
    return t, view, Pitched(view.data_ptr(), raw[0] * es, raw[1])


def time_launches(fn, stream, reps, warmup=5):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for _ in range(reps):
        fn()
    e1.record(stream)
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--reps", type=int, default=50)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("time_reduce.py needs a CUDA device")
    os.makedirs(args.out, exist_ok=True)
    torch.cuda.set_device(0)
    hbm, hbm_src = peak()
    info = gpu_info()
    stream = torch.cuda.Stream()
    ws = R.Workspace(0)
    rows = []
    lines = [f"GPU: {info}", f"peak for the share: {hbm:.1f} GB/s ({hbm_src}); also shown: share of the measured copy rate {MEASURED_COPY_GBS} GB/s", ""]

    def record(name, ms, nbytes, extra=None):
        gbs = nbytes / ms / 1e6
        row = dict(case=name, ms=round(ms, 5), bytes=nbytes, gbs=round(gbs, 1), share_of_peak=round(gbs / hbm, 4), peak_source=hbm_src,
                   share_of_measured_copy=round(gbs / MEASURED_COPY_GBS, 4))  # fmt: skip
        row.update(extra or {})
        rows.append(row)
        line = f"{name:<44s} {ms:8.4f} ms  {nbytes / 1e9:6.3f} GB  {gbs:7.1f} GB/s  {100 * gbs / hbm:5.1f} % of {hbm_src}  {100 * gbs / MEASURED_COPY_GBS:5.1f} % of measured copy"
        lines.append(line)
        print(line, flush=True)

    def reduce_case(name, kind, ptrs, es, acc, lo, hi):
        cells = R.cells(lo, hi)
        ms = time_launches(lambda: ws.launch(kind, ptrs, es, acc, lo, hi, stream), stream, args.reps)
        record(name, ms, len(ptrs) * es * cells)
        return ws.result(stream)

    n = 512
    raw = (n + 2,) * 3
    acc, lo, hi = (-1, -1, -1), (0, 0, 0), (n, n, n)
    keep_a, va, pa = field(raw, np.float64, 8, 1)  # LocalDomain.lead_bytes: 8 for FP64 radius 1
    res = reduce_case("512^3 FP64 VALUE (r=1, lead 8)", R.VALUE, [pa], 8, acc, lo, hi)
    inner = va[1:-1, 1:-1, 1:-1]
    mn, mx = torch.aminmax(inner)
    assert res[0] == mn.item() and res[1] == mx.item(), "VALUE min/max differ from torch.aminmax"
    keep_b, vb, pb = field(raw, np.float64, 8, 2)
    reduce_case("512^3 FP64 DIFF", R.DIFF, [pa, pb], 8, acc, lo, hi)

    # the existing sqdiff kernel on the same operands (float atomics, one division per element)
    out = torch.zeros(1, dtype=torch.float64, device="cuda:0")
    fn = lib().sb_sqdiff
    args_sq = (pa, pb, 8, i3(acc), i3(lo), i3(hi), C.c_void_p(out.data_ptr()), stream_ptr(stream))
    ms = time_launches(lambda: check(fn(*args_sq)), stream, args.reps)
    record("512^3 FP64 sb_sqdiff (existing)", ms, 2 * 8 * n**3)

    # what a user does today: torch reductions on the strided compute-region view
    def torch_value():
        with torch.cuda.stream(stream):
            torch.aminmax(inner)
            inner.sum()
            (inner * inner).sum()

    ms = time_launches(torch_value, stream, max(5, args.reps // 5))
    record("512^3 FP64 torch aminmax+sum+sum(x*x) (view)", ms, 8 * n**3, dict(note="same 1 read of the field counted; torch reads it 4 times and writes x*x"))
    del keep_b, vb, pb, inner
    keep_a = va = pa = None
    torch.cuda.empty_cache()

    keep_f, vf, pf = field(raw, np.float32, 0, 3)  # 2056-byte rows: two 16-byte phases
    reduce_case("512^3 FP32 VALUE (r=1, alternating phases)", R.VALUE, [pf], 4, acc, lo, hi)
    keep_f = vf = pf = None
    torch.cuda.empty_cache()

    m = 256
    raw3 = (m + 6,) * 3
    vec = [field(raw3, np.float64, 8, 10 + i) for i in range(3)]
    reduce_case("256^3 FP64 VECTOR (r=3, lead 8)", R.VECTOR, [v[2] for v in vec], 8, (-3, -3, -3), (0, 0, 0), (m, m, m))
    del vec
    torch.cuda.empty_cache()

    from stencil_b200 import astaroth as ac

    dd = sb.DistributedDomain(m, m, m)
    dd.set_gpus([0])
    dd.set_radius(3)
    handles = [dd.add_data(np.float64, nm) for nm in ac.FIELDS]
    dd.realize()
    d = dd.domains()[0]
    rng = np.random.default_rng(0)
    for q in range(8):
        d.quantity_from_host(q, 0.1 * rng.standard_normal(tuple(reversed(d.raw_size()))))
    sim = ac.Astaroth(dd, handles)
    for _ in range(3):
        sim.diagnostics()
    reps = max(10, args.reps // 5)
    t0 = time.perf_counter()
    for _ in range(reps):
        sim.diagnostics()
    ms = (time.perf_counter() - t0) * 1e3 / reps
    record("256^3 FP64 Astaroth.diagnostics() (9 reductions)", ms, 11 * 8 * m**3, dict(note="host wall clock per call, includes 9 host waits"))
    dd.close()
    ws.free()

    with open(os.path.join(args.out, "time_reduce.json"), "w") as f:
        json.dump(dict(gpu=info, reps=args.reps, rows=rows), f, indent=1)
    with open(os.path.join(args.out, "time_reduce.txt"), "w") as f:
        f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
