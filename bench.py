#!/usr/bin/env python
"""bench.py -- jacobi3d cells/s at 512^3 per GPU, radius 1, FP64 (BASELINE.json configs[1]).

    python bench.py --gpus 1 --steps 20 --warmup 5
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
        bench.py --gpus N --steps K --warmup W
    python bench.py --impl reference ...      # the CPU arm (oracle port, all host cores)

A "step" is one iteration of the reference driver's loop (bin/jacobi3d.cu:296-368): interior kernel
|| halo exchange -> exterior slabs -> stream sync -> swap.  One JSON line on stdout (rank 0).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "jacobi3d_cells_per_s"
UNIT = "cells/s"


def parse():
    p = argparse.ArgumentParser()
    p.add_argument("--gpus", type=int, default=1)
    p.add_argument("--steps", type=int, default=20)
    p.add_argument("--warmup", type=int, default=5)
    p.add_argument("--impl", default="ours", choices=["ours", "reference"])
    p.add_argument("--size", type=int, default=512, help="per-GPU cube edge (BASELINE: 512)")
    p.add_argument("--dtype", default="f64", choices=["f32", "f64"])
    p.add_argument("--grow", default="yz", choices=["yz", "cube", "x"], help="which axes the weak-scaling rule grows (see grown_size)")
    p.add_argument("--no-cpu-baseline", action="store_true")
    p.add_argument("--no-e2e", action="store_true")
    p.add_argument("--no-overlap", action="store_true")
    p.add_argument("--no-exchange-bench", action="store_true", help="skip the halo-exchange latency leg (BASELINE metric part 2, configs[2])")
    p.add_argument("--no-parity", action="store_true", help="skip the bit-exact check against the oracle that follows the timed region")
    p.add_argument("--schedule", default="fused", choices=["fused", "queued", "host-sync"],
                   help="fused: one kernel per iteration = jacobi update + halo push into the neighbours' ghost cells (Jacobi3D.step_fused); "
                   "queued: interior || exchange -> exterior with CUDA-event dependencies (step_async); host-sync: the reference's loop (step)")
    p.add_argument("--host-sync", action="store_true", help="block the host after the exchange and after the exterior kernels like bin/jacobi3d.cu:337-365 (default: iterations queue back to back, dependencies as CUDA events)")
    p.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write the field they computed as DIR/jacobi_field_sample.npy (see dump_outputs)")
    args = p.parse_args()
    if args.steps < 1:
        p.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        p.error("--dump-outputs needs --impl ours")
    return args


def measured_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return json.load(f)["hbm_gbs"], "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def ncu_traffic(fused, n, dtype):
    """DRAM bytes per launch of the dominant kernel from the committed ncu summary (profiles/), with the file's hash so that
    a stale citation is detectable."""
    import hashlib

    if n != 512 or dtype != "f64":
        return {"traffic": None, "traffic_source": None}
    name = "jacobi_fused_r2.summary.txt" if fused else "jacobi_march_r1.summary.txt"
    path = os.path.join(ROOT, "profiles", name)
    try:
        text = open(path).read()
        for ln in text.splitlines():
            if ln.startswith("traffic = dram read + write (bytes)"):
                return {"traffic": int(float(ln.split()[-1])), "traffic_source": {"file": "profiles/" + name, "sha256": hashlib.sha256(text.encode()).hexdigest()[:16]}}
    except OSError:
        pass
    return {"traffic": None, "traffic_source": None}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md)."""

    Q = "index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, device: int):
        self.device, self.proc, self.lines = device, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100", "-i", str(self.device)],
                stdout=subprocess.PIPE,
                stderr=subprocess.DEVNULL,
                text=True,
            )
            self.t = threading.Thread(target=self._pump, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons, power = [], [], set(), []
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                mx.append(float(f[2]))
                power.append(float(f[3]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {
            "sm_mhz": float(np.median(sm)) if sm else None,
            "sm_max_mhz": max(mx) if mx else None,
            "power_w_max": max(power) if power else None,
            "samples": len(sm),
            "reasons": sorted(reasons),
        }


# --------------------------------------------------------------------------------------------- CPU arm
def time_cpu(n, dtype_name, steps, warmup, budget_s=0.0):
    """The oracle port of the same loop on one periodic n^3 subdomain (C + OpenMP, oracle/stencil_oracle.c), timed in its
    own process with a pinned OpenMP environment (oracle/cpu_bench.py: one thread per physical core of the affinity mask,
    capped by the cgroup quota; OMP_PROC_BIND=close, OMP_PLACES=cores; first touch with the compute loops' schedule).
    Used for `cpu_baseline` and for `--impl reference` (SURVEY.md fact 1: the reference has no runnable CPU path;
    BASELINE.md 2a: the CPU baseline is this restatement)."""
    from oracle import cpu_bench

    return cpu_bench.run_in_subprocess(n, dtype_name, steps, warmup, budget_s)


def cpu_model():
    try:
        for ln in open("/proc/cpuinfo"):
            if ln.startswith("model name"):
                return ln.split(":", 1)[1].strip()
    except OSError:
        pass
    return "unknown"


def run_reference(args, rank, world):
    """--impl reference: the reference's CPU implementation of the path = the oracle port (see CpuJacobi)."""
    if rank != 0:
        return
    n = args.size
    res = time_cpu(n, args.dtype, args.steps, max(args.warmup, 1))
    line = {
        "impl": "reference",
        "metric": METRIC,
        "value": res["value"],
        "unit": UNIT,
        "n_gpus": args.gpus,
        "steps": res["steps"],
        "warmup": max(args.warmup, 1),
        "ms_per_step": res["ms_per_step"],
        "higher_is_better": True,
        "scaling": "weak",
        "vs_baseline": None,
        "dtype": args.dtype,
        "data": "synthetic",
        "config": {
            "workload": f"jacobi3d {n}^3 radius-1 {args.dtype.upper()} (BASELINE configs[1]), one periodic subdomain on the host",
            "note": "reference has no runnable CPU path (SURVEY.md fact 1); this is the oracle port: C + OpenMP restatement of bin/jacobi3d.cu:296-368",
            "cpu": cpu_model(),
        },
        "cpu_baseline": {
            "value": res["value"],
            "unit": UNIT,
            "cores": res["cores"],
            "kind": "port",
            "sample": f"{res['steps']} full iterations of {n}^3 (interior + 6-face periodic exchange + exterior)",
            "host": res["host"],
            "omp": res["omp"],
        },
        "e2e": {"value": res["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# --------------------------------------------------------------------------------------------- halo exchange leg
def trimean(v):
    q1, q2, q3 = np.percentile(np.asarray(v, dtype=np.float64), [25, 50, 75])
    return float((q1 + 2 * q2 + q3) / 4)


def halo_exchange_metric(rank, world, gpus, ngpu, iters=30):
    """BASELINE metric part 2 / configs[2]: `dd.exchange(); dd.swap();` on 512^3 TOTAL, uniform radius 2, 3 x float,
    over this run's GPUs -- the timing loop of bin/bench_exchange.cu:39-54 (barrier, wall clock, trimean of 30, max
    over ranks).  Beside it the UNMODIFIED reference library on the same box and GPUs (oracle/_ref/ref_exchange_uniform,
    one process x N GPUs, its only mode here: no MPI in this image): its default transports (PeerAccessSender /
    PeerCopySender: pack -> cudaMemcpyPeerAsync -> unpack) and Method::CudaMpi (tx_cuda_aware_mpi; the single-process
    shim turns the device-pointer Isend/Irecv into a cudaMemcpyAsync, which favours the reference), and the same driver
    source linked against OUR C++ library (bin/exchange_uniform) when bin/ was built."""
    import torch
    import torch.distributed as td

    import stencil_b200 as sb

    size, q, r = (512, 512, 512), 3, 2
    dd = sb.DistributedDomain(*size)
    dd.set_gpus(gpus)
    dd.set_radius(sb.Radius.constant(r))
    for _ in range(q):
        dd.add_data(np.float32)
    dd.realize()
    host = td.new_group(backend="gloo") if world > 1 else None  # host-side barriers: no spinning NCCL kernel on the GPUs

    def barrier():
        if host is not None:
            td.barrier(group=host)

    times = []
    for i in range(iters + 3):
        torch.cuda.synchronize()
        barrier()
        t0 = time.perf_counter()
        dd.exchange()
        dd.swap()
        dt = time.perf_counter() - t0
        if i >= 3:
            times.append(dt)
    t = torch.tensor(times, dtype=torch.float64, device="cuda")
    if world > 1:
        td.all_reduce(t, op=td.ReduceOp.MAX)
    times = t.cpu().numpy()
    total = dd.exchange_bytes_for_method(sb.Method.Default)
    peer = dd.exchange_bytes_for_method(sb.Method.CudaMemcpyPeer)
    tb = torch.tensor([total, peer], dtype=torch.float64, device="cuda")
    if world > 1:
        td.all_reduce(tb)  # every rank counts what it sends
    total, peer = float(tb[0]), float(tb[1])
    dd.close()
    us = trimean(times) * 1e6
    out = {
        "workload": "bench_exchange 512^3 total, uniform radius 2, 3 x float (BASELINE configs[2]); dd.exchange(); dd.swap(); trimean of %d, max over ranks" % iters,
        "us": us,
        "min_us": float(times.min()) * 1e6,
        "bytes": int(total),
        "cross_gpu_bytes": int(peer),
        # payload every GPU sends (= receives) over NVLink per exchange / exchange time
        "nvlink_gbs_per_dir": (peer / ngpu) / (us * 1e-6) / 1e9 if peer > 0 else 0.0,
        "nvlink_peak_gbs_per_dir": 900.0,
        "transport": "fused direct write into the neighbours' ghost cells (peer access / CUDA IPC), thin rows staged; ready/done flags on the device",
    }
    barrier()
    if rank == 0:  # the reference library, one process x N GPUs, while the other ranks wait on the host
        def ref(exe, how):
            path = os.path.join(ROOT, exe)
            if not os.path.exists(path):
                return None
            env = dict(os.environ, CUDA_VISIBLE_DEVICES=",".join(str(g) for g in range(ngpu)))
            for k in ("RANK", "WORLD_SIZE", "LOCAL_RANK", "OMPI_COMM_WORLD_SIZE", "PMI_SIZE"):
                env.pop(k, None)
            try:
                o = subprocess.run([path, "512", "512", "512", str(q), str(r), str(iters), how], cwd="/tmp", env=env, capture_output=True, text=True, timeout=300)
                row = [ln for ln in o.stdout.splitlines() if "_exchange," in ln][-1].split(",")
                return float(row[-2]) * 1e6  # trimean seconds -> us
            except Exception as e:  # the reference aborting is a result, not a bench failure
                return "failed: %s" % (str(e)[:80],)

        out["reference_us"] = ref("oracle/_ref/ref_exchange_uniform", "default")
        out["reference_cudampi_us"] = ref("oracle/_ref/ref_exchange_uniform", "cudampi")
        out["ours_cpp_one_process_us"] = ref("bin/exchange_uniform", "default")
        out["reference_note"] = "reference library unmodified, 1 process x %d GPU(s) (no MPI here); cudampi = Method::CudaMpi over the single-process shim" % ngpu
    barrier()
    return out


# --------------------------------------------------------------------------------------------- GPU arm
def grown_size(n, ngpu, grow):
    """The global size for `ngpu` subdomains of n^3.
    --grow yz (default): the weak-scaling rule of bin/jacobi3d.cu:189-199 -- multiply the prime factors of the subdomain
        count into the currently smallest axis -- restricted to the two slow axes (ties to z): x, the contiguous axis,
        whose faces are single cells one row pitch apart, is never cut.  1 / 2 / 4 / 8 GPUs: 512^3, 512x512x1024,
        512x1024x1024, 512x1024x2048 (partition 1x2x4).
    --grow cube: the rule on all three axes with ties to z first (8 GPUs: 1024^3, partition 2x2x2);
    --grow x: the reference's literal order, ties to x first (the same shapes as `cube`, mirrored)."""
    from stencil_b200.domain import prime_factors
    from stencil_b200.jacobi import scaled_size

    if grow == "yz":
        y = z = n
        for pf in prime_factors(ngpu):
            if z <= y:
                z *= pf
            else:
                y *= pf
        return n, y, z
    X, Y, Z = scaled_size(n, n, n, ngpu)
    return (Z, Y, X) if grow == "cube" else (X, Y, Z)


DUMP_POINTS = 1 << 22  # 32 MiB of FP64: the 512^3 field itself is 1 GiB
DUMP_SEED = 20240517


def dump_outputs(out_dir, dd, h, size, dtype, rank, world):
    """--dump-outputs: the field the timed steps left in curr (what a caller of the jacobi loop reads back), at DUMP_POINTS
    cells drawn with a fixed seed from the global X x Y x Z domain -- the same cells for every partition, process count and
    build -- in the run's dtype, as out_dir/jacobi_field_sample.npy on rank 0."""
    import torch
    import torch.distributed as td

    X, Y, Z = size
    rng = np.random.default_rng(DUMP_SEED)
    pts = np.stack([rng.integers(0, Z, DUMP_POINTS), rng.integers(0, Y, DUMP_POINTS), rng.integers(0, X, DUMP_POINTS)], axis=1)  # z, y, x
    vals = np.zeros(DUMP_POINTS, dtype=dtype)
    for d in dd.domains():
        lo = np.array(d.origin()[::-1])
        inside = np.all((pts >= lo) & (pts < lo + np.array(d.size()[::-1])), axis=1)
        q = pts[inside] - lo
        vals[inside] = d.interior_to_host(h.id)[q[:, 0], q[:, 1], q[:, 2]]
    if world > 1:
        t = torch.from_numpy(vals).cuda()
        td.all_reduce(t)  # every cell lives on one rank; the others add zeros
        vals = t.cpu().numpy()
    if rank == 0:
        os.makedirs(out_dir, exist_ok=True)
        np.save(os.path.join(out_dir, "jacobi_field_sample.npy"), vals)


def run_ours(args, rank, world):
    import torch
    import torch.distributed as td

    import stencil_b200 as sb
    from stencil_b200.jacobi import Jacobi3D, jacobi_radius, scaled_size

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- stencil_b200 has no CPU fallback")
    local = int(os.environ.get("LOCAL_RANK", 0))
    torch.cuda.set_device(local)
    L = sb.lib()
    dtype = np.float64 if args.dtype == "f64" else np.float32
    es = np.dtype(dtype).itemsize
    n = args.size
    ngpu = args.gpus
    if world == 1 and ngpu > 1:
        gpus = list(range(ngpu))  # one process driving N GPUs (the reference's 1 rank x N GPUs mode)
    else:
        gpus = [local]
    X, Y, Z = grown_size(n, ngpu, args.grow)
    cut = os.environ.get("SB_BENCH_CUT", "")  # diagnostics: one cut along a chosen axis at 2 ranks
    if cut:
        X, Y, Z = {"x": (2 * n, n, n), "y": (n, 2 * n, n), "z": (n, n, 2 * n)}[cut] if ngpu == 2 else (X, Y, Z)

    dd = sb.DistributedDomain(X, Y, Z)
    dd.set_gpus(gpus)
    dd.set_radius(jacobi_radius())
    h = dd.add_data(dtype, "d")
    dd.realize()
    jac = Jacobi3D(dd, h, overlap=not args.no_overlap)
    jac.init(0.5)

    def barrier():
        for d in dd.domains():
            sb._lib.check(L.sb_device_sync(d.gpu()))
        if world > 1:
            td.barrier()
            torch.cuda.synchronize()

    schedule = "host-sync" if (args.host_sync or not jac.overlap) else args.schedule
    if schedule == "fused" and os.environ.get("SB_FORCE_NCCL") == "1":
        schedule = "queued"  # the fused schedule stores into peer memory
    queued = schedule == "queued"
    fused = schedule == "fused"
    for _ in range(max(args.warmup, 3)):
        if fused:
            jac.step_fused()
        elif queued:
            jac.step_async()
        else:
            jac.step()
    jac.synchronize()
    if fused and not getattr(jac, "fused_supported", True):
        # x faces cross ranks: Jacobi3D.step_fused delegates to the queued schedule (measured faster, see jacobi.py)
        schedule, fused, queued = "queued", False, True

    # ---- device-resident timed region -------------------------------------------------------
    cs0 = jac.streams[0]
    k0 = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps)]
    k1 = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps)]
    ev_a, ev_b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
        time.sleep(0.3)
    barrier()
    launches0 = L.sb_launch_count()
    t_wall0 = time.perf_counter()
    ev_a.record(cs0)
    for i in range(args.steps):
        if fused:
            jac.step_fused(timing=(k0[i], k1[i]))
            continue
        if queued:
            jac.step_async(timing=(k0[i], k1[i]))
            continue
        k0[i].record(cs0)
        if jac.overlap:
            jac.launch_interior()
            k1[i].record(cs0)
            dd.exchange()
            jac.launch_exterior()
        else:
            dd.exchange()
            jac.launch_whole()
            k1[i].record(cs0)
        jac.synchronize()
        dd.swap()
    if queued:
        # the last iteration ends with the exterior kernels: bring them onto the timed stream
        for e in jac._ev_ext:
            cs0.wait_event(e)
    if fused:
        for e in list(jac._ev_fused or ()) + list(getattr(jac, "_ev_fused_x", None) or ()):  # other subdomains, last x exchange
            cs0.wait_event(e)
    ev_b.record(cs0)
    barrier()
    t_wall = time.perf_counter() - t_wall0
    launches = L.sb_launch_count() - launches0
    clocks = sampler.stop() if rank == 0 else None
    ms_total = ev_a.elapsed_time(ev_b)
    kern_ms = float(np.mean([a.elapsed_time(b) for a, b in zip(k0, k1)]))
    t = torch.tensor([ms_total, t_wall * 1e3], dtype=torch.float64, device="cuda")
    if world > 1:
        td.all_reduce(t, op=td.ReduceOp.MAX)
    ms_total, wall_ms = float(t[0]), float(t[1])
    ms_step = ms_total / args.steps
    cells = X * Y * Z
    value = cells / (ms_step * 1e-3)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, dd, h, (X, Y, Z), dtype, rank, world)

    # ---- roofline of the dominant kernel (interior jacobi) ----------------------------------
    peak, peak_src = measured_peaks()
    dom_cells = jac.interior_cells if (jac.overlap and not fused) else sum(int(np.prod(d.size())) for d in dd.domains())
    if world == 1 and len(dd.domains()) > 1:
        # events sit on the first GPU's stream: attribute that subdomain's cells only
        dom_cells = dom_cells // len(dd.domains())
    alg_bytes = 2 * es * dom_cells
    achieved = alg_bytes / (kern_ms * 1e-3) / 1e9
    roofline = {
        "bound": "hbm",
        "kernel": "jacobi_fused_kernel (whole region + halo push + rank handshake)" if fused else ("jacobi_march_kernel (interior region)" if jac.overlap else "jacobi_march_kernel (whole region)"),
        "achieved": achieved,
        "peak": peak,
        "unit": "GB/s",
        "frac": achieved / peak,
        "peak_source": peak_src,
        "algorithmic_bytes_per_launch": alg_bytes,
        "kernel_ms": kern_ms,
        # dram__bytes_read.sum + dram__bytes_write.sum of one launch of this kernel, read from the committed `ncu --set full`
        # summary named in traffic_source (not re-measured by this run; null when no capture of this configuration exists)
        **ncu_traffic(fused, n, args.dtype),
        "step_frac_of_roofline": (2 * es * cells / ngpu) / (ms_step * 1e-3) / 1e9 / peak,
    }

    # ---- end to end: host buffers in, host result out, every step ---------------------------
    e2e = None
    if not args.no_e2e:
        d0 = dd.domains()[0]
        raw = d0.raw_size()
        nbytes = raw[0] * raw[1] * raw[2] * es
        pin_in = torch.empty(nbytes, dtype=torch.uint8, pin_memory=True)
        pin_out = torch.empty(8, dtype=torch.uint8, pin_memory=True)
        host_field = pin_in.numpy().view(dtype).reshape(raw[::-1])
        host_field[...] = 0.5
        res_dev = torch.zeros(1, dtype=torch.float64, device=f"cuda:{d0.gpu()}")
        lo, hi = d0.get_compute_region()
        steps_e = max(3, min(args.steps, 10))

        def e2e_step():
            # host field -> curr (pinned H2D on the compute stream), one iteration, residual -> host
            sb._lib.check(L.sb_memcpy(d0.curr_[0], pin_in.data_ptr(), nbytes, d0.gpu(), sb._lib.stream_ptr(cs0)))
            cs0.synchronize()
            jac.step()
            sb._lib.check(
                L.sb_sqdiff(d0.curr_data(0), d0.next_data(0), es, sb._lib.i3(d0.accessor_origin()), sb._lib.i3(lo), sb._lib.i3(hi), res_dev.data_ptr(), sb._lib.stream_ptr(cs0))
            )
            sb._lib.check(L.sb_memcpy(pin_out.data_ptr(), res_dev.data_ptr(), 8, d0.gpu(), sb._lib.stream_ptr(cs0)))
            cs0.synchronize()

        for _ in range(2):
            e2e_step()
        barrier()
        t0 = time.perf_counter()
        for _ in range(steps_e):
            e2e_step()
        barrier()
        te = torch.tensor([(time.perf_counter() - t0) / steps_e], dtype=torch.float64, device="cuda")
        if world > 1:
            td.all_reduce(te, op=td.ReduceOp.MAX)
        e2e = {
            "value": cells / float(te[0]),
            "unit": UNIT,
            "h2d_bytes_per_step": int(nbytes) * max(1, len(dd.domains())) * world,
            "d2h_bytes_per_step": 8 * world,
            "ms_per_step": float(te[0]) * 1e3,
            "steps": steps_e,
            "definition": "every step: pinned-host field -> curr (H2D), one jacobi iteration through DistributedDomain, L2 residual -> host (D2H)",
        }

    # ---- CPU baseline (rank 0, N=1, bounded sample) -----------------------------------------
    cpu = None
    if rank == 0 and ngpu == 1 and not args.no_cpu_baseline:
        r = time_cpu(n, args.dtype, steps=50, warmup=1, budget_s=12.0)
        cpu = {
            "value": r["value"],
            "unit": UNIT,
            "cores": r["cores"],
            "kind": "port",
            "sample": f"{r['steps']} full iterations of {n}^3 {args.dtype} (<=12 s), oracle/stencil_oracle.c with OpenMP on {cpu_model()}",
            "host": r["host"],
            "omp": r["omp"],
        }

    if rank == 0:
        line = {
            "metric": METRIC,
            "value": value,
            "unit": UNIT,
            "n_gpus": ngpu,
            "steps": args.steps,
            "warmup": max(args.warmup, 3),
            "ms_per_step": ms_step,
            "higher_is_better": True,
            "scaling": "weak",
            "vs_baseline": None,
            "dtype": args.dtype,
            "data": "synthetic",
            "per_gpu": value / ngpu,
            "wall_ms_per_step": wall_ms / args.steps,
            "config": {
                "workload": f"jacobi3d {n}^3 per GPU radius-1 {args.dtype.upper()} (BASELINE configs[1]); global {X}x{Y}x{Z} (weak-scaling rule of bin/jacobi3d.cu:189-199, --grow {args.grow})",
                "parallelism": f"{world} process(es) x {len(gpus)} GPU(s), 3-D domain decomposition, fused P2P halo write",
                "overlap": jac.overlap,
                "schedule": schedule,
                "iteration_sync": {
                    "fused": "one kernel per iteration: update + halo push into the neighbours' ghost cells; ranks ordered inside the kernel (its first CTA publishes the iteration number to every neighbour rank, boundary tiles poll the neighbour's word), subdomains of one process by CUDA events (Jacobi3D.step_fused)",
                    "queued": "interior || exchange -> exterior, dependencies as CUDA events + ready/done flags (Jacobi3D.step_async)",
                    "host-sync": "host-side after exchange and exterior (Jacobi3D.step, the reference's loop)",
                }[schedule],
                "l2": "inputs larger than L2 (2 x %.2f GiB per GPU vs 126 MB)" % (2 * es * (n + 2) ** 3 / 2**31),
                "init": "0.5 everywhere, hot/cold spheres (bin/jacobi3d.cu:18-63)",
            },
            "roofline": roofline,
            "cpu_baseline": cpu,
            "e2e": e2e,
            "gpu_launches": int(launches),
            "clocks": clocks,
        }
    jac.close()
    dd.close()
    # ---- parity (outside every timed region): the same schedule on 128^3 per GPU against the single-address-space
    # oracle, bit for bit, on every rank -- the analogue of the reference's whole-subdomain exchange check
    # (test/test_cuda_mpi_exchange.cu:193-245) for the loop of bin/jacobi3d.cu:296-368
    parity = None
    if not args.no_parity:
        sys.path.insert(0, os.path.join(ROOT, "tests"))
        from jacobi_parity import check_jacobi_parity

        kinds = {"fused": ("fused",) * 6 + ("queued",) * 2, "queued": ("queued",) * 6 + ("host-sync",) * 2, "host-sync": ("host-sync",) * 4}[schedule]
        parity = check_jacobi_parity(grown_size(128, ngpu, args.grow), gpus, dtype, kinds, world)

    xchg = None
    if not args.no_exchange_bench:
        xchg = halo_exchange_metric(rank, world, gpus, ngpu)
    if rank == 0:
        line["parity_check"] = parity
        line["halo_exchange"] = xchg
        print(json.dumps(line), flush=True)
    if parity is not None and not parity["bit_exact"]:
        raise SystemExit(f"bench.py: parity check FAILED: {parity}")


def main():
    args = parse()
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    if world > 1:
        import torch
        import torch.distributed as td

        torch.cuda.set_device(int(os.environ.get("LOCAL_RANK", 0)))
        td.init_process_group("nccl", device_id=torch.device("cuda", int(os.environ.get("LOCAL_RANK", 0))))
    try:
        run_ours(args, rank, world)
    finally:
        if world > 1:
            import torch.distributed as td

            td.destroy_process_group()


if __name__ == "__main__":
    main()
