"""The C++ API (include/stencil/*.hpp + lib/libstencil.a) on a GPU: our jacobi3d_b200 driver (the reference loop over
stencil::FusedJacobi3d) compared with the reference's own kernel through stored golden vectors, our multi-rank exchange
check, and -- when `make drivers REF=<reference checkout>` has built them (__graft_entry__.build() does so when
STENCIL_REFERENCE names a checkout) -- the REFERENCE's own Catch2 suites and drivers compiled unchanged against our
headers and library.  Match: test/test_exchange.cu:37-220, test/test_cuda_*.cu, bin/jacobi3d.cu, bin/bench_exchange.cu."""
import os
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BIN = os.path.join(ROOT, "bin")
pytestmark = pytest.mark.gpu


def need(*names):
    """The reference's drivers and suites: they exist only where `make drivers REF=<reference checkout>` ran."""
    missing = [n for n in names if not os.path.exists(os.path.join(ROOT, n))]
    if missing:
        pytest.skip("reference drivers not built: " + ", ".join(missing) + " missing -- `make drivers REF=<reference checkout>`")


def built(*names):
    """This repository's own drivers: `make` builds them, so a missing one is a build failure."""
    missing = [n for n in names if not os.path.exists(os.path.join(ROOT, n))]
    assert not missing, ", ".join(missing) + " missing -- run `make`"


def run(cmd, tmp_path, timeout=900):
    out = subprocess.run(cmd, cwd=tmp_path, capture_output=True, text=True, timeout=timeout)
    assert out.returncode == 0, (cmd, out.stdout[-3000:], out.stderr[-3000:])
    return out


def test_reference_host_suite_against_our_library(tmp_path):
    need("bin/test_cpu")
    out = run([os.path.join(BIN, "test_cpu")], tmp_path)
    assert "All tests passed" in out.stdout, out.stdout[-2000:]


def test_reference_cuda_suite_against_our_library(tmp_path):
    """pack / packer / translate (4 back-ends) / local_domain / rcstream / align / gpu_topo / test_exchange."""
    need("bin/test_cuda")
    out = run([os.path.join(BIN, "test_cuda")], tmp_path)
    assert "All tests passed" in out.stdout, out.stdout[-2000:]


def test_reference_jacobi3d_driver_runs_unchanged(tmp_path):
    need("bin/jacobi3d")
    out = run([os.path.join(BIN, "jacobi3d"), "64", "64", "64", "-n", "5"], tmp_path)
    line = [ln for ln in out.stdout.splitlines() if ln.startswith("jacobi3d,")]
    assert line, out.stdout[-2000:]
    f = line[-1].split(",")
    assert float(f[-1]) > 0 and float(f[-2]) > 0  # trimean and min iteration time


def test_reference_bench_exchange_driver_runs_unchanged(tmp_path):
    need("bin/bench_exchange")
    out = run([os.path.join(BIN, "bench_exchange"), "--x", "64", "--y", "64", "--z", "64", "--q", "3", "--fr", "2", "--er", "2", "--cr", "2", "--iters", "5"], tmp_path)
    rows = [ln for ln in out.stdout.splitlines() if ln.startswith("64-64-64/")]
    assert [r.split(",")[0].split("/")[1] for r in rows] == ["px", "x", "faces", "face&edge", "uniform"], out.stdout[-2000:]
    assert all(float(r.split(",")[2]) > 0 for r in rows)  # trimean seconds per exchange + swap


@pytest.mark.parametrize("shape", [(64, 64, 64), (96, 80, 72)])
def test_jacobi3d_b200_matches_the_reference_kernel(tmp_path, shape):
    """Our C++ fast path (FusedJacobi3d: fused kernel; and its reference-schedule fallback) against the reference's own
    stencil_kernel built with IEEE division (tests/golden/jacobi_ref.npz, ieee_*), bit for bit after 10 iterations."""
    built("bin/jacobi3d_b200")
    gold = np.load(os.path.join(ROOT, "tests", "golden", "jacobi_ref.npz"))
    si = [tuple(s) for s in gold["shapes"].tolist()].index(shape)
    want = gold[f"ieee_{si}"][list(gold["iters"]).index(10)].ravel()
    n = [str(v) for v in shape]
    # the driver scales the size by the prime factors of the GPU count (bin/jacobi3d.cu:189-199): pin it to one GPU
    env = dict(os.environ, CUDA_VISIBLE_DEVICES=os.environ.get("CUDA_VISIBLE_DEVICES", "0").split(",")[0])
    for extra in ([], ["--reference-schedule"]):
        got_f = tmp_path / "got.bin"
        out = subprocess.run([os.path.join(BIN, "jacobi3d_b200"), *n, "-n", "5", "--dump", str(got_f)] + extra, cwd=tmp_path, env=env, capture_output=True, text=True, timeout=600)
        assert out.returncode == 0, out.stderr[-3000:]
        got = np.fromfile(got_f, dtype=np.float32)  # 5 timed + 5 queued iterations = 10
        assert got.shape == want.shape and np.array_equal(got, want), (shape, extra, int(np.count_nonzero(got != want)))
        assert float(np.ptp(got)) > 0


def mpirun_env():
    return {k: v for k, v in os.environ.items() if k not in ("WORLD_SIZE", "RANK", "LOCAL_RANK")}


@pytest.mark.parametrize("ranks", [2, 4])
def test_cpp_multi_rank_exchange(tmp_path, ranks):
    """One process per rank through the C++ API (bin/sb_mpirun = this repo's node-local MPI stand-in): allocations, staging
    buffers and flag mailboxes are shared through CUDA IPC handles sent over MPI, the exchange is the fused direct write +
    device-side ready/done flags.  Every rank checks the WHOLE allocation of its subdomains (ghost cells included) against
    the periodically wrapped field, 5 radius shapes x 3 quantities x 3 rounds with swaps.  With fewer GPUs than ranks the
    ranks share GPUs (the reference's rule, src/stencil.cu:76-85), so this runs on a 1-GPU box as well.
    Match: test/test_cuda_mpi_exchange.cu:193-245, include/stencil/tx_cuda.cuh:185-492, src/tx_colocated.cu."""
    built("bin/sb_mpirun", "bin/test_exchange_multigpu")
    out = subprocess.run([os.path.join(BIN, "sb_mpirun"), "-n", str(ranks), os.path.join(BIN, "test_exchange_multigpu")], cwd=tmp_path, env=mpirun_env(),
                         capture_output=True, text=True, timeout=900)  # fmt: skip
    assert out.returncode == 0 and "ALL OK" in out.stdout, out.stdout[-3000:] + out.stderr[-3000:]
    assert f"on {ranks} rank(s)" in out.stdout


def test_reference_jacobi3d_driver_one_rank_per_gpu(tmp_path):
    """The reference's unchanged jacobi3d driver as 2 ranks (what `mpirun -n 2 jacobi3d` is on a machine with MPI)."""
    built("bin/sb_mpirun")
    need("bin/jacobi3d")
    out = subprocess.run([os.path.join(BIN, "sb_mpirun"), "-n", "2", os.path.join(BIN, "jacobi3d"), "64", "64", "64", "-n", "5"], cwd=tmp_path, env=mpirun_env(),
                         capture_output=True, text=True, timeout=600)  # fmt: skip
    assert out.returncode == 0, out.stdout[-2000:] + out.stderr[-3000:]
    line = [ln for ln in out.stdout.splitlines() if ln.startswith("jacobi3d,")]
    assert line and line[-1].split(",")[2] == "2", out.stdout[-2000:]  # world size 2
