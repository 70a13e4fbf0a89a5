"""Host-side logic of bench.py that decides WHAT is measured (no GPU): the weak-scaling shapes and how the partitioner
cuts them.  bin/jacobi3d.cu:189-199 is the size rule, partition.hpp:157-255 the partitioner (oracle/geometry.py)."""
import importlib.util
import os

import pytest

from oracle import geometry as g

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def bench():
    spec = importlib.util.spec_from_file_location("bench_module", os.path.join(ROOT, "bench.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod


@pytest.mark.parametrize("n", [64, 128, 512])
@pytest.mark.parametrize("ngpu", [1, 2, 3, 4, 6, 8])
@pytest.mark.parametrize("grow", ["yz", "cube", "x"])
def test_every_gpu_gets_an_n_cubed_subdomain(bench, n, ngpu, grow):
    size = bench.grown_size(n, ngpu, grow)
    assert size[0] * size[1] * size[2] == ngpu * n**3
    part = g.NodePartition(size, g.Radius.constant(1), 1, ngpu)
    dim = part.dim()
    assert dim[0] * dim[1] * dim[2] == ngpu
    if grow == "yz":
        assert size[0] == n and dim[0] == 1  # x, the contiguous axis, is never grown and never cut
    sizes = {tuple(part.subdomain_size(i)) for i in part.all_indices()}
    if ngpu in (1, 2, 4, 8):
        assert sizes == {(n, n, n)}


def test_reference_order_is_the_size_rule_of_the_driver(bench):
    # bin/jacobi3d.cu:189-199 restated in oracle/geometry.py
    for ngpu in (1, 2, 4, 8):
        assert tuple(bench.grown_size(512, ngpu, "x")) == tuple(g.jacobi_scaled_size(512, 512, 512, ngpu))
    assert tuple(bench.grown_size(512, 8, "yz")) == (512, 1024, 2048)
    assert tuple(bench.grown_size(512, 4, "yz")) == (512, 1024, 1024)
    assert tuple(bench.grown_size(512, 2, "yz")) == (512, 512, 1024)
    assert tuple(bench.grown_size(512, 2, "cube")) == (512, 512, 1024)
    assert tuple(bench.grown_size(512, 8, "cube")) == (1024, 1024, 1024)


def test_dump_outputs_samples_the_global_field(bench, tmp_path, monkeypatch):
    """--dump-outputs reads each seeded global cell from the subdomain that owns it, whatever the partition."""
    import numpy as np

    X, Y, Z = 40, 30, 50
    field = np.random.default_rng(0).standard_normal((Z, Y, X))

    class Sub:
        def __init__(self, origin, size):
            self.o, self.s = origin, size

        def origin(self):
            return self.o

        def size(self):
            return self.s

        def interior_to_host(self, q):
            (x, y, z), (sx, sy, sz) = self.o, self.s
            return field[z : z + sz, y : y + sy, x : x + sx].copy()

    class Dom:
        def domains(self):
            return [Sub((0, 0, 0), (40, 30, 20)), Sub((0, 0, 20), (40, 16, 30)), Sub((0, 16, 20), (40, 14, 30))]

    class Handle:
        id = 0

    monkeypatch.setattr(bench, "DUMP_POINTS", 5000)
    bench.dump_outputs(str(tmp_path), Dom(), Handle(), (X, Y, Z), np.float64, 0, 1)
    got = np.load(tmp_path / "jacobi_field_sample.npy")
    rng = np.random.default_rng(bench.DUMP_SEED)
    z, y, x = rng.integers(0, Z, 5000), rng.integers(0, Y, 5000), rng.integers(0, X, 5000)
    assert got.dtype == np.float64 and np.array_equal(got, field[z, y, x])
