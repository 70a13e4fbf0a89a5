"""Run under torchrun with 2 ranks (one GPU each): DistributedDomain.reduce gives the same bits on both ranks, and the
same bits as one process driving the same two-subdomain partition on one GPU (set_gpus([g, g])).
    python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 --master-port 29541 tests/mp_reduce_check.py"""
import os
import struct
import sys

import numpy as np
import torch
import torch.distributed as td

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import stencil_b200 as sb  # noqa: E402
from oracle import np_oracle as no  # noqa: E402
from stencil_b200 import reduce as R  # noqa: E402

SIZE = (96, 64, 80)
KINDS = [(R.VALUE, [0]), (R.EXP, [1]), (R.VECTOR, [0, 1, 2]), (R.ALFVEN, [0, 1, 2, 3]), (R.DIFF, [(0, "curr"), (0, "next")])]


def run(gpus, dtype):
    """Every kind over the whole domain, as tuples of the bit patterns of (min, max, sum, sum2) and the count."""
    dd = sb.DistributedDomain(*SIZE)
    dd.set_gpus(gpus)
    dd.set_radius(sb.Radius.constant(2))
    hs = [dd.add_data(dtype) for _ in range(4)]
    dd.realize()
    rng = np.random.default_rng(8)
    glob = [rng.uniform(-2.0, 2.0, SIZE[::-1]).astype(dtype) for _ in range(5)]
    for d in dd.domains():
        for q, which in [(0, "curr"), (1, "curr"), (2, "curr"), (3, "curr"), (0, "next")]:
            host = np.zeros(tuple(reversed(d.raw_size())), dtype=dtype)
            no.box(host, (2, 2, 2), d.size())[...] = no.box(glob[q if which == "curr" else 4], d.origin(), d.size())
            d.quantity_from_host(q, host, which)
    out = []
    for kind, ops in KINDS:
        s = dd.reduce(kind, [hs[o] if isinstance(o, int) else (hs[o[0]], o[1]) for o in ops])
        out.append(tuple(struct.pack("<d", v) for v in (s.min, s.max, s.sum, s.sum2)) + (s.count,))
    dd.close()
    return out


def main():
    local = int(os.environ.get("LOCAL_RANK", 0))
    torch.cuda.set_device(local)
    # before the process group exists: one process, the same two-subdomain partition on this rank's GPU
    single = {dt: run([local, local], dt) for dt in (np.float64, np.float32)}
    td.init_process_group("nccl", device_id=torch.device("cuda", local))
    rank, world = td.get_rank(), td.get_world_size()
    assert world == 2, "run with --nproc-per-node 2"
    for dt in (np.float64, np.float32):
        mine = run([local], dt)
        everyone = [None, None]
        td.all_gather_object(everyone, mine)
        assert everyone[0] == everyone[1], (rank, dt)
        assert mine == single[dt], (rank, dt, mine, single[dt])
    td.barrier()
    if rank == 0:
        print("mp_reduce_check OK: 2 ranks bit-identical to each other and to one process", flush=True)
    td.destroy_process_group()


if __name__ == "__main__":
    main()
