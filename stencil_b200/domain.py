"""Host-side mirror of the reference's domain API for the halo-exchange path, over the C ABI.

Names and argument meaning follow cwpearson/stencil (include/stencil/stencil.hpp:33-225,
local_domain.cuh:34-276, radius.hpp, method.hpp) so that tests read like the reference's own:

    dd = DistributedDomain(512, 512, 512)
    dd.set_radius(Radius.face_edge_corner(1, 0, 0))
    h = dd.add_data(np.float64, "d")
    dd.realize()
    dd.exchange(); dd.swap()

Two deployment modes, one code path:
  * one process driving several GPUs (the reference's 1 rank x N GPUs, src/stencil.cu:74-85):
    peer access is enabled all-pairs and each source GPU runs ONE fused kernel that writes every
    outgoing halo straight into the neighbours' ghost cells;
  * one process per GPU under torch.distributed (torchrun): allocations and completion flags are
    shared through CUDA IPC handles exchanged with all_gather_object; the same fused kernel writes
    through the IPC mappings over NVLink, ordered by device-side ready/done flags (no host barrier
    in the exchange).

All arithmetic on coordinates is delegated to the C ABI (sb_halo_pos, sb_node_partition, ...);
this module only sequences calls.  No CPU fallback exists.
"""
from __future__ import annotations

import ctypes as C
import enum
import os
from typing import Dict, List, Optional, Sequence, Tuple

import numpy as np

from . import _lib
from ._lib import BoxCopy, I27, Pitched, check, i3, lib, o3, stream_ptr, t3

Vec = Tuple[int, int, int]

ALL_DIRS: List[Vec] = [
    (x, y, z) for z in (-1, 0, 1) for y in (-1, 0, 1) for x in (-1, 0, 1) if (x, y, z) != (0, 0, 0)
]


def _neg(d: Vec) -> Vec:
    return (-d[0], -d[1], -d[2])


class Method(enum.IntFlag):
    """include/stencil/method.hpp:5-16.  On one NVSwitch node every message takes the fused
    direct-write path; the flags are kept so reference call sites (set_methods) keep working and
    so exchange_bytes_for_method can attribute bytes the way the reference does."""

    NONE = 0
    CudaMpi = 1
    ColoPackMemcpyUnpack = 2
    ColoQuantityKernel = 4
    ColoRegionKernel = 8
    ColoMemcpy3d = 16
    ColoDomainKernel = 32
    CudaMemcpyPeer = 64
    CudaKernel = 128
    Default = 1 + 2 + 64 + 128


class PlacementStrategy(enum.Enum):
    NodeAware = 0
    Trivial = 1
    IntraNodeRandom = 2


class Radius:
    """include/stencil/radius.hpp -- 27 radii; x(d)/y(d)/z(d) read the face entries."""

    def __init__(self):
        self._r: Dict[Vec, int] = {(x, y, z): 0 for z in (-1, 0, 1) for y in (-1, 0, 1) for x in (-1, 0, 1)}

    @staticmethod
    def constant(r: int) -> "Radius":
        out = Radius()
        for k in out._r:
            out._r[k] = int(r)
        return out

    @staticmethod
    def face_edge_corner(face: int, edge: int, corner: int) -> "Radius":
        out = Radius()
        for d in out._r:
            out._r[d] = (0, face, edge, corner)[sum(1 for c in d if c)]
        return out

    def dir(self, x, y=None, z=None) -> int:
        d = tuple(x) if y is None else (x, y, z)
        return self._r[d]

    def set_dir(self, d: Vec, v: int) -> None:
        self._r[tuple(d)] = int(v)

    def x(self, d: int) -> int:
        return self._r[(d, 0, 0)]

    def y(self, d: int) -> int:
        return self._r[(0, d, 0)]

    def z(self, d: int) -> int:
        return self._r[(0, 0, d)]

    def set_face(self, r: int) -> None:
        for d in self._r:
            if sum(1 for c in d if c) == 1:
                self._r[d] = int(r)

    def set_edge(self, r: int) -> None:
        for d in self._r:
            if sum(1 for c in d if c) == 2:
                self._r[d] = int(r)

    def set_corner(self, r: int) -> None:
        for d in self._r:
            if sum(1 for c in d if c) == 3:
                self._r[d] = int(r)

    def c27(self) -> I27:
        return I27(*[self._r[(x, y, z)] for z in (-1, 0, 1) for y in (-1, 0, 1) for x in (-1, 0, 1)])

    def __eq__(self, o) -> bool:
        return isinstance(o, Radius) and self._r == o._r


class DataHandle:
    """DataHandle<T>, local_domain.cuh:18-26"""

    def __init__(self, idx: int, dtype, name: str = ""):
        self.id = idx
        self.dtype = np.dtype(dtype)
        self.name = name


# ------------------------------------------------------------------------------------------ geometry (C ABI)
def halo_pos(d: Vec, sz: Vec, radius: Radius, halo: bool) -> Vec:
    out = o3()
    check(lib().sb_halo_pos(i3(d), i3(sz), radius.c27(), int(bool(halo)), out))
    return t3(out)


def halo_extent(d: Vec, sz: Vec, radius: Radius) -> Vec:
    out = o3()
    check(lib().sb_halo_extent(i3(d), i3(sz), radius.c27(), out))
    return t3(out)


def raw_size(sz: Vec, radius: Radius) -> Vec:
    out = o3()
    check(lib().sb_raw_size(i3(sz), radius.c27(), out))
    return t3(out)


def prime_factors(n: int) -> List[int]:
    buf = (C.c_int64 * 64)()
    k = check(lib().sb_prime_factors(int(n), buf, 64))
    return [int(buf[i]) for i in range(k)]


class Partition:
    """NodePartition (default) or RankPartition ("trivial") through the C ABI."""

    def __init__(self, size: Vec, radius: Radius, n_nodes: int, gpus_per_node: int, trivial: bool = False):
        dim, base, rem = o3(), o3(), o3()
        if trivial:
            check(lib().sb_rank_partition(i3(size), n_nodes * gpus_per_node, dim, base, rem))
            self.sys_dim, self.node_dim = (1, 1, 1), t3(dim)
        else:
            sysd, noded = o3(), o3()
            check(lib().sb_node_partition(i3(size), radius.c27(), n_nodes, gpus_per_node, sysd, noded, base, rem))
            self.sys_dim, self.node_dim = t3(sysd), t3(noded)
        self.dim = tuple(self.sys_dim[a] * self.node_dim[a] for a in range(3))
        self._base, self._rem = base, rem

    def subdomain_size(self, idx: Vec) -> Vec:
        out = o3()
        check(lib().sb_subdomain_size(self._base, self._rem, i3(idx), out))
        return t3(out)

    def subdomain_origin(self, idx: Vec) -> Vec:
        out = o3()
        check(lib().sb_subdomain_origin(self._base, self._rem, i3(idx), out))
        return t3(out)

    def indices(self) -> List[Vec]:
        d = self.dim
        return [(x, y, z) for z in range(d[2]) for y in range(d[1]) for x in range(d[0])]


def get_neighbor(idx: Vec, d: Vec, dim: Vec) -> Vec:
    """Topology::get_neighbor with periodic boundaries (src/topology.cpp:5-18)."""
    return tuple((idx[a] + d[a]) % dim[a] for a in range(3))


# ------------------------------------------------------------------------------------------ LocalDomain
class LocalDomain:
    """One subdomain on one GPU: curr/next allocation per quantity (local_domain.cuh:34-276,
    src/local_domain.cu).  Rows are unpitched (pitch == raw_x * elem_size) exactly like the
    reference, because astaroth-style kernels index i + j*mx + k*mx*my."""

    def __init__(self, sz: Vec, origin: Vec, dev: int):
        self.sz_ = tuple(int(v) for v in sz)
        self.origin_ = tuple(int(v) for v in origin)
        self.dev_ = int(dev)
        self.radius_ = Radius.constant(0)
        self.elem_sizes_: List[int] = []
        self.dtypes_: List[np.dtype] = []
        self.names_: List[str] = []
        self.curr_: List[int] = []  # device addresses
        self.next_: List[int] = []
        self._owned = False

    # -- configuration
    def set_radius(self, r) -> None:
        self.radius_ = r if isinstance(r, Radius) else Radius.constant(int(r))

    def add_data(self, dtype, name: str = "") -> DataHandle:
        dt = np.dtype(dtype)
        self.dtypes_.append(dt)
        self.elem_sizes_.append(dt.itemsize)
        self.names_.append(name)
        return DataHandle(len(self.dtypes_) - 1, dt, name)

    def lead_bytes(self, es: int) -> int:
        """HBM layout rule (DESIGN.md section 1): when every row has the same 16-byte phase (pitch % 16 == 0) the
        allocation starts `lead` bytes into its cudaMalloc block so that the first COMPUTE cell of every row is 16-byte
        aligned -- 512 FP64 cells are then exactly 256 aligned vectors (8 warp strips) and the halo rows of the y / z
        faces are 128-bit copyable.  The reference starts at the block (src/local_domain.cu:187-203); the layout inside
        the allocation (x fastest, unpitched) is unchanged.  SB_ALLOC_ALIGN=0 restores the reference placement."""
        import os

        if os.environ.get("SB_ALLOC_ALIGN", "1") == "0":
            return 0
        raw = self.raw_size()
        if (raw[0] * es) % 16 != 0:
            return 0
        return (16 - (self.radius_.x(-1) * es) % 16) % 16

    def realize(self) -> None:
        raw = self.raw_size()
        self._base_of = {}  # pointer handed out -> cudaMalloc block (for free and CUDA IPC)
        for es in self.elem_sizes_:
            nbytes = raw[0] * raw[1] * raw[2] * es
            lead = self.lead_bytes(es)
            for store in (self.curr_, self.next_):
                p = C.c_void_p()
                check(lib().sb_malloc(C.byref(p), nbytes + 32, self.dev_))
                check(lib().sb_memset(p, 0, nbytes + 32, self.dev_, None))
                store.append(int(p.value) + lead)
                self._base_of[int(p.value) + lead] = int(p.value)
        check(lib().sb_device_sync(self.dev_))
        self._owned = True

    def free(self) -> None:
        if self._owned:
            for p in self.curr_ + self.next_:
                lib().sb_free(C.c_void_p(self._base_of.get(p, p)), self.dev_)
            self.curr_, self.next_, self._owned = [], [], False

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass

    # -- queries
    def gpu(self) -> int:
        return self.dev_

    def size(self) -> Vec:
        return self.sz_

    def origin(self) -> Vec:
        return self.origin_

    def radius(self) -> Radius:
        return self.radius_

    def num_data(self) -> int:
        return len(self.elem_sizes_)

    def elem_size(self, q: int) -> int:
        return self.elem_sizes_[q]

    def raw_size(self) -> Vec:
        return raw_size(self.sz_, self.radius_)

    def halo_pos(self, d: Vec, halo: bool) -> Vec:
        return halo_pos(d, self.sz_, self.radius_, halo)

    def halo_extent(self, d: Vec) -> Vec:
        return halo_extent(d, self.sz_, self.radius_)

    def halo_bytes(self, d: Vec, q: int) -> int:
        e = self.halo_extent(d)
        return self.elem_sizes_[q] * e[0] * e[1] * e[2]

    def get_compute_region(self) -> Tuple[Vec, Vec]:
        return self.origin_, tuple(self.origin_[a] + self.sz_[a] for a in range(3))

    def accessor_origin(self) -> Vec:
        """Accessor origin: subdomain origin minus the negative-side radius (local_domain.cuh:153-173)."""
        r = self.radius_
        return (self.origin_[0] - r.x(-1), self.origin_[1] - r.y(-1), self.origin_[2] - r.z(-1))

    def pitched(self, q: int, which: str = "curr") -> Pitched:
        raw = self.raw_size()
        ptr = (self.curr_ if which == "curr" else self.next_)[q]
        return Pitched(ptr, raw[0] * self.elem_sizes_[q], raw[1])

    def curr_data(self, q: int) -> Pitched:
        return self.pitched(q, "curr")

    def next_data(self, q: int) -> Pitched:
        return self.pitched(q, "next")

    def swap(self) -> None:
        """LocalDomain::swap, src/local_domain.cu:67-84"""
        self.curr_, self.next_ = self.next_, self.curr_

    # -- host transfers (test / IO helpers; reference region_to_host etc., src/local_domain.cu:131-157)
    def quantity_to_host(self, q: int, which: str = "curr") -> np.ndarray:
        raw = self.raw_size()
        out = np.empty(raw[::-1], dtype=self.dtypes_[q])
        p = (self.curr_ if which == "curr" else self.next_)[q]
        check(lib().sb_memcpy(out.ctypes.data, C.c_void_p(p), out.nbytes, self.dev_, None))
        check(lib().sb_stream_sync(self.dev_, None))
        return out

    def interior_to_host(self, q: int) -> np.ndarray:
        full = self.quantity_to_host(q)
        p = self.halo_pos((0, 0, 0), True)
        e = self.sz_
        return np.ascontiguousarray(full[p[2] : p[2] + e[2], p[1] : p[1] + e[1], p[0] : p[0] + e[0]])

    def quantity_from_host(self, q: int, arr: np.ndarray, which: str = "curr") -> None:
        raw = self.raw_size()
        arr = np.ascontiguousarray(arr, dtype=self.dtypes_[q])
        assert arr.shape == raw[::-1], (arr.shape, raw)
        p = (self.curr_ if which == "curr" else self.next_)[q]
        check(lib().sb_memcpy(C.c_void_p(p), arr.ctypes.data, arr.nbytes, self.dev_, None))
        check(lib().sb_stream_sync(self.dev_, None))


# ------------------------------------------------------------------------------------------ copy plans
class CopyPlan:
    """sb_copy_plan: many box copies, one launch."""

    def __init__(self, device: int, copies: Sequence[BoxCopy]):
        arr = (BoxCopy * max(1, len(copies)))(*copies)
        h = C.c_void_p()
        check(lib().sb_copy_plan_create(C.byref(h), device, arr, len(copies)))
        self._h = h
        self.device = device
        self.bytes = int(lib().sb_copy_plan_bytes(h))
        self.num_tiles = int(lib().sb_copy_plan_num_tiles(h))
        self.num_tma_segments = int(lib().sb_copy_plan_num_tma_segments(h))

    def launch(self, stream=None) -> None:
        check(lib().sb_copy_plan_launch(self._h, stream_ptr(stream)))

    def destroy(self) -> None:
        if self._h:
            lib().sb_copy_plan_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.destroy()
        except Exception:
            pass


def box_copy(dst: Pitched, dst_pos: Vec, src: Pitched, src_pos: Vec, ext: Vec, es: int) -> BoxCopy:
    return BoxCopy(dst, i3(dst_pos), src, i3(src_pos), i3(ext), es)


# ------------------------------------------------------------------------------------------ DistributedDomain
class DistributedDomain:
    """include/stencil/stencil.hpp:33-225 / src/stencil.cu for one NVSwitch node."""

    def __init__(self, x: int, y: int, z: int):
        self.size_ = (int(x), int(y), int(z))
        self.radius_ = Radius.constant(0)
        self.dtypes_: List[np.dtype] = []
        self.names_: List[str] = []
        self.gpus_: Optional[List[int]] = None
        self.flags_ = Method.Default
        self.strategy_ = PlacementStrategy.NodeAware
        self.domains_: List[LocalDomain] = []
        self.domain_idx_: List[Vec] = []
        self.partition_: Optional[Partition] = None
        self._plans: List[List[CopyPlan]] = []  # [parity][local domain]
        self._parity = 0
        self._streams = []
        self._bytes_kernel = 0
        self._bytes_peer = 0
        self._remote = None  # CUDA-IPC mappings of the other ranks (dist.RemoteDomains)
        self._nccl = None  # NCCL fallback (dist.NcclExchange)
        self._use_nccl = False
        self._epoch = 0
        self._reduce_ws = {}  # local subdomain -> reduce.Workspace, allocated by the first reduce()

    # -- configuration (call before realize)
    def set_radius(self, r) -> None:
        self.radius_ = r if isinstance(r, Radius) else Radius.constant(int(r))

    def add_data(self, dtype, name: str = "") -> DataHandle:
        self.dtypes_.append(np.dtype(dtype))
        self.names_.append(name)
        return DataHandle(len(self.dtypes_) - 1, dtype, name)

    def set_methods(self, flags: Method) -> None:
        if (flags & Method.ColoQuantityKernel) and (flags & Method.ColoPackMemcpyUnpack):
            raise _lib.StencilError("can't use Direct Access and Pack-Memcpy-Unpack for colocated ranks")  # stencil.cu:192-197
        self.flags_ = flags

    def set_placement(self, strategy: PlacementStrategy) -> None:
        self.strategy_ = strategy

    def set_gpus(self, cuda_ids: Sequence[int]) -> None:
        self.gpus_ = [int(g) for g in cuda_ids]

    # -- queries
    def size(self) -> Vec:
        return self.size_

    def domains(self) -> List[LocalDomain]:
        return self.domains_

    def get_compute_region(self) -> Tuple[Vec, Vec]:
        return (0, 0, 0), self.size_

    def get_origin(self, i: int) -> Vec:
        return self.domains_[i].origin()

    def get_interior(self) -> List[Tuple[Vec, Vec]]:
        out = []
        for d in self.domains_:
            lo, hi = d.get_compute_region()
            ilo, ihi = o3(), o3()
            check(lib().sb_interior(i3(lo), i3(hi), self.radius_.c27(), ilo, ihi))
            out.append((t3(ilo), t3(ihi)))
        return out

    def get_exterior(self) -> List[List[Tuple[Vec, Vec]]]:
        out = []
        for d in self.domains_:
            lo, hi = d.get_compute_region()
            elo, ehi = (C.c_int64 * 18)(), (C.c_int64 * 18)()
            n = check(lib().sb_exterior(i3(lo), i3(hi), self.radius_.c27(), elo, ehi))
            out.append([(tuple(elo[3 * k : 3 * k + 3]), tuple(ehi[3 * k : 3 * k + 3])) for k in range(n)])
        return out

    def exchange_bytes_for_method(self, method: Method) -> int:
        """src/stencil.cu:139-161: same-GPU messages count as CudaKernel, cross-GPU as CudaMemcpyPeer
        (the transport that carries them here is the fused direct write in both cases)."""
        total = 0
        if method & Method.CudaKernel:
            total += self._bytes_kernel
        if method & Method.CudaMemcpyPeer:
            total += self._bytes_peer
        return total

    # -- realize
    def do_placement(self) -> None:
        from . import dist as _dist

        world = _dist.world()
        if self.gpus_ is None:
            n = C.c_int(0)
            check(lib().sb_device_count(C.byref(n)))
            if world.size > 1:
                self.gpus_ = [world.local_device]
            else:
                self.gpus_ = list(range(n.value))
        n_sub = len(self.gpus_) * world.size
        trivial = self.strategy_ == PlacementStrategy.Trivial
        # one node: NodePartition(size, radius, 1 node, n_sub gpus)  (partition.hpp:157-211)
        self.partition_ = Partition(self.size_, self.radius_, 1, n_sub, trivial=trivial)
        self._world = world
        self._assign_owners()

    def realize(self) -> None:
        from . import dist as _dist

        self.do_placement()
        world = self._world
        part = self.partition_
        all_idx = part.indices()
        my = [idx for idx in all_idx if self._owner[idx][0] == world.rank]
        for slot, idx in enumerate(my):
            d = LocalDomain(part.subdomain_size(idx), part.subdomain_origin(idx), self.gpus_[slot])
            d.set_radius(self.radius_)
            for dt, nm in zip(self.dtypes_, self.names_):
                d.add_data(dt, nm)
            d.realize()
            self.domains_.append(d)
            self.domain_idx_.append(idx)
        # peer access between all local GPUs (src/stencil.cu:123-127)
        for a in set(self.gpus_):
            for b in set(self.gpus_):
                ok = C.c_int(0)
                check(lib().sb_enable_peer(a, b, C.byref(ok)))
                if not ok.value:
                    raise _lib.StencilError(f"GPU {a} cannot map GPU {b}: P2P unavailable (NCCL fallback not selected)")
        self._remote, self._nccl = None, None
        self._alloc_staging()
        if world.size > 1:
            force_nccl = os.environ.get("SB_FORCE_NCCL", "0") == "1"
            if not force_nccl:
                try:
                    self._remote = _dist.share_domains(self, world)
                except _lib.StencilError as e:  # no IPC / peer mapping between these GPUs
                    import warnings

                    warnings.warn(f"CUDA IPC mapping unavailable ({e}); falling back to NCCL send/recv")
                    force_nccl = True
            self._use_nccl = force_nccl
            if force_nccl:
                self._drop_remote_staging()
        else:
            self._use_nccl = False
        self._build_plans()
        if self._use_nccl:
            self._nccl = _dist.NcclExchange(self, world)
        import torch

        self._streams = [torch.cuda.Stream(device=d.gpu(), priority=-1) for d in self.domains_]

    def _pitched_of(self, idx: Vec, q: int, parity: int) -> Tuple[Pitched, int]:
        """(pitched ptr, device) of the CURR buffer of quantity q of subdomain idx when the local swap
        parity is `parity` (every rank swaps in lock step)."""
        rank, slot = self._owner[idx]
        if rank == self._world.rank:
            d = self.domains_[slot]
            which = "curr" if parity == 0 else "next"
            # parity 1 means swap() was called an odd number of times: what is now curr was next at realize
            base = (d._curr0 if which == "curr" else d._next0)[q]
            raw = d.raw_size()
            return Pitched(base, raw[0] * d.elem_size(q), raw[1]), d.gpu()
        return self._remote.pitched(idx, q, parity)

    def _elem_sizes(self) -> List[int]:
        return [dt.itemsize for dt in self.dtypes_]

    def _gpu_key(self, idx: Vec):
        """Identity of the GPU holding subdomain idx (for 'same GPU?' decisions)."""
        rank, slot = self._owner[tuple(idx)]
        if rank == self._world.rank:
            return (rank, self.gpus_[slot])
        return (rank, -1 - slot)

    def _drop_remote_staging(self) -> None:
        """NCCL mode: messages from other ranks arrive packed through NCCL, not through staging buffers."""
        for key in [k for k in self._recv_local if self._owner[k[0]][0] != self._world.rank]:
            lib().sb_free(C.c_void_p(self._recv_local.pop(key)), self.domains_[0].gpu())
            self._recv_entries.pop(key)

    def _alloc_staging(self) -> None:
        """Receive buffers (on MY GPUs) for the thin messages other GPUs send to my subdomains (dist.staging_layout)."""
        from . import dist as _dist

        self._recv_local: Dict[tuple, int] = {}
        self._recv_entries: Dict[tuple, list] = {}
        if os.environ.get("SB_NO_STAGING", "0") == "1":
            return
        for di, dst_idx in enumerate(self.domain_idx_):
            srcs = {get_neighbor(dst_idx, d, self.partition_.dim) for d in ALL_DIRS}
            for src_idx in sorted(srcs):
                if self._gpu_key(src_idx) == self._gpu_key(dst_idx):
                    continue
                total, entries = _dist.staging_layout(self, src_idx, dst_idx)
                if total == 0:
                    continue
                p = C.c_void_p()
                check(lib().sb_malloc(C.byref(p), total, self.domains_[di].gpu()))
                self._recv_local[(tuple(src_idx), tuple(dst_idx))] = int(p.value)
                self._recv_entries[(tuple(src_idx), tuple(dst_idx))] = entries

    def _staging_target(self, src_idx: Vec, dst_idx: Vec):
        """Address of the staging buffer for (src -> dst), wherever dst lives; None if this pair is not staged."""
        key = (tuple(src_idx), tuple(dst_idx))
        if key in self._recv_local:
            return self._recv_local[key]
        if self._remote is not None and key in self._remote.recv:
            return self._remote.recv[key]
        return None

    def plan_messages(self) -> List[dict]:
        """The send plan of this rank (pure geometry, no GPU): one entry per (local subdomain, direction)
        with a non-zero receiving radius -- src/stencil.cu:327-412.  dict(src_slot, src_idx, dst_idx,
        dst_rank, dst_slot, dir, src_pos, dst_pos, ext)."""
        part = self.partition_
        my = [idx for idx in part.indices() if self._owner[idx][0] == self._world.rank]
        out = []
        for slot, idx in enumerate(my):
            sz = part.subdomain_size(idx)
            for dirv in ALL_DIRS:
                if self.radius_.dir(_neg(dirv)) == 0:
                    continue  # src/stencil.cu:344
                dst_idx = get_neighbor(idx, dirv, part.dim)
                dst_sz = part.subdomain_size(dst_idx)
                ext = halo_extent(_neg(dirv), dst_sz, self.radius_)  # stencil.cu:361-363
                if ext[0] * ext[1] * ext[2] == 0:
                    continue
                out.append(
                    dict(
                        src_slot=slot,
                        src_idx=idx,
                        dst_idx=dst_idx,
                        dst_rank=self._owner[dst_idx][0],
                        dst_slot=self._owner[dst_idx][1],
                        dir=dirv,
                        src_pos=halo_pos(dirv, sz, self.radius_, False),
                        dst_pos=halo_pos(_neg(dirv), dst_sz, self.radius_, True),
                        ext=ext,
                    )
                )
        return out

    def _assign_owners(self) -> None:
        # subdomain k of the node (linear order of the partition) lives on (rank, local gpu slot),
        # rank-major: the reference's global id = node*gpusPerNode + id with an identity placement
        # (NVSwitch is uniform, so the QAP of partition.hpp:706-716 is permutation-invariant -- DESIGN.md)
        per_rank = len(self.gpus_)
        self._owner = {idx: (k // per_rank, k % per_rank) for k, idx in enumerate(self.partition_.indices())}

    def _build_plans(self) -> None:
        """Phase 1 (one launch per local subdomain): every outgoing halo region is stored either straight into the
        neighbour's ghost cells (same GPU, or wide rows over NVLink) or, for thin rows bound for another GPU, into
        the neighbour's dense staging buffer.  Phase 2 (one launch per local subdomain that has staged senders):
        scatter the staging buffers into the ghost cells."""
        from . import dist as _dist

        for d in self.domains_:
            d._curr0, d._next0 = list(d.curr_), list(d.next_)
        self._plans, self._unpack_plans = [], []
        self._bytes_kernel = self._bytes_peer = 0
        self._staged_bytes = 0
        msgs = self.plan_messages()
        for parity in (0, 1):
            plans, unplans = [], []
            for di, d in enumerate(self.domains_):
                copies: List[BoxCopy] = []
                for m in msgs:
                    if m["src_slot"] != di:
                        continue
                    remote = m["dst_rank"] != self._world.rank
                    if self._use_nccl and remote:
                        if parity == 0:
                            self._bytes_peer += sum(d.elem_size(q) for q in range(d.num_data())) * m["ext"][0] * m["ext"][1] * m["ext"][2]
                        continue  # carried by the NCCL fallback, not by the fused kernel
                    stage_base = None if self._gpu_key(m["src_idx"]) == self._gpu_key(m["dst_idx"]) else self._staging_target(m["src_idx"], m["dst_idx"])
                    staged = {}
                    if stage_base is not None:
                        _, entries = _dist.staging_layout(self, m["src_idx"], m["dst_idx"])
                        staged = {e["q"]: e for e in entries if e["dir"] == m["dir"]}
                    for q in range(d.num_data()):
                        es = d.elem_size(q)
                        src_p, _ = self._pitched_of(m["src_idx"], q, parity)
                        nbytes = es * m["ext"][0] * m["ext"][1] * m["ext"][2]
                        if q in staged:
                            dense = Pitched(stage_base + staged[q]["offset"], m["ext"][0] * es, m["ext"][1])
                            copies.append(box_copy(dense, (0, 0, 0), src_p, m["src_pos"], m["ext"], es))
                            if parity == 0:
                                self._staged_bytes += nbytes
                        else:
                            dst_p, _ = self._pitched_of(m["dst_idx"], q, parity)
                            copies.append(box_copy(dst_p, m["dst_pos"], src_p, m["src_pos"], m["ext"], es))
                        if parity == 0:
                            if self._gpu_key(m["src_idx"]) == self._gpu_key(m["dst_idx"]):
                                self._bytes_kernel += nbytes
                            else:
                                self._bytes_peer += nbytes
                plans.append(CopyPlan(d.gpu(), copies))
                # phase 2 of this subdomain as a receiver
                ucopies: List[BoxCopy] = []
                for (src_idx, dst_idx), base in self._recv_local.items():
                    if dst_idx != tuple(self.domain_idx_[di]):
                        continue
                    for e in self._recv_entries[(src_idx, dst_idx)]:
                        dst_p, _ = self._pitched_of(dst_idx, e["q"], parity)
                        dense = Pitched(base + e["offset"], e["ext"][0] * e["es"], e["ext"][1])
                        ucopies.append(box_copy(dst_p, e["dst_pos"], dense, (0, 0, 0), e["ext"], e["es"]))
                unplans.append(CopyPlan(d.gpu(), ucopies) if ucopies else None)
            self._plans.append(plans)
            self._unpack_plans.append(unplans)
        # in-process senders of each local receiver (for the phase-1 -> phase-2 stream dependency)
        self._stage_senders: List[List[int]] = []
        for di, dst_idx in enumerate(self.domain_idx_):
            snd = set()
            for (src_idx, d_idx) in self._recv_local:
                if d_idx == tuple(dst_idx) and self._owner[src_idx][0] == self._world.rank:
                    snd.add(self._owner[src_idx][1])
            self._stage_senders.append(sorted(snd))

    # -- the hot path
    def exchange_async(self) -> None:
        """Enqueue the halo exchange on the library's high-priority streams (one per local subdomain)."""
        import torch

        plans, unplans = self._plans[self._parity], self._unpack_plans[self._parity]
        if self._remote is not None:
            self._epoch += 1
            self._remote.begin(self._epoch, self._streams)
        for plan, s in zip(plans, self._streams):
            plan.launch(s)
        if self._remote is not None:
            self._remote.finish(self._epoch, self._streams)  # every remote sender's phase 1 has landed
            if len(self._streams) > 1:
                ev0 = torch.cuda.Event()
                ev0.record(self._streams[0])
                for o in self._streams[1:]:
                    o.wait_event(ev0)
        if self._nccl is not None:
            self._nccl.exchange(self._parity, self._streams[0])
        # phase 2: scatter what other GPUs staged for my subdomains
        if any(u is not None for u in unplans):
            events = {}
            for di, snd in enumerate(self._stage_senders):
                for sj in snd:
                    if sj not in events and sj != di:
                        ev = torch.cuda.Event()
                        ev.record(self._streams[sj])
                        events[sj] = ev
            for di, u in enumerate(unplans):
                if u is None:
                    continue
                for sj in self._stage_senders[di]:
                    if sj != di:
                        self._streams[di].wait_event(events[sj])
                u.launch(self._streams[di])

    def exchange(self) -> None:
        """DistributedDomain::exchange (src/stencil.cu:1002-1186): returns when every ghost cell of
        every local subdomain holds its neighbour's current value."""
        self.exchange_async()
        for d, s in zip(self.domains_, self._streams):
            check(lib().sb_stream_sync(d.gpu(), stream_ptr(s)))

    def exchange_streams(self):
        return self._streams

    def swap(self) -> None:
        """DistributedDomain::swap (src/stencil.cu:852-872).  The exchange plans exist for both
        parities, so -- unlike the reference's captured pack graphs (SURVEY.md 4, latent bug) -- the
        next exchange reads the new curr buffers."""
        for d in self.domains_:
            d.swap()
        self._parity ^= 1

    def reduce(self, kind: int, handles, which: str = "curr", streams=None):
        """Reduction of `kind` (stencil_b200.reduce: VALUE, DIFF, VECTOR, EXP, ALFVEN) over the whole compute region ->
        reduce.Stats.  `handles` are the operands in order, each a DataHandle (read from `which` buffer) or a
        (DataHandle, "curr" | "next") pair; they must share one dtype.  One launch per local subdomain on streams[i] (default:
        each GPU's current torch stream), waited for here.  Collective like exchange(): every rank must call it, and every
        rank gets the same bits -- the per-subdomain results are combined in global subdomain index order, so the result
        also does not depend on how the subdomains are spread over ranks and GPUs."""
        from . import reduce as _r

        ops = [(h, which) if isinstance(h, DataHandle) else (h[0], h[1]) for h in handles]
        if len({np.dtype(self.dtypes_[h.id]) for h, _ in ops}) > 1:
            raise _lib.StencilError("reduction operands must have the same dtype")
        if any(w not in ("curr", "next") for _, w in ops):
            raise ValueError("which must be 'curr' or 'next'")
        if streams is None:
            import torch

            streams = [torch.cuda.current_stream(d.gpu()) for d in self.domains_]
        for di, (d, s) in enumerate(zip(self.domains_, streams)):
            if di not in self._reduce_ws:
                self._reduce_ws[di] = _r.Workspace(d.gpu())
            lo, hi = d.get_compute_region()
            self._reduce_ws[di].launch(kind, [d.pitched(h.id, w) for h, w in ops], d.elem_size(ops[0][0].id), d.accessor_origin(), lo, hi, s)
        local = {}
        for di, (d, s) in enumerate(zip(self.domains_, streams)):
            lo, hi = d.get_compute_region()
            local[tuple(self.domain_idx_[di])] = self._reduce_ws[di].result(s) + (_r.cells(lo, hi),)
        return _r.combine_ranks(local, self.partition_.indices(), self._world.size)

    def close(self) -> None:
        for ws in self._reduce_ws.values():
            ws.free()
        self._reduce_ws = {}
        for plans in self._plans + getattr(self, "_unpack_plans", []):
            for p in plans:
                if p is not None:
                    p.destroy()
        self._plans, self._unpack_plans = [], []

        if self._remote is not None:
            self._remote.close()
            self._remote = None
        if getattr(self, "_nccl", None) is not None:
            self._nccl.close()
            self._nccl = None
        # staging buffers: only after every peer has unmapped them (barrier inside RemoteDomains.close)
        for ptr in getattr(self, "_recv_local", {}).values():
            lib().sb_free(C.c_void_p(ptr), self.domains_[0].gpu() if self.domains_ else 0)
        self._recv_local = {}
        for d in self.domains_:
            d.free()
        self.domains_ = []


# ------------------------------------------------------------------------------------------ jacobi helpers
def _set_current_device(dev: int) -> None:
    """LocalDomain::set_device: kernels launched on a stream need that stream's device to be current."""
    import torch

    if torch.cuda.current_device() != dev:
        torch.cuda.set_device(dev)


def jacobi3d(d: LocalDomain, h: DataHandle, region: Tuple[Vec, Vec], compute_region: Tuple[Vec, Vec], stream=None) -> None:
    """One application of the reference's stencil_kernel (bin/jacobi3d.cu:40-85) to `region` of
    subdomain d: reads curr, writes next."""
    _set_current_device(d.gpu())
    check(
        lib().sb_jacobi3d(
            d.next_data(h.id),
            d.curr_data(h.id),
            d.elem_size(h.id),
            i3(d.accessor_origin()),
            i3(region[0]),
            i3(region[1]),
            i3(compute_region[0]),
            i3(compute_region[1]),
            stream_ptr(stream),
        )
    )


def fill(d: LocalDomain, h: DataHandle, region: Tuple[Vec, Vec], value: float, which: str = "curr", stream=None) -> None:
    """init_kernel (bin/jacobi3d.cu:18-29)."""
    _set_current_device(d.gpu())
    check(
        lib().sb_fill(d.pitched(h.id, which), d.elem_size(h.id), i3(d.accessor_origin()), i3(region[0]), i3(region[1]), float(value), stream_ptr(stream))
    )
