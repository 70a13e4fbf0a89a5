"""The jacobi3d iteration of the reference driver (bin/jacobi3d.cu:296-377) over DistributedDomain.

    interior kernel on a compute stream  ||  dd.exchange() on the library's high-priority streams
    exterior slabs (after the exchange)  ->  stream sync  ->  dd.swap()

All ctypes argument packs are built once per swap parity so the per-iteration host work is a
handful of foreign calls.
"""
from __future__ import annotations

import ctypes as C
import math
from typing import Tuple

import numpy as np

from ._lib import HaloPush, Pitched, check, i3, lib, stream_ptr
from .domain import DataHandle, DistributedDomain, Radius


def jacobi_radius() -> Radius:
    """faces only, radius 1 (bin/jacobi3d.cu:237-246)"""
    return Radius.face_edge_corner(1, 0, 0)


def scaled_size(x: int, y: int, z: int, num_subdoms: int) -> Tuple[int, int, int]:
    """Weak-scaling size rule of bin/jacobi3d.cu:189-199 (one node): multiply the prime factors of the
    subdomain count into the currently smallest dimension."""
    from .domain import prime_factors

    for pf in prime_factors(num_subdoms):
        if x <= y and x <= z:
            x *= pf
        elif y <= z:
            y *= pf
        else:
            z *= pf
    return x, y, z


FACE_DIRS = ((-1, 0, 0), (1, 0, 0), (0, -1, 0), (0, 1, 0), (0, 0, -1), (0, 0, 1))


def fused_x_mode(part, owner, elem_size: int, radius: Radius, mode: str = "") -> str:
    """How the fused schedule moves x faces for a given partition / ownership (pure: every rank computes the same).

    "direct": no x face crosses ranks -- the kernel stores boundary cells into the neighbour's ghost cells (own memory or
              a peer GPU of this process) or reads a periodic self-neighbour in place;
    "dense":  x faces cross ranks and travel as 256-byte lines into dense receive arrays (kernel mode XPUSH): needs whole warp
              strips along x and rows of one 16-byte phase (mode "0" = SB_FUSED_IPC=0 switches it off);
    "queued": fall back to the queued schedule (Jacobi3D.step_async)."""
    from .domain import get_neighbor

    def crosses(dirs):
        return any(owner[tuple(i)][0] != owner[tuple(get_neighbor(i, dv, part.dim))][0] for i in part.indices() for dv in dirs)

    if not crosses(FACE_DIRS[:2]):
        return "direct"
    strip = 32 * (16 // elem_size)
    layout = all(
        part.subdomain_size(i)[0] % strip == 0 and ((part.subdomain_size(i)[0] + radius.x(-1) + radius.x(1)) * elem_size) % 16 == 0
        for i in part.indices()
    )
    return "dense" if (layout and mode != "0") else "queued"


def fused_schedule(dd, elem_size: int, mode: str = "") -> str:
    """Which schedule Jacobi3D.step_fused runs -- "fused" or "queued" -- as a pure function of the GLOBAL partition,
    radius and transport, so that every rank takes the same one (a rank on another schedule would wait on flags the
    others never write)."""
    r = dd.radius_
    if any(r.dir(d6) != 1 for d6 in FACE_DIRS):
        return "queued"  # the fused kernel pushes face radius 1 (bin/jacobi3d.cu:237-246)
    if getattr(dd, "_use_nccl", False):
        return "queued"  # it stores into peer memory: not available on the NCCL fallback
    part = dd.partition_
    if any(part.subdomain_size(i)[0] < 16 for i in part.indices()):
        return "queued"
    return "queued" if fused_x_mode(part, dd._owner, elem_size, r, mode) == "queued" else "fused"


class Jacobi3D:
    def __init__(self, dd: DistributedDomain, h: DataHandle, overlap: bool = True):
        import torch

        self.dd, self.h, self.overlap = dd, h, overlap
        self.creg = dd.get_compute_region()
        self.streams = [torch.cuda.Stream(device=d.gpu()) for d in dd.domains()]
        # the exterior slabs only depend on the exchange, not on the interior kernel: they run on their
        # own stream so that they (and their launch latency) hide behind the interior kernel's tail
        self.ext_streams = [torch.cuda.Stream(device=d.gpu()) for d in dd.domains()]
        interiors, exteriors = dd.get_interior(), dd.get_exterior()
        L = lib()
        self._fn = L.sb_jacobi3d
        self._fn_regions = L.sb_jacobi3d_regions
        # calls[parity][domain] = (interior args, [exterior args...], whole args)
        self._calls = []
        for parity in (0, 1):
            per_dom = []
            for di, d in enumerate(dd.domains()):
                src = d.pitched(h.id, "curr" if parity == 0 else "next")
                dst = d.pitched(h.id, "next" if parity == 0 else "curr")
                if parity == 1:
                    # pitched() reads the CURRENT curr_/next_ lists; parity 1 = after one swap
                    pass
                acc = i3(d.accessor_origin())
                clo, chi = i3(self.creg[0]), i3(self.creg[1])
                s = stream_ptr(self.streams[di])

                def pack(reg):
                    return (dst, src, d.elem_size(h.id), acc, i3(reg[0]), i3(reg[1]), clo, chi, s)

                ne = len(exteriors[di])
                elo = (C.c_int64 * (3 * max(ne, 1)))(*[v for r in exteriors[di] for v in r[0]])
                ehi = (C.c_int64 * (3 * max(ne, 1)))(*[v for r in exteriors[di] for v in r[1]])
                ext_pack = (dst, src, d.elem_size(h.id), acc, ne, elo, ehi, clo, chi, stream_ptr(self.ext_streams[di]))
                per_dom.append((pack(interiors[di]), ext_pack, pack(d.get_compute_region())))
            self._calls.append(per_dom)
        # like the reference driver (d.set_device() before every launch, bin/jacobi3d.cu:310), the CUDA device
        # must be current when launching on one of its streams; only matters with several GPUs per process
        self._devs = [d.gpu() for d in dd.domains()]
        self._multi_dev = len(set(self._devs)) > 1
        self._set_device = torch.cuda.set_device
        import os

        dbg = os.environ.get("SB_DEBUG_SKIP", "")
        self._debug_skip = {"both": ("ext", "xchg")}.get(dbg, (dbg,) if dbg else ())
        self._ghosts_current = False  # step_fused: do the ghost cells of curr hold the neighbours' current values?
        self._ev_ext = None  # step_async: exterior-done events of the previous iteration (one per subdomain)
        self._ev_int = None
        self.interior_cells = sum(int(np.prod([hi[a] - lo[a] for a in range(3)])) for lo, hi in interiors)
        self._parity0 = dd._parity

    def _args(self):
        return self._calls[(self.dd._parity - self._parity0) & 1]

    def launch_interior(self) -> None:
        for dev, a in zip(self._devs, self._args()):
            if self._multi_dev:
                self._set_device(dev)
            check(self._fn(*a[0]))

    def launch_exterior(self) -> None:
        """All exterior slabs of a subdomain in ONE launch (the reference issues up to six)."""
        for dev, a in zip(self._devs, self._args()):
            if self._multi_dev:
                self._set_device(dev)
            check(self._fn_regions(*a[1]))

    def launch_whole(self) -> None:
        for dev, a in zip(self._devs, self._args()):
            if self._multi_dev:
                self._set_device(dev)
            check(self._fn(*a[2]))

    def step(self) -> None:
        """One iteration, exactly the loop body of bin/jacobi3d.cu:296-368."""
        dd = self.dd
        self._ghosts_current = False
        if self._ev_ext is not None or getattr(self, "_ev_fused", None) is not None:
            self.synchronize()  # drain iterations queued by step_async / step_fused
            self._ev_fused = None
        if self.overlap:
            self.launch_interior()
            dd.exchange()
            self.launch_exterior()
        else:
            dd.exchange()
            self.launch_whole()
        self.synchronize()
        self._ev_ext = self._ev_int = None
        dd.swap()

    def step_async(self, timing=None) -> None:
        """The same iteration with every dependency expressed as a CUDA event instead of a host-side stream
        synchronisation, so consecutive iterations queue back to back on the device (the reference blocks the host
        in exchange() and after the exterior kernels, bin/jacobi3d.cu:337-365).  Per subdomain, iteration i
        (curr = A, next = B):

            interior i   reads A, writes B interior      after exterior i-1 (wrote A's boundary, read B near it)
            exchange i   reads A boundary, writes ghosts  after exterior i-1 of every sending subdomain
            exterior i   reads A + ghosts, writes B rim   after exchange i, and after interior i-1 (read B's rim)

        Remote ranks are ordered by the device-side ready/done flags of the exchange itself (dist.RemoteDomains):
        `ready` is signalled on the exchange stream, i.e. after this rank's exterior i-1.  Results are bitwise
        those of step().  `timing` = (event, event) recorded around subdomain 0's interior kernel."""
        import torch

        if not self.overlap:
            raise RuntimeError("step_async needs the overlapped (interior/exterior) schedule")
        dd = self.dd
        self._ghosts_current = False
        if getattr(self, "_ev_fused", None) is not None:
            self.synchronize()
            self._ev_fused = None
        skip = self._debug_skip  # timing diagnostics only (SB_DEBUG_SKIP=ext|xchg|both): results are wrong when set
        nd = len(self._devs)
        prev_ext, prev_int = self._ev_ext, self._ev_int
        xs = dd.exchange_streams()
        ev_int = []
        for di, (dev, a) in enumerate(zip(self._devs, self._args())):
            if self._multi_dev:
                self._set_device(dev)
            s = self.streams[di]
            if prev_ext is not None:
                s.wait_event(prev_ext[di])
            if timing is not None and di == 0:
                timing[0].record(s)
            check(self._fn(*a[0]))
            if timing is not None and di == 0:
                timing[1].record(s)
            e = torch.cuda.Event()
            e.record(s)
            ev_int.append(e)
        if prev_ext is not None:
            for x in xs:
                for e in prev_ext:
                    x.wait_event(e)
        if "xchg" not in skip:
            dd.exchange_async()
        ev_x = []
        for di, x in enumerate(xs):
            if self._multi_dev:
                self._set_device(self._devs[di])
            e = torch.cuda.Event()
            e.record(x)
            ev_x.append(e)
        ev_ext = []
        for di, (dev, a) in enumerate(zip(self._devs, self._args())):
            if self._multi_dev:
                self._set_device(dev)
            s = self.ext_streams[di]
            for e in ev_x:
                s.wait_event(e)
            if prev_int is not None:
                s.wait_event(prev_int[di])
            if "ext" not in skip:
                check(self._fn_regions(*a[1]))
            e = torch.cuda.Event()
            e.record(s)
            ev_ext.append(e)
        self._ev_ext, self._ev_int = ev_ext, ev_int
        dd.swap()

    # ------------------------------------------------------------------ fused schedule
    def _build_fused(self) -> bool:
        """Argument packs of sb_jacobi3d_fused_sync per swap parity: the whole compute region + the six face neighbours'
        output allocations (own memory, a peer GPU of this process, or another rank's IPC mapping), the dense x arrays and
        the mailboxes of the in-kernel handshake.  Returns False (on every rank alike) if the fused schedule does not
        apply after all."""
        import os

        from . import dist as _dist
        from ._lib import FUSED_MAX_GROUPS, StepSync
        from .domain import CopyPlan, box_copy, get_neighbor

        dd, h = self.dd, self.h
        r = dd.radius_
        dirs = FACE_DIRS
        part = dd.partition_
        es = dd.domains()[0].elem_size(h.id)
        L = lib()
        me = dd._world.rank
        multi_rank = dd._remote is not None

        def gather(obj):
            return _dist.all_gather_object(obj) if multi_rank else [obj]

        # An x face is one cell per row: 8 bytes every 4112.  Stored cell by cell into another GPU it is one tiny NVLink
        # transaction per row (78 us per iteration through CUDA-IPC mappings, profiles/README.md section 6.1), so towards
        # any OTHER subdomain the column travels as a dense [y][z] array (z fastest, like the march): the shipping CTA
        # writes 256-byte lines into the neighbour's receive array (double buffered by swap parity) and the neighbour's
        # edge lanes read their x ghosts from it.  Needs whole warp strips along x and a 16-byte aligned first compute
        # cell; otherwise the column goes into the ghost column (inside a process) or the schedule is "queued" (across
        # ranks, decided by fused_schedule).  One decision for the whole job: every rank evaluates the same inputs.
        strip = 32 * (16 // es)
        layout = all(part.subdomain_size(i)[0] % strip == 0 and ((part.subdomain_size(i)[0] + r.x(-1) + r.x(1)) * es) % 16 == 0 for i in part.indices())
        aligned = all((d.pitched(h.id, w).ptr + r.x(-1) * es) % 16 == 0 for d in dd.domains() for w in ("curr", "next"))
        dense = layout and all(gather(bool(aligned)))
        x_crosses_ranks = fused_x_mode(part, dd._owner, es, r, os.environ.get("SB_FUSED_IPC", "")) != "direct"
        if x_crosses_ranks and not dense:
            return False

        self._xbuf, self._xopened = [], []

        def dev_alloc(nbytes, gpu):
            pbuf = C.c_void_p()
            check(L.sb_malloc(C.byref(pbuf), nbytes, gpu))
            check(L.sb_memset(pbuf, 0, nbytes, gpu, None))
            self._xbuf.append((int(pbuf.value), gpu))
            return int(pbuf.value)

        def export(ptr):
            hb = (C.c_char * 64)()
            check(L.sb_ipc_export(C.c_void_p(ptr), hb))
            return bytes(hb)

        def nbr_of(di, k):
            idx = tuple(dd.domain_idx_[di])
            nidx = tuple(get_neighbor(idx, dirs[k], part.dim))
            return idx, nidx, dd._owner[nidx]

        # receive arrays: one per local subdomain, x side and swap parity, where the x neighbour is another subdomain
        recv = {}
        if dense:
            for di, d in enumerate(dd.domains()):
                raw = d.raw_size()
                for side in (0, 1):
                    idx, nidx, _ = nbr_of(di, side)
                    if nidx != idx:
                        recv[(idx, side)] = [dev_alloc(raw[1] * raw[2] * es, d.gpu()) for _ in range(2)]
        # mailboxes of the in-kernel handshake: one subdomain per rank (the torchrun layout) with neighbours on other ranks
        inkernel = multi_rank and len(dd.domains()) == 1 and os.environ.get("SB_FUSED_INKERNEL", "1") != "0"
        mailbox = dev_alloc(6 * FUSED_MAX_GROUPS * 4, dd.domains()[0].gpu()) if inkernel else 0
        for _, gpu in self._xbuf:
            check(L.sb_device_sync(gpu))
        remote_recv, remote_mail = {}, {}
        if multi_rank:
            mine = {"recv": {key: [export(p_) for p_ in ptrs] for key, ptrs in recv.items()}, "mail": export(mailbox) if mailbox else None}
            wanted = set()  # the receive arrays my subdomains write into: side 1 - s of my neighbour on side s
            for di in range(len(dd.domains())):
                for s_ in (0, 1):
                    idx, nidx, (nrank, _) = nbr_of(di, s_)
                    if nrank != me:
                        wanted.add((nidx, 1 - s_))
            nbr_ranks = {nbr_of(di, k)[2][0] for di in range(len(dd.domains())) for k in range(6)} - {me}
            gpu0 = dd.domains()[0].gpu()

            def open_(hnd):
                out = C.c_void_p()
                check(L.sb_ipc_import(hnd, gpu0, C.byref(out)))
                self._xopened.append(int(out.value))
                return int(out.value)

            for rank, table in enumerate(gather(mine)):
                if rank == me:
                    continue
                for key, handles in table["recv"].items():
                    key = (tuple(key[0]), key[1])
                    if key in wanted:
                        remote_recv[key] = [open_(hnd) for hnd in handles]
                if inkernel and rank in nbr_ranks and table["mail"] is not None:
                    remote_mail[rank] = open_(table["mail"])

        self._fused_calls, self._init_plans = [], []
        self._fused_nbr_slots = []  # in-process neighbours of each local subdomain (stream dependencies)
        for rel in (0, 1):
            absolute = (self._parity0 + rel) & 1
            per_dom, inits = [], []
            for di, d in enumerate(dd.domains()):
                src = d.pitched(h.id, "curr" if rel == 0 else "next")
                dst = d.pitched(h.id, "next" if rel == 0 else "curr")
                push = HaloPush()
                slots = set()
                init_copies = []
                myraw = d.raw_size()
                for k in range(6):
                    idx, nidx, (rank, slot) = nbr_of(di, k)
                    # the neighbour's NEXT buffer at this parity is its curr buffer of the other parity
                    pn, _ = dd._pitched_of(nidx, h.id, absolute ^ 1)
                    if rank == me:
                        raw = dd.domains_[slot].raw_size()
                        slots.add(slot)
                    else:
                        raw = dd._remote.raw_of(nidx)
                    push.nbr[k] = Pitched(pn.ptr, pn.pitch, pn.ysize)
                    push.nbr_zsize[k] = raw[2]
                    if k < 2 and (idx, k) in recv:
                        target = recv[(nidx, 1 - k)] if rank == me else remote_recv[(nidx, 1 - k)]
                        # iteration `rel` writes what the neighbour reads in the next one (parity rel ^ 1)
                        push.nbr[k] = Pitched(target[rel ^ 1], es, myraw[1])
                        push.nbr_zsize[k] = myraw[2]
                        push.x_dense[k] = 1
                        push.x_recv[k] = recv[(idx, k)][rel]
                        # before the first fused iteration at this parity: the neighbour needs my column of curr itself
                        lo3 = (r.x(-1), r.y(-1), r.z(-1))
                        sz3 = d.size()
                        xcol = lo3[0] if k == 0 else lo3[0] + sz3[0] - 1
                        for zz in range(lo3[2], lo3[2] + sz3[2]):
                            col = Pitched(target[rel] + zz * es, myraw[2] * es, myraw[1])  # element (0, y, 0) -> [y][zz]
                            init_copies.append(box_copy(col, (0, lo3[1], 0), src, (xcol, lo3[1], zz), (1, sz3[1], 1), es))
                    if os.environ.get("SB_DEBUG_NOPUSH"):  # timing diagnostics only: results are wrong
                        push.nbr[k] = Pitched(None, 0, 0)
                creg = d.get_compute_region()
                clo, chi = i3(self.creg[0]), i3(self.creg[1])
                pack = (dst, src, d.elem_size(h.id), i3(d.accessor_origin()), i3(creg[0]), i3(creg[1]), clo, chi, push, stream_ptr(self.streams[di]))
                per_dom.append(pack)
                inits.append(CopyPlan(d.gpu(), init_copies) if init_copies else None)
                if rel == 0:
                    self._fused_nbr_slots.append(sorted(slots))
            self._fused_calls.append(per_dom)
            self._init_plans.append(inits)
        self._fn_fused = L.sb_jacobi3d_fused_sync
        self._fused_epoch = 0
        self._ev_fused = None
        self._ghosts_current = False
        # Ordering between ranks.  One subdomain per rank: inside the kernel -- its first CTA publishes the iteration number
        # in every neighbour's mailbox, boundary CTAs poll the word of the neighbour across their face
        # (sb_jacobi3d_fused_sync); no extra launch.  Several subdomains per rank: one counter per rank, signalled by a tiny
        # kernel after all of them (dist.RemoteDomains.signal_step / wait_step).
        self._sync = None
        if inkernel and remote_mail:
            sy = StepSync()
            row = FUSED_MAX_GROUPS * 4
            for k in range(6):
                _, _, (rank, _) = nbr_of(0, k)
                if rank != me:
                    sy.wait_rows[k] = mailbox + k * row  # written by the neighbour across face k ...
                    sy.signal_rows[k] = remote_mail[rank] + (k ^ 1) * row  # ... which sees me across its face k ^ 1
            self._sync = sy
        return True

    def step_fused(self, timing=None) -> None:
        """One iteration as ONE kernel per subdomain: the jacobi update of the whole compute region, with every boundary
        cell also stored into the ghost cell of the face neighbour that reads it next iteration (sb_jacobi3d_fused).
        The halo exchange of bin/jacobi3d.cu:337 is thereby part of the previous iteration's kernel; what remains
        between iterations is ordering -- CUDA events between the subdomains of this process, one device-side
        counter per neighbour rank (dist.RemoteDomains.signal_step / wait_step).  Bitwise the results of step().
        The first fused iteration after construction (or after step / step_async) runs a regular exchange()."""
        import ctypes as C

        import torch

        if not hasattr(self, "_fused_calls"):
            import os

            es = self.dd.domains()[0].elem_size(self.h.id)
            self._fused_calls = []
            # a pure function of the global partition; _build_fused adds one all-gathered layout check (the same everywhere)
            self.fused_supported = fused_schedule(self.dd, es, os.environ.get("SB_FUSED_IPC", "")) == "fused" and self._build_fused()
        if not self.fused_supported:  # the queued schedule computes the same iteration
            return self.step_async(timing=timing)
        dd = self.dd
        if self._ev_ext is not None:
            self.synchronize()
            self._ev_ext = self._ev_int = None
        if not self._ghosts_current:
            self.synchronize()
            dd.exchange()  # ghost cells of curr, once; afterwards every iteration leaves them filled for the next
            rel0 = (dd._parity - self._parity0) & 1
            for di, plan in enumerate(self._init_plans[rel0]):  # dense x columns for neighbour ranks (SB_FUSED_IPC=1)
                if plan is not None:
                    plan.launch(self.streams[di])
            self.synchronize()
            if dd._remote is not None:
                import torch.distributed as td

                td.barrier()  # every rank's exchange has landed before anybody's first fused kernel
            self._ghosts_current = True
            self._ev_fused = None
        calls = self._fused_calls[(dd._parity - self._parity0) & 1]
        prev = self._ev_fused
        remote = dd._remote
        events = []
        for di, (dev, a) in enumerate(zip(self._devs, calls)):
            if self._multi_dev:
                self._set_device(dev)
            s = self.streams[di]
            if prev is not None:
                for sj in self._fused_nbr_slots[di]:
                    if sj != di:
                        s.wait_event(prev[sj])
            sync = self._sync
            if sync is not None:
                # the kernel of iteration e (of this object: its mailboxes start at zero) publishes e when it starts -- "my
                # iterations before e are complete" -- and its boundary tiles wait for e from the neighbour across their face
                sync.wait_value = sync.signal_value = self._fused_epoch & 0xFFFFFFFF
            elif remote is not None:
                remote.wait_step(remote.step_epoch, s)
            if timing is not None and di == 0:
                timing[0].record(s)
            check(self._fn_fused(a[0], a[1], a[2], a[3], a[4], a[5], a[6], a[7], C.byref(a[8]), C.byref(sync) if sync is not None else None, a[9]))
            if timing is not None and di == 0:
                timing[1].record(s)
            e = torch.cuda.Event()
            e.record(s)
            events.append(e)
        self._fused_epoch += 1
        if remote is not None:
            remote.step_epoch += 1
            if self._sync is None:
                # one counter per rank: signal after ALL local subdomains of this iteration are done
                s0 = self.streams[0]
                for e in events[1:]:
                    s0.wait_event(e)
                remote.signal_step(remote.step_epoch, s0)
        self._ev_fused = events
        dd.swap()

    def capture_fused(self, iterations: int = 2):
        """Capture `iterations` (even: both swap parities) fused iterations into ONE CUDA graph and return it; `graph.replay()`
        then advances the solution by that many iterations with a single launch from the host (SURVEY.md section 8 f3; the
        reference captures its pack kernels the same way, src/packer.cu:96-106).  Single-process runs only: across ranks the
        iteration number travels in the kernel arguments.  The Python-side swap state is unchanged by a replay (the parity
        returns to where it was), so step_fused() / step() may be mixed with replays freely."""
        import torch

        if iterations < 2 or iterations % 2:
            raise ValueError("capture an even number of iterations (both swap parities)")
        if self.dd._remote is not None:
            raise RuntimeError("capture_fused: single-process runs only (the cross-rank handshake passes the iteration number by value)")
        self.step_fused()  # builds the argument packs, fills the ghost cells, allocates the group counters (no allocation may happen during capture)
        self.step_fused()
        if not self.fused_supported:
            raise RuntimeError("capture_fused: the fused schedule does not apply to this domain")
        self.synchronize()
        graph = torch.cuda.CUDAGraph()
        s0 = self.streams[0]
        with torch.cuda.graph(graph, stream=s0):
            # the other subdomains' streams join the capture through the event dependencies step_fused records
            for o in self.streams[1:]:
                o.wait_stream(s0)
            self._ev_fused = None
            for _ in range(iterations):
                self.step_fused()
            for o in self.streams[1:]:
                s0.wait_stream(o)
        self._ev_fused = None  # events recorded during capture are not waitable outside it; replays are ordered by s0

        class _FusedGraph:
            """replay() launches the captured iterations on the solver's own stream (ordered with step_fused / synchronize)."""

            def __init__(self, g, stream, iters):
                self.graph, self.stream, self.iterations = g, stream, iters

            def replay(self):
                with torch.cuda.stream(self.stream):
                    self.graph.replay()

        return _FusedGraph(graph, s0, iterations)

    def close(self) -> None:
        """Drain the queued work; release the dense x receive arrays and mailboxes of the fused schedule."""
        self.synchronize()
        self._sync = None
        if not getattr(self, "_xbuf", None) and not getattr(self, "_xopened", None):
            return
        multi_rank = self.dd._remote is not None
        if multi_rank:
            import torch.distributed as td
        for plans in getattr(self, "_init_plans", []):
            for p in plans:
                if p is not None:
                    p.destroy()
        self._init_plans = []
        if multi_rank:
            td.barrier()  # nobody unmaps or frees while a neighbour could still write
        for ptr in self._xopened:
            lib().sb_ipc_close(C.c_void_p(ptr), self.dd.domains()[0].gpu())
        if multi_rank:
            td.barrier()
        for ptr, dev in self._xbuf:
            lib().sb_free(C.c_void_p(ptr), dev)
        self._xbuf, self._xopened = [], []
        if hasattr(self, "_fused_calls"):
            del self._fused_calls  # a later step_fused() builds everything again

    def synchronize(self) -> None:
        """Wait for the compute streams (bin/jacobi3d.cu:363-365)."""
        for s in self.streams:
            s.synchronize()
        if self.overlap:
            for s in self.ext_streams:
                s.synchronize()

    def residual(self) -> float:
        """||curr - next||_2 over the whole distributed compute region: after a step, the change of the last iteration
        (u_{n+1} - u_n), accumulated in FP64.  Waits for the queued iterations; collective across ranks."""
        from . import reduce as _r

        self.synchronize()
        h = self.h
        return math.sqrt(self.dd.reduce(_r.DIFF, [(h, "curr"), (h, "next")], streams=self.streams).sum2)

    def init(self, value: float = 0.5) -> None:
        """init_kernel (bin/jacobi3d.cu:18-29) on curr; ghost cells are filled by the first exchange."""
        from .domain import fill

        for d in self.dd.domains():
            fill(d, self.h, d.get_compute_region(), value)
            check(lib().sb_device_sync(d.gpu()))
