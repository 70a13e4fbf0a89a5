"""The astaroth MHD iteration of the reference's second driver (astaroth/astaroth.cu:551-640) over DistributedDomain.

    for substep in 0..2:   interior solve<substep> || dd.exchange()  ->  exterior solve<substep>  ->  stream sync
    dd.swap()

Eight fields (lnrho, uux, uuy, uuz, ax, ay, az, entropy; astaroth/astaroth.cu:427-434), radius 3 everywhere, FP64 in the
reference (AcReal = double) and FP32 as well here.  The kernel is `sb_astaroth_substep` (stencil_b200/csrc/astaroth.cu).
"""
from __future__ import annotations

import ctypes as C
from typing import Optional, Sequence

import numpy as np

from ._lib import AstarothParams, check, i3, lib, stream_ptr
from .domain import DataHandle, DistributedDomain

FIELDS = ("lnrho", "uux", "uuy", "uuz", "ax", "ay", "az", "entropy")
NGHOST = 3  # STENCIL_ORDER / 2, astaroth/astaroth.h:8-9
AUTO, CELL, TILE, TEAM, TEAM_TMA, TEAM3_TMA = 0, 1, 2, 3, 4, 5


def conf_params(dt: float = 1e-8) -> AstarothParams:
    """What the reference driver's device constants end up holding: astaroth/astaroth.conf:10-67 for the keys the file
    sets, the *_DEFAULT_VALUE statics (astaroth/user_kernels.h:30-35, 329, 367) for the ones it leaves out (the loader
    NaN-fills the config and acDeviceLoadScalarUniform skips invalid values, astaroth/astaroth_utils.cu:100-106,
    astaroth/kernels.cu:96-100), dt = 1e-8 from astaroth/astaroth.cu:578."""
    ds = 0.04908738521
    return AstarothParams(1.0 / ds, 1.0 / ds, 1.0 / ds, dt, 1.0, 0.5, 1.0, 1.3, 1.2, 1.4, 5e-3, 0.01, 5e-3)


def substep(step: int, fin: Sequence[int], fout: Sequence[int], dtype_size: int, raw, lo, hi, params: AstarothParams, variant: int = AUTO,
            stream=None) -> None:  # fmt: skip
    """integrate_substep (astaroth/kernels.cu:62-87) on raw device pointers; [lo, hi) in memory-offset coordinates."""
    pin = (C.c_void_p * 8)(*fin)
    pout = (C.c_void_p * 8)(*fout)
    check(lib().sb_astaroth_substep(step, pin, pout, dtype_size, i3(raw), i3(lo), i3(hi), C.byref(params), variant, stream_ptr(stream)))


class Astaroth:
    """Drives the 8-field RK3 iteration on a realized DistributedDomain whose first 8 quantities are FIELDS."""

    def __init__(self, dd: DistributedDomain, handles: Sequence[DataHandle], params: Optional[AstarothParams] = None,
                 overlap: Optional[bool] = None, variant: int = AUTO):  # fmt: skip
        """overlap=None picks the faster schedule measured on B200 (profiles/README.md section 5): the tile kernel fills
        every SM's shared memory, so a concurrent exchange only waits for it -- exchange first, then one launch over the
        whole region (FP64 7.07 vs 7.34 ms, FP32 3.64 vs 3.85 ms per iteration at 256^3); overlap=True is the
        interior || exchange -> exterior split of the reference driver."""
        import torch

        if overlap is None:
            overlap = False

        if len(handles) != 8:
            raise ValueError("astaroth needs the 8 fields " + ", ".join(FIELDS))
        self.dd, self.handles, self.overlap, self.variant = dd, list(handles), overlap, variant
        self.params = params if params is not None else conf_params()
        self.streams = [torch.cuda.Stream(device=d.gpu()) for d in dd.domains()]
        self.ext_streams = [torch.cuda.Stream(device=d.gpu()) for d in dd.domains()]
        self._devs = [d.gpu() for d in dd.domains()]
        self._multi_dev = len(set(self._devs)) > 1
        self._set_device = torch.cuda.set_device
        self._fn = lib().sb_astaroth_substep
        interiors, exteriors = dd.get_interior(), dd.get_exterior()
        # argument packs per swap parity and subdomain: regions move from global to memory-offset coordinates
        # (cr.lo += acOff - origin, astaroth/astaroth.cu:563-566)
        self._calls = []
        for parity in (0, 1):
            per_dom = []
            for di, d in enumerate(dd.domains()):
                es = d.elem_size(handles[0].id)
                cur = [d.pitched(h.id, "curr" if parity == 0 else "next").ptr for h in handles]
                nxt = [d.pitched(h.id, "next" if parity == 0 else "curr").ptr for h in handles]
                pin, pout = (C.c_void_p * 8)(*cur), (C.c_void_p * 8)(*nxt)
                raw = i3(d.raw_size())
                org = d.origin()

                def box(reg):
                    lo = [reg[0][a] - org[a] + NGHOST for a in range(3)]
                    hi = [reg[1][a] - org[a] + NGHOST for a in range(3)]
                    return i3(lo), i3(hi)

                s, se = stream_ptr(self.streams[di]), stream_ptr(self.ext_streams[di])
                pp = C.byref(self.params)
                interior = (pin, pout, es, raw, *box(interiors[di]), pp, variant, s)
                exterior = [(pin, pout, es, raw, *box(r), pp, variant, se) for r in exteriors[di]]
                whole = (pin, pout, es, raw, *box(d.get_compute_region()), pp, variant, s)
                per_dom.append((interior, exterior, whole))
            self._calls.append(per_dom)
        self._parity0 = dd._parity
        self.cells = sum(int(np.prod(d.size())) for d in dd.domains())

    def _args(self):
        return self._calls[(self.dd._parity - self._parity0) & 1]

    def _launch(self, step: int, which: int) -> None:
        for dev, a in zip(self._devs, self._args()):
            if self._multi_dev:
                self._set_device(dev)
            packs = a[which] if which == 1 else [a[which]]
            for p in packs:
                check(self._fn(step, p[0], p[1], p[2], p[3], p[4], p[5], p[6], p[7], p[8]))

    def synchronize(self) -> None:
        for s in self.streams + self.ext_streams:
            s.synchronize()

    def diagnostics(self) -> dict:
        """What an astaroth run reports between iterations: {"uu": Stats of the length of (uux, uuy, uuz), and for each of
        FIELDS: Stats of its values} over the whole distributed compute region (stencil_b200.reduce: min, max, sum, rms).
        Waits for the solver's queued work first; collective across ranks like DistributedDomain.reduce."""
        from . import reduce as _r

        self.synchronize()
        out = {"uu": self.dd.reduce(_r.VECTOR, self.handles[1:4], streams=self.streams)}
        for name, h in zip(FIELDS, self.handles):
            out[name] = self.dd.reduce(_r.VALUE, [h], streams=self.streams)
        return out

    def step(self) -> None:
        """One iteration = three substeps + swap, exactly the loop body of astaroth/astaroth.cu:551-640 (the exchange
        of every substep re-sends the same `curr`: the reference never swaps between substeps)."""
        dd = self.dd
        for sub in range(3):
            if self.overlap:
                self._launch(sub, 0)
                dd.exchange()
                self._launch(sub, 1)
            else:
                dd.exchange()
                self._launch(sub, 2)
            self.synchronize()
        dd.swap()
