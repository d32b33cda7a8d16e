"""Device-resident driver: physics_state chunks kept in HBM as torch tensors (torch is plumbing:
allocation, streams, torch.distributed), the C ABI's *_dev entry points do the work."""
from __future__ import annotations

import ctypes as C
import torch

from . import zm_conv as Z


def _ptr(t: torch.Tensor):
    return C.c_void_p(t.data_ptr())


class DeviceTend:
    """Holds one rank's chunk set on the GPU and runs zm_conv_tend on it."""

    def __init__(self, ch, device="cuda", ncnst=0, hist=None):
        """ncnst > 0 adds the constituent arrays of BASELINE config 4 (convtran over the tracer set as zm_conv_intr
        runs it from tphysbc): constituents 2,3 (cloud liquid / ice) are transported by convtran1 inside zm_conv_tend
        (zm_conv_intr.F90:865-880), 4..ncnst by convtran2 in zm_conv_tend_2 (:955-1028), every third of those 'dry'.
        hist = True or an iterable of zm_conv.HIST_FIELDS names: every step also writes those history fields into the
        device tensors self.hist[name] (zm_conv_tend_hist_fields)."""
        p = Z._params
        if p is None:
            raise Z.ZmError("zm_init has not been called")
        self.nch, self.pc, self.L = ch.nchunks, p.pcols, p.pver
        self.ztodt = float(ch.ztodt)
        self.device = torch.device(device)
        host = dict(t=ch.t, q=ch.q, u=ch.u, v=ch.v, pmid=ch.pmid, pint=ch.pint, pdel=ch.pdel, zm=ch.zm,
                    zi=ch.zi, phis=ch.phis, pblh=ch.pblh, tpert=ch.tpert, landfrac=ch.landfrac, cld=ch.cld)
        self.host_in = {k: torch.from_numpy(v).pin_memory() for k, v in host.items()}
        self.host_ncol = torch.from_numpy(ch.ncol.astype("int32")).pin_memory()
        self.ncol = self.host_ncol.to(self.device)
        self.inp = {k: v.to(self.device) for k, v in self.host_in.items()}
        nch, pc, L = self.nch, self.pc, self.L
        f64 = dict(dtype=torch.float64, device=self.device)
        i32 = dict(dtype=torch.int32, device=self.device)
        self.out = {}
        for k in Z.TEND_OUT_2D:
            self.out[k] = torch.zeros((nch, L, pc), **f64)
        for k in Z.TEND_OUT_2DP:
            self.out[k] = torch.zeros((nch, L + 1, pc), **f64)
        for k in Z.TEND_OUT_1D:
            self.out[k] = torch.zeros((nch, pc), **f64)
        for k in Z.TEND_OUT_INT:
            self.out[k] = torch.zeros((nch, pc), **i32)
        self.out["lengath"] = torch.zeros(nch, **i32)
        self.hist = {k: torch.zeros(Z.hist_shape(k, nch, L, pc), **f64) for k in Z.hist_names(hist)}
        self.in_bytes = sum(v.numel() * v.element_size() for v in self.host_in.values()) + self.host_ncol.numel() * 4
        self.ncnst = int(ncnst)
        if self.ncnst:
            import numpy as np
            from . import soundings as S
            if self.ncnst < 4:
                raise Z.ZmError("ncnst must be >= 4 (water vapour, cloud liquid, cloud ice, one tracer)")
            q3, fracis, pdeldry = S.make_tracers(ch, self.ncnst)
            self.tr = {k: torch.from_numpy(v).to(self.device) for k, v in dict(q=q3, fracis=fracis, pdeldry=pdeldry).items()}
            self.ptend_qc = torch.zeros_like(self.tr["q"])
            self.do1 = np.zeros(self.ncnst, np.int32); self.do1[1:3] = 1            # cnst_is_convtran1
            self.do2 = np.zeros(self.ncnst, np.int32); self.do2[3:] = 1             # cnst_is_convtran2
            self.dry = np.zeros(self.ncnst, np.int32); self.dry[3::3] = 1           # cnst_get_type_byind == 'dry'

    def upload(self, stream=None):
        """H2D of the step's inputs from pinned host memory (part of the e2e timed region)."""
        for k, v in self.host_in.items():
            self.inp[k].copy_(v, non_blocking=True)
        self.ncol.copy_(self.host_ncol, non_blocking=True)

    def step(self):
        """Enqueue one zm_conv_tend on torch's current stream (no host sync)."""
        s = torch.cuda.current_stream(self.device).cuda_stream
        if self.ncnst:
            Z.lib().zm_convtran1_fields(C.c_int(self.ncnst), self.do1.ctypes.data_as(Z.c_ip),
                                        self.dry.ctypes.data_as(Z.c_ip), _ptr(self.tr["q"]), _ptr(self.tr["fracis"]),
                                        _ptr(self.ptend_qc))
        if self.hist:
            Z.lib().zm_conv_tend_hist_fields(*[(_ptr(self.hist[k]) if k in self.hist else None) for k in Z.HIST_FIELDS])
        args = [C.c_int(self.nch), _ptr(self.ncol)] + [_ptr(self.inp[k]) for k in Z.TEND_IN_ORDER]
        args += [C.c_double(self.ztodt)] + [_ptr(self.out[k]) for k in Z.TEND_ARG_ORDER] + [C.c_void_p(s)]
        rc = Z.lib().zm_conv_tend_batch_dev(*args)
        if rc != 0:
            raise Z.ZmError(f"zm_conv_tend_batch_dev rc={rc}: {Z.last_error()}")

    def step2(self):
        """Enqueue zm_conv_tend_2 (dpdry gather + convtran2) on torch's current stream, from this step's pbuf fields."""
        s = torch.cuda.current_stream(self.device).cuda_stream
        o = self.out
        rc = Z.lib().zm_conv_tend_2_batch_dev(
            C.c_int(self.nch), self.do2.ctypes.data_as(Z.c_ip), _ptr(self.tr["q"]), C.c_int(self.ncnst),
            _ptr(self.tr["pdeldry"]), _ptr(self.tr["fracis"]), _ptr(self.ptend_qc), C.c_double(self.ztodt),
            self.dry.ctypes.data_as(Z.c_ip), *[_ptr(o[k]) for k in ("mu", "md", "du", "eu", "ed", "dp", "dsubcld", "jt",
                                                                    "maxg", "ideep", "lengath")], C.c_void_p(s))
        if rc != 0:
            raise Z.ZmError(f"zm_conv_tend_2_batch_dev rc={rc}: {Z.last_error()}")

    def checksums(self) -> torch.Tensor:
        """One wrap-around 64-bit sum of the bit patterns per output field (device tensor): equal checksums on two
        devices mean bit-identical outputs up to a collision."""
        sums = []
        for k in Z.TEND_ARG_ORDER:
            t = self.out[k]
            sums.append(t.view(torch.int64).sum() if t.dtype == torch.float64 else t.to(torch.int64).sum())
        if self.ncnst:
            sums.append(self.ptend_qc.view(torch.int64).sum())
        return torch.stack(sums)

    def conservation(self) -> torch.Tensor:
        """Enqueue the per-rank budget reduction; returns the 6-double device tensor."""
        if not hasattr(self, "_cons"):
            self._cons = torch.zeros(6, dtype=torch.float64, device=self.device)
        s = torch.cuda.current_stream(self.device).cuda_stream
        o = self.out
        rc = Z.lib().zm_conservation_dev(C.c_int(self.nch), _ptr(self.ncol), _ptr(self.inp["pdel"]),
                                         _ptr(o["ptend_q"]), _ptr(o["ptend_s"]), _ptr(o["prec"]),
                                         _ptr(o["snow"]), _ptr(o["rliq"]), _ptr(o["lengath"]),
                                         _ptr(self._cons), C.c_void_p(s))
        if rc != 0:
            raise Z.ZmError(f"zm_conservation_dev rc={rc}: {Z.last_error()}")
        return self._cons

    def check(self):
        s = torch.cuda.current_stream(self.device).cuda_stream
        rc = Z.lib().zm_sync_check(C.c_void_p(s))
        if rc > 0:
            raise Z.ZmEndrun(Z.last_error())
        return rc
