"""Host-side mirror of the reference's `module zm_conv` public interface
(physics/zm_conv.F90:33-37) over the C ABI of libzmconv_b200.so (include/zmconv_b200.h).

Same procedure names, argument meaning and error behaviour as the reference:
    zm_convi      zm_conv.F90:115    (call site zm_conv_intr.F90:376-379)
    zm_convr      zm_conv.F90:231    (zm_conv_intr.F90:662-673)
    zm_conv_evap  zm_conv.F90:1712   (zm_conv_intr.F90:764-769)
    momtran       zm_conv.F90:2315   (zm_conv_intr.F90:822-826)
    convtran      zm_conv.F90:1976   (zm_conv_intr.F90:875-879, 1020-1024)
The only difference is batching: every array carries a leading chunk dimension
`[nchunks, (ncnst,) nlev, pcols]` (C order == the reference's Fortran chunk arrays back to
back); `nchunks = 1` is the reference's per-chunk call.  A Brent non-convergence raises
`ZmEndrun` (the reference calls endrun, zm_conv.F90:5401-5410).

There is NO CPU fallback: if the CUDA library cannot be loaded this module raises.
"""
from __future__ import annotations

import ctypes as C
import os
import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIBPATH = os.path.join(_HERE, "libzmconv_b200.so")

c_dp = C.POINTER(C.c_double)
c_ip = C.POINTER(C.c_int)


class ZmParams(C.Structure):
    """zm_params_t (include/zmconv_b200.h)."""
    _fields_ = [
        ("pcols", C.c_int), ("pver", C.c_int), ("limcnv", C.c_int), ("num_cin", C.c_int),
        ("zm_org", C.c_int), ("microp", C.c_int), ("no_deep_pbl", C.c_int), ("lparcel_pbl", C.c_int),
        ("cam3", C.c_int), ("masterproc", C.c_int),
        ("c0_lnd", C.c_double), ("c0_ocn", C.c_double), ("ke", C.c_double), ("ke_lnd", C.c_double),
        ("momcu", C.c_double), ("momcd", C.c_double), ("tiedke_add", C.c_double),
        ("capelmt", C.c_double), ("dmpdz", C.c_double), ("tau", C.c_double),
        ("cpair", C.c_double), ("epsilo", C.c_double), ("gravit", C.c_double), ("latice", C.c_double),
        ("latvap", C.c_double), ("tmelt", C.c_double), ("rair", C.c_double), ("cpwv", C.c_double),
        ("cpliq", C.c_double), ("rh2o", C.c_double), ("cpvir", C.c_double), ("zvir", C.c_double),
    ]


class ZmEndrun(RuntimeError):
    """The reference's `call endrun(...)` (fatal)."""


class ZmError(RuntimeError):
    pass


_lib = None


def lib() -> C.CDLL:
    """Loads libzmconv_b200.so; fails loudly (no fallback path exists)."""
    global _lib
    if _lib is None:
        if not os.path.exists(_LIBPATH):
            raise ZmError(f"{_LIBPATH} is missing: run `python -m cam_nor_physics_b200.build` "
                          "(or __graft_entry__.build()); there is no CPU fallback")
        _lib = C.CDLL(_LIBPATH)
        _lib.zm_fp64_peak_flops.restype = C.c_double
        _lib.zm_build_info.restype = C.c_char_p
        _lib.zm_launch_count.restype = C.c_longlong
    return _lib


EXPORTS = [
    "zm_params_default", "zm_init", "zm_finalize", "zm_last_error", "zm_convr_batch",
    "zm_convr_batch_dev", "zm_conv_evap_batch", "zm_conv_evap_batch_dev", "zm_momtran_batch",
    "zm_momtran_batch_dev", "zm_convtran_batch", "zm_convtran_batch_dev", "zm_sync_check",
    "zm_conv_tend_batch", "zm_conv_tend_batch_dev", "zm_microbench", "zm_conservation_dev",
    "zm_conv_tend_2_batch", "zm_tend_trace", "zm_org_fields", "zm_geopotential_t_batch", "zm_geopotential_t_batch_dev",
    "zm_geopotential_t_gen_batch", "zm_geopotential_t_gen_batch_dev", "zm_convect_diagnostics_batch",
    "zm_convect_diagnostics_batch_dev",
    "zm_math_eval_dev", "zm_math_eval_host", "zm_thermo_eval_dev", "zm_fp64_peak_flops",
    "zm_set_profiling", "zm_get_kernel_times", "zm_launch_count",
    "zm_convtran1_fields", "zm_conv_tend_diag_batch", "zm_conv_tend_diag_batch_dev", "zm_get_timers",
    "zm_conv_tend_2_batch_dev", "zm_tend_transfer_bytes", "zm_build_info", "zm_conv_tend_hist_fields",
    "zm_conv_tend_batch_gathered", "zm_conv_tend_2_batch_gathered", "zm_tend_2_transfer_bytes",
]


def last_error() -> str:
    buf = C.create_string_buffer(1024)
    lib().zm_last_error(buf, 1024)
    return buf.value.decode(errors="replace")


def _check(rc: int, what: str):
    if rc < 0:
        raise ZmError(f"{what}: rc={rc}: {last_error()}")
    if rc > 0:
        raise ZmEndrun(f"**** ZM_CONV {what}: Tmix did not converge ****  {last_error()}")


def _dp(a):
    return a.ctypes.data_as(c_dp)


def _ip(a):
    return a.ctypes.data_as(c_ip)


def _f(a):
    return np.ascontiguousarray(a, dtype=np.float64)


def _i(a):
    return np.ascontiguousarray(a, dtype=np.int32)


_params: ZmParams | None = None


def default_params(pcols: int, pver: int, limcnv: int) -> ZmParams:
    p = ZmParams()
    lib().zm_params_default(C.byref(p), pcols, pver, limcnv)
    return p


def zm_convi(limcnv_in, zmconv_c0_lnd, zmconv_c0_ocn, zmconv_ke, zmconv_ke_lnd, zmconv_momcu,
             zmconv_momcd, zmconv_num_cin, zmconv_org, zmconv_microp_in, no_deep_pbl_in,
             zmconv_tiedke_add, zmconv_capelmt, zmconv_dmpdz, zmconv_parcel_pbl, zmconv_tau,
             *, pcols: int, pver: int, masterproc: bool = True, cam3: bool = False) -> ZmParams:
    """zm_convi with the reference's 16-argument list (zm_conv.F90:115-120); ppgrid's pcols/pver
    (module parameters in the reference) come as keywords."""
    p = default_params(pcols, pver, limcnv_in)
    p.c0_lnd, p.c0_ocn, p.ke, p.ke_lnd = zmconv_c0_lnd, zmconv_c0_ocn, zmconv_ke, zmconv_ke_lnd
    p.momcu, p.momcd, p.num_cin = zmconv_momcu, zmconv_momcd, int(zmconv_num_cin)
    p.zm_org, p.microp, p.no_deep_pbl = int(bool(zmconv_org)), int(bool(zmconv_microp_in)), int(bool(no_deep_pbl_in))
    p.tiedke_add, p.capelmt, p.dmpdz = zmconv_tiedke_add, zmconv_capelmt, zmconv_dmpdz
    p.lparcel_pbl, p.tau = int(bool(zmconv_parcel_pbl)), zmconv_tau
    p.masterproc, p.cam3 = int(masterproc), int(cam3)
    return zm_init(p)


def zm_init(p: ZmParams) -> ZmParams:
    global _params
    rc = lib().zm_init(C.byref(p))
    if rc != 0:
        raise ZmEndrun(f"zm_convi: {last_error()}") if rc in (-3,) else ZmError(f"zm_init rc={rc}: {last_error()}")
    _params = p
    return p


def _grid():
    if _params is None:
        raise ZmError("zm_convi/zm_init has not been called")
    return _params.pcols, _params.pver


def zm_org_fields(org, orgt, org2d):
    """Attach the pointer dummies org / orgt / org2d of zm_convr (zm_conv.F90:421-423) for the next zm_convr /
    zm_conv_tend call of this thread (needed iff zmconv_org)."""
    _check(lib().zm_org_fields(_dp(org), _dp(orgt), _dp(org2d)), "zm_org_fields")


def zm_convr(ncol, t, qh, pblh, zm, geos, zi, pap, paph, dpp, delt, tpert, landfrac, org=None):
    """zm_convr (zm_conv.F90:231).  Inputs `[nchunks, nlev, pcols]` / `[nchunks, pcols]`;
    returns a dict with every intent(out) dummy of the reference by its Fortran name (plus `orgt`, `org2d`
    when the organisation tracer `org` is passed, zmconv_org)."""
    pc, L = _grid()
    ncol = _i(ncol)
    nch = ncol.shape[0]
    z2 = lambda n=L: np.zeros((nch, n, pc))
    z1 = lambda: np.zeros((nch, pc))
    o = dict(prec=z1(), jctop=z1(), jcbot=z1(), qtnd=z2(), heat=z2(), mcon=z2(L + 1), cme=z2(),
             cape=z1(), eurt=z2(), dlf=z2(), pflx=z2(L + 1), zdu=z2(), rprd=z2(), mu=z2(), md=z2(),
             du=z2(), eu=z2(), ed=z2(), dp=z2(), dsubcld=z1(),
             jt=np.zeros((nch, pc), np.int32), maxg=np.zeros((nch, pc), np.int32),
             ideep=np.zeros((nch, pc), np.int32), lengath=np.zeros(nch, np.int32),
             ql=z2(), rliq=z1(), dif=z2(), dnlf=z2(), dnif=z2(), rice=z1())
    t, qh, pblh, zm, geos, zi, pap, paph, dpp, tpert, landfrac = map(
        _f, (t, qh, pblh, zm, geos, zi, pap, paph, dpp, tpert, landfrac))
    assert t.shape == (nch, L, pc) and paph.shape == (nch, L + 1, pc) and geos.shape == (nch, pc)
    if org is not None:
        org = _f(org)
        o["orgt"], o["org2d"] = z2(), z2()
        zm_org_fields(org, o["orgt"], o["org2d"])
    rc = lib().zm_convr_batch(
        C.c_int(nch), _ip(ncol), _dp(t), _dp(qh), _dp(o["prec"]), _dp(o["jctop"]), _dp(o["jcbot"]),
        _dp(pblh), _dp(zm), _dp(geos), _dp(zi), _dp(o["qtnd"]), _dp(o["heat"]), _dp(pap), _dp(paph),
        _dp(dpp), C.c_double(delt), _dp(o["mcon"]), _dp(o["cme"]), _dp(o["cape"]), _dp(o["eurt"]),
        _dp(tpert), _dp(o["dlf"]), _dp(o["pflx"]), _dp(o["zdu"]), _dp(o["rprd"]), _dp(o["mu"]),
        _dp(o["md"]), _dp(o["du"]), _dp(o["eu"]), _dp(o["ed"]), _dp(o["dp"]), _dp(o["dsubcld"]),
        _ip(o["jt"]), _ip(o["maxg"]), _ip(o["ideep"]), _ip(o["lengath"]), _dp(o["ql"]), _dp(o["rliq"]),
        _dp(landfrac), _dp(o["dif"]), _dp(o["dnlf"]), _dp(o["dnif"]), _dp(o["rice"]))
    _check(rc, "zm_convr")
    return o


def zm_conv_evap(ncol, t, pmid, pdel, q, landfrac, prdprec, cldfrc, deltat, prec):
    """zm_conv_evap (zm_conv.F90:1712); `prec` is inout (m/s), returned updated."""
    pc, L = _grid()
    ncol = _i(ncol)
    nch = ncol.shape[0]
    o = dict(tend_s=np.zeros((nch, L, pc)), tend_s_snwprd=np.zeros((nch, L, pc)),
             tend_s_snwevmlt=np.zeros((nch, L, pc)), tend_q=np.zeros((nch, L, pc)),
             prec=_f(prec).copy(), snow=np.zeros((nch, pc)), ntprprd=np.zeros((nch, L, pc)),
             ntsnprd=np.zeros((nch, L, pc)), flxprec=np.zeros((nch, L + 1, pc)),
             flxsnow=np.zeros((nch, L + 1, pc)))
    t, pmid, pdel, q, landfrac, prdprec, cldfrc = map(_f, (t, pmid, pdel, q, landfrac, prdprec, cldfrc))
    rc = lib().zm_conv_evap_batch(
        C.c_int(nch), _ip(ncol), _dp(t), _dp(pmid), _dp(pdel), _dp(q), _dp(landfrac), _dp(o["tend_s"]),
        _dp(o["tend_s_snwprd"]), _dp(o["tend_s_snwevmlt"]), _dp(o["tend_q"]), _dp(prdprec), _dp(cldfrc),
        C.c_double(deltat), _dp(o["prec"]), _dp(o["snow"]), _dp(o["ntprprd"]), _dp(o["ntsnprd"]),
        _dp(o["flxprec"]), _dp(o["flxsnow"]))
    _check(rc, "zm_conv_evap")
    return o


def momtran(ncol, domomtran, q, mu, md, du, eu, ed, dp, dsubcld, jt, mx, ideep, lengath, dt):
    """momtran (zm_conv.F90:2315); q = winds `[nchunks, 2, nlev, pcols]`, il1g=1, il2g=lengath."""
    pc, L = _grid()
    ncol = _i(ncol)
    nch = ncol.shape[0]
    q = _f(q)
    ncnst = q.shape[1]
    o = dict(dqdt=np.zeros_like(q), pguall=np.zeros_like(q), pgdall=np.zeros_like(q),
             icwu=np.zeros_like(q), icwd=np.zeros_like(q), seten=np.zeros((nch, L, pc)))
    mu, md, du, eu, ed, dp, dsubcld = map(_f, (mu, md, du, eu, ed, dp, dsubcld))
    rc = lib().zm_momtran_batch(
        C.c_int(nch), _ip(ncol), _ip(_i(domomtran)), _dp(q), C.c_int(ncnst), _dp(mu), _dp(md), _dp(du),
        _dp(eu), _dp(ed), _dp(dp), _dp(dsubcld), _ip(_i(jt)), _ip(_i(mx)), _ip(_i(ideep)),
        _ip(_i(lengath)), _dp(o["dqdt"]), _dp(o["pguall"]), _dp(o["pgdall"]), _dp(o["icwu"]),
        _dp(o["icwd"]), C.c_double(dt), _dp(o["seten"]))
    _check(rc, "momtran")
    return o


def convtran(doconvtran, q, mu, md, du, eu, ed, dp, dsubcld, jt, mx, ideep, lengath, fracis, dpdry,
             dt, cnst_is_dry, dqdt=None):
    """convtran (zm_conv.F90:1976); q/fracis `[nchunks, ncnst, nlev, pcols]`.  Returns dqdt; slices
    of inactive constituents keep the values of the `dqdt` argument (reference: untouched)."""
    pc, L = _grid()
    q = _f(q)
    nch, ncnst = q.shape[0], q.shape[1]
    dqdt = np.zeros_like(q) if dqdt is None else _f(dqdt).copy()
    mu, md, du, eu, ed, dp, dsubcld, fracis, dpdry = map(_f, (mu, md, du, eu, ed, dp, dsubcld, fracis, dpdry))
    rc = lib().zm_convtran_batch(
        C.c_int(nch), _ip(_i(doconvtran)), _dp(q), C.c_int(ncnst), _dp(mu), _dp(md), _dp(du), _dp(eu),
        _dp(ed), _dp(dp), _dp(dsubcld), _ip(_i(jt)), _ip(_i(mx)), _ip(_i(ideep)), _ip(_i(lengath)),
        _dp(fracis), _dp(dqdt), _dp(dpdry), C.c_double(dt), _ip(_i(cnst_is_dry)))
    _check(rc, "convtran")
    return dqdt


TEND_OUT_2D = ["ptend_s", "ptend_q", "ptend_u", "ptend_v", "cme", "zdu", "ql", "rprd", "evapcdp", "dlf",
               "mu", "md", "du", "eu", "ed", "dp"]
TEND_OUT_2DP = ["mcon", "pflx", "flxprec", "flxsnow"]
TEND_OUT_1D = ["rliq", "rice", "jctop", "jcbot", "prec", "snow", "dsubcld", "cape"]
TEND_OUT_INT = ["jt", "maxg", "ideep"]
# order of the output pointers in zm_conv_tend_batch[_dev] (include/zmconv_b200.h)
TEND_ARG_ORDER = ["ptend_s", "ptend_q", "ptend_u", "ptend_v", "mcon", "cme", "pflx", "zdu", "rliq", "rice",
                  "jctop", "jcbot", "prec", "snow", "ql", "rprd", "evapcdp", "flxprec", "flxsnow", "dlf",
                  "mu", "md", "du", "eu", "ed", "dp", "dsubcld", "jt", "maxg", "ideep", "lengath", "cape"]
TEND_IN_ORDER = ["t", "q", "u", "v", "pmid", "pint", "pdel", "zm", "zi", "phis", "pblh", "tpert",
                 "landfrac", "cld"]
# zm_conv_tend's history fields, in the argument order of zm_conv_tend_hist_fields: zm_convr's, zm_conv_evap's and
# momtran's own outputs inside the step (zm_conv_intr.F90:676-857)
HIST_FIELDS = ["heat", "qtnd", "eurt", "dif", "dnlf", "dnif", "tend_s", "tend_s_snwprd", "tend_s_snwevmlt",
               "ntprprd", "ntsnprd", "seten", "pguall", "pgdall", "icwu", "icwd"]
HIST_3D = ("pguall", "pgdall", "icwu", "icwd")          # (pcols,pver,2) per chunk: component 1 = u, 2 = v


def hist_names(hist) -> list:
    """The history fields selected by `hist`: True = all, False/None = none, else an iterable of names."""
    if hist is None or hist is False:
        return []
    if hist is True:
        return list(HIST_FIELDS)
    names = list(hist)
    bad = [k for k in names if k not in HIST_FIELDS]
    if bad:
        raise ZmError(f"unknown history fields {bad}; known: {HIST_FIELDS}")
    return [k for k in HIST_FIELDS if k in names]


def hist_shape(name: str, nch: int, L: int, pc: int) -> tuple:
    return (nch, 2, L, pc) if name in HIST_3D else (nch, L, pc)


def zm_conv_tend_2(doconvtran, q, pdeldry, fracis, ztodt, cnst_is_dry, ptend_q=None):
    """zm_conv_tend_2 (zm_conv_intr.F90:955): convtran2 with the mass-flux fields taken from the device
    mirror left by this thread's last zm_conv_tend call."""
    q = _f(q)
    nch, pcnst = q.shape[0], q.shape[1]
    dq = np.zeros_like(q) if ptend_q is None else _f(ptend_q).copy()
    rc = lib().zm_conv_tend_2_batch(C.c_int(nch), _ip(_i(doconvtran)), _dp(q), C.c_int(pcnst), _dp(_f(pdeldry)),
                                    _dp(_f(fracis)), _dp(dq), C.c_double(ztodt), _ip(_i(cnst_is_dry)))
    _check(rc, "zm_conv_tend_2")
    return dq


# ---- zm_conv_tend_2 on the convective columns' records (zm_conv_tend_2_batch_gathered) ----------------------------
def convtran2_active(doconvtran, pcnst: int) -> np.ndarray:
    """0-based indices m >= 1 with doconvtran[m] (the reference's m = 2..pcnst loop), ascending: the constituent axis
    of the records."""
    do = np.asarray(doconvtran)
    return np.array([m for m in range(1, pcnst) if do[m]], dtype=np.int64)


def convtran2_offsets(lengath, pver: int, nact: int) -> np.ndarray:
    """[nchunks + 1] offsets (doubles) of the chunks' blocks in q_rec / fracis_rec / dqdt_rec: nact*pver*base(c) with
    base(c) = sum(lengath(1:c-1)); the last entry is the records' total size.  pdeldry_rec's are these / nact."""
    lg = np.asarray(lengath, dtype=np.int64)
    return nact * pver * np.concatenate([[0], np.cumsum(lg)])


def convtran2_records(q, fracis, pdeldry, ideep, lengath, doconvtran, cnst_is_dry=None):
    """The caller's pack (loop 1 of the batched Fortran binding in gathered mode): q, fracis `[nchunks, pcnst, pver,
    pcols]` and pdeldry `[nchunks, pver, pcols]` of each chunk's convective columns ideep(1:lengath) and flagged
    constituents.  Returns (q_rec, fracis_rec, pdeldry_rec) as 1-D float64 arrays; pdeldry_rec is None when no flagged
    constituent is dry.  Chunk c's block is g(n, pver, nact) in Fortran order (include/zmconv_b200.h)."""
    q, fracis = np.asarray(q), np.asarray(fracis)
    nch, pcnst, L, _ = q.shape
    lengath = np.asarray(lengath)
    act = convtran2_active(doconvtran, pcnst)
    off = convtran2_offsets(lengath, L, len(act))
    any_dry = cnst_is_dry is not None and len(act) > 0 and bool(np.asarray(cnst_is_dry)[act].any())
    q_rec, f_rec = np.empty(off[-1]), np.empty(off[-1])
    p_rec = np.empty(off[-1] // max(len(act), 1)) if any_dry else None
    for c in range(nch):
        n = int(lengath[c])
        if n == 0 or len(act) == 0:
            continue
        cols = np.asarray(ideep[c][:n]) - 1
        q_rec[off[c]:off[c + 1]] = q[c][act][:, :, cols].ravel()
        f_rec[off[c]:off[c + 1]] = fracis[c][act][:, :, cols].ravel()
        if any_dry:
            o = off[c] // len(act)
            p_rec[o:o + L * n] = np.asarray(pdeldry[c])[:, cols].ravel()
    return q_rec, f_rec, p_rec


def scatter_convtran2(dqdt_rec, ideep, lengath, doconvtran, pcnst: int, pver: int | None = None):
    """The caller's scatter (loop 2): the dense `[nchunks, pcnst, pver, pcols]` tendency zm_conv_tend_2 returns, rebuilt
    from dqdt_rec -- zero everywhere except the flagged constituents' convective columns.  pver defaults to the records'
    size over sum(lengath)*nact (or zm_init's pver when there are no records)."""
    ideep, lengath = np.asarray(ideep), np.asarray(lengath)
    nch, pc = ideep.shape
    act = convtran2_active(doconvtran, pcnst)
    nact = len(act)
    tot = int(lengath.astype(np.int64).sum())
    L = pver if pver is not None else (np.asarray(dqdt_rec).size // (tot * nact) if tot and nact else _grid()[1])
    off = convtran2_offsets(lengath, L, nact)
    out = np.zeros((nch, pcnst, L, pc))
    for c in range(nch):
        n = int(lengath[c])
        if n == 0 or nact == 0:
            continue
        cols = ideep[c][:n] - 1
        out[c][act[:, None, None], np.arange(L)[None, :, None], cols[None, None, :]] = \
            dqdt_rec[off[c]:off[c + 1]].reshape(nact, L, n)
    return out


def zm_conv_tend_2_gathered(lengath, doconvtran, pcnst, cnst_is_dry, q_rec, fracis_rec, pdeldry_rec, ztodt,
                            out=None):
    """zm_conv_tend_2 on the records of convtran2_records (zm_conv_tend_2_batch_gathered), the mass-flux fields taken
    from the device mirror of this thread's last zm_conv_tend call.  Returns dqdt_rec (sum(lengath)*pver*nact doubles,
    scatter_convtran2 gives the dense tendency).  `out` may be a preallocated 1-D float64 buffer (e.g. page-locked) of
    at least that size; the result is then a view of it."""
    _, L = _grid()
    lengath = _i(lengath)
    nch = lengath.shape[0]
    do = _i(doconvtran)
    nact = len(convtran2_active(do, pcnst))
    need = int(lengath.astype(np.int64).sum()) * L * nact
    if out is None:
        out = np.empty(need)
    if out.dtype != np.float64 or out.ndim != 1 or not out.flags.c_contiguous:
        raise ZmError("out must be a 1-D C-contiguous float64 array")
    # converted copies are bound to names: the library reads them through raw pointers while the call runs
    dry = _i(cnst_is_dry) if cnst_is_dry is not None else None
    qr, fr = _f(q_rec), _f(fracis_rec)
    pr = _f(pdeldry_rec) if pdeldry_rec is not None else None
    rc = lib().zm_conv_tend_2_batch_gathered(
        C.c_int(nch), _ip(lengath), _ip(do), C.c_int(pcnst), _ip(dry) if dry is not None else None, _dp(qr), _dp(fr),
        _dp(pr) if pr is not None else None, _dp(out), C.c_longlong(out.size), C.c_double(ztodt))
    _check(rc, "zm_conv_tend_2_gathered")
    return out[:need]


def last_tend_2_transfer_bytes():
    """(host->device, device->host) bytes the last zm_conv_tend_2[_gathered] call of this thread moved over PCIe."""
    a, b = C.c_longlong(0), C.c_longlong(0)
    lib().zm_tend_2_transfer_bytes(C.byref(a), C.byref(b))
    return {"h2d": int(a.value), "d2h": int(b.value)}


def zm_conv_tend(ncol, state: dict, ztodt: float, out: dict | None = None, keep_pbuf_on_device: bool = False,
                 convtran1: dict | None = None, hist=None):
    """zm_conv_tend (zm_conv_intr.F90:390) over host arrays: zm_convr -> physics_update ->
    zm_conv_evap -> momtran [-> convtran1] with everything resident on the device in between.
    `state` holds t,q,u,v,pmid,pint,pdel,zm,zi,phis,pblh,tpert,landfrac,cld in chunk layout.
    convtran1 = dict(doconvtran=cnst_is_convtran1 flags [pcnst], cnst_is_dry=[pcnst] or None,
    q=state%q [nchunks,pcnst,pver,pcols], fracis=same shape[, ptend_q=initial ptend_all%q]) adds the transport of
    cloud liquid / ice (zm_conv_intr.F90:865-880); the result comes back as out["ptend_qc"].
    hist = True (all) or an iterable of HIST_FIELDS names returns those history fields in `out` under their names
    (zm_conv_tend_hist_fields): [nchunks, pver, pcols], or [nchunks, 2, pver, pcols] for pguall, pgdall, icwu, icwd.
    Arrays already in `out` under those names are written in place."""
    pc, L = _grid()
    ncol = _i(ncol)
    nch = ncol.shape[0]
    if out is None:
        out = {}
        for k in TEND_OUT_2D:
            out[k] = np.zeros((nch, L, pc))
        for k in TEND_OUT_2DP:
            out[k] = np.zeros((nch, L + 1, pc))
        for k in TEND_OUT_1D:
            out[k] = np.zeros((nch, pc))
        for k in TEND_OUT_INT:
            out[k] = np.zeros((nch, pc), np.int32)
        out["lengath"] = np.zeros(nch, np.int32)
    args, names, alive = _tend_inputs(ncol, state, ztodt, out, convtran1, hist)
    mirror_only = {"mu", "md", "du", "eu", "ed", "dp", "dsubcld", "jt", "maxg"} if keep_pbuf_on_device else set()
    for k in TEND_ARG_ORDER:
        a = out[k]
        if k in mirror_only:
            args.append(None)       # stays in the device mirror for zm_conv_tend_2 (no D2H)
        else:
            args.append(_ip(a) if a.dtype == np.int32 else _dp(a))
    _attach_hist(out, names)
    rc = lib().zm_conv_tend_batch(*args)
    del alive                   # the attached org / convtran1 arrays had to outlive the step
    _check(rc, "zm_conv_tend")
    return out


def _tend_inputs(ncol, state, ztodt, out, convtran1, hist):
    """Marshalling shared by zm_conv_tend and zm_conv_tend_gathered: the input arguments, the org / convtran1
    attachments, the history arrays in `out` (created or checked).  Returns (argument list, history names, arrays the
    library holds raw pointers to: the caller keeps them alive until the step has returned)."""
    pc, L = _grid()
    nch = ncol.shape[0]
    ins = [_f(state[k]) for k in TEND_IN_ORDER]
    args = [C.c_int(nch), _ip(ncol)] + [_dp(a) for a in ins] + [C.c_double(ztodt)]
    alive = []                              # attached arrays: _f may have made a copy that nothing else references
    if "org" in state:                      # zmconv_org: organisation tracer in, its tendency and column mean out
        org = _f(state["org"])
        if "orgt" not in out:
            out["orgt"], out["org2d"] = np.zeros_like(org), np.zeros_like(org)
        zm_org_fields(org, out["orgt"], out["org2d"])
        alive.append(org)
    if convtran1 is not None:
        q3, f3 = _f(convtran1["q"]), _f(convtran1["fracis"])
        pcnst = q3.shape[1]
        out["ptend_qc"] = np.zeros_like(q3) if convtran1.get("ptend_q") is None else _f(convtran1["ptend_q"]).copy()
        dry = convtran1.get("cnst_is_dry")
        alive += [q3, f3]
        lib().zm_convtran1_fields(C.c_int(pcnst), _ip(_i(convtran1["doconvtran"])),
                                  _ip(_i(dry)) if dry is not None else None, _dp(q3), _dp(f3), _dp(out["ptend_qc"]))
    names = hist_names(hist)
    for k in names:
        shape = hist_shape(k, nch, L, pc)
        if k not in out:
            out[k] = np.zeros(shape)
        a = out[k]
        if a.shape != shape or a.dtype != np.float64 or not a.flags.c_contiguous:
            raise ZmError(f"out[{k!r}] must be a C-contiguous float64 array of shape {shape}")
    return args, names, alive


def _attach_hist(out, names):
    if names:       # attached last, right before the step: nothing may fail and leave the attachment to a later call
        lib().zm_conv_tend_hist_fields(*[(_dp(out[k]) if k in names else None) for k in HIST_FIELDS])


# Record of one convective column in zm_conv_tend_batch_gathered (include/zmconv_b200.h): the fields indexed by the
# column ideep(slot), then -- with the pbuf fields in the records -- the slot-indexed pbuf fields.
GATHERED_FIELDS = ["ptend_s", "ptend_q", "ptend_u", "ptend_v", "cme", "zdu", "ql", "rprd", "evapcdp", "dlf",
                   "mcon", "pflx", "flxprec", "flxsnow"]
GATHERED_PBUF = ["mu", "md", "du", "eu", "ed", "dp"]
GATHERED_COL_OUT = ["rliq", "rice", "jctop", "jcbot", "prec", "snow", "cape", "dsubcld"]


def gathered_layout(pver: int, with_pbuf: bool):
    """({field: (offset, nlev)} in doubles, rec_len) of a zm_conv_tend_batch_gathered record."""
    lay, off = {}, 0
    for k in GATHERED_FIELDS + (GATHERED_PBUF if with_pbuf else []):
        n = pver + 1 if k in TEND_OUT_2DP else pver
        lay[k] = (off, n)
        off += n
    return lay, off


def zm_conv_tend_gathered(ncol, state: dict, ztodt: float, keep_pbuf_on_device: bool = False,
                          convtran1: dict | None = None, hist=None, out: dict | None = None):
    """zm_conv_tend with the (pcols,pver[p]) outputs returned as one record per convective column
    (zm_conv_tend_batch_gathered).  Returns the per-column outputs (rliq, rice, jctop, jcbot, prec, snow, cape,
    dsubcld, jt, maxg, ideep, lengath), `pbuf_in_records` and `rec`, a [sum(lengath), rec_len] view, chunk after
    chunk in gathered order; gathered_layout gives the fields' offsets, scatter_gathered the dense arrays of zm_conv_tend.
    keep_pbuf_on_device: mu..dp stay out of the records and, with dsubcld, jt, maxg, in the device mirror only (those
    three are then left as found).  convtran1 / hist as in zm_conv_tend (their arrays travel whole).  Arrays already in
    `out` are written in place; out["rec_buf"] may be a 1-D float64 buffer of at least nchunks*pcols*rec_len doubles that
    the records are written into (e.g. page-locked once and reused)."""
    pc, L = _grid()
    ncol = _i(ncol)
    nch = ncol.shape[0]
    _, rec_len = gathered_layout(L, not keep_pbuf_on_device)
    out = {} if out is None else out
    for k in GATHERED_COL_OUT:
        out.setdefault(k, np.zeros((nch, pc)))
    for k in ("jt", "maxg", "ideep"):
        out.setdefault(k, np.zeros((nch, pc), np.int32))
    out.setdefault("lengath", np.zeros(nch, np.int32))
    buf = out.get("rec_buf")
    if buf is None:
        buf = out["rec_buf"] = np.empty(nch * pc * rec_len)
    if buf.dtype != np.float64 or buf.ndim != 1 or not buf.flags.c_contiguous:
        raise ZmError("out['rec_buf'] must be a 1-D C-contiguous float64 array")
    args, names, alive = _tend_inputs(ncol, state, ztodt, out, convtran1, hist)
    mirror_only = {"dsubcld", "jt", "maxg"} if keep_pbuf_on_device else set()
    for k in GATHERED_COL_OUT + ["jt", "maxg", "ideep", "lengath"]:
        a = out[k]
        args.append(None if k in mirror_only else (_ip(a) if a.dtype == np.int32 else _dp(a)))
    args += [C.c_int(0 if keep_pbuf_on_device else 1), _dp(buf), C.c_longlong(buf.size)]
    _attach_hist(out, names)
    rc = lib().zm_conv_tend_batch_gathered(*args)
    del alive                   # the attached org / convtran1 arrays had to outlive the step
    _check(rc, "zm_conv_tend_gathered")
    n = int(out["lengath"].sum())
    out["rec"] = buf[:n * rec_len].reshape(n, rec_len)
    out["pbuf_in_records"] = int(not keep_pbuf_on_device)
    return out


def scatter_gathered(res: dict) -> dict:
    """zm_conv_tend's dense output dict rebuilt from a zm_conv_tend_gathered result: zeros, then every record's fields
    into column ideep(slot) (slot row for the pbuf fields) of its chunk.  Without the pbuf fields in the records,
    mu..dp are 0, as zm_conv_tend returns them with keep_pbuf_on_device."""
    lengath, ideep, rec = res["lengath"], res["ideep"], res["rec"]
    nch, pc = ideep.shape
    with_pbuf = bool(res["pbuf_in_records"])
    L = (rec.shape[1] - 4) // (20 if with_pbuf else 14)
    lay, rec_len = gathered_layout(L, with_pbuf)
    assert rec.shape == (int(lengath.sum()), rec_len), rec.shape
    chunk = np.repeat(np.arange(nch), lengath)
    slot = np.arange(rec.shape[0]) - np.repeat(np.cumsum(lengath) - lengath, lengath)
    col = ideep[chunk, slot] - 1
    out = {}
    for k in TEND_OUT_2D + TEND_OUT_2DP:
        n = L + 1 if k in TEND_OUT_2DP else L
        out[k] = np.zeros((nch, n, pc))
        if k in lay:
            o, _ = lay[k]
            out[k][chunk, :, slot if k in GATHERED_PBUF else col] = rec[:, o:o + n]
    for k in GATHERED_COL_OUT + ["jt", "maxg", "ideep", "lengath"]:
        out[k] = res[k]
    return out


def zm_conv_tend_diag(ncol, ps, pmid, mu=None, md=None, jt=None, maxg=None, ideep=None, lengath=None):
    """freqzm, mu_out, md_out, pcont, pconb of zm_conv_tend (zm_conv_intr.F90:685-688, 700-706, 721-729).  With the
    mass-flux fields left out they come from the device mirror of this thread's last zm_conv_tend call."""
    pc, L = _grid()
    ncol = _i(ncol)
    nch = ncol.shape[0]
    o = dict(freqzm=np.zeros((nch, pc)), mu_out=np.zeros((nch, L, pc)), md_out=np.zeros((nch, L, pc)),
             pcont=np.zeros((nch, pc)), pconb=np.zeros((nch, pc)))
    given = mu is not None
    a = [(_dp(_f(x)) if given else None) for x in (mu, md)] + [(_ip(_i(x)) if given else None) for x in (jt, maxg, ideep, lengath)]
    rc = lib().zm_conv_tend_diag_batch(C.c_int(nch), _ip(ncol), _dp(_f(ps)), _dp(_f(pmid)), *a, _dp(o["freqzm"]),
                                       _dp(o["mu_out"]), _dp(o["md_out"]), _dp(o["pcont"]), _dp(o["pconb"]))
    _check(rc, "zm_conv_tend_diag")
    return o


def timers():
    """Device times (ms) of the last profiled zm_conv_tend / zm_conv_tend_2 call under the reference's GPTL timer
    names (zm_conv_intr.F90:654-880, 1019-1025): zm_convr, zm_conv_evap, momtran, convtran1, convtran2."""
    n = C.c_int(8)
    names = (C.c_char_p * 8)()
    ms = (C.c_float * 8)()
    lib().zm_get_timers(C.byref(n), names, ms)
    return {names[i].decode(): float(ms[i]) for i in range(n.value)}


def geopotential_t(ncol, piln, pmln, pint, pmid, pdel, rpdel, t, q, rair, gravit, zvir, dycore_lr=True):
    """geopotential_t (physics/geopotential.F90:153); returns (zi, zm)."""
    pc, L = _grid()
    ncol = _i(ncol)
    nch = ncol.shape[0]
    zi, zm = np.zeros((nch, L + 1, pc)), np.zeros((nch, L, pc))
    piln, pmln, pint, pmid, pdel, rpdel, t, q, rair, zvir = map(_f, (piln, pmln, pint, pmid, pdel, rpdel, t, q, rair, zvir))
    rc = lib().zm_geopotential_t_batch(C.c_int(nch), _ip(ncol), C.c_int(int(dycore_lr)), _dp(piln), _dp(pmln),
                                       _dp(pint), _dp(pmid), _dp(pdel), _dp(rpdel), _dp(t), _dp(q), _dp(rair),
                                       C.c_double(gravit), _dp(zvir), _dp(zi), _dp(zm))
    _check(rc, "geopotential_t")
    return zi, zm


def geopotential_t_gen(ncol, piln, pmln, pint, pmid, pdel, rpdel, t, q3, rair, gravit, zvir, species_idx,
                       dycore_lr=False):
    """geopotential_t, generalized-virtual-temperature branch (physics/geopotential.F90:248-310; dycore MPAS / SE).
    q3: (nchunks, ncnst, pver, pcols); species_idx: 1-based thermodynamic_active_species_idx.  Returns (zi, zm)."""
    pc, L = _grid()
    ncol = _i(ncol)
    nch = ncol.shape[0]
    zi, zm = np.zeros((nch, L + 1, pc)), np.zeros((nch, L, pc))
    piln, pmln, pint, pmid, pdel, rpdel, t, q3, rair, zvir = map(_f, (piln, pmln, pint, pmid, pdel, rpdel, t, q3, rair, zvir))
    sp = _i(species_idx)
    rc = lib().zm_geopotential_t_gen_batch(C.c_int(nch), _ip(ncol), C.c_int(int(dycore_lr)), C.c_int(q3.shape[1]),
                                           C.c_int(sp.shape[0]), _ip(sp), _dp(piln), _dp(pmln), _dp(pint), _dp(pmid),
                                           _dp(pdel), _dp(rpdel), _dp(t), _dp(q3), _dp(rair), C.c_double(gravit),
                                           _dp(zvir), _dp(zi), _dp(zm))
    _check(rc, "geopotential_t")
    return zi, zm


def convect_diagnostics_calc(ncol, cmfmc, qc, rliq, pmid, rprddp, cnt, cnb):
    """convect_diagnostics_calc (physics/convect_diagnostics.F90:115) with shallow_scheme='CLUBB_SGS'.
    Returns a dict with the updated inout fields and the outputs."""
    pc, L = _grid()
    ncol = _i(ncol)
    nch = ncol.shape[0]
    o = dict(cmfmc=_f(cmfmc).copy(), qc=_f(qc).copy(), qc2=np.ones((nch, L, pc)), rliq=_f(rliq).copy(),
             rliq2=np.ones((nch, pc)), cnt=_f(cnt).copy(), cnb=_f(cnb).copy(), cmfmc2=np.ones((nch, L + 1, pc)),
             rprdsh=np.ones((nch, L, pc)), rprdtot=np.zeros((nch, L, pc)), pcnt=np.zeros((nch, pc)),
             pcnb=np.zeros((nch, pc)))
    pmid, rprddp = _f(pmid), _f(rprddp)
    rc = lib().zm_convect_diagnostics_batch(C.c_int(nch), _ip(ncol), _dp(o["cmfmc"]), _dp(o["qc"]), _dp(o["qc2"]),
                                            _dp(o["rliq"]), _dp(o["rliq2"]), _dp(pmid), _dp(rprddp), _dp(o["cnt"]),
                                            _dp(o["cnb"]), _dp(o["cmfmc2"]), _dp(o["rprdsh"]), _dp(o["rprdtot"]),
                                            _dp(o["pcnt"]), _dp(o["pcnb"]))
    _check(rc, "convect_diagnostics_calc")
    return o


# ---- diagnostics ---------------------------------------------------------------------------------
def math_eval(fid: int, x, y=None, device: bool = True):
    x = _f(x)
    y = _f(x if y is None else y)
    out = np.empty_like(x)
    fn = lib().zm_math_eval_dev if device else lib().zm_math_eval_host
    rc = fn(C.c_int(fid), C.c_int(x.size), _dp(x), _dp(y), _dp(out))
    _check(rc, "math_eval")
    return out


def thermo_eval(fid: int, a, b, c=None, d=None, e=None):
    a = _f(a)
    z = np.zeros_like(a)
    b, c, d, e = (_f(v) if v is not None else z for v in (b, c, d, e))
    o0, o1 = np.empty_like(a), np.empty_like(a)
    rc = lib().zm_thermo_eval_dev(C.c_int(fid), C.c_int(a.size), _dp(a), _dp(b), _dp(c), _dp(d), _dp(e),
                                  _dp(o0), _dp(o1))
    _check(rc, "thermo_eval")
    return o0, o1


def tend_trace():
    """Timeline (ms) of the last zm_conv_tend call on this thread: rows = sub-batches, columns = inputs on device,
    late inputs on device, zm_convr done, kernels done, zm_convr outputs on host, all outputs on host."""
    buf = (C.c_double * 48)()
    nb = lib().zm_tend_trace(buf, C.c_int(48))
    return np.array(buf[:6 * nb]).reshape(nb, 6)


def last_transfer_bytes():
    """(host->device, device->host) bytes the last zm_conv_tend call of this thread moved over PCIe."""
    a, b = C.c_longlong(0), C.c_longlong(0)
    lib().zm_tend_transfer_bytes(C.byref(a), C.byref(b))
    return {"h2d": int(a.value), "d2h": int(b.value)}


def fp64_peak_flops(iters: int = 20000) -> float:
    return float(lib().zm_fp64_peak_flops(C.c_int(iters)))


def kernel_times():
    n = C.c_int(24)
    names = (C.c_char_p * 24)()
    ms = (C.c_float * 24)()
    lib().zm_get_kernel_times(C.byref(n), names, ms)
    return [(names[i].decode(), float(ms[i])) for i in range(n.value)]
