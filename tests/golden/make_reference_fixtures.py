"""Generates tests/golden/reftext_*.npz: outputs of the REFERENCE'S OWN SOURCE TEXT for seeded inputs.

physics/zm_conv.F90 is read from the CAM-Nor source tree named by $CAM_NOR_SRC, every routine on the hot path is translated
mechanically to Python by fortran_exec.py (statement by statement; nothing is re-derived by hand) and executed:
zm_convi, zm_convr (-> buoyan_dilute, parcel_dilute, entropy, enthalpy, ientropy, ienthalpy, qsat_hPa, cldprp,
closure, q1q2_pjr, buoyan for cam3), zm_conv_evap, momtran, convtran.  Inputs, namelist values and outputs are stored;
tests/test_oracle.py::test_oracle_equals_reference_source_text compares the CPU oracle with them bit for bit (glibc
libm flavour), tests/test_gpu_parity.py compares the CUDA library within the north-star tolerance.

The externals that are NOT part of the reference tree (wv_saturation::qsat_water / qsat, cloud_fraction::cldfrc_fice,
physconst values, constituents::cnst_get_type_byind) are supplied here in Python with the formulas SURVEY.md 8c
lists -- those stay unpinned (there is no reference text for them).

usage:  CAM_NOR_SRC=<CAM-Nor checkout> python tests/golden/make_reference_fixtures.py        (~1 minute)
"""
import math
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, HERE); sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "tests"))
import fortran_exec as F                      # noqa: E402
from cam_nor_physics_b200 import soundings as S   # noqa: E402

PHYSICS = os.path.join(os.environ.get("CAM_NOR_SRC", ""), "physics")
if not os.environ.get("CAM_NOR_SRC") or not os.path.isfile(os.path.join(PHYSICS, "zm_conv.F90")):
    raise SystemExit("CAM_NOR_SRC must name a CAM-Nor source tree (with physics/zm_conv.F90); it is %r"
                     % os.environ.get("CAM_NOR_SRC"))
SRC = os.path.join(PHYSICS, "zm_conv.F90")
INTR = os.path.join(PHYSICS, "zm_conv_intr.F90")
PTYPES = os.path.join(PHYSICS, "physics_types.F90")
ROUTINES = ["zm_convi", "qsat_hpa", "entropy", "enthalpy", "ientropy", "ienthalpy", "parcel_dilute", "buoyan_dilute",
            "buoyan", "cldprp", "closure", "q1q2_pjr", "zm_convr", "zm_conv_evap", "momtran", "convtran"]


# ---- externals (not in the reference tree; SURVEY.md 8c) -----------------------------------------------------
def physconst():
    boltz, avogad = 1.38065e-23, 6.02214e26
    rgas = avogad * boltz
    mwdair, mwwv = 28.966, 18.016
    c = dict(cpair=1.00464e3, epsilo=mwwv / mwdair, gravit=9.80616, latice=3.337e5, latvap=2.501e6, tmelt=273.15,
             rair=rgas / mwdair, cpwv=1.810e3, cpliq=4.188e3, rh2o=rgas / mwwv)
    c["cpvir"] = c["cpwv"] / c["cpair"] - 1.0
    c["zvir"] = c["rh2o"] / c["rair"] - 1.0
    return c


def gg_water(t):
    tb = 373.16
    return 10.0 ** (-7.90298 * (tb / t - 1.0) + 5.02808 * math.log10(tb / t)
                    - 1.3816e-7 * (10.0 ** (11.344 * (1.0 - t / tb)) - 1.0)
                    + 8.1328e-3 * (10.0 ** (-3.49149 * (tb / t - 1.0)) - 1.0) + math.log10(1013.246)) * 100.0


def gg_ice(t):
    t3 = 273.16
    return 10.0 ** (-9.09718 * (t3 / t - 1.0) - 3.56654 * math.log10(t3 / t) + 0.876793 * (1.0 - t / t3)
                    + math.log10(6.1071)) * 100.0


class Externals:
    def __init__(self, c):
        self.c = c
        tmelt, ttrice = c["tmelt"], 20.0
        tmin, tmax = 127.16, 375.16
        n = int(tmax - tmin + 1) + 1
        self.tmin, self.tmax = tmin, tmax
        self.estbl = []
        for i in range(n):
            t = tmin + i
            if t < tmelt - ttrice:
                w = 1.0
            elif t < tmelt:
                w = (tmelt - t) / ttrice
            else:
                w = 0.0
            if w >= 1.0:
                es = gg_ice(t)
            elif w <= 0.0:
                es = gg_water(t)
            else:
                es = w * gg_ice(t) + (1.0 - w) * gg_water(t)
            self.estbl.append(es)

    def svp_to_qsat(self, es, p):
        eps = self.c["epsilo"]
        if (p - es) <= 0.0:
            return 1.0
        return eps * es / (p - (1.0 - eps) * es)

    def qsat_water(self, t, p, es=None, qs=None):
        e = gg_water(t)
        q = self.svp_to_qsat(e, p)
        return min(e, p), q

    def qsat(self, t, p, es, qs, ncol):
        """wv_saturation::qsat (table version) on (ncol) vectors: es, qs are filled in place.  The caller passes array
        sections (t(1:ncol,k) ...), which arrive here as 0-based numpy views of the Fortran arrays."""
        for i in range(ncol):
            tt = max(min(t[i], self.tmax) - self.tmin, 0.0)
            j = int(tt)
            w = tt - math.trunc(tt)
            e = (1.0 - w) * self.estbl[j] + w * self.estbl[j + 1]
            qs[i] = self.svp_to_qsat(e, p[i])
            es[i] = min(e, p[i])

    def cldfrc_fice(self, ncol, t, fice, fsnow):
        tmelt = self.c["tmelt"]
        tmax_fice, tmin_fice = tmelt - 10.0, tmelt - 40.0
        tmax_fsnow, tmin_fsnow = tmelt, tmelt - 5.0
        for k in range(1, t.shape[1] + 1):
            for i in range(1, ncol + 1):
                tt = t[i, k]
                if tt > tmax_fice:
                    fice[i, k] = 0.0
                elif tt < tmin_fice:
                    fice[i, k] = 1.0
                else:
                    fice[i, k] = (tmax_fice - tt) / (tmax_fice - tmin_fice)
                if tt > tmax_fsnow:
                    fsnow[i, k] = 0.0
                elif tt < tmin_fsnow:
                    fsnow[i, k] = 1.0
                else:
                    fsnow[i, k] = (tmax_fsnow - tt) / (tmax_fsnow - tmin_fsnow)


def build_module(pcols, pver, masterproc=True, cam3=False, dry_of=None):
    c = physconst()
    ext = Externals(c)
    ns = dict(c)
    ns.update(pcols=pcols, pver=pver, pverp=pver + 1, masterproc=masterproc, iulog=6,
              qsat_water=ext.qsat_water, qsat=ext.qsat, cldfrc_fice=ext.cldfrc_fice,
              _OUTS={"qsat_water": [2, 3]},
              get_rlat_p=lambda *a: 0.0, get_rlon_p=lambda *a: 0.0,
              cam_physpkg_is=lambda s: bool(cam3) and s == "cam3",
              cnst_get_type_byind=(lambda m: "dry" if (dry_of and dry_of[m - 1]) else "wet"))
    m = F.Module(SRC, ns)
    m.module_parameters(40, 108)
    m.load(*ROUTINES)
    return m, c


def FA(a, dtype=float):
    """numpy [.., nlev, pcols] chunk array -> FArr view indexed (i, k[, m]) like the Fortran dummy."""
    if a.ndim == 1:
        return F.FArr(a.shape, dtype=dtype, data=a)
    return F.FArr(a.T.shape, dtype=dtype, data=a.T)


def run_case(name, ncols, pver, p_conv, nl, ncol_used=None, org=False, cam3=False, col0=0, ncnst=6, pcols=16,
             transform=None, tracer_edge=False):
    """One chunk.  nl: namelist overrides of zm_convi."""
    L = pver
    # cam3: zm_convr tests `cin` (zm_conv.F90:909) although buoyan never defines it -- undefined behaviour in the
    # reference.  Undefined local reals read as 0.0 for that case (what fresh stack memory usually holds, and what
    # the oracle / CUDA library define, DESIGN.md section 8); NaN everywhere else, so that no other result can
    # silently depend on an undefined value.
    F.FArr.UNDEFINED = 0.0 if cam3 else np.nan
    ch = S.make_chunks(ncols, L, pcols, p_conv=p_conv, col0=col0)
    ncol = int(ch.ncol[0]) if ncol_used is None else ncol_used
    do = [0] + [1, 1, 0, 1, 1, 1, 1][:ncnst - 1]
    dry = [0] + [0, 1, 0, 1, 0, 1, 0][:ncnst - 1]
    m, c = build_module(pcols, L, masterproc=nl.get("masterproc", True), cam3=cam3, dry_of=dry)
    p = dict(limcnv=S.limcnv_for(L), c0_lnd=0.0075, c0_ocn=0.03, ke=5.0e-6, ke_lnd=1.0e-5, momcu=0.7, momcd=0.7,
             num_cin=1, zm_org=bool(org), microp=False, no_deep_pbl=False, tiedke_add=0.5, capelmt=70.0,
             dmpdz=-1.0e-3, lparcel_pbl=False, tau=3600.0)
    p.update({k: v for k, v in nl.items() if k != "masterproc"})
    m.ns["zm_convi"](p["limcnv"], p["c0_lnd"], p["c0_ocn"], p["ke"], p["ke_lnd"], p["momcu"], p["momcd"], p["num_cin"],
                     p["zm_org"], p["microp"], p["no_deep_pbl"], p["tiedke_add"], p["capelmt"], p["dmpdz"],
                     p["lparcel_pbl"], p["tau"])
    z2 = lambda n=L: np.zeros((n, pcols))      # noqa: E731
    z1 = lambda: np.zeros(pcols)               # noqa: E731
    o = dict(prec=z1(), jctop=z1(), jcbot=z1(), qtnd=z2(), heat=z2(), mcon=z2(L + 1), cme=z2(), cape=z1(), eurt=z2(),
             dlf=z2(), pflx=z2(L + 1), zdu=z2(), rprd=z2(), mu=z2(), md=z2(), du=z2(), eu=z2(), ed=z2(), dp=z2(),
             dsubcld=z1(), jt=np.zeros(pcols, np.int64), maxg=np.zeros(pcols, np.int64),
             ideep=np.zeros(pcols, np.int64), ql=z2(), rliq=z1(), dif=z2(), dnlf=z2(), dnif=z2(), rice=z1())
    inp = {k: np.ascontiguousarray(getattr(ch, k)[0]) for k in
           ("t", "q", "u", "v", "pmid", "pint", "pdel", "zm", "zi", "phis", "pblh", "tpert", "landfrac", "cld")}
    if transform:                                   # stress cases: unusual soundings (inputs are stored, not regenerated)
        STRESS[transform](inp, c)
    orgf = orgt = org2d = None
    if org:
        rng = np.random.default_rng(17)
        orgf = np.maximum(rng.uniform(-0.3, 1.0, (L, pcols)), 0.0)
        orgt, org2d = np.full((L, pcols), 7.0), np.zeros((L, pcols))
    delt = 0.5 * float(ch.ztodt)
    A = lambda k, dt=float: FA(o[k], dt)       # noqa: E731
    lengath, = m.ns["zm_convr"](
        1, ncol, FA(inp["t"]), FA(inp["q"]), A("prec"), A("jctop"), A("jcbot"), FA(inp["pblh"]), FA(inp["zm"]),
        FA(inp["phis"]), FA(inp["zi"]), A("qtnd"), A("heat"), FA(inp["pmid"]), FA(inp["pint"]), FA(inp["pdel"]), delt,
        A("mcon"), A("cme"), A("cape"), A("eurt"), FA(inp["tpert"]), A("dlf"), A("pflx"), A("zdu"), A("rprd"), A("mu"),
        A("md"), A("du"), A("eu"), A("ed"), A("dp"), A("dsubcld"), A("jt", int), A("maxg", int), A("ideep", int), None,
        A("ql"), A("rliq"), FA(inp["landfrac"]), FA(orgf) if org else None, FA(orgt) if org else None,
        FA(org2d) if org else None, A("dif"), A("dnlf"), A("dnif"), F.FStruct(), F.FStruct(), A("rice"))
    fx = {"nl_" + k: np.asarray(v) for k, v in p.items()}
    fx.update(nl_masterproc=np.asarray(bool(nl.get("masterproc", True))), nl_cam3=np.asarray(bool(cam3)),
              pcols=np.asarray(pcols), pver=np.asarray(L), ncol=np.asarray(ncol), ztodt=np.asarray(float(ch.ztodt)))
    fx.update({"in_" + k: v for k, v in inp.items()})
    fx.update({"convr_" + k: v for k, v in o.items()})
    fx["convr_lengath"] = np.asarray(int(lengath))
    if org:
        fx.update(in_org=orgf, convr_orgt=orgt, convr_org2d=org2d)

    # ---- glue statements of zm_conv_tend, executed from the reference text one statement block at a time ----
    # mcon unit conversion (zm_conv_intr.F90:693)
    tmcon = o["mcon"].copy()
    mi = F.Module(INTR, dict(ncol=ncol, pver=L, pverp=L + 1, gravit=c["gravit"], mcon=FA(tmcon)))
    mi.run_lines(693, 693)
    fx["tend_mcon"] = tmcon
    # physics_update of state1 with zm_convr's ptend (physics_types.F90:321-323 for q, :426-430 for t; the qneg3
    # clip at qmin(1) = 1e-12 that follows :322 is an external and applied by hand)
    st, pt = F.FStruct(), F.FStruct()
    q3, dq3 = inp["q"][None].copy(), o["qtnd"][None].copy()
    t1 = inp["t"].copy()
    st.q, pt.q = F.FArr(q3.T.shape, data=q3.T), F.FArr(dq3.T.shape, data=dq3.T)
    st.t, pt.s = FA(t1), FA(o["heat"])
    pt.top_level, pt.bot_level = 1, L
    cpv = np.full((L, pcols), c["cpair"])
    mp_ = F.Module(PTYPES, dict(ncol=ncol, pver=L, m=1, dt=float(ch.ztodt), state=st, ptend=pt, tend=None,
                               cpairv_loc=FA(cpv)))
    mp_.run_lines(321, 323)
    mp_.run_lines(426, 430)
    q1 = np.maximum(q3[0], 1e-12)
    assert np.array_equal(t1[:, :ncol], (inp["t"] + o["heat"] * float(ch.ztodt) / c["cpair"])[:, :ncol])
    t1[:, ncol:] = inp["t"][:, ncol:]; q1[:, ncol:] = np.maximum(inp["q"][:, ncol:], 1e-12)

    # ---- zm_conv_evap on that state (zm_conv_intr.F90:764-769) ----
    ev = dict(tend_s=z2(), tend_s_snwprd=z2(), tend_s_snwevmlt=z2(), tend_q=z2(), prec=o["prec"].copy(), snow=z1(),
              ntprprd=z2(), ntsnprd=z2(), flxprec=z2(L + 1), flxsnow=z2(L + 1))
    E = lambda k: FA(ev[k])                    # noqa: E731
    m.ns["zm_conv_evap"](ncol, 1, FA(t1), FA(inp["pmid"]), FA(inp["pdel"]), FA(q1), FA(inp["landfrac"]), E("tend_s"),
                         E("tend_s_snwprd"), E("tend_s_snwevmlt"), E("tend_q"), FA(o["rprd"]), FA(inp["cld"]),
                         float(ch.ztodt), E("prec"), E("snow"), E("ntprprd"), E("ntsnprd"), E("flxprec"), E("flxsnow"))
    fx.update(evap_in_t=t1, evap_in_q=q1)
    fx.update({"evap_" + k: v for k, v in ev.items()})
    if org:
        # organisation tendency (zm_conv_intr.F90:773-777) from the reference text
        st2, pt2 = F.FStruct(), F.FStruct()
        o3, t3 = orgf[None].copy(), np.zeros((1, L, pcols))
        st2.q, pt2.q = F.FArr(o3.T.shape, data=o3.T), F.FArr(t3.T.shape, data=t3.T)
        mo_ = F.Module(INTR, dict(ncol=ncol, pver=L, ixorg=1, ztodt=float(ch.ztodt), zmconv_org=True, state=st2,
                                  ptend_loc=pt2, evapcdp=FA(ev["tend_q"])))
        mo_.run_lines(773, 777)
        fx["tend_orgt"] = t3[0]

    # ---- momtran (zm_conv_intr.F90:811-826) ----
    winds = np.stack([inp["u"], inp["v"]], axis=0)                     # [2][L][pcols] == Fortran (pcols,pver,2)
    mo = dict(dqdt=np.zeros((2, L, pcols)), pguall=np.zeros((2, L, pcols)), pgdall=np.zeros((2, L, pcols)),
              icwu=np.zeros((2, L, pcols)), icwd=np.zeros((2, L, pcols)), seten=z2())
    F3 = lambda a: F.FArr(a.T.shape, data=a.T)     # noqa: E731
    domom = F.FArr((2,), dtype=int, data=np.array([1, 1]))
    m.ns["momtran"](1, ncol, domom, F3(winds), 2, FA(o["mu"]), FA(o["md"]), FA(o["du"]), FA(o["eu"]), FA(o["ed"]),
                    FA(o["dp"]), FA(o["dsubcld"]), FA(o["jt"], int), FA(o["maxg"], int), FA(o["ideep"], int), 1,
                    int(lengath), 0, F3(mo["dqdt"]), F3(mo["pguall"]), F3(mo["pgdall"]), F3(mo["icwu"]), F3(mo["icwd"]),
                    float(ch.ztodt), FA(mo["seten"]))
    fx.update({"momtran_" + k: v for k, v in mo.items()})

    # ---- convtran (zm_conv_intr.F90:1014-1024 dpdry gather; :875 / :1020 call) ----
    qtr, fracis, pdeldry = S.make_tracers(ch, ncnst)
    qtr, fracis, pdeldry = qtr[0], fracis[0], pdeldry[0]
    if tracer_edge:       # exact zeros, tiny and slightly negative mixing ratios: the chat branches of :2119-2139
        u = np.random.default_rng(5).uniform(size=qtr.shape)
        qtr[u < 0.08] = 0.0
        qtr[(u >= 0.08) & (u < 0.12)] *= -0.01
        qtr[(u >= 0.12) & (u < 0.16)] *= 1e-25
    dpdry = np.zeros((L, pcols))
    n = int(lengath)
    idx = o["ideep"][:n] - 1
    dpdry[:, :n] = pdeldry[:, idx] / 100.0
    dq = np.full((ncnst, L, pcols), 7.25)
    m.ns["convtran"](1, F.FArr((ncnst,), dtype=int, data=np.array(do)), F3(qtr), ncnst, FA(o["mu"]), FA(o["md"]),
                     FA(o["du"]), FA(o["eu"]), FA(o["ed"]), FA(o["dp"]), FA(o["dsubcld"]), FA(o["jt"], int),
                     FA(o["maxg"], int), FA(o["ideep"], int), 1, int(lengath), 0, F3(fracis), F3(dq), FA(dpdry),
                     float(ch.ztodt))
    fx.update(convtran_in_q=qtr, convtran_in_fracis=fracis, convtran_in_dpdry=dpdry,
              convtran_in_doconvtran=np.array(do, np.int32), convtran_in_is_dry=np.array(dry, np.int32),
              convtran_dqdt=dq)
    path = os.path.join(HERE, "reftext_%s.npz" % name)
    np.savez_compressed(path, **fx)
    print("%-22s ncol %2d  lengath %2d  prec mean %.3e  -> %s (%d KB)" %
          (name, ncol, int(lengath), float(o["prec"].mean()), os.path.basename(path), os.path.getsize(path) // 1024))


def run_geopotential():
    """geopotential_t (physics/geopotential.F90:153, SURVEY N4) for the FV ('LR') and the Eulerian branch."""
    pcols, L = 16, 32
    F.FArr.UNDEFINED = np.nan
    ch = S.make_chunks(13, L, pcols, p_conv=0.5, col0=7000)
    c = physconst()
    fx = {}
    for lr in (1, 0):
        m = F.Module(os.path.join(PHYSICS, "geopotential.F90"),
                     dict(pcols=pcols, pver=L, pverp=L + 1, dycore_is=(lambda s, lr=lr: s == "LR" if lr else s == "EUL")),
                     lenient=True)       # the MPAS/SE branch uses module data that is not in scope: kept as run-time stops
        m.load("geopotential_t")
        pint, pmid, pdel, t, q = (np.ascontiguousarray(getattr(ch, k)[0]) for k in ("pint", "pmid", "pdel", "t", "q"))
        piln, pmln, rpdel = np.log(pint), np.log(pmid), 1.0 / pdel
        rair = np.full((L, pcols), c["rair"]); zvir = np.full((L, pcols), c["zvir"])
        zi, zm = np.zeros((L + 1, pcols)), np.zeros((L, pcols))
        q3 = q[None]                                            # (pcols,pver,1)
        m.ns["geopotential_t"](FA(piln), FA(pmln), FA(pint), FA(pmid), FA(pdel), FA(rpdel), FA(t),
                               F.FArr(q3.T.shape, data=q3.T), FA(rair), c["gravit"], FA(zvir), FA(zi), FA(zm), 13)
        fx.update({"in_piln": piln, "in_pint": pint, "in_pmid": pmid, "in_pdel": pdel, "in_rpdel": rpdel, "in_t": t,
                   "in_q": q, "in_rair": rair, "in_zvir": zvir, "gravit": np.asarray(c["gravit"]), "ncol": np.asarray(13),
                   "zi_lr%d" % lr: zi, "zm_lr%d" % lr: zm})
    path = os.path.join(HERE, "reftext_geopotential_t.npz")
    np.savez_compressed(path, **fx)
    print("geopotential_t -> %s (%d KB)" % (os.path.basename(path), os.path.getsize(path) // 1024))


def run_geopotential_gen():
    """geopotential_t, generalized-virtual-temperature branch (physics/geopotential.F90:248-310): dycore 'SE' (EUL-type
    hydrostatic elements) and, for the inner LR test of the same branch (:283-287), a dycore that answers true to
    both 'SE' and 'LR'.  thermodynamic_active_species_num / _idx come from air_composition, which is not in the
    reference tree: supplied here (water vapour + two condensates out of five constituents)."""
    pcols, L, ncnst = 16, 32, 5
    species = np.array([1, 2, 4], np.int32)
    F.FArr.UNDEFINED = np.nan
    ch = S.make_chunks(13, L, pcols, p_conv=0.5, col0=7000)
    c = physconst()
    fx = {}
    pint, pmid, pdel, t, q = (np.ascontiguousarray(getattr(ch, k)[0]) for k in ("pint", "pmid", "pdel", "t", "q"))
    rng = np.random.default_rng(20261019)
    q3 = np.zeros((ncnst, L, pcols))
    q3[0] = q
    q3[1] = 2e-4 * rng.random((L, pcols)) * (pmid > 4e4)           # cloud liquid
    q3[2] = 1e-6 * rng.random((L, pcols))                           # not thermodynamically active
    q3[3] = 1e-4 * rng.random((L, pcols)) * (pmid < 6e4)           # cloud ice
    q3[4] = 1e-9 * rng.random((L, pcols))
    for lr in (0, 1):
        names = ("SE", "LR") if lr else ("SE",)
        sp = F.FArr((len(species),), data=species.astype(np.int64)) if hasattr(F, "FArr") else species
        m = F.Module(os.path.join(PHYSICS, "geopotential.F90"),
                     dict(pcols=pcols, pver=L, pverp=L + 1, dycore_is=(lambda s, names=names: s in names),
                          thermodynamic_active_species_num=len(species), thermodynamic_active_species_idx=sp),
                     lenient=True)
        m.load("geopotential_t")
        piln, pmln, rpdel = np.log(pint), np.log(pmid), 1.0 / pdel
        rair = np.full((L, pcols), c["rair"]); zvir = np.full((L, pcols), c["zvir"])
        zi, zm = np.zeros((L + 1, pcols)), np.zeros((L, pcols))
        m.ns["geopotential_t"](FA(piln), FA(pmln), FA(pint), FA(pmid), FA(pdel), FA(rpdel), FA(t),
                               F.FArr(q3.T.shape, data=np.ascontiguousarray(q3.T)), FA(rair), c["gravit"], FA(zvir),
                               FA(zi), FA(zm), 13)
        fx.update({"in_piln": piln, "in_pint": pint, "in_pmid": pmid, "in_pdel": pdel, "in_rpdel": rpdel, "in_t": t,
                   "in_q3": q3, "in_rair": rair, "in_zvir": zvir, "gravit": np.asarray(c["gravit"]), "ncol": np.asarray(13),
                   "species_idx": species, "zi_lr%d" % lr: zi, "zm_lr%d" % lr: zm})
    path = os.path.join(HERE, "reftext_geopotential_t_gen.npz")
    np.savez_compressed(path, **fx)
    print("geopotential_t (generalized Tv) -> %s (%d KB)" % (os.path.basename(path), os.path.getsize(path) // 1024))


def run_convect_diagnostics():
    """convect_diagnostics_calc (physics/convect_diagnostics.F90:115-249, SURVEY N4), shallow_scheme = 'CLUBB_SGS'.
    The physics buffer is a dict of FArr; pbuf_get_field / pbuf_set_field are two-line shims."""
    pcols, L, ncol = 16, 32, 14
    F.FArr.UNDEFINED = np.nan
    rng = np.random.default_rng(23)
    ch = S.make_chunks(ncol, L, pcols, p_conv=0.5, col0=8000)
    names = ["icwmrsh", "rprddp", "rprdsh", "nevapr_shcu", "cldtop", "cldbot", "prec_sh", "snow_sh", "cmfmc_sh", "rprdtot"]
    idx = {n + "_idx": i for i, n in enumerate(names)}
    arr2 = lambda n=L: rng.uniform(0.0, 1.0e-3, (n, pcols))      # noqa: E731
    pb = {"icwmrsh": arr2(), "rprddp": arr2(), "rprdsh": arr2(), "nevapr_shcu": arr2(),
          "cldtop": np.floor(rng.uniform(3, L - 4, pcols)), "cldbot": np.floor(rng.uniform(L - 6, L + 1, pcols)),
          "prec_sh": rng.uniform(0, 1e-7, pcols), "snow_sh": rng.uniform(0, 1e-8, pcols), "cmfmc_sh": arr2(L + 1),
          "rprdtot": np.zeros((L, pcols))}
    pb["cldbot"][::5] = 1.0                                       # exercises `if (cnb == 1) cnb = cnt`
    fx = {"pb_in_" + k: v.copy() for k, v in pb.items()}
    pbuf = {idx[k + "_idx"]: FA(v) for k, v in pb.items()}

    hist = {}

    def pbuf_get_field(pbuf, i, ptr=None):
        return (pbuf[i],)

    def outfld(name, field, idim, lchnk):
        hist[name] = np.array(field.a, copy=True)

    def pbuf_set_field(pbuf, i, val, start=None, kount=None):
        a = pbuf[i]
        a.a[start[0] - 1:start[0] - 1 + kount[0], start[1] - 1:start[1] - 1 + kount[1]] = val

    ns = dict(idx)
    ns.update(pcols=pcols, pver=L, pverp=L + 1, shallow_scheme="CLUBB_SGS", pbuf_get_field=pbuf_get_field,
              pbuf_set_field=pbuf_set_field, outfld=outfld, _OUTS={"pbuf_get_field": [2]})
    m = F.Module(os.path.join(PHYSICS, "convect_diagnostics.F90"), ns, lenient=True)
    m.load("convect_diagnostics_calc")
    state = F.FStruct()
    state.lchnk, state.ncol = 1, ncol
    pmid = np.ascontiguousarray(ch.pmid[0])
    state.pmid = FA(pmid)
    cmfmc, qc, rliq = arr2(L + 1), arr2(), rng.uniform(0, 1e-7, pcols)
    qc2, rliq2 = np.ones((L, pcols)), np.ones(pcols)
    fx.update(in_cmfmc=cmfmc.copy(), in_qc=qc.copy(), in_rliq=rliq.copy(), in_pmid=pmid, ncol=np.asarray(ncol))
    m.ns["convect_diagnostics_calc"](1800.0, FA(cmfmc), FA(qc), FA(qc2), FA(rliq), FA(rliq2), state, pbuf)
    fx.update(out_cmfmc=cmfmc, out_qc=qc, out_qc2=qc2, out_rliq=rliq, out_rliq2=rliq2,
              out_pcnt=hist["PCLDTOP"], out_pcnb=hist["PCLDBOT"])
    fx.update({"pb_out_" + k: v for k, v in pb.items()})
    path = os.path.join(HERE, "reftext_convect_diagnostics.npz")
    np.savez_compressed(path, **fx)
    print("convect_diagnostics_calc -> %s (%d KB)" % (os.path.basename(path), os.path.getsize(path) // 1024))


def run_sweep(nchunks=32, col0=20000, p_conv=0.5):
    """zm_convr of the reference text over many chunks of mixed soundings (default namelist): broad branch coverage.
    Inputs are NOT stored -- they are soundings.make_chunks(16*nchunks, 32, 16, p_conv, col0=col0), seeded."""
    pcols, L = 16, 32
    F.FArr.UNDEFINED = np.nan
    ch = S.make_chunks(pcols * nchunks - 5, L, pcols, p_conv=p_conv, col0=col0)     # last chunk ragged
    m, c = build_module(pcols, L)
    m.ns["zm_convi"](S.limcnv_for(L), 0.0075, 0.03, 5.0e-6, 1.0e-5, 0.7, 0.7, 1, False, False, False, 0.5, 70.0, -1.0e-3,
                     False, 3600.0)
    keys2 = ["qtnd", "heat", "cme", "eurt", "dlf", "zdu", "rprd", "mu", "md", "du", "eu", "ed", "dp", "ql", "dif", "dnlf",
             "dnif"]
    keys2p = ["mcon", "pflx"]
    keys1 = ["prec", "jctop", "jcbot", "cape", "dsubcld", "rliq", "rice"]
    keysi = ["jt", "maxg", "ideep"]
    out = {k: np.zeros((nchunks, L, pcols)) for k in keys2}
    out.update({k: np.zeros((nchunks, L + 1, pcols)) for k in keys2p})
    out.update({k: np.zeros((nchunks, pcols)) for k in keys1})
    out.update({k: np.zeros((nchunks, pcols), np.int64) for k in keysi})
    out["lengath"] = np.zeros(nchunks, np.int64)
    for cc in range(nchunks):
        I = lambda k: FA(np.ascontiguousarray(getattr(ch, k)[cc]))       # noqa: E731
        A = lambda k, dt=float: FA(out[k][cc], dt)                        # noqa: E731
        out["lengath"][cc], = m.ns["zm_convr"](
            cc + 1, int(ch.ncol[cc]), I("t"), I("q"), A("prec"), A("jctop"), A("jcbot"), I("pblh"), I("zm"), I("phis"),
            I("zi"), A("qtnd"), A("heat"), I("pmid"), I("pint"), I("pdel"), 0.5 * float(ch.ztodt), A("mcon"), A("cme"),
            A("cape"), A("eurt"), I("tpert"), A("dlf"), A("pflx"), A("zdu"), A("rprd"), A("mu"), A("md"), A("du"),
            A("eu"), A("ed"), A("dp"), A("dsubcld"), A("jt", int), A("maxg", int), A("ideep", int), None, A("ql"),
            A("rliq"), I("landfrac"), None, None, None, A("dif"), A("dnlf"), A("dnif"), F.FStruct(), F.FStruct(),
            A("rice"))
    fx = {"convr_" + k: v for k, v in out.items()}
    fx.update(nchunks=np.asarray(nchunks), col0=np.asarray(col0), p_conv=np.asarray(p_conv),
              ncols=np.asarray(pcols * nchunks - 5))
    path = os.path.join(HERE, "reftext_sweep_L32.npz")
    np.savez_compressed(path, **fx)
    print("sweep: %d chunks, %d convective columns -> %s (%d KB)" %
          (nchunks, int(out["lengath"].sum()), os.path.basename(path), os.path.getsize(path) // 1024))


def _st_cold(inp, c):
    inp["t"] -= 14.0
    inp["q"] *= 0.42


def _st_near_saturated(inp, c):
    L, pc = inp["t"].shape
    for k in range(L):
        for i in range(pc):
            if inp["pmid"][k, i] > 3.0e4:
                e = gg_water(inp["t"][k, i])
                qs = c["epsilo"] * e / (inp["pmid"][k, i] - (1.0 - c["epsilo"]) * e)
                inp["q"][k, i] = 0.97 * qs


def _st_low_pbl_big_tpert(inp, c):
    inp["pblh"][:] = 60.0
    inp["tpert"][:] = 3.0


def _st_high_pbl(inp, c):
    inp["pblh"][:] = 3500.0
    inp["landfrac"][:] = np.linspace(0.0, 1.0, inp["landfrac"].size)


def _pick_columns(inp, cols, col0=20000, p_conv=0.1):
    """Replace the chunk by hand-picked columns of the seeded generator (column j <- global column col0 + cols[j])."""
    L = inp["t"].shape[0]
    for j, idx in enumerate(cols):
        one = S.make_chunks(1, L, 1, p_conv=p_conv, col0=col0 + idx)
        for k in inp:
            inp[k][..., j] = getattr(one, k)[0][..., 0]


# cam3: columns 969, 4568, 8331, 18573, 20141 (+20000) have an undilute CAPE of 10-24 J/kg (below capelmt) and a dilute
# CAPE of 0 -- they show what the second buoyan_dilute call (zm_conv.F90:1080-1091, all ncol columns) does to columns
# outside the first gather, and that a chunk without any first-gather column returns before it (zm_conv.F90:917).
def _st_cam3_partial(inp, c):
    _pick_columns(inp, [969, 8, 4568, 22, 0, 8331, 24, 1, 18573, 28, 20141, 36, 2, 37, 3, 39])


def _st_cam3_idle(inp, c):
    _pick_columns(inp, [969, 0, 4568, 1, 8331, 2, 18573, 3, 20141, 4, 5, 6, 7, 9, 10, 11])


STRESS = {"cam3_partial": _st_cam3_partial, "cam3_idle": _st_cam3_idle, "cold": _st_cold, "near_saturated": _st_near_saturated, "low_pbl_big_tpert": _st_low_pbl_big_tpert,
          "high_pbl": _st_high_pbl}

CASES = [
    dict(name="config1_L32", ncols=16, pver=32, p_conv=1.0, nl={}),
    dict(name="mixed_ragged_L32", ncols=11, pver=32, p_conv=0.5, nl={}, col0=4000),
    dict(name="parcel_pbl_L58", ncols=16, pver=58, p_conv=0.7, nl={"lparcel_pbl": True}, col0=900),
    dict(name="num_cin3_L32", ncols=16, pver=32, p_conv=0.7, nl={"num_cin": 3}, col0=1700),
    dict(name="no_deep_pbl_L32", ncols=16, pver=32, p_conv=0.7, nl={"no_deep_pbl": True}, col0=2500),
    dict(name="not_master_L32", ncols=16, pver=32, p_conv=0.7, nl={"masterproc": False, "dmpdz": -0.5e-3}, col0=3300),
    dict(name="zm_org_L32", ncols=16, pver=32, p_conv=0.7, nl={}, org=True, col0=5100),
    dict(name="cam3_L32", ncols=16, pver=32, p_conv=0.7, nl={"num_cin": 5}, cam3=True, col0=6000),
    dict(name="parcel_pbl_numcin5_L32", ncols=16, pver=32, p_conv=0.9,
         nl={"lparcel_pbl": True, "num_cin": 5, "tiedke_add": 0.0, "capelmt": 30.0}, col0=9100),
    dict(name="pcols24_L26", ncols=19, pver=26, p_conv=0.8, nl={}, col0=9900, pcols=24),
    dict(name="single_column_L32", ncols=1, pver=32, p_conv=1.0, nl={}, col0=10700),
    dict(name="strong_entrainment_L32", ncols=16, pver=32, p_conv=1.0,
         nl={"dmpdz": -2.5e-3, "tau": 1800.0, "c0_lnd": 0.0059, "c0_ocn": 0.045, "ke": 1.0e-6, "momcu": 0.4,
             "momcd": 0.4}, col0=11500, tracer_edge=True),
    dict(name="cam3_partial_second_pass_L32", ncols=16, pver=32, p_conv=0.1, nl={"num_cin": 5}, cam3=True, col0=20000,
         transform="cam3_partial"),
    dict(name="cam3_idle_chunk_L32", ncols=16, pver=32, p_conv=0.1, nl={"num_cin": 5}, cam3=True, col0=20000,
         transform="cam3_idle"),
    dict(name="stress_cold_L32", ncols=16, pver=32, p_conv=1.0, nl={}, col0=12300, transform="cold"),
    dict(name="stress_near_saturated_L32", ncols=16, pver=32, p_conv=1.0, nl={}, col0=13100, transform="near_saturated"),
    dict(name="stress_low_pbl_L32", ncols=16, pver=32, p_conv=1.0, nl={}, col0=13900, transform="low_pbl_big_tpert"),
    dict(name="stress_high_pbl_L32", ncols=16, pver=32, p_conv=1.0, nl={"lparcel_pbl": True}, col0=14700,
         transform="high_pbl"),
]

if __name__ == "__main__":
    only = sys.argv[1:]
    for cs in CASES:
        if only and cs["name"] not in only:
            continue
        run_case(**cs)
    if not only or "geopotential_t" in only:
        run_geopotential()
    if not only or "geopotential_t_gen" in only:
        run_geopotential_gen()
    if not only or "convect_diagnostics" in only:
        run_convect_diagnostics()
    if not only or "sweep" in only:
        run_sweep()
