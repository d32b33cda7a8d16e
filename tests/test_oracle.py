"""CPU tests of the oracle: golden vectors, property tests derived from the reference code
(SURVEY.md section 4), agreement of the two math flavours, error conventions."""
import os
import numpy as np
import pytest

from cam_nor_physics_b200 import soundings as S
from helpers import (get_oracle, state_of, assert_same, TEND_KEYS, CONVR_KEYS, masked, dpdry_gathered,
                     near_threshold_columns, RTOL, ATOL, REFTEXT_CASES, REFTEXT_CONVR, reftext_overrides)

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


class _Ch:
    """Rebuilds a soundings.Chunks-like object from a golden file."""
    def __init__(self, g):
        for k in ["t", "q", "u", "v", "pmid", "pint", "pdel", "zm", "zi", "phis", "pblh", "tpert", "landfrac", "cld"]:
            setattr(self, k, g["in_" + k])
        self.ncol = g["in_ncol"]; self.ztodt = float(g["in_ztodt"])
        self.nchunks = self.t.shape[0]; self.pver = self.t.shape[1]; self.pcols = self.t.shape[2]
        self.ncols_total = int(self.ncol.sum())


@pytest.mark.parametrize("name", ["config1_L32_pcols16", "mixed4_L32_pcols16"])
@pytest.mark.parametrize("math", ["libm", "pm"])
def test_oracle_matches_golden(built, name, math):
    g = np.load(os.path.join(GOLD, name + ".npz"))
    ch = _Ch(g)
    o, p, rc = get_oracle(math, 16, 32)
    assert rc == 0
    out = o.conv_tend_batch(ch)
    assert out["rc"] == 0
    ref = {k[5:]: g[k] for k in g.files if k.startswith("tend_")}
    # integer outputs exact; reals within the BASELINE tolerance (libm flavour reproduces bit for bit
    # on the same glibc; the portable-math flavour differs by <= 1 ulp per transcendental)
    assert_same(out, ref, TEND_KEYS, 16, exact=False, what=f"oracle[{math}] vs golden {name}")
    cv = o.convr_batch(ch)
    refc = {k[6:]: g[k] for k in g.files if k.startswith("convr_")}
    assert_same(cv, refc, CONVR_KEYS, 16, exact=False, what=f"oracle[{math}] convr vs golden {name}")
    dq = np.stack([o.convtran(g["in_doconvtran"], g["in_tracers"][c], ref["mu"][c], ref["md"][c], ref["du"][c],
                              ref["eu"][c], ref["ed"][c], ref["dp"][c], ref["dsubcld"][c], ref["jt"][c],
                              ref["maxg"][c], ref["ideep"][c], ref["lengath"][c], g["in_fracis"][c],
                              g["in_dpdry"][c], ch.ztodt, g["in_cnst_is_dry"]) for c in range(ch.nchunks)])
    assert np.allclose(dq, g["convtran_dqdt"], rtol=RTOL, atol=1e-30)


def test_math_flavours_agree(built):
    """oracle(glibc libm) vs oracle(portable zm_math.h): ints exact, reals within 1e-10 rel / 1e-14 abs."""
    ch = S.make_chunks(16 * 40, 32, 16, p_conv=0.6)
    a, _, _ = get_oracle("libm", 16, 32)
    b, _, _ = get_oracle("pm", 16, 32)
    ra, rb = a.conv_tend_batch(ch), b.conv_tend_batch(ch)
    assert ra["rc"] == 0 and rb["rc"] == 0
    assert len(near_threshold_columns(ra["cape"])) == 0
    assert_same(rb, ra, TEND_KEYS, 16, exact=False, what="pm vs libm")


def test_inverse_identities(oracle_libm):
    """ienthalpy(enthalpy(T)) ~ T and ientropy(entropy(T)) ~ T within Brent's tol (zm_conv.F90:5027-5028,5342)."""
    o = oracle_libm
    rng = np.random.default_rng(3)
    for _ in range(200):
        T = rng.uniform(200.0, 310.0); p = rng.uniform(150.0, 1000.0); q = rng.uniform(1e-5, 0.02); z = rng.uniform(0, 1.5e4)
        tfg = T + rng.uniform(-5, 5)
        rc, t1, qs1 = o.ientropy(o.entropy(T, p, q), p, q, tfg)
        assert rc == 0 and abs(t1 - T) < 2e-3
        rc, t2, qs2 = o.ienthalpy(o.enthalpy(T, p, q, z), p, z, q, tfg)
        assert rc == 0 and abs(t2 - T) < 2e-3
        es, qs = o.qsat_hpa(t2, p)
        assert qs == qs2            # T is a point where F was evaluated: qst is qsat_hPa(T,p)


def test_water_closure_and_zero_rows(oracle_libm):
    """prec = max(0, -sum dpp*dq - sum dpp*dlf*2dt)/(g*2dt*1000) (zm_conv.F90:1629-1638) =>
    sum dpp*(qtnd+dlf)/g + 1000*prec = 0 when unclipped; rows above jt are exactly zero."""
    o = oracle_libm
    ch = S.make_chunks(16 * 20, 32, 16, p_conv=0.8)
    r = o.convr_batch(ch)
    g = o.params.gravit
    col = (ch.pdel * (r["qtnd"] + r["dlf"])).sum(axis=1) / g + 1000.0 * r["prec"]
    conv = r["prec"] > 0
    assert conv.sum() > 50
    assert np.all(np.abs(col[conv]) <= 1e-10 * 1000.0 * r["prec"][conv] + 1e-18)
    for c in range(ch.nchunks):
        for gi in range(int(r["lengath"][c])):
            i = r["ideep"][c, gi] - 1
            jt, mx = r["jt"][c, gi], r["maxg"][c, gi]
            assert np.all(r["qtnd"][c, : jt - 1, i] == 0.0) and np.all(r["heat"][c, : jt - 1, i] == 0.0)
            assert np.all(r["mu"][c, :jt, gi] == 0.0)          # mu(jt) = 0 (zm_conv.F90:3640-3644)
            assert r["jctop"][c, i] == jt and r["jcbot"][c, i] == mx
            # below the launch level tendencies repeat the launch-level value (zm_conv.F90:4413-4416)
            assert np.all(r["qtnd"][c, mx - 1:, i] == r["qtnd"][c, mx - 1, i])
    # ideep is strictly increasing over 1..lengath and zero beyond (zm_conv.F90:906-915)
    for c in range(ch.nchunks):
        n = int(r["lengath"][c])
        assert np.all(np.diff(r["ideep"][c, :n]) > 0) and np.all(r["ideep"][c, n:] == 0)


def test_no_convection_defaults(oracle_libm):
    """lengath = 0 => all tendencies 0, jctop = pver, jcbot = 1 (zm_conv.F90:559-563, 781-782, 917)."""
    o = oracle_libm
    ch = S.make_chunks(32, 32, 16, p_conv=0.0)
    r = o.convr_batch(ch)
    assert r["lengath"].sum() == 0 and np.all(r["ideep"] == 0)
    for k in ["qtnd", "heat", "mcon", "dlf", "pflx", "cme", "rprd", "zdu", "ql", "prec", "rliq", "eurt"]:
        assert np.all(r[k] == 0.0), k
    assert np.all(r["jctop"] == 32) and np.all(r["jcbot"] == 1)


def test_transport_zero_outside_cloud(oracle_libm):
    """convtran / momtran give exactly 0 tendency above jt and below mx (zm_conv.F90:2249-2252)."""
    o = oracle_libm
    ch = S.make_chunks(64, 32, 16, p_conv=0.7)
    r = o.conv_tend_batch(ch)
    q, fracis, pdeldry = S.make_tracers(ch, 4)
    dpdry = dpdry_gathered(ch, r, pdeldry)
    for c in range(ch.nchunks):
        dq = o.convtran([0, 1, 1, 1], q[c], r["mu"][c], r["md"][c], r["du"][c], r["eu"][c], r["ed"][c], r["dp"][c],
                        r["dsubcld"][c], r["jt"][c], r["maxg"][c], r["ideep"][c], r["lengath"][c], fracis[c],
                        dpdry[c], ch.ztodt, [0, 0, 1, 0])
        assert np.all(dq[0] == 0.0)                       # constituent 1 is never transported (m = 2, ncnst)
        for gi in range(int(r["lengath"][c])):
            i = r["ideep"][c, gi] - 1
            jt, mx = r["jt"][c, gi], r["maxg"][c, gi]
            assert np.all(dq[1:, : jt - 1, i] == 0.0) and np.all(dq[1:, mx:, i] == 0.0)
            assert np.any(dq[1:, jt - 1: mx, i] != 0.0)
        nonconv = np.setdiff1d(np.arange(16), r["ideep"][c][: r["lengath"][c]] - 1)
        assert np.all(dq[:, :, nonconv] == 0.0)
        assert np.all(r["ptend_u"][c][:, nonconv] == 0.0)


def test_zm_convi_error_conventions(built):
    _, _, rc = get_oracle("libm", 16, 32, num_cin=6)
    assert rc != 0                                        # endrun: NUM_CIN must not exceed 5 (zm_conv.F90:200)
    _, _, rc = get_oracle("libm", 16, 32, microp=1)
    assert rc != 0                                        # zmconv_microp is out of scope
    get_oracle("libm", 16, 32)


def test_brent_failure_is_reported(built):
    """Non-convergence is fatal in the reference (zm_conv.F90:5401-5410): the oracle returns a count."""
    o, _, _ = get_oracle("libm", 16, 32)
    rc, t, qs = o.ientropy(250.0, 900.0, 0.01, float("nan"))   # NaN first guess never converges
    assert rc == 1


def test_geopotential_reproduces_the_input_heights(oracle_libm):
    """soundings.py builds zm/zi with the FV branch of geopotential_t (geopotential.F90:218-247); the oracle's
    restatement must give the same heights from the same t,q,p (operation order differs only in rog*tv)."""
    o = oracle_libm
    ch = S.make_chunks(32, 32, 16, p_conv=0.5)
    zvir = np.full_like(ch.t, S.ZVIR); rair = np.full_like(ch.t, S.RAIR)
    for c in range(ch.nchunks):
        zi, zm = o.geopotential_t(16, True, np.log(ch.pint[c]), ch.pint[c], ch.pmid[c], ch.pdel[c], 1.0 / ch.pdel[c],
                                  ch.t[c], ch.q[c], rair[c], S.GRAVIT, zvir[c])
        assert np.allclose(zi, ch.zi[c], rtol=1e-12, atol=1e-9) and np.allclose(zm, ch.zm[c], rtol=1e-12, atol=1e-9)
        assert np.all(zi[-1] == 0.0)


def test_zm_org_branches_oracle():
    """zmconv_org (SURVEY N3; zm_conv.F90:555-556, 793-819, 5066-5074, 1860-1864; zm_conv_intr.F90:773-777).
    org = 0 with all-ocean/all-land columns reproduces the zm_org = .false. zm_convr bit for bit; a positive
    organisation reduces the test-parcel entrainment, so CAPE can only grow; org2d is the pressure-weighted mean
    over org > 0; the tendency relaxes org toward min(1, 5e7 |evapcdp| - org/10800)."""
    o0, _, _ = get_oracle("pm", 16, 32)
    ch = S.make_chunks(640, 32, 16, p_conv=0.6)
    ch.landfrac[:] = np.round(ch.landfrac)
    base = o0.convr_batch(ch)
    o1, p1, rc = get_oracle("pm", 16, 32, zm_org=1)
    assert rc == 0
    zero = np.zeros_like(ch.t)
    r0 = o1.convr_batch(ch, org=zero)
    for k in CONVR_KEYS:
        assert np.array_equal(masked(r0, k, r0["lengath"], 16) if k in ("mu", "md", "du", "eu", "ed", "dp", "dsubcld", "jt", "maxg")
                              else r0[k], masked(base, k, base["lengath"], 16) if k in ("mu", "md", "du", "eu", "ed", "dp", "dsubcld", "jt", "maxg")
                              else base[k]), k
    assert np.all(r0["orgt"] == 0.0) and np.all(r0["org2d"] == 0.0)
    rng = np.random.default_rng(11)
    org = np.maximum(rng.uniform(-0.3, 1.0, ch.t.shape), 0.0)      # the tracer lives in [0, 1]; ~23 % exact zeros
    r1 = o1.convr_batch(ch, org=org)
    assert np.all(r1["orgt"] == 0.0)
    # org2d: weighted mean over org > 0
    w = np.where(org > 0, ch.pdel, 0.0)
    mean = (w * org).sum(axis=1) / np.maximum(w.sum(axis=1), 1e-300)
    assert np.allclose(r1["org2d"], np.repeat(mean[:, None, :], 32, axis=1), rtol=1e-13)
    # less entrainment where org > 0 cannot lower the trigger count by much; CAPE of triggered columns grows
    assert r1["lengath"].sum() >= base["lengath"].sum()
    t1 = o1.conv_tend_batch(ch, org=org)
    assert t1["rc"] == 0
    tgt = np.minimum(1.0, np.maximum(0.0, 5e7 * np.abs(t1["evapcdp"]) - org / 10800.0))
    assert np.allclose(t1["orgt"], (tgt - org) / ch.ztodt, rtol=1e-13, atol=1e-18)


@pytest.mark.parametrize("case", REFTEXT_CASES)
def test_oracle_equals_reference_source_text(case):
    """THE PIN: tests/golden/reftext_*.npz hold what the reference's own Fortran text computes (translated
    statement by statement and executed by tests/golden/fortran_exec.py, see make_reference_fixtures.py) for
    zm_convr (with buoyan_dilute / parcel_dilute / Brent inversions / cldprp / closure / q1q2_pjr inside),
    zm_conv_evap, momtran and convtran.  The oracle built with glibc libm must reproduce every output BIT FOR BIT."""
    g = np.load(os.path.join(GOLD, "reftext_%s.npz" % case))
    pc, L, ncol = int(g["pcols"]), int(g["pver"]), int(g["ncol"])
    o, p, rc = get_oracle("libm", pc, L, **reftext_overrides(g))
    assert rc == 0 and int(g["nl_limcnv"]) == p.limcnv
    ztodt = float(g["ztodt"])

    class Ch:      # one chunk in the layout convr_batch expects
        nchunks, ztodt = 1, float(g["ztodt"])
    ch = Ch()
    ch.ncol = np.array([ncol], np.int32)
    for k in ("t", "q", "pmid", "pint", "pdel", "zm", "zi", "phis", "pblh", "tpert", "landfrac"):
        setattr(ch, k, g["in_" + k][None])
    org = g["in_org"][None] if "in_org" in g.files else None
    r = o.convr_batch(ch, org=org)
    assert r["rc"] == 0
    n = int(g["convr_lengath"])
    assert int(r["lengath"][0]) == n
    bad = []
    for k in REFTEXT_CONVR:
        a, b = r[k][0], g["convr_" + k]
        if k in ("mu", "md", "du", "eu", "ed", "dp", "dsubcld", "jt", "maxg"):
            a, b = a[..., :n], b[..., :n]
        if k in ("jctop", "jcbot", "ideep", "jt", "maxg"):     # defined for i <= ncol / gathered entries
            a, b = a[..., :ncol] if k in ("jctop", "jcbot") else a, b[..., :ncol] if k in ("jctop", "jcbot") else b
        if not np.array_equal(np.asarray(a, float), np.asarray(b, float)):
            bad.append(k)
    if org is not None:
        assert np.array_equal(r["orgt"][0], g["convr_orgt"]) and np.array_equal(r["org2d"][0][:, :ncol], g["convr_org2d"][:, :ncol])
    assert not bad, "zm_convr outputs differ from the reference text: %s" % bad
    # zm_conv_evap
    ev = o.conv_evap(ncol, g["evap_in_t"], g["in_pmid"], g["in_pdel"], g["evap_in_q"], g["in_landfrac"],
                     g["convr_rprd"], g["in_cld"], ztodt, g["convr_prec"])
    for k in ("tend_s", "tend_s_snwprd", "tend_s_snwevmlt", "tend_q", "prec", "snow", "ntprprd", "ntsnprd", "flxprec",
              "flxsnow"):
        assert np.array_equal(ev[k][..., :ncol], g["evap_" + k][..., :ncol]), ("zm_conv_evap", k)
    # momtran
    winds = np.stack([g["in_u"], g["in_v"]], axis=0)
    mo = o.momtran(ncol, [1, 1], winds, g["convr_mu"], g["convr_md"], g["convr_du"], g["convr_eu"], g["convr_ed"],
                   g["convr_dp"], g["convr_dsubcld"], g["convr_jt"], g["convr_maxg"], g["convr_ideep"], n, ztodt)
    for k in ("dqdt", "pguall", "pgdall", "icwu", "icwd", "seten"):
        assert np.array_equal(mo[k][..., :ncol], g["momtran_" + k][..., :ncol]), ("momtran", k)
    # convtran
    do, dry = g["convtran_in_doconvtran"], g["convtran_in_is_dry"]
    dq = o.convtran(do, g["convtran_in_q"], g["convr_mu"], g["convr_md"], g["convr_du"], g["convr_eu"], g["convr_ed"],
                    g["convr_dp"], g["convr_dsubcld"], g["convr_jt"], g["convr_maxg"], g["convr_ideep"], n,
                    g["convtran_in_fracis"], g["convtran_in_dpdry"], ztodt, dry)
    for mth in range(1, len(do)):
        if do[mth]:
            assert np.array_equal(dq[mth], g["convtran_dqdt"][mth]), ("convtran", mth)
        else:
            assert np.all(g["convtran_dqdt"][mth] == 7.25)      # the reference leaves inactive constituents untouched
    # the zm_conv_tend sequence: the oracle's fused driver against the pieces above combined the way zm_conv_intr.F90
    # does (ptend_all = sum of the three ptend_loc, :736/:803/:833), with the glue statements (:693 mcon units,
    # physics_update arithmetic, :773-777 organisation tendency) taken from the reference text as well
    for k in ("u", "v", "cld"):
        setattr(ch, k, g["in_" + k][None])
    tr = o.conv_tend_batch(ch, org=org)
    assert tr["rc"] == 0
    c = slice(0, ncol)
    assert np.array_equal(tr["mcon"][0][:, c], g["tend_mcon"][:, c])
    if bool(g["nl_cam3"]):      # momentum transport is non-cam3 physics (zm_conv_intr.F90:808): no wind tendency, no seten
        assert np.array_equal(tr["ptend_s"][0][:, c], (g["convr_heat"] + g["evap_tend_s"])[:, c])
        assert np.all(tr["ptend_u"][0] == 0.0) and np.all(tr["ptend_v"][0] == 0.0)
    else:
        assert np.array_equal(tr["ptend_s"][0][:, c], ((g["convr_heat"] + g["evap_tend_s"]) + g["momtran_seten"])[:, c])
        assert np.array_equal(tr["ptend_u"][0][:, c], g["momtran_dqdt"][0][:, c])
        assert np.array_equal(tr["ptend_v"][0][:, c], g["momtran_dqdt"][1][:, c])
    assert np.array_equal(tr["ptend_q"][0][:, c], (g["convr_qtnd"] + g["evap_tend_q"])[:, c])
    # convtran1 inside the fused driver (zm_conv_intr.F90:865-880) against the reference text's convtran on the same
    # constituents: fake_dpdry = 0 only differs for 'dry' species, so the fixture's moist ones are compared
    do, dry = np.asarray(g["convtran_in_doconvtran"]), np.asarray(g["convtran_in_is_dry"])
    moist = [int(m) for m in range(1, len(do)) if do[m] and not dry[m]]
    if moist:
        do1 = np.zeros_like(do); do1[moist] = 1
        tr1 = o.conv_tend_batch(ch, org=org, convtran1=dict(doconvtran=do1, cnst_is_dry=np.zeros_like(do),
                                                           q=g["convtran_in_q"][None], fracis=g["convtran_in_fracis"][None]))
        for m in moist:
            assert np.array_equal(tr1["ptend_qc"][0, m], g["convtran_dqdt"][m]), ("convtran1", m)
    for k in ("prec", "snow", "flxprec", "flxsnow"):
        assert np.array_equal(tr[k][0][..., c], g["evap_" + k][..., c]), k
    assert np.array_equal(tr["evapcdp"][0][:, c], g["evap_tend_q"][:, c])
    if org is not None:
        assert np.array_equal(tr["orgt"][0][:, c], g["tend_orgt"][:, c])


def test_oracle_geopotential_t_equals_reference_source_text():
    """geopotential_t (physics/geopotential.F90:153-247, SURVEY N4): reference text executed through the translator."""
    g = np.load(os.path.join(GOLD, "reftext_geopotential_t.npz"))
    o, _, _ = get_oracle("libm", 16, 32)
    for lr in (1, 0):
        zi, zm = o.geopotential_t(int(g["ncol"]), lr, g["in_piln"], g["in_pint"], g["in_pmid"], g["in_pdel"], g["in_rpdel"],
                                  g["in_t"], g["in_q"], g["in_rair"], float(g["gravit"]), g["in_zvir"])
        n = int(g["ncol"])
        assert np.array_equal(zi[:, :n], g["zi_lr%d" % lr][:, :n]) and np.array_equal(zm[:, :n], g["zm_lr%d" % lr][:, :n]), lr


def test_oracle_geopotential_t_generalized_tv_equals_reference_source_text():
    """geopotential_t, generalized-virtual-temperature branch (physics/geopotential.F90:248-310; dycore MPAS / SE), with
    both hydrostatic-element variants of that branch (:283-298): reference text executed through the translator."""
    g = np.load(os.path.join(GOLD, "reftext_geopotential_t_gen.npz"))
    o, _, _ = get_oracle("libm", 16, 32)
    n = int(g["ncol"])
    plain = np.load(os.path.join(GOLD, "reftext_geopotential_t.npz"))
    for lr in (0, 1):
        zi, zm = o.geopotential_t_gen(n, lr, g["in_piln"], g["in_pint"], g["in_pmid"], g["in_pdel"], g["in_rpdel"],
                                      g["in_t"], g["in_q3"], g["in_rair"], float(g["gravit"]), g["in_zvir"],
                                      g["species_idx"])
        assert np.array_equal(zi[:, :n], g["zi_lr%d" % lr][:, :n]) and np.array_equal(zm[:, :n], g["zm_lr%d" % lr][:, :n]), lr
        # the branch is not the plain one in disguise: condensate loading lowers the heights by up to metres
        d = np.abs(zi[:, :n] - plain["zi_lr%d" % lr][:, :n])
        assert 0.1 < d.max() < 50.0
    # no active species: qfac = sum = 1 and the factor is 1 + (zvir+1)*q  (:303)
    zi0, _ = o.geopotential_t_gen(n, 0, g["in_piln"], g["in_pint"], g["in_pmid"], g["in_pdel"], g["in_rpdel"], g["in_t"],
                                  g["in_q3"], g["in_rair"], float(g["gravit"]), g["in_zvir"], np.zeros(0, np.int32))
    assert np.all(zi0[:-1, :n] > g["zi_lr0"][:-1, :n])


def test_oracle_convect_diagnostics_equals_reference_source_text():
    """convect_diagnostics_calc (physics/convect_diagnostics.F90:115-249, SURVEY N4), CLUBB_SGS branch."""
    g = np.load(os.path.join(GOLD, "reftext_convect_diagnostics.npz"))
    o, _, _ = get_oracle("libm", 16, 32)
    n = int(g["ncol"])
    r = o.convect_diagnostics(n, g["in_cmfmc"], g["in_qc"], g["in_rliq"], g["in_pmid"], g["pb_in_rprddp"],
                              g["pb_in_cldtop"], g["pb_in_cldbot"])
    assert np.array_equal(r["cmfmc"][:, :n], g["out_cmfmc"][:, :n]) and np.array_equal(r["qc"][:, :n], g["out_qc"][:, :n])
    assert np.array_equal(r["rliq"][:n], g["out_rliq"][:n])
    assert np.all(r["qc2"] == 0.0) and np.all(g["out_qc2"] == 0.0) and np.all(r["rliq2"] == 0.0)
    assert np.array_equal(r["cnt"][:n], g["pb_out_cldtop"][:n]) and np.array_equal(r["cnb"][:n], g["pb_out_cldbot"][:n])
    assert np.array_equal(r["pcnt"][:n], g["out_pcnt"][:n]) and np.array_equal(r["pcnb"][:n], g["out_pcnb"][:n])
    assert np.array_equal(r["rprdtot"][:, :n], g["pb_out_rprdtot"][:, :n])
    assert np.all(r["cmfmc2"] == 0.0) and np.all(r["rprdsh"] == 0.0)


def test_oracle_equals_reference_source_text_sweep():
    """507 columns of mixed soundings (32 chunks, the last one ragged) through the reference text's zm_convr: the
    glibc-libm oracle must reproduce every output bit for bit (inputs are regenerated from the seeded generator)."""
    g = np.load(os.path.join(GOLD, "reftext_sweep_L32.npz"))
    o, _, _ = get_oracle("libm", 16, 32)
    ch = S.make_chunks(int(g["ncols"]), 32, 16, p_conv=float(g["p_conv"]), col0=int(g["col0"]))
    r = o.convr_batch(ch)
    assert r["rc"] == 0
    assert np.array_equal(r["lengath"], g["convr_lengath"]) and r["lengath"].sum() > 200
    bad = []
    for k in REFTEXT_CONVR:
        a, b = r[k], g["convr_" + k]
        if k in ("mu", "md", "du", "eu", "ed", "dp", "dsubcld", "jt", "maxg"):
            a, b = masked(r, k, g["convr_lengath"], 16), masked({k: b}, k, g["convr_lengath"], 16)
        if k in ("jctop", "jcbot"):
            m = np.arange(16)[None, :] < ch.ncol[:, None]
            a, b = a * m, b * m
        if not np.array_equal(np.asarray(a, float), np.asarray(b, float)):
            bad.append(k)
    assert not bad, bad


@pytest.mark.skipif(not os.path.isfile(os.path.join(os.environ.get("CAM_NOR_SRC", "/nonexistent"), "physics",
                                                    "zm_conv.F90")),
                    reason="executes the reference source text: set CAM_NOR_SRC to a CAM-Nor source tree")
def test_oracle_equals_reference_source_text_random_chunks():
    """A short run of tests/golden/reference_text_fuzz.py: random chunks / namelist values / zm_org / cam3 / perturbed
    soundings through the reference text and the glibc-libm oracle, bit for bit (the 300-case run of round 1 is
    profiles/reference_text_fuzz_r1_*.log)."""
    import subprocess, sys, json
    r = subprocess.run([sys.executable, os.path.join(GOLD, "reference_text_fuzz.py"), "8", "515"],
                       capture_output=True, text=True, timeout=1200)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    s = json.loads(r.stdout.strip().splitlines()[-1])
    assert s["cases"] == 8 and s["oracle_equals_reference_text_bit_for_bit"]
