"""GPU parity tests (run on the B200 box with -m gpu).  Everything goes through the C ABI
(include/zmconv_b200.h) via cam_nor_physics_b200.zm_conv.  The checker is the CPU oracle:
  * oracle built with the same portable math header  -> bit-exact comparison of every output;
  * oracle built with glibc libm / committed golden vectors -> integer outputs exact, r8 outputs within
    1e-10 relative / 1e-14 absolute (BASELINE.json north_star), near-threshold columns reported."""
import os

import numpy as np
import pytest

from cam_nor_physics_b200 import soundings as S
from helpers import (get_oracle, init_cuda, state_of, assert_same, cuda_convr, dpdry_gathered, CONVR_KEYS,
                     TEND_KEYS, near_threshold_columns, REFTEXT_CASES, REFTEXT_CONVR, reftext_overrides, RTOL, ATOL,
                     GATHERED_2D, GATHERED_1D, INT_KEYS)

pytestmark = pytest.mark.gpu
GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def test_portable_math_device_equals_host(built):
    from cam_nor_physics_b200 import zm_conv as Z
    rng = np.random.default_rng(0)
    n = 200000
    for fid, x, y in [(0, np.exp(rng.uniform(-40, 40, n)), None), (1, rng.uniform(0.5, 4, n), None),
                      (2, rng.uniform(-60, 60, n), None), (3, rng.uniform(-9, 9, n), None),
                      (4, rng.uniform(0.3, 50, n), rng.uniform(-3, 3, n))]:
        assert np.array_equal(Z.math_eval(fid, x, y, device=True), Z.math_eval(fid, x, y, device=False)), fid
    # trimmed variants used by the state function (shared-memory tables, no special-case selects, divisions by
    # refined reciprocals) against the GENERAL host functions / IEEE division
    xs = np.concatenate([np.exp(rng.uniform(-700, 700, n)), rng.uniform(0.5, 2.0, n)])
    assert np.array_equal(Z.math_eval(5, xs, device=True), Z.math_eval(0, xs, device=False))
    assert np.array_equal(Z.math_eval(6, xs, device=True), Z.math_eval(1, xs, device=False))
    xp = np.concatenate([rng.uniform(-300, 300, n), rng.uniform(-3, 8, n)])
    assert np.array_equal(Z.math_eval(7, xp, device=True), Z.math_eval(3, xp, device=False))
    a = np.concatenate([rng.uniform(50, 1000, n), np.exp(rng.uniform(-50, 50, n))])
    for b in (373.16, 1000.0, 273.15):
        assert np.array_equal(Z.math_eval(8, a, np.full_like(a, b), device=True), a / b), b
    b = np.exp(rng.uniform(-50, 50, a.size))
    assert np.array_equal(Z.math_eval(9, a, b, device=True), a / b)          # div_hot == IEEE quotient
    # saturation vapour pressure: global-memory and shared-memory table paths, cell edges, formula fallback
    ts = np.concatenate([rng.uniform(100, 400, n), np.arange(139, 352) + 0.5, np.arange(139, 352) + 0.5 - 1e-13,
                         np.arange(139, 352) + 0.5 + 1e-13, np.arange(139, 352) + 0.0])
    host = Z.math_eval(10, ts, device=False)
    assert np.array_equal(Z.math_eval(10, ts, device=True), host)
    assert np.array_equal(Z.math_eval(12, ts, device=True), host)
    assert np.array_equal(Z.math_eval(11, ts, device=True), Z.math_eval(11, ts, device=False))


def test_thermo_scalars_match_oracle(built):
    Z = init_cuda(16, 32)
    o, _, _ = get_oracle("pm", 16, 32)
    rng = np.random.default_rng(5)
    n = 3000
    T = rng.uniform(170, 330, n); p = rng.uniform(60, 1050, n); q = rng.uniform(1e-7, 0.03, n)
    q[::7] = np.exp(rng.uniform(np.log(1e-12), np.log(1e-6), q[::7].size))        # very dry parcels
    z = rng.uniform(0, 1.6e4, n); tfg = T + rng.uniform(-6, 6, n)
    s0, _ = Z.thermo_eval(0, T, p, q)
    h0, _ = Z.thermo_eval(1, T, p, q, z)
    assert np.array_equal(s0, [o.entropy(*a) for a in zip(T, p, q)])
    assert np.array_equal(h0, [o.enthalpy(*a) for a in zip(T, p, q, z)])
    t1, q1 = Z.thermo_eval(2, s0, p, q, tfg)
    ref = [o.ientropy(*a) for a in zip(s0, p, q, tfg)]
    assert np.array_equal(t1, [r[1] for r in ref]) and np.array_equal(q1, [r[2] for r in ref])
    t2, q2 = Z.thermo_eval(3, h0, p, z, q, tfg)
    ref = [o.ienthalpy(*a) for a in zip(h0, p, z, q, tfg)]
    assert np.array_equal(t2, [r[1] for r in ref]) and np.array_equal(q2, [r[2] for r in ref])
    es, qs = Z.thermo_eval(5, T, p * 100.0)
    ref = [o.qsat_table(a, b * 100.0) for a, b in zip(T, p)]
    assert np.array_equal(es, [r[0] for r in ref]) and np.array_equal(qs, [r[1] for r in ref])


@pytest.mark.parametrize("ncols,pconv,pver,over", [
    (16, 1.0, 32, {}),                          # BASELINE config 1: one pcols=16 chunk of tropical soundings
    (4096, 0.5, 32, {}),                        # mixed grid
    (1000, 0.6, 32, {}),                        # ragged: last chunk has 8 of 16 columns
    (320, 0.0, 32, {}),                         # no convection anywhere (lengath = 0 in every chunk)
    (2048, 0.6, 58, {"lparcel_pbl": 1}),        # L58 with the PBL-mixed launch parcel (BASELINE config 5 setup)
    (512, 0.6, 72, {}),                         # > 64 levels: the 128-level instantiation of the plume kernels
    (1024, 0.7, 32, {"num_cin": 3}),            # several negative-buoyancy regions allowed
    (1024, 0.7, 32, {"no_deep_pbl": 1}),
    (1024, 0.7, 32, {"masterproc": 0, "dmpdz": -0.5e-3}),   # tentrm quirk (zm_conv.F90:213)
    (2048, 0.6, 32, {"cam3": 1, "num_cin": 5}),  # cam3: undilute buoyan as first trigger pass (zm_conv.F90:871)
])
def test_zm_convr_bit_exact_vs_oracle(built, ncols, pconv, pver, over):
    Z = init_cuda(16, pver, **over)
    o, _, rc = get_oracle("pm", 16, pver, **over)
    assert rc == 0
    ch = S.make_chunks(ncols, pver, 16, p_conv=pconv)
    ref = o.convr_batch(ch)
    assert ref["rc"] == 0
    out = cuda_convr(Z, ch)
    assert_same(out, ref, CONVR_KEYS, 16, exact=True, what=f"zm_convr {ncols}x{pver} {over}")
    if pconv == 0.0:
        assert out["lengath"].sum() == 0
    else:
        assert out["lengath"].sum() > 0


@pytest.mark.parametrize("pver,pcols,ncols,pconv,seed", [
    (72, 16, 4643, 0.1, 2145566664),     # two columns with a small undilute CAPE (7, 18 J/kg) and a dilute CAPE of 0
    (58, 8, 2926, 0.0, 1233135682),      # a chunk without any first-gather column keeps its undilute CAPE
])
def test_cam3_second_pass_coverage(built, pver, pcols, ncols, pconv, seed):
    """cam3: the first trigger pass is the undilute buoyan, so the dilute second call (zm_conv.F90:1080-1091, all ncol
    columns) changes cape / tp / qstp of columns that did NOT trigger too -- but only in chunks that have a
    convective column after the first gather (zm_conv.F90:917 returns otherwise).  Both found by
    scripts/parity_fuzz.py."""
    over = {"cam3": 1, "num_cin": 5}
    Z = init_cuda(pcols, pver, **over)
    o, _, rc = get_oracle("pm", pcols, pver, **over)
    assert rc == 0
    ch = S.make_chunks(ncols, pver, pcols, p_conv=pconv, seed=seed)
    ref = o.convr_batch(ch)
    out = cuda_convr(Z, ch)
    assert_same(out, ref, CONVR_KEYS, pcols, exact=True, what="cam3 fuzz case")
    init_cuda(16, 32)


def test_large_pcols_chunk(built):
    """pcols = 128 (CAM allows large pcols): compaction spans several warp sweeps."""
    Z = init_cuda(128, 32)
    o, _, _ = get_oracle("pm", 128, 32)
    ch = S.make_chunks(128 * 6 - 37, 32, 128, p_conv=0.5)
    ref = o.convr_batch(ch)
    out = cuda_convr(Z, ch)
    assert_same(out, ref, CONVR_KEYS, 128, exact=True, what="pcols=128")


@pytest.mark.parametrize("name", ["config1_L32_pcols16", "mixed4_L32_pcols16"])
def test_against_golden_vectors(built, name):
    g = np.load(os.path.join(GOLD, name + ".npz"))
    Z = init_cuda(16, 32)
    st = {k[3:]: g[k] for k in g.files if k.startswith("in_") and k[3:] in Z.TEND_IN_ORDER}
    out = Z.zm_conv_tend(g["in_ncol"], st, float(g["in_ztodt"]))
    ref = {k[5:]: g[k] for k in g.files if k.startswith("tend_")}
    assert len(near_threshold_columns(ref["cape"])) == 0
    assert_same(out, ref, TEND_KEYS, 16, exact=False, what=f"CUDA zm_conv_tend vs golden {name}")
    dq = Z.convtran(g["in_doconvtran"], g["in_tracers"], ref["mu"], ref["md"], ref["du"], ref["eu"], ref["ed"],
                    ref["dp"], ref["dsubcld"], ref["jt"], ref["maxg"], ref["ideep"], ref["lengath"],
                    g["in_fracis"], g["in_dpdry"], float(g["in_ztodt"]), g["in_cnst_is_dry"])
    assert np.allclose(dq, g["convtran_dqdt"], rtol=1e-10, atol=1e-30)


def test_evap_momtran_convtran_bit_exact(built):
    Z = init_cuda(16, 32)
    o, p, _ = get_oracle("pm", 16, 32)
    ch = S.make_chunks(1500, 32, 16, p_conv=0.6)
    ref = o.convr_batch(ch)
    nch = ch.nchunks
    t1 = ch.t + ref["heat"] * ch.ztodt / p.cpair
    q1 = np.maximum(ch.q + ref["qtnd"] * ch.ztodt, 1e-12)
    ev = Z.zm_conv_evap(ch.ncol, t1, ch.pmid, ch.pdel, q1, ch.landfrac, ref["rprd"], ch.cld, ch.ztodt, ref["prec"])
    for c in range(nch):
        r = o.conv_evap(int(ch.ncol[c]), t1[c], ch.pmid[c], ch.pdel[c], q1[c], ch.landfrac[c], ref["rprd"][c],
                        ch.cld[c], ch.ztodt, ref["prec"][c])
        n = int(ch.ncol[c])
        for k in r:
            assert np.array_equal(ev[k][c][..., :n], r[k][..., :n]), (c, k)
    winds = np.stack([ch.u, ch.v], axis=1)
    mo = Z.momtran(ch.ncol, [1, 1], winds, ref["mu"], ref["md"], ref["du"], ref["eu"], ref["ed"], ref["dp"],
                   ref["dsubcld"], ref["jt"], ref["maxg"], ref["ideep"], ref["lengath"], ch.ztodt)
    for c in range(nch):
        r = o.momtran(int(ch.ncol[c]), [1, 1], winds[c], ref["mu"][c], ref["md"][c], ref["du"][c], ref["eu"][c],
                      ref["ed"][c], ref["dp"][c], ref["dsubcld"][c], ref["jt"][c], ref["maxg"][c], ref["ideep"][c],
                      ref["lengath"][c], ch.ztodt)
        n = int(ch.ncol[c])
        for k in r:
            assert np.array_equal(mo[k][c][..., :n], r[k][..., :n]), (c, k)
    ncnst = 9
    q, fracis, pdeldry = S.make_tracers(ch, ncnst)
    do = [0, 1, 1, 0, 1, 1, 0, 1, 1]
    dry = [0, 0, 1, 0, 0, 1, 1, 0, 1]
    dpdry = dpdry_gathered(ch, ref, pdeldry)
    sentinel = np.full_like(q, 7.25)
    dq = Z.convtran(do, q, ref["mu"], ref["md"], ref["du"], ref["eu"], ref["ed"], ref["dp"], ref["dsubcld"],
                    ref["jt"], ref["maxg"], ref["ideep"], ref["lengath"], fracis, dpdry, ch.ztodt, dry, dqdt=sentinel)
    for c in range(nch):
        r = o.convtran(do, q[c], ref["mu"][c], ref["md"][c], ref["du"][c], ref["eu"][c], ref["ed"][c], ref["dp"][c],
                       ref["dsubcld"][c], ref["jt"][c], ref["maxg"][c], ref["ideep"][c], ref["lengath"][c],
                       fracis[c], dpdry[c], ch.ztodt, dry)
        for m in range(ncnst):
            if do[m] and m >= 1:
                assert np.array_equal(dq[c, m], r[m]), (c, m)
            else:
                assert np.all(dq[c, m] == 7.25)          # inactive constituents are not touched (zm_conv.F90:2298)
    assert np.count_nonzero(dq[:, 1]) > 0
    # lengath = 0 everywhere: transport returns zeros for active constituents
    zero = np.zeros_like(ref["lengath"])
    dq0 = Z.convtran(do, q, ref["mu"], ref["md"], ref["du"], ref["eu"], ref["ed"], ref["dp"], ref["dsubcld"],
                     ref["jt"], ref["maxg"], ref["ideep"], zero, fracis, dpdry, ch.ztodt, dry)
    assert np.all(dq0 == 0.0)


def test_f09_full_step_vs_oracle(built):
    """BASELINE configs 2-3 at full size: 55,296 columns L32 through zm_conv_tend (convr+evap+momtran)."""
    Z = init_cuda(16, 32)
    o, _, _ = get_oracle("pm", 16, 32)
    ch = S.make_chunks(55296, 32, 16, p_conv=0.35)
    ref = o.conv_tend_batch(ch)
    assert ref["rc"] == 0
    out = Z.zm_conv_tend(ch.ncol, state_of(ch), ch.ztodt)
    assert_same(out, ref, TEND_KEYS, 16, exact=True, what="f09 zm_conv_tend")
    frac = ref["lengath"].sum() / 55296
    assert 0.2 < frac < 0.5
    # and against the glibc-libm flavour (the gfortran-like one): tolerance of the north star
    o2, _, _ = get_oracle("libm", 16, 32)
    ref2 = o2.conv_tend_batch(ch)
    near = near_threshold_columns(ref2["cape"])
    print("near-threshold columns (reported, left out of the comparison):", near.tolist())
    # ptend_s / ptend_q are sums of zm_convr's and zm_conv_evap's tendencies that largely cancel below cloud base:
    # the tolerance is taken against the magnitude of the terms (which are themselves compared against it)
    cv = o2.convr_batch(ch)
    cvo = cuda_convr(Z, ch)
    assert_same(cvo, cv, CONVR_KEYS, 16, exact=False, what="f09 zm_convr vs libm oracle", skip_cols=near,
                scales={"cape": np.full_like(cv["cape"], 70.0)})
    scales = {"ptend_s": np.abs(cv["heat"]) + np.abs(ref2["ptend_s"] - cv["heat"]),
              "ptend_q": np.abs(cv["qtnd"]) + np.abs(ref2["evapcdp"]), "cape": np.full_like(ref2["cape"], 70.0)}
    if not len(near):          # gathered outputs shift when a column enters or leaves ideep
        assert_same(out, ref2, TEND_KEYS, 16, exact=False, what="f09 zm_conv_tend vs libm oracle", scales=scales)
    else:
        keys = [k for k in TEND_KEYS if k not in GATHERED_2D + GATHERED_1D + INT_KEYS]
        assert_same(out, ref2, keys, 16, exact=False, what="f09 zm_conv_tend vs libm oracle", scales=scales,
                    skip_cols=near)


def test_config5_shard_L58_full_step_vs_oracle(built):
    """BASELINE config 5, one GPU's shard at full size (131,072 columns, L58, parcel_pbl, 40 % convective) through
    zm_conv_tend: bit for bit against the portable-math oracle, within the north-star tolerance against the
    glibc-libm one (near-threshold columns reported and left out)."""
    over = dict(lparcel_pbl=1)
    Z = init_cuda(16, 58, **over)
    ch = S.make_chunks(131072, 58, 16, p_conv=0.4)
    out = Z.zm_conv_tend(ch.ncol, state_of(ch), ch.ztodt)
    o, _, _ = get_oracle("pm", 16, 58, **over)
    ref = o.conv_tend_batch(ch)
    assert ref["rc"] == 0
    assert_same(out, ref, TEND_KEYS, 16, exact=True, what="config-5 shard zm_conv_tend")
    assert 0.1 < ref["lengath"].sum() / 131072 < 0.6
    o2, _, _ = get_oracle("libm", 16, 58, **over)
    ref2 = o2.conv_tend_batch(ch)
    near = near_threshold_columns(ref2["cape"])
    print("near-threshold columns (reported, left out of the comparison):", near.tolist())
    cv = o2.convr_batch(ch)
    # cape is a sum of signed buoyancy terms (zm_conv.F90:4785-4796), each of the order of the trigger threshold or
    # larger, that can cancel to a fraction of a J/kg: the tolerance is taken against capelmt, the number it is
    # compared with (zm_conv.F90:908)
    scales = {"ptend_s": np.abs(cv["heat"]) + np.abs(ref2["ptend_s"] - cv["heat"]),
              "ptend_q": np.abs(cv["qtnd"]) + np.abs(ref2["evapcdp"]), "cape": np.full_like(ref2["cape"], 70.0)}
    keys = TEND_KEYS if not len(near) else [k for k in TEND_KEYS if k not in GATHERED_2D + GATHERED_1D + INT_KEYS]
    assert_same(out, ref2, keys, 16, exact=False, what="config-5 shard vs libm oracle", scales=scales,
                skip_cols=near if len(near) else None)


def test_config4_f09_convtran_41_constituents_vs_oracle(built):
    """BASELINE config 4 at full size: the f09 grid with a 41-constituent stand-in for the OsloAero tracer set --
    convtran1 (2 constituents) inside zm_conv_tend and convtran2 (38, every third 'dry') in zm_conv_tend_2 from the
    device pbuf mirror -- bit for bit against the oracle's batch drivers."""
    Z = init_cuda(16, 32)
    o, _, _ = get_oracle("pm", 16, 32)
    ch = S.make_chunks(55296, 32, 16, p_conv=0.35)
    pcnst = 41
    q, fracis, pdeldry = S.make_tracers(ch, pcnst)
    do1 = np.zeros(pcnst, np.int32); do1[1:3] = 1
    do2 = np.zeros(pcnst, np.int32); do2[3:] = 1
    dry = np.zeros(pcnst, np.int32); dry[3::3] = 1
    t1 = dict(doconvtran=do1, cnst_is_dry=dry, q=q, fracis=fracis)
    ref = o.conv_tend_batch(ch, convtran1=t1)
    refq = o.conv_tend_2_batch(do2, q, pdeldry, fracis, ch.ztodt, dry, ref, ptend_q=ref["ptend_qc"])
    out = Z.zm_conv_tend(ch.ncol, state_of(ch), ch.ztodt, keep_pbuf_on_device=True, convtran1=t1)
    dq = Z.zm_conv_tend_2(do2, q, pdeldry, fracis, ch.ztodt, dry, ptend_q=out["ptend_qc"])
    assert np.array_equal(out["ptend_qc"], ref["ptend_qc"])
    assert np.array_equal(dq, refq)
    assert np.count_nonzero(dq[:, 3:]) > 0 and np.count_nonzero(dq[:, 1:3]) > 0 and not dq[:, 0].any()


def test_sharding_invariance_and_properties_L58_large(built):
    """BASELINE config 5 shard (131,072 columns L58, 10-60% convective): size-independent properties --
    chunk partition invariance, water closure, sorted ideep, zero rows outside the cloud."""
    Z = init_cuda(16, 58, lparcel_pbl=1)
    n = 131072
    ch = S.make_chunks(n, 58, 16, p_conv=0.4)
    out = cuda_convr(Z, ch)
    half = n // 2
    a = cuda_convr(Z, S.make_chunks(half, 58, 16, p_conv=0.4))
    b = cuda_convr(Z, S.make_chunks(half, 58, 16, p_conv=0.4, col0=half))
    for k in ["qtnd", "heat", "prec", "ideep", "lengath", "mu", "jt", "cape", "pflx"]:
        assert np.array_equal(np.concatenate([a[k], b[k]]), out[k]), k
    frac = out["lengath"].sum() / n
    assert 0.1 < frac < 0.6
    g = 9.80616
    col = (ch.pdel * (out["qtnd"] + out["dlf"])).sum(axis=1) / g + 1000.0 * out["prec"]
    conv = out["prec"] > 0
    assert np.all(np.abs(col[conv]) <= 1e-10 * 1000.0 * out["prec"][conv] + 1e-18)
    nz = np.arange(16)[None, :] < out["lengath"][:, None]
    srt = np.where(nz, out["ideep"], 1 << 20)
    assert np.all(np.diff(srt, axis=1)[nz[:, 1:]] > 0)
    assert np.all(out["ideep"][~nz] == 0)
    nonconv = np.ones((ch.nchunks, 16), bool)
    ci, gi = np.nonzero(nz)
    nonconv[ci, out["ideep"][ci, gi] - 1] = False
    assert np.all(out["qtnd"].transpose(0, 2, 1)[nonconv] == 0.0)
    assert np.all(out["jctop"][nonconv] == 58) and np.all(out["jcbot"][nonconv] == 1)


def test_error_conventions(built):
    from cam_nor_physics_b200 import zm_conv as Z
    with pytest.raises(Z.ZmEndrun):
        init_cuda(16, 32, num_cin=6)                       # zm_conv.F90:200
    with pytest.raises(Z.ZmError):
        init_cuda(16, 32, microp=1)
    Z = init_cuda(16, 32)
    ch = S.make_chunks(16, 32, 16)
    t = ch.t.copy(); t[0, :, 3] = np.nan                  # NaN sounding -> Brent cannot converge -> endrun
    with pytest.raises(Z.ZmEndrun) as e:
        Z.zm_convr(ch.ncol, t, ch.q, ch.pblh, ch.zm, ch.phis, ch.zi, ch.pmid, ch.pint, ch.pdel, 900.0, ch.tpert, ch.landfrac)
    assert "icol=4" in str(e.value)


def test_device_resident_path_and_conservation(built):
    import torch
    from cam_nor_physics_b200.device import DeviceTend
    Z = init_cuda(16, 32)
    o, _, _ = get_oracle("pm", 16, 32)
    ch = S.make_chunks(4096, 32, 16, p_conv=0.5)
    ref = o.conv_tend_batch(ch)
    dev = DeviceTend(ch)
    dev.step(); cons = dev.conservation(); assert dev.check() == 0
    for k in ["ptend_s", "ptend_q", "ptend_u", "prec", "snow", "mcon", "ideep", "lengath"]:
        assert np.array_equal(dev.out[k].cpu().numpy(), ref[k]), k
    c = cons.cpu().numpy()
    g = 9.80616
    assert np.isclose(c[0], (ch.pdel / g * ref["ptend_q"]).sum(), rtol=1e-12)
    assert np.isclose(c[1], 1000.0 * (ref["prec"] + ref["rliq"]).sum(), rtol=1e-12)
    assert c[4] == ref["lengath"].sum() and c[5] == 4096
    assert np.isclose(c[2], (ch.pdel / g * ref["ptend_s"]).sum(), rtol=1e-11)
    assert np.isclose(c[3], 1000.0 * (2.501e6 * (ref["prec"] + ref["rliq"]) + 3.337e5 * ref["snow"]).sum(), rtol=1e-12)
    # deterministic: a fixed grid and a fixed order of additions -- the same bits every time
    c2 = dev.conservation().cpu().numpy()
    assert np.array_equal(c.view(np.int64), c2.view(np.int64))


def test_momtran_component_flags_and_reentrancy(built):
    """domomtran(m) = .false. leaves that component's outputs untouched (zm_conv.F90:2458); and the
    library is re-entrant: two host threads driving different chunk sets concurrently get the same
    answers as serial calls (reference call pattern: OpenMP threads, physpkg.F90:1147)."""
    import threading
    Z = init_cuda(16, 32)
    o, _, _ = get_oracle("pm", 16, 32)
    ch = S.make_chunks(640, 32, 16, p_conv=0.7)
    ref = o.convr_batch(ch)
    winds = np.stack([ch.u, ch.v], axis=1)
    mo = Z.momtran(ch.ncol, [1, 0], winds, ref["mu"], ref["md"], ref["du"], ref["eu"], ref["ed"], ref["dp"],
                   ref["dsubcld"], ref["jt"], ref["maxg"], ref["ideep"], ref["lengath"], ch.ztodt)
    for c in range(ch.nchunks):
        r = o.momtran(int(ch.ncol[c]), [1, 0], winds[c], ref["mu"][c], ref["md"][c], ref["du"][c], ref["eu"][c],
                      ref["ed"][c], ref["dp"][c], ref["dsubcld"][c], ref["jt"][c], ref["maxg"][c], ref["ideep"][c],
                      ref["lengath"][c], ch.ztodt)
        for k in ["dqdt", "pguall", "pgdall", "icwu", "icwd", "seten"]:
            assert np.array_equal(mo[k][c], r[k]), (c, k)
    res = {}

    def work(tag, lo, hi):
        sub = S.make_chunks(16 * (hi - lo), 32, 16, p_conv=0.7, col0=16 * lo)
        res[tag] = cuda_convr(Z, sub)

    ths = [threading.Thread(target=work, args=(i, 10 * i, 10 * i + 10)) for i in range(4)]
    [t.start() for t in ths]; [t.join() for t in ths]
    for i in range(4):
        sub = {k: v[10 * i: 10 * i + 10] for k, v in ref.items() if k != "rc"}
        assert_same(res[i], sub, ["qtnd", "heat", "prec", "ideep", "lengath", "mu", "jt", "maxg", "pflx"], 16,
                    exact=True, what=f"thread {i}")


def test_next_rows_geopotential_and_convect_diagnostics(built):
    """SURVEY.md 8f N4: geopotential_t (both hydrostatic branches) and convect_diagnostics_calc, bit-exact."""
    Z = init_cuda(16, 32)
    o, _, _ = get_oracle("pm", 16, 32)
    ch = S.make_chunks(1000, 32, 16, p_conv=0.5)
    zvir = np.full_like(ch.t, S.ZVIR); rair = np.full_like(ch.t, S.RAIR)
    piln, rpdel = np.log(ch.pint), 1.0 / ch.pdel
    for lr in (True, False):
        zi, zm = Z.geopotential_t(ch.ncol, piln, np.log(ch.pmid), ch.pint, ch.pmid, ch.pdel, rpdel, ch.t, ch.q, rair,
                                  S.GRAVIT, zvir, dycore_lr=lr)
        for c in range(ch.nchunks):
            n = int(ch.ncol[c])
            rzi, rzm = o.geopotential_t(n, lr, piln[c], ch.pint[c], ch.pmid[c], ch.pdel[c], rpdel[c], ch.t[c], ch.q[c],
                                        rair[c], S.GRAVIT, zvir[c])
            assert np.array_equal(zi[c][:, :n], rzi[:, :n]) and np.array_equal(zm[c][:, :n], rzm[:, :n]), (lr, c)
    ref = o.conv_tend_batch(ch)
    out = Z.convect_diagnostics_calc(ch.ncol, ref["mcon"], ref["dlf"], ref["rliq"], ch.pmid, ref["rprd"], ref["jctop"],
                                     ref["jcbot"])
    for c in range(ch.nchunks):
        n = int(ch.ncol[c])
        r = o.convect_diagnostics(n, ref["mcon"][c], ref["dlf"][c], ref["rliq"][c], ch.pmid[c], ref["rprd"][c],
                                  ref["jctop"][c], ref["jcbot"][c])
        for k in r:
            assert np.array_equal(out[k][c][..., :n], r[k][..., :n]), (c, k)
    assert np.all(out["cnb"][ch.ncol[:, None] > np.arange(16)[None, :]] >= 1)


def test_geopotential_t_generalized_tv(built):
    """geopotential_t, generalized-virtual-temperature branch (physics/geopotential.F90:248-310, SURVEY N4): bit-exact
    against the oracle on 1000 columns x 7 constituents, both hydrostatic variants, several species lists (incl. none);
    equal to the reference text's own output on the committed fixture; bad species indices are refused."""
    Z = init_cuda(16, 32)
    o, _, _ = get_oracle("pm", 16, 32)
    ch = S.make_chunks(1000, 32, 16, p_conv=0.5)
    zvir = np.full_like(ch.t, S.ZVIR); rair = np.full_like(ch.t, S.RAIR)
    piln, rpdel = np.log(ch.pint), 1.0 / ch.pdel
    rng = np.random.default_rng(7)
    ncnst = 7
    q3 = 1e-4 * rng.random((ch.nchunks, ncnst, 32, 16))
    q3[:, 0] = ch.q
    for species in ([1, 2, 3], [1], [1, 6, 2, 7, 4], []):
        sp = np.array(species, np.int32)
        for lr in (False, True):
            zi, zm = Z.geopotential_t_gen(ch.ncol, piln, np.log(ch.pmid), ch.pint, ch.pmid, ch.pdel, rpdel, ch.t, q3, rair,
                                          S.GRAVIT, zvir, sp, dycore_lr=lr)
            for c in range(0, ch.nchunks, 3):
                n = int(ch.ncol[c])
                rzi, rzm = o.geopotential_t_gen(n, lr, piln[c], ch.pint[c], ch.pmid[c], ch.pdel[c], rpdel[c], ch.t[c],
                                                q3[c], rair[c], S.GRAVIT, zvir[c], sp)
                assert np.array_equal(zi[c][:, :n], rzi[:, :n]) and np.array_equal(zm[c][:, :n], rzm[:, :n]), (species, lr, c)
    g = np.load(os.path.join(GOLD, "reftext_geopotential_t_gen.npz"))
    n = int(g["ncol"])
    one = lambda k: g[k][None]
    for lr in (0, 1):
        zi, zm = Z.geopotential_t_gen(np.array([n], np.int32), one("in_piln"), np.log(one("in_pmid")), one("in_pint"),
                                      one("in_pmid"), one("in_pdel"), one("in_rpdel"), one("in_t"), one("in_q3"),
                                      one("in_rair"), float(g["gravit"]), one("in_zvir"), g["species_idx"], dycore_lr=lr)
        assert np.array_equal(zi[0][:, :n], g["zi_lr%d" % lr][:, :n]) and np.array_equal(zm[0][:, :n], g["zm_lr%d" % lr][:, :n])
    with pytest.raises(Z.ZmError):
        Z.geopotential_t_gen(ch.ncol, piln, np.log(ch.pmid), ch.pint, ch.pmid, ch.pdel, rpdel, ch.t, q3, rair, S.GRAVIT, zvir,
                             np.array([1, ncnst + 1], np.int32))


def test_conv_tend_2_uses_device_mirror(built):
    """zm_conv_tend with the pbuf fields kept on the device, then zm_conv_tend_2 (convtran2,
    zm_conv_intr.F90:955-1028) from that mirror: bit-exact vs oracle convtran on the oracle's fields."""
    Z = init_cuda(16, 32)
    o, _, _ = get_oracle("pm", 16, 32)
    ch = S.make_chunks(800, 32, 16, p_conv=0.6)
    ref = o.conv_tend_batch(ch)
    out = Z.zm_conv_tend(ch.ncol, state_of(ch), ch.ztodt, keep_pbuf_on_device=True)
    assert np.all(out["mu"] == 0.0) and np.all(out["jt"] == 0)       # not copied back
    assert_same(out, ref, ["lengath", "ideep", "ptend_s", "ptend_q", "prec", "mcon"], 16, exact=True, what="tend")
    pcnst = 8
    q, fracis, pdeldry = S.make_tracers(ch, pcnst)
    do = [0, 0, 1, 1, 0, 1, 1, 1]
    dry = [0, 0, 1, 0, 0, 1, 0, 1]
    dq = Z.zm_conv_tend_2(do, q, pdeldry, fracis, ch.ztodt, dry)
    dpdry = dpdry_gathered(ch, ref, pdeldry)
    for c in range(ch.nchunks):
        r = o.convtran(do, q[c], ref["mu"][c], ref["md"][c], ref["du"][c], ref["eu"][c], ref["ed"][c], ref["dp"][c],
                       ref["dsubcld"][c], ref["jt"][c], ref["maxg"][c], ref["ideep"][c], ref["lengath"][c], fracis[c],
                       dpdry[c], ch.ztodt, dry)
        for m in range(pcnst):
            if do[m]:
                assert np.array_equal(dq[c, m], r[m]), (c, m)
            else:
                assert np.all(dq[c, m] == 0.0)
    assert np.count_nonzero(dq) > 0
    # a second tend call with another nchunks invalidates the mirror for the old size
    ch2 = S.make_chunks(160, 32, 16, p_conv=0.6)
    Z.zm_conv_tend(ch2.ncol, state_of(ch2), ch2.ztodt)
    with pytest.raises(Z.ZmError):
        Z.zm_conv_tend_2(do, q, pdeldry, fracis, ch.ztodt, dry)


def test_pbuf_mirror_survives_the_calls_between_tend_and_tend_2(built):
    """The model runs geopotential_t / convect_diagnostics_calc (and anything else that stages host arrays) between
    zm_conv_tend and zm_conv_tend_2 (physpkg.F90:2820, 2885, 1988): the device pbuf mirror must survive them, whatever
    their sizes.  A failed tend call leaves no mirror."""
    Z = init_cuda(16, 32)
    o, _, _ = get_oracle("pm", 16, 32)
    ch = S.make_chunks(640, 32, 16, p_conv=0.6)
    ref = o.conv_tend_batch(ch)
    Z.zm_conv_tend(ch.ncol, state_of(ch), ch.ztodt, keep_pbuf_on_device=True)
    # same-size and larger host-pointer calls in between: each restages the thread's staging arena
    big = S.make_chunks(4000, 32, 16, p_conv=0.5)
    for cc in (ch, big):
        piln, pmln, rpdel = np.log(cc.pint), np.log(cc.pmid), 1.0 / cc.pdel
        rair = np.full_like(cc.t, 287.04); zvir = np.full_like(cc.t, 0.608)
        Z.geopotential_t(cc.ncol, piln, pmln, cc.pint, cc.pmid, cc.pdel, rpdel, cc.t, cc.q, rair, 9.80616, zvir)
        cuda_convr(Z, cc)
        n = cc.nchunks
        Z.convect_diagnostics_calc(cc.ncol, np.zeros((n, 33, 16)), np.zeros((n, 32, 16)), np.zeros((n, 16)), cc.pmid,
                                   np.zeros((n, 32, 16)), np.full((n, 16), 20.0), np.full((n, 16), 30.0))
    pcnst = 6
    q, fracis, pdeldry = S.make_tracers(ch, pcnst)
    do, dry = [0, 1, 1, 0, 1, 1], [0, 0, 1, 0, 1, 0]
    dq = Z.zm_conv_tend_2(do, q, pdeldry, fracis, ch.ztodt, dry)
    dpdry = dpdry_gathered(ch, ref, pdeldry)
    for c in range(ch.nchunks):
        r = o.convtran(do, q[c], ref["mu"][c], ref["md"][c], ref["du"][c], ref["eu"][c], ref["ed"][c], ref["dp"][c],
                       ref["dsubcld"][c], ref["jt"][c], ref["maxg"][c], ref["ideep"][c], ref["lengath"][c], fracis[c],
                       dpdry[c], ch.ztodt, dry)
        for m in range(pcnst):
            assert np.array_equal(dq[c, m], r[m] if do[m] else np.zeros_like(r[m])), (c, m)
    assert np.count_nonzero(dq) > 0
    # the diagnostics of zm_conv_tend from the same mirror (zm_conv_intr.F90:685-729)
    ps = ch.pint[:, -1, :]
    dg = Z.zm_conv_tend_diag(ch.ncol, ps, ch.pmid)
    dg2 = Z.zm_conv_tend_diag(ch.ncol, ps, ch.pmid, ref["mu"], ref["md"], ref["jt"], ref["maxg"], ref["ideep"], ref["lengath"])
    for c in range(ch.nchunks):
        r = o.conv_tend_diag(ch.ncol[c], ps[c], ch.pmid[c], ref["mu"][c], ref["md"][c], ref["jt"][c], ref["maxg"][c],
                             ref["ideep"][c], ref["lengath"][c])
        for k in r:
            assert np.array_equal(dg[k][c], r[k]) and np.array_equal(dg2[k][c], r[k]), (c, k)
    assert dg["freqzm"].sum() == ref["lengath"].sum() and np.any(dg["pcont"] < ps)
    # a tend call that fails (zm_org without attached fields) leaves no mirror behind
    Z2 = init_cuda(16, 32, zm_org=1)
    with pytest.raises(Z2.ZmError):
        Z2.zm_conv_tend(ch.ncol, state_of(ch), ch.ztodt, keep_pbuf_on_device=True)
    with pytest.raises(Z2.ZmError):
        Z2.zm_conv_tend_2(do, q, pdeldry, fracis, ch.ztodt, dry)


@pytest.mark.parametrize("ncols,cam3", [(1600, False), (16 * 1100, False), (900, True)])
def test_conv_tend_with_convtran1_and_cam3(built, ncols, cam3):
    """zm_conv_tend including convtran1 (zm_conv_intr.F90:865-880: cloud liquid / ice on state1%q, fake_dpdry = 0),
    unpipelined and pipelined (sub-batches move only the flagged constituent slices), and the cam3 package, which
    skips momtran (zm_conv_intr.F90:808): every output bit for bit against the oracle."""
    over = dict(cam3=1, num_cin=5) if cam3 else {}
    Z = init_cuda(16, 32, **over)
    o, _, _ = get_oracle("pm", 16, 32, **over)
    ch = S.make_chunks(ncols, 32, 16, p_conv=0.55)
    pcnst = 7
    q, fracis, _ = S.make_tracers(ch, pcnst)
    q[:, 0] = ch.q
    t1 = dict(doconvtran=[1, 1, 1, 0, 0, 1, 0], cnst_is_dry=[0] * pcnst, q=q, fracis=fracis,
              ptend_q=np.full_like(q, 3.0))
    ref = o.conv_tend_batch(ch, convtran1=t1)
    out = Z.zm_conv_tend(ch.ncol, state_of(ch), ch.ztodt, convtran1=t1)
    assert_same(out, ref, TEND_KEYS, 16, exact=True, what="zm_conv_tend + convtran1")
    assert np.array_equal(out["ptend_qc"], ref["ptend_qc"])
    assert np.all(out["ptend_qc"][:, [0, 3, 4, 6]] == 3.0)          # water vapour and unflagged slices untouched
    assert np.count_nonzero(out["ptend_qc"][:, [1, 2, 5]]) > 0 and not np.any(out["ptend_qc"][:, [1, 2, 5]] == 3.0)
    if cam3:
        assert np.all(out["ptend_u"] == 0.0) and np.all(out["ptend_v"] == 0.0)
    else:
        assert np.count_nonzero(out["ptend_u"]) > 0
    # the attachment is one-shot
    out2 = Z.zm_conv_tend(ch.ncol, state_of(ch), ch.ztodt)
    assert "ptend_qc" not in out2 and np.array_equal(out2["ptend_s"], out["ptend_s"])


@pytest.mark.parametrize("pcols,pver", [(16, 32), (13, 29), (24, 26)])
def test_conv_tend_glue_any_shape_and_alignment(built, monkeypatch, pcols, pver):
    """The fused step's glue has one form for every shape and alignment: momtran reads state%u / state%v and writes
    ptend_u / ptend_v itself, zm_conv_evap applies physics_update and stores the summed tendencies, the last kernel adds
    seten.  (13,29) gives an odd nchunks*pcols*pver; a device-resident step with ptend_s and ptend_u one element off
    16-byte alignment launches exactly the kernels of the aligned one.  All bit for bit against the oracle,
    host-pointer and device-resident calls."""
    import torch
    Z = init_cuda(pcols, pver)
    o, _, _ = get_oracle("pm", pcols, pver)
    from cam_nor_physics_b200.device import DeviceTend
    ch = S.make_chunks(pcols * 91 - 3, pver, pcols, p_conv=0.6)      # 91 chunks: 13 x 29 x 91 elements are odd
    ref = o.conv_tend_batch(ch)
    assert int(ref["lengath"].sum()) > 100
    monkeypatch.setenv("ZM_DEV_GRAPH", "0")
    out = Z.zm_conv_tend(ch.ncol, state_of(ch), ch.ztodt)
    assert_same(out, ref, TEND_KEYS, pcols, exact=True, what="host-pointer step")
    L = Z.lib()
    dev = DeviceTend(ch)
    L.zm_launch_count(1)
    dev.step()
    assert dev.check() == 0
    n_step = L.zm_launch_count(1)
    dout = {k: v.cpu().numpy() for k, v in dev.out.items()}
    assert_same(dout, ref, TEND_KEYS, pcols, exact=True, what="device-resident step")
    # ptend_s (the seten sum) and ptend_u (the zero-fill) 8 bytes past a 16-byte boundary, pre-filled with garbage
    for k in ("ptend_s", "ptend_u"):
        a = dev.out[k]
        buf = torch.full((a.numel() + 1,), 1.25, dtype=a.dtype, device=a.device)
        dev.out[k] = buf[1:].view(a.shape)
        assert dev.out[k].data_ptr() % 16 == 8
    dev.step()
    assert dev.check() == 0
    assert L.zm_launch_count(1) == n_step
    dout = {k: v.cpu().numpy() for k, v in dev.out.items()}
    assert_same(dout, ref, TEND_KEYS, pcols, exact=True, what="device-resident step, misaligned ptend_s and ptend_u")
    assert np.count_nonzero(ref["ptend_u"]) > 0 and np.count_nonzero(ref["mcon"]) > 0


@pytest.mark.parametrize("ncols", [16 * 70, 16 * 1100 + 5])
def test_dense_return_defines_every_element(built, ncols):
    """zm_conv_tend_batch copies the outputs device->host whole: every element is defined, whatever the arrays held
    before, with and without the pbuf fields kept on the device, and equals the oracle bit for bit."""
    Z = init_cuda(16, 32)
    ch = S.make_chunks(ncols, 32, 16, p_conv=0.45)
    out = None
    for rep in range(2):                   # the second call finds garbage in the arrays
        if out is not None:
            for k, a in out.items():
                a[...] = 7 if a.dtype.kind == "i" else 1.25
        out = Z.zm_conv_tend(ch.ncol, state_of(ch), ch.ztodt, out)
    dense = {k: v.copy() for k, v in out.items()}
    moved = Z.last_transfer_bytes()
    assert moved["d2h"] >= sum(v.nbytes for v in out.values())
    out = Z.zm_conv_tend(ch.ncol, state_of(ch), ch.ztodt, keep_pbuf_on_device=True)
    for k in dense:
        if k in ("mu", "md", "du", "eu", "ed", "dp", "dsubcld", "jt", "maxg"):
            assert not out[k].any()
        else:
            assert np.array_equal(out[k], dense[k]), k
    o, _, _ = get_oracle("pm", 16, 32)
    assert_same(dense, o.conv_tend_batch(ch), TEND_KEYS, 16, exact=True, what="dense return vs oracle")


def test_finalize_releases_and_reinit_reproduces(built):
    """zm_finalize frees the thread's arenas/streams; a fresh zm_init + step gives the same bits, and the
    pipelined host API (default: 4 equal sub-batches; an explicit 1,1,2,4,4,4-sixteenths ramp; 8 equal ones) equals
    the unpipelined one."""
    Z = init_cuda(16, 32)
    ch = S.make_chunks(16 * 1100, 32, 16, p_conv=0.5)         # 1100 chunks: enough for the default schedule
    out1 = Z.zm_conv_tend(ch.ncol, state_of(ch), ch.ztodt)
    tr = Z.tend_trace()
    assert tr.shape == (4, 6) and np.all(tr >= 0.0)
    assert np.all(tr[:, 5] >= tr[:, 2])                        # outputs leave after zm_convr finished
    assert Z.lib().zm_finalize() == 0
    with pytest.raises(Z.ZmError):
        Z.zm_conv_tend(ch.ncol, state_of(ch), ch.ztodt)
    Z = init_cuda(16, 32)
    for var, val, shape in (("ZM_TEND_SUBBATCHES", "1", (1, 6)), ("ZM_TEND_SUBBATCHES", "8", (8, 6)),
                            ("ZM_TEND_SCHEDULE", "1,1,2,4,4,4", (6, 6)), ("ZM_TEND_SCHEDULE", "-4,20", (4, 6)),
                            ("ZM_TEND_SCHEDULE", "1,1,1,1,1,1,1,1,8", (4, 6))):
        os.environ[var] = val                      # invalid lists (non-positive entries, too many) fall back to the default
        try:
            out2 = Z.zm_conv_tend(ch.ncol, state_of(ch), ch.ztodt)
            assert Z.tend_trace().shape == shape, (var, val)
        finally:
            del os.environ[var]
        for k in out1:
            assert np.array_equal(out1[k], out2[k]), (var, val, k)
    assert out1["lengath"].sum() > 0


def test_zm_org_bit_exact_vs_oracle(built):
    """zmconv_org branches (SURVEY N3): zm_convr and the zm_conv_tend sequence with an organisation tracer."""
    Z = init_cuda(16, 32, zm_org=1)
    o, _, rc = get_oracle("pm", 16, 32, zm_org=1)
    assert rc == 0
    ch = S.make_chunks(16 * 300 - 5, 32, 16, p_conv=0.6)
    org = np.maximum(np.random.default_rng(3).uniform(-0.3, 1.0, ch.t.shape), 0.0)   # tracer in [0,1], ~23 % zeros
    ref = o.convr_batch(ch, org=org)
    out = Z.zm_convr(ch.ncol, ch.t, ch.q, ch.pblh, ch.zm, ch.phis, ch.zi, ch.pmid, ch.pint, ch.pdel,
                     0.5 * ch.ztodt, ch.tpert, ch.landfrac, org=org)
    assert_same(out, ref, CONVR_KEYS + ["orgt", "org2d"], 16, exact=True, what="zm_convr zm_org")
    assert out["lengath"].sum() > 0 and np.any(out["org2d"] > 0)
    st = state_of(ch); st["org"] = org
    tref = o.conv_tend_batch(ch, org=org)
    tout = Z.zm_conv_tend(ch.ncol, st, ch.ztodt)
    assert_same(tout, tref, TEND_KEYS + ["orgt", "org2d"], 16, exact=True, what="zm_conv_tend zm_org")
    assert np.any(tout["orgt"] != 0.0)
    # a call without the fields attached fails loudly
    with pytest.raises(Z.ZmError):
        Z.zm_conv_tend(ch.ncol, state_of(ch), ch.ztodt)
    init_cuda(16, 32)                   # back to the default configuration for the tests that follow


def test_device_resident_step_graph_replay(built):
    """Device-pointer API: the 1st call runs directly, the 2nd identical call is captured into a CUDA graph, later
    calls replay it.  All of them, on the default stream and on a side stream, must equal the host-pointer API
    (which equals the oracle) bit for bit; changed inputs must be picked up by a replay (same pointers)."""
    import torch
    from cam_nor_physics_b200.device import DeviceTend
    Z = init_cuda(16, 32)
    ch = S.make_chunks(16 * 200, 32, 16, p_conv=0.5)
    ref = Z.zm_conv_tend(ch.ncol, state_of(ch), ch.ztodt)
    dev = DeviceTend(ch)
    l0 = Z.lib().zm_launch_count(1)
    per_step = []
    for it in range(4):
        for v in dev.out.values():
            v.fill_(-7)                                # stale values must be overwritten by every step
        dev.step()
        assert dev.check() == 0
        per_step.append(Z.lib().zm_launch_count(1))
        for k in TEND_KEYS:
            got = dev.out[k].cpu().numpy()
            assert_same({k: got, "lengath": dev.out["lengath"].cpu().numpy()}, ref, [k], 16, exact=True,
                        what=f"device step {it}")
    assert len(set(per_step)) == 1 and per_step[0] > 0     # replayed steps report the same kernel count
    # new input values behind the same pointers: a replayed graph must compute the new answer
    ch2 = S.make_chunks(16 * 200, 32, 16, p_conv=0.2, col0=50000)
    ref2 = Z.zm_conv_tend(ch2.ncol, state_of(ch2), ch2.ztodt)
    for k in Z.TEND_IN_ORDER:
        dev.inp[k].copy_(torch.from_numpy(np.ascontiguousarray(getattr(ch2, k))))
    st = torch.cuda.Stream()
    torch.cuda.synchronize()
    with torch.cuda.stream(st):
        dev.step()
        assert dev.check() == 0
    torch.cuda.synchronize()
    for k in ["lengath", "ideep", "ptend_s", "ptend_q", "ptend_u", "prec", "mcon"]:
        assert_same({k: dev.out[k].cpu().numpy(), "lengath": dev.out["lengath"].cpu().numpy()}, ref2, [k], 16,
                    exact=True, what="device step after input change")


@pytest.mark.parametrize("pver,over", [(58, {"lparcel_pbl": 1}), (72, {}), (24, {})])
def test_zm_conv_tend_other_level_counts(built, pver, over):
    """The whole zm_conv_tend sequence (zm_convr + physics_update + zm_conv_evap + momtran) at level counts where
    a lane owns more than one level (L58, L72) or fewer lanes than a warp are busy (L24)."""
    Z = init_cuda(16, pver, **over)
    o, _, rc = get_oracle("pm", 16, pver, **over)
    assert rc == 0
    ch = S.make_chunks(16 * 40 - 3, pver, 16, p_conv=0.6)
    ref = o.conv_tend_batch(ch)
    assert ref["rc"] == 0
    out = Z.zm_conv_tend(ch.ncol, state_of(ch), ch.ztodt)
    assert_same(out, ref, TEND_KEYS, 16, exact=True, what=f"zm_conv_tend L{pver}")
    assert out["lengath"].sum() > 0
    init_cuda(16, 32)


@pytest.mark.parametrize("case", REFTEXT_CASES)
def test_cuda_vs_reference_source_text(built, case):
    """CUDA library against the outputs of the reference's own Fortran text (tests/golden/reftext_*.npz, produced by
    tests/golden/make_reference_fixtures.py): integer outputs exact, r8 outputs within the north-star tolerance
    (the fixtures were computed with glibc log/exp/pow, the library uses its portable math)."""
    g = np.load(os.path.join(GOLD, "reftext_%s.npz" % case))
    pc, L, ncol = int(g["pcols"]), int(g["pver"]), int(g["ncol"])
    Z = init_cuda(pc, L, **reftext_overrides(g))
    ztodt = float(g["ztodt"])
    ncols = np.array([ncol], np.int32)
    I = lambda k: g["in_" + k][None]          # noqa: E731
    org = g["in_org"][None] if "in_org" in g.files else None
    r = Z.zm_convr(ncols, I("t"), I("q"), I("pblh"), I("zm"), I("phis"), I("zi"), I("pmid"), I("pint"), I("pdel"),
                   0.5 * ztodt, I("tpert"), I("landfrac"), org=org)
    n = int(g["convr_lengath"])
    assert len(near_threshold_columns(g["convr_cape"])) == 0
    assert int(r["lengath"][0]) == n
    bad = []
    for k in REFTEXT_CONVR:
        a, b = r[k][0], g["convr_" + k]
        if k in ("mu", "md", "du", "eu", "ed", "dp", "dsubcld", "jt", "maxg"):
            a, b = a[..., :n], b[..., :n]
        if k in ("jctop", "jcbot"):
            a, b = a[..., :ncol], b[..., :ncol]
        if k in ("ideep", "jt", "maxg", "jctop", "jcbot"):
            ok = np.array_equal(np.asarray(a, float), np.asarray(b, float))
        else:
            ok = np.allclose(a, b, rtol=RTOL, atol=ATOL)
        if not ok:
            bad.append(k)
    assert not bad, "zm_convr vs reference text: %s" % bad
    if org is not None:
        assert np.all(r["orgt"] == 0.0)
        assert np.allclose(r["org2d"][0][:, :ncol], g["convr_org2d"][:, :ncol], rtol=RTOL, atol=ATOL)
    # downstream routines on the REFERENCE's zm_convr outputs
    G = lambda k: g["convr_" + k][None]       # noqa: E731
    ev = Z.zm_conv_evap(ncols, g["evap_in_t"][None], I("pmid"), I("pdel"), g["evap_in_q"][None], I("landfrac"),
                        G("rprd"), I("cld"), ztodt, G("prec"))
    for k in ("tend_s", "tend_s_snwprd", "tend_s_snwevmlt", "tend_q", "prec", "snow", "ntprprd", "ntsnprd", "flxprec",
              "flxsnow"):
        assert np.allclose(ev[k][0][..., :ncol], g["evap_" + k][..., :ncol], rtol=RTOL, atol=ATOL), ("evap", k)
    winds = np.stack([g["in_u"], g["in_v"]], axis=0)[None]
    ilen = np.array([n], np.int32)
    mo = Z.momtran(ncols, [1, 1], winds, G("mu"), G("md"), G("du"), G("eu"), G("ed"), G("dp"), G("dsubcld"),
                   G("jt").astype(np.int32), G("maxg").astype(np.int32), G("ideep").astype(np.int32), ilen, ztodt)
    for k in ("dqdt", "pguall", "pgdall", "icwu", "icwd", "seten"):
        assert np.allclose(mo[k][0][..., :ncol], g["momtran_" + k][..., :ncol], rtol=RTOL, atol=1e-13), ("momtran", k)
    do, dry = g["convtran_in_doconvtran"], g["convtran_in_is_dry"]
    dq = Z.convtran(do, g["convtran_in_q"][None], G("mu"), G("md"), G("du"), G("eu"), G("ed"), G("dp"), G("dsubcld"),
                    G("jt").astype(np.int32), G("maxg").astype(np.int32), G("ideep").astype(np.int32), ilen,
                    g["convtran_in_fracis"][None], g["convtran_in_dpdry"][None], ztodt, dry)
    for mth in range(1, len(do)):
        if do[mth]:
            assert np.allclose(dq[0, mth], g["convtran_dqdt"][mth], rtol=RTOL, atol=1e-30), ("convtran", mth)
    init_cuda(16, 32)


def test_cuda_vs_reference_source_text_sweep(built):
    """507 mixed columns: CUDA zm_convr against the reference text's outputs (integers exact, r8 within tolerance)."""
    g = np.load(os.path.join(GOLD, "reftext_sweep_L32.npz"))
    Z = init_cuda(16, 32)
    ch = S.make_chunks(int(g["ncols"]), 32, 16, p_conv=float(g["p_conv"]), col0=int(g["col0"]))
    assert len(near_threshold_columns(g["convr_cape"])) == 0
    out = cuda_convr(Z, ch)
    ref = {k[6:]: g[k] for k in g.files if k.startswith("convr_")}
    ref["lengath"] = ref["lengath"].astype(np.int32)
    m = np.arange(16)[None, :] < ch.ncol[:, None]
    for k in ("jctop", "jcbot"):
        out[k] = out[k] * m
        ref[k] = ref[k] * m
    assert_same(out, ref, [k for k in REFTEXT_CONVR] + ["lengath"], 16, exact=False, what="CUDA vs reference text (sweep)")


def test_convtran_zero_and_negative_tracers(built):
    """Tracer columns with exact zeros, tiny values and slightly negative entries (CAM tracers do go negative before
    qneg3): the interface-value branches of zm_conv.F90:2119-2139 (minc < 0, both zero, one zero) bit-exact vs oracle."""
    Z = init_cuda(16, 32)
    o, p, _ = get_oracle("pm", 16, 32)
    ch = S.make_chunks(640, 32, 16, p_conv=0.7, col0=31000)
    ref = o.convr_batch(ch)
    ncnst = 7
    q, fracis, pdeldry = S.make_tracers(ch, ncnst)
    rng = np.random.default_rng(77)
    u = rng.uniform(size=q.shape)
    q[(u < 0.06)] = 0.0
    q[(u >= 0.06) & (u < 0.09)] *= -0.01
    q[(u >= 0.09) & (u < 0.12)] *= 1e-25
    q[:, 5] = 0.0                                   # an all-zero constituent
    do = [0, 1, 1, 1, 1, 1, 1]
    dry = [0, 0, 1, 0, 1, 0, 1]
    dpdry = dpdry_gathered(ch, ref, pdeldry)
    dq = Z.convtran(do, q, ref["mu"], ref["md"], ref["du"], ref["eu"], ref["ed"], ref["dp"], ref["dsubcld"],
                    ref["jt"], ref["maxg"], ref["ideep"], ref["lengath"], fracis, dpdry, ch.ztodt, dry)
    for c in range(ch.nchunks):
        r = o.convtran(do, q[c], ref["mu"][c], ref["md"][c], ref["du"][c], ref["eu"][c], ref["ed"][c], ref["dp"][c],
                       ref["dsubcld"][c], ref["jt"][c], ref["maxg"][c], ref["ideep"][c], ref["lengath"][c],
                       fracis[c], dpdry[c], ch.ztodt, dry)
        for m in range(1, ncnst):
            assert np.array_equal(dq[c, m], r[m]), (c, m)
    assert np.all(dq[:, 5] == 0.0) and np.count_nonzero(dq) > 0 and np.all(np.isfinite(dq))


def test_randomised_parity_sweep(built):
    """A short run of scripts/parity_fuzz.py (random seeds, sizes, pcols, level counts, options, perturbed soundings;
    zm_convr / zm_conv_tend / zm_org / device mirror + zm_conv_tend_2 / convtran / N4 routines, bit-exact vs the
    oracle).  The 160-case run of round 1 is profiles/parity_fuzz_r1_*.log."""
    import subprocess, sys, json
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, os.path.join(root, "scripts", "parity_fuzz.py"), "24", "101"],
                       capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    summary = json.loads(r.stdout.strip().splitlines()[-1])
    assert summary["cases"] == 24 and summary["all_bit_exact"]
    init_cuda(16, 32)
