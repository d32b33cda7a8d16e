"""zm_conv_tend_2_batch_gathered: convtran2 (zm_conv_tend_2) on the convective columns' records of the flagged
constituents, for the caller's own pack (loop 1) and scatter (loop 2).

The contract rests on a premise that is asserted first, on the dense zm_conv_tend_2: for a flagged constituent the
tendency is exactly 0 outside the convective columns ideep(1:lengath), for an unflagged one it is 0 everywhere.  Then
the scattered records must equal the dense tendency and the oracle's convtran bit for bit, with the device mirror
left by the dense or by the gathered zm_conv_tend step, and only the records may cross PCIe."""
import ctypes as C
import threading

import numpy as np
import pytest

from cam_nor_physics_b200 import soundings as S
from cam_nor_physics_b200 import zm_conv as Z
from helpers import dpdry_gathered, get_oracle, init_cuda, state_of
from test_tend_gathered import make_case, same_bits


def _synthetic(rng, nch, pc, L, pcnst):
    lengath = rng.integers(0, pc + 1, nch).astype(np.int32)
    lengath[0], lengath[-1] = 0, pc
    ideep = np.zeros((nch, pc), np.int32)
    for c in range(nch):
        ideep[c, :lengath[c]] = rng.permutation(pc)[:lengath[c]] + 1
    q = rng.standard_normal((nch, pcnst, L, pc))
    fracis = rng.uniform(size=q.shape)
    pdeldry = rng.uniform(1.0, 2.0, (nch, L, pc))
    return lengath, ideep, q, fracis, pdeldry


def _flags(kind, pcnst):
    do, dry = np.zeros(pcnst, np.int32), np.zeros(pcnst, np.int32)
    if kind == "one_moist":
        do[pcnst // 2] = 1
    elif kind == "one_dry":
        do[1] = 1; dry[1] = 1
    elif kind == "all_mixed":                         # nact = pcnst - 1
        do[:] = 1; dry[2::2] = 1
    elif kind == "water_flag_ignored":                # entry 1 is not a convtran2 constituent whatever its flag
        do[0] = 1; do[3:] = 1; dry[0] = 1
    return do, dry


# ---- CPU -----------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("shape", [(37, 13, 29, 6), (20, 16, 32, 9), (5, 4, 7, 2)])
@pytest.mark.parametrize("kind", ["one_moist", "one_dry", "all_mixed", "water_flag_ignored"])
def test_records_round_trip(shape, kind):
    """convtran2_records then scatter_convtran2 gives back exactly the flagged constituents' convective columns and
    zeros elsewhere; pdeldry_rec exists iff a flagged constituent is dry."""
    nch, pc, L, pcnst = shape
    rng = np.random.default_rng(nch * 7 + pcnst)
    lengath, ideep, q, fracis, pdeldry = _synthetic(rng, nch, pc, L, pcnst)
    do, dry = _flags(kind, pcnst)
    act = Z.convtran2_active(do, pcnst)
    assert list(act) == [m for m in range(1, pcnst) if do[m]]
    qr, fr, pr = Z.convtran2_records(q, fracis, pdeldry, ideep, lengath, do, dry)
    n = int(lengath.sum())
    assert qr.shape == fr.shape == (n * L * len(act),)
    assert (pr is not None) == bool(dry[act].any())
    mask = np.zeros(q.shape, bool)
    for c in range(nch):
        for m in act:
            mask[c, m][:, ideep[c, :lengath[c]] - 1] = True
    for rec, dense in ((qr, q), (fr, fracis)):
        # pver comes from the records' size, or must be given when there are none (nact = 0)
        back = Z.scatter_convtran2(rec, ideep, lengath, do, pcnst, pver=None if len(act) else L)
        assert same_bits(back, np.where(mask, dense, 0.0))
    # without dry constituents no pdeldry travels; the moist call of the same columns gives the same q records
    qm, _, pm = Z.convtran2_records(q, fracis, pdeldry, ideep, lengath, do, None)
    assert pm is None and same_bits(qm, qr)


def test_record_offsets_follow_the_header_formula():
    """Element (slot i, level k, active constituent a) of chunk c is at nact*pver*base(c) + (a*pver + k)*n + i, with
    base(c) = sum(lengath(1:c-1)); pdeldry_rec's (i, k) at pver*base(c) + k*n + i."""
    nch, pc, L, pcnst = 23, 13, 11, 7
    rng = np.random.default_rng(3)
    lengath, ideep, q, fracis, pdeldry = _synthetic(rng, nch, pc, L, pcnst)
    do, dry = np.array([0, 1, 0, 1, 1, 0, 1], np.int32), np.array([0, 0, 0, 1, 0, 0, 0], np.int32)
    act = Z.convtran2_active(do, pcnst)
    nact = len(act)
    qr, fr, pr = Z.convtran2_records(q, fracis, pdeldry, ideep, lengath, do, dry)
    off = Z.convtran2_offsets(lengath, L, nact)
    base = 0
    for c in range(nch):
        n = int(lengath[c])
        assert off[c] == nact * L * base
        for a, m in enumerate(act):
            for k in range(L):
                for i in range(n):
                    col = ideep[c, i] - 1
                    e = nact * L * base + (a * L + k) * n + i
                    assert qr[e] == q[c, m, k, col] and fr[e] == fracis[c, m, k, col]
                    assert pr[L * base + k * n + i] == pdeldry[c, k, col]
        base += n
    assert off[-1] == qr.size == nact * L * base


# ---- GPU -----------------------------------------------------------------------------------------------------------
CASES = ["p16_L32_1100", "odd_13x29", "pcols128", "L58_parcel_pbl", "cam3", "zm_org", "lengath_0_and_full",
         "config4_41"]


def _case(name):
    if name == "config4_41":                  # BASELINE config 4's flags: 41 constituents, 38 transported, every third dry
        pc, L, over, org = 16, 32, {}, None
        ch = S.make_chunks(16 * 300 - 5, L, pc, p_conv=0.4)
        pcnst = 41
        do = np.zeros(pcnst, np.int32); do[3:] = 1
        dry = np.zeros(pcnst, np.int32); dry[3::3] = 1
        return pc, L, over, ch, org, pcnst, do, dry
    pc, L, over, ch, org = make_case(name)
    pcnst = 8
    do = np.array([0, 0, 1, 1, 0, 1, 1, 1], np.int32)
    dry = np.array([0, 0, 1, 0, 0, 1, 0, 1], np.int32)
    return pc, L, over, ch, org, pcnst, do, dry


def _st(ch, org):
    st = state_of(ch)
    if org is not None:
        st["org"] = org
    return st


def _expected_bytes(lengath, L, do, dry, pcnst):
    act = Z.convtran2_active(do, pcnst)
    n = int(np.asarray(lengath, np.int64).sum())
    any_dry = int(bool(np.asarray(dry)[act].any())) if len(act) else 0
    return {"h2d": (2 * len(act) + any_dry) * L * n * 8, "d2h": len(act) * L * n * 8 + 4 * len(lengath)}


@pytest.mark.gpu
@pytest.mark.parametrize("name", CASES)
def test_tend_2_gathered(built, name):
    pc, L, over, ch, org, pcnst, do, dry = _case(name)
    Z_ = init_cuda(pc, L, **over)
    st = _st(ch, org)
    o, _, rc = get_oracle("pm", pc, L, **over)
    assert rc == 0
    ref = o.conv_tend_batch(ch, org=org)
    assert ref["rc"] == 0
    q, fracis, pdeldry = S.make_tracers(ch, pcnst)
    res = Z_.zm_conv_tend(ch.ncol, st, ch.ztodt, keep_pbuf_on_device=True)
    lg, ideep = res["lengath"].copy(), res["ideep"].copy()
    assert int(lg.sum()) > 0 and np.array_equal(lg, ref["lengath"]) and np.array_equal(ideep, ref["ideep"])
    if name == "lengath_0_and_full":
        assert (lg == 0).any() and (lg == pc).any(), lg
    dense = Z_.zm_conv_tend_2(do, q, pdeldry, fracis, ch.ztodt, dry)
    b_dense = Z_.last_tend_2_transfer_bytes()
    n3, n2 = q.size, pdeldry.size
    assert b_dense == {"h2d": (3 * n3 + n2) * 8, "d2h": n3 * 8}
    # the premise
    incol = np.zeros((ch.nchunks, pc), bool)
    for c in range(ch.nchunks):
        incol[c, ideep[c, :lg[c]] - 1] = True
    for m in range(pcnst):
        if m >= 1 and do[m]:
            assert not dense[:, m][np.broadcast_to(~incol[:, None, :], dense[:, m].shape)].any(), (name, m)
        else:
            assert not dense[:, m].any(), (name, m)
    assert np.count_nonzero(dense) > 0
    # the oracle's convtran on the oracle's fields (every chunk of the smaller cases, every 7th of the larger)
    dpdry = dpdry_gathered(ch, ref, pdeldry)
    for c in range(0, ch.nchunks, 1 if ch.nchunks <= 200 else 7):
        r = o.convtran(do, q[c], ref["mu"][c], ref["md"][c], ref["du"][c], ref["eu"][c], ref["ed"][c], ref["dp"][c],
                       ref["dsubcld"][c], ref["jt"][c], ref["maxg"][c], ref["ideep"][c], ref["lengath"][c], fracis[c],
                       dpdry[c], ch.ztodt, dry)
        for m in range(1, pcnst):
            if do[m]:
                assert same_bits(dense[c, m], r[m]), (name, c, m)

    qr, fr, pr = Z_.convtran2_records(q, fracis, pdeldry, ideep, lg, do, dry)
    expect = _expected_bytes(lg, L, do, dry, pcnst)
    for source in ("dense", "gathered"):
        if source == "gathered":         # the mirror of the gathered tend step
            g = Z_.zm_conv_tend_gathered(ch.ncol, st, ch.ztodt, keep_pbuf_on_device=True)
            assert same_bits(g["lengath"], lg) and same_bits(g["ideep"], ideep)
        Z_.lib().zm_launch_count(1)
        rec = Z_.zm_conv_tend_2_gathered(lg, do, pcnst, dry, qr, fr, pr, ch.ztodt)
        launches = int(Z_.lib().zm_launch_count(1))
        assert launches == 3 + int(pr is not None), (name, launches)     # scan, [dpdry], chunk bounds, convtran
        assert Z_.last_tend_2_transfer_bytes() == expect, (name, source)
        back = Z_.scatter_convtran2(rec, ideep, lg, do, pcnst)
        assert same_bits(back, dense), (name, source)
    # the records in a larger, NaN-filled buffer: only sum(lengath)*pver*nact doubles are written
    buf = np.full(qr.size + 1000, np.nan)
    rec = Z_.zm_conv_tend_2_gathered(lg, do, pcnst, dry, qr, fr, pr, ch.ztodt, out=buf)
    assert np.isfinite(rec).all() and np.isnan(buf[qr.size:]).all()
    assert same_bits(Z_.scatter_convtran2(rec, ideep, lg, do, pcnst), dense)
    # timers keep the GPTL name
    Z_.lib().zm_set_profiling(1)
    Z_.zm_conv_tend_2_gathered(lg, do, pcnst, dry, qr, fr, pr, ch.ztodt)
    Z_.lib().zm_set_profiling(0)
    assert Z_.timers()["convtran2"] > 0.0


def _raw(Z_, nch, lengath, do, pcnst, dry, qr, fr, pr, out, cap, ztodt):
    return Z_.lib().zm_conv_tend_2_batch_gathered(
        C.c_int(nch), Z_._ip(lengath), Z_._ip(do), C.c_int(pcnst), Z_._ip(dry) if dry is not None else None,
        Z_._dp(qr), Z_._dp(fr), Z_._dp(pr) if pr is not None else None, Z_._dp(out), C.c_longlong(cap),
        C.c_double(ztodt))


@pytest.mark.gpu
def test_tend_2_gathered_refusals(built):
    """Every refusal returns an error and leaves a NaN-filled dqdt_rec untouched; nact = 0 writes nothing."""
    Z_ = init_cuda(16, 32)
    ch = S.make_chunks(16 * 120 - 3, 32, 16, p_conv=0.6)
    pcnst = 6
    do = np.array([0, 1, 0, 1, 1, 0], np.int32)
    dry = np.array([0, 0, 0, 1, 0, 0], np.int32)
    q, fracis, pdeldry = S.make_tracers(ch, pcnst)
    res = Z_.zm_conv_tend(ch.ncol, state_of(ch), ch.ztodt, keep_pbuf_on_device=True)
    lg, ideep = res["lengath"].copy(), res["ideep"].copy()
    qr, fr, pr = Z_.convtran2_records(q, fracis, pdeldry, ideep, lg, do, dry)
    need = qr.size
    nch = ch.nchunks

    def refused(rc, code, what):
        assert rc == code, (what, rc, Z_.last_error())
        assert np.isnan(out).all(), what

    out = np.full(need, np.nan)
    bad = lg.copy()
    c = int(np.argmax(lg))
    bad[c] -= 1
    refused(_raw(Z_, nch, bad, do, pcnst, dry, qr, fr, pr, out, need, ch.ztodt), -9, "lengath")
    assert "lengath" in Z_.last_error()
    refused(_raw(Z_, nch, lg, do, pcnst, dry, qr, fr, pr, out, need - 1, ch.ztodt), -9, "rec_cap")
    assert "rec_cap" in Z_.last_error()
    refused(_raw(Z_, nch, lg, do, pcnst, dry, qr, fr, None, out, need, ch.ztodt), -9, "pdeldry_rec")
    refused(_raw(Z_, nch - 1, lg[:-1], do, pcnst, dry, qr, fr, pr, out, need, ch.ztodt), -7, "nchunks")
    # nact = 0: returns 0, writes and moves nothing
    none = np.zeros(pcnst, np.int32); none[0] = 1
    assert _raw(Z_, nch, lg, none, pcnst, dry, qr, fr, pr, out, need, ch.ztodt) == 0 and np.isnan(out).all()
    assert Z_.last_tend_2_transfer_bytes() == {"h2d": 0, "d2h": 0}
    # a moist flag set needs no pdeldry_rec
    moist = np.array([0, 1, 0, 0, 1, 0], np.int32)
    qm, fm, pm = Z_.convtran2_records(q, fracis, pdeldry, ideep, lg, moist, dry)
    assert pm is None
    dm = Z_.zm_conv_tend_2(moist, q, pdeldry, fracis, ch.ztodt, dry)
    got = Z_.zm_conv_tend_2_gathered(lg, moist, pcnst, dry, qm, fm, None, ch.ztodt)
    assert same_bits(Z_.scatter_convtran2(got, ideep, lg, moist, pcnst), dm)
    # the call after the refusals succeeds
    ok = _raw(Z_, nch, lg, do, pcnst, dry, qr, fr, pr, out, need, ch.ztodt)
    assert ok == 0 and np.isfinite(out).all()
    # no mirror at all
    Z_.lib().zm_finalize()
    Z_ = init_cuda(16, 32)
    out[:] = np.nan
    refused(_raw(Z_, nch, lg, do, pcnst, dry, qr, fr, pr, out, need, ch.ztodt), -7, "no mirror")


@pytest.mark.gpu
def test_tend_2_gathered_two_threads(built):
    """Two host threads, each with its own batch and device mirror, give the single-threaded results."""
    Z_ = init_cuda(16, 32)
    pcnst = 9
    do = np.array([0, 1, 1, 0, 1, 1, 1, 0, 1], np.int32)
    dry = np.array([0, 0, 1, 0, 0, 1, 0, 0, 1], np.int32)
    batches = {"a": S.make_chunks(16 * 700, 32, 16, p_conv=0.5),
               "b": S.make_chunks(16 * 90 - 7, 32, 16, p_conv=0.7, col0=7 * 10 ** 5)}
    inputs, serial = {}, {}
    for key, ch in batches.items():
        q, fracis, pdeldry = S.make_tracers(ch, pcnst)
        res = Z_.zm_conv_tend(ch.ncol, state_of(ch), ch.ztodt, keep_pbuf_on_device=True)
        lg, ideep = res["lengath"].copy(), res["ideep"].copy()
        inputs[key] = (lg, ideep) + Z_.convtran2_records(q, fracis, pdeldry, ideep, lg, do, dry)
        serial[key] = Z_.zm_conv_tend_2(do, q, pdeldry, fracis, ch.ztodt, dry)
    results, errors = {}, []

    def worker(key):
        try:
            ch = batches[key]
            lg, ideep, qr, fr, pr = inputs[key]
            for _ in range(3):
                Z_.zm_conv_tend(ch.ncol, state_of(ch), ch.ztodt, keep_pbuf_on_device=True)
                rec = Z_.zm_conv_tend_2_gathered(lg, do, pcnst, dry, qr, fr, pr, ch.ztodt)
                results[key] = Z_.scatter_convtran2(rec, ideep, lg, do, pcnst)
        except Exception as e:      # noqa: BLE001 (reported below)
            errors.append(repr(e))

    th = [threading.Thread(target=worker, args=(k,)) for k in batches]
    for t in th:
        t.start()
    for t in th:
        t.join()
    assert not errors, errors
    for key in batches:
        assert same_bits(results[key], serial[key]), key
