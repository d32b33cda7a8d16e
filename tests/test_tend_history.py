"""History fields of the fused zm_conv_tend step (zm_conv_tend_hist_fields): zm_convr's heat, qtnd, eurt, dif, dnlf,
dnif, zm_conv_evap's tend_s and snow / net-production diagnostics, momtran's seten, pguall, pgdall, icwu, icwd.

The reference values come from the oracle's unfused procedures chained the way zm_conv_tend chains them
(zm_conv_intr.F90:662-836): zm_convr -> the physics_update statements -> zm_conv_evap on state1 -> momtran on
state1%u/v.  The CPU test pins that chain to the oracle's own zm_conv_tend; the GPU tests compare every attached
field with it bit for bit and check that attaching changes none of the regular outputs."""
import numpy as np
import pytest

from cam_nor_physics_b200 import soundings as S
from helpers import TEND_KEYS, assert_same, get_oracle, init_cuda, state_of

HIST = ["heat", "qtnd", "eurt", "dif", "dnlf", "dnif", "tend_s", "tend_s_snwprd", "tend_s_snwevmlt", "ntprprd",
        "ntsnprd", "seten", "pguall", "pgdall", "icwu", "icwd"]
MOM = ["seten", "pguall", "pgdall", "icwu", "icwd"]
SENTINEL = -777.25


def chain_reference(o, p, ch, org=None):
    """The history fields of zm_conv_tend from the oracle's unfused procedures, chunk by chunk; padding columns and,
    with cam3, the momtran fields stay 0.  Returns (history fields, zm_convr result, per-chunk evap / momtran)."""
    nch, L, pc = ch.nchunks, p.pver, p.pcols
    r = o.convr_batch(ch, org=org)
    assert r["rc"] == 0
    h = {k: np.zeros((nch, 2, L, pc) if k in ("pguall", "pgdall", "icwu", "icwd") else (nch, L, pc)) for k in HIST}
    for k in ("heat", "qtnd", "eurt", "dif", "dnlf", "dnif"):
        h[k][...] = r[k]
    ev_all, mt_all = [], []
    for c in range(nch):
        n = int(ch.ncol[c])
        t1 = ch.t[c] + r["heat"][c] * ch.ztodt / p.cpair             # physics_types.F90:427
        qn = ch.q[c] + r["qtnd"][c] * ch.ztodt                        # :322-329, qneg3 clip at qmin = 1e-12
        q1 = np.where(qn < 1.e-12, 1.e-12, qn)
        ev = o.conv_evap(n, t1, ch.pmid[c], ch.pdel[c], q1, ch.landfrac[c], r["rprd"][c], ch.cld[c], ch.ztodt,
                         r["prec"][c])
        for k in ("tend_s", "tend_s_snwprd", "tend_s_snwevmlt", "ntprprd", "ntsnprd"):
            h[k][c] = ev[k]
        ev_all.append(ev)
        if not p.cam3:
            mt = o.momtran(n, [1, 1], np.stack([ch.u[c], ch.v[c]]), r["mu"][c], r["md"][c], r["du"][c], r["eu"][c],
                           r["ed"][c], r["dp"][c], r["dsubcld"][c], r["jt"][c], r["maxg"][c], r["ideep"][c],
                           r["lengath"][c], ch.ztodt)
            for k in MOM:
                h[k][c] = mt[k]
            mt_all.append(mt)
    return h, r, ev_all, mt_all


def assert_hist(out, ref, names, ch, what):
    bad = [k for k in names if not np.array_equal(out[k], ref[k])]
    assert not bad, f"{what}: history fields differ from the unfused chain: {bad}"
    for k in names:
        for c in range(ch.nchunks):
            assert not out[k][c, ..., int(ch.ncol[c]):].any(), f"{what}: {k} padding of chunk {c} not 0"


def sentinel_out(nch, L, pc, names):
    return {k: np.full((nch, 2, L, pc) if k in ("pguall", "pgdall", "icwu", "icwd") else (nch, L, pc), SENTINEL)
            for k in names}


# ---- CPU: the reference chain is the oracle's zm_conv_tend -------------------------------------------------------
@pytest.mark.parametrize("over", [{}, {"cam3": 1, "num_cin": 5}])
def test_chain_reference_reproduces_oracle_conv_tend(built, over):
    """Summed the way zm_conv_tend sums them (ptend_s = (heat + tend_s) + seten, ptend_q = qtnd + tend_q,
    ptend_u/v = momtran's dqdt), the unfused chain's intermediates give the oracle's fused step bit for bit; so the
    history values the tests below expect are the ones inside the oracle's zm_conv_tend."""
    o, p, rc = get_oracle("pm", 16, 32, **over)
    assert rc == 0
    ch = S.make_chunks(16 * 12 - 5, 32, 16, p_conv=0.6)
    h, r, ev, mt = chain_reference(o, p, ch)
    ref = o.conv_tend_batch(ch)
    assert ref["rc"] == 0 and int(ref["lengath"].sum()) > 20
    ps = (h["heat"] + h["tend_s"]) + (0.0 if p.cam3 else h["seten"])
    assert np.array_equal(ps, ref["ptend_s"])
    assert np.array_equal(h["qtnd"] + np.stack([e["tend_q"] for e in ev]), ref["ptend_q"])
    assert np.array_equal(np.stack([e["flxprec"] for e in ev]), ref["flxprec"])
    assert np.array_equal(np.stack([e["prec"] for e in ev]), ref["prec"])
    if p.cam3:
        assert not ref["ptend_u"].any()
    else:
        assert np.array_equal(np.stack([m["dqdt"][0] for m in mt]), ref["ptend_u"])
        assert np.array_equal(np.stack([m["dqdt"][1] for m in mt]), ref["ptend_v"])
        assert np.count_nonzero(h["pguall"]) > 0 and np.count_nonzero(h["icwd"]) > 0
    assert np.count_nonzero(h["tend_s_snwprd"]) > 0 and np.count_nonzero(h["eurt"]) > 0


# ---- GPU: host-pointer step ---------------------------------------------------------------------------------------
CONFIGS = {
    "default": (16, 32, {}, 16 * 90 - 3),
    "cam3": (16, 32, {"cam3": 1, "num_cin": 5}, 16 * 90 - 3),
    "zm_org": (16, 32, {"zm_org": 1}, 16 * 90 - 3),
    "L58_parcel_pbl": (16, 58, {"lparcel_pbl": 1}, 16 * 40 - 3),
    "odd_13x29": (13, 29, {}, 13 * 91 - 3),          # odd pcols*pver: packed winds and the unfused evap kernel
}


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(CONFIGS))
def test_host_step_history_fields(built, name):
    pc, L, over, ncols = CONFIGS[name]
    Z = init_cuda(pc, L, **over)
    o, p, rc = get_oracle("pm", pc, L, **over)
    assert rc == 0
    ch = S.make_chunks(ncols, L, pc, p_conv=0.6)
    st = state_of(ch)
    org = None
    if over.get("zm_org"):
        org = np.maximum(np.random.default_rng(3).uniform(-0.3, 1.0, ch.t.shape), 0.0)
        st["org"] = org
    href, _, _, _ = chain_reference(o, p, ch, org=org)
    ref = o.conv_tend_batch(ch, org=org)
    out = Z.zm_conv_tend(ch.ncol, st, ch.ztodt, hist=True)
    keys = TEND_KEYS + (["orgt", "org2d"] if org is not None else [])
    assert_same(out, ref, keys, pc, exact=True, what=f"{name}: regular outputs with history attached")
    assert_hist(out, href, HIST, ch, name)
    if over.get("cam3"):
        assert all(not out[k].any() for k in MOM)
    else:
        assert np.count_nonzero(out["icwu"]) > 0 and np.count_nonzero(out["pgdall"]) > 0
    # every element is written, whatever the arrays held
    regular = {k: v.copy() for k, v in out.items() if k not in HIST}
    out2 = Z.zm_conv_tend(ch.ncol, st, ch.ztodt, out={**regular, **sentinel_out(ch.nchunks, L, pc, HIST)}, hist=True)
    assert_hist(out2, href, HIST, ch, name + " (sentinel-filled arrays)")


@pytest.mark.gpu
def test_pipelined_history_fields_and_transfer_bytes(built, monkeypatch):
    """1,100 chunks: the default schedule of four sub-batches slices the history arrays like every other output;
    they travel whole (also under ZM_TEND_RETURN=sparse) and are exactly the extra device->host bytes."""
    Z = init_cuda(16, 32)
    o, p, _ = get_oracle("pm", 16, 32)
    ch = S.make_chunks(16 * 1100, 32, 16, p_conv=0.5)
    ref = o.conv_tend_batch(ch)
    href, _, _, _ = chain_reference(o, p, ch)
    for ret in ("dense", "sparse"):
        monkeypatch.setenv("ZM_TEND_RETURN", ret)
        plain = Z.zm_conv_tend(ch.ncol, state_of(ch), ch.ztodt)
        b0 = Z.last_transfer_bytes()
        out = {k: np.full_like(v, 7 if v.dtype.kind == "i" else SENTINEL) for k, v in plain.items()}
        out.update(sentinel_out(ch.nchunks, 32, 16, HIST))
        out = Z.zm_conv_tend(ch.ncol, state_of(ch), ch.ztodt, out=out, hist=True)
        b1 = Z.last_transfer_bytes()
        assert Z.tend_trace().shape[0] == 4
        for k in plain:
            assert np.array_equal(out[k], plain[k]), (ret, k)
        assert_same(out, ref, TEND_KEYS, 16, exact=True, what=f"pipelined ({ret}) regular outputs")
        assert_hist(out, href, HIST, ch, f"pipelined ({ret})")
        assert b1["h2d"] == b0["h2d"]
        assert b1["d2h"] - b0["d2h"] == sum(out[k].nbytes for k in HIST), ret


# ---- GPU: isolation -------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("split", ["1", "0"])
def test_subset_attach_and_one_shot(built, monkeypatch, split):
    """A subset attaches only itself (the other arrays keep their contents); the attachment is one-shot and leaves
    the next step exactly a never-attached step, launch count included.  With every field attached the zero-fill list
    of the split-wind step is at its limit (an overflow would fail the call)."""
    monkeypatch.setenv("ZM_TEND_SPLIT_WINDS", split)
    Z = init_cuda(16, 32)
    ch = S.make_chunks(16 * 150 - 7, 32, 16, p_conv=0.6)
    st = state_of(ch)
    L = Z.lib()
    L.zm_launch_count(1)
    plain = Z.zm_conv_tend(ch.ncol, st, ch.ztodt)
    n_plain = L.zm_launch_count(1)
    full = Z.zm_conv_tend(ch.ncol, st, ch.ztodt, hist=True)
    n_full = L.zm_launch_count(1)
    assert n_full == n_plain + 1                           # the in-cloud wind initialisation
    sub = ["tend_s", "icwd"]
    out = {k: v.copy() for k, v in plain.items()}
    out.update(sentinel_out(ch.nchunks, 32, 16, HIST))
    out = Z.zm_conv_tend(ch.ncol, st, ch.ztodt, out=out, hist=sub)
    for k in HIST:
        if k in sub:
            assert np.array_equal(out[k], full[k]), k
        else:
            assert np.all(out[k] == SENTINEL), k
    L.zm_launch_count(1)
    after = Z.zm_conv_tend(ch.ncol, st, ch.ztodt)
    assert L.zm_launch_count(1) == n_plain
    assert not any(k in after for k in HIST)
    for k in plain:
        assert np.array_equal(after[k], plain[k]) and np.array_equal(full[k], plain[k]), k


# ---- GPU: device-resident step ----------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("subbatches", ["1", "2"])
def test_device_step_history_graph_replay(built, monkeypatch, subbatches):
    """DeviceTend(hist=True): direct, captured and replayed steps all write every history field (sentinel-filled
    before each step) with the host-pointer step's values; other pointers attached force a new capture, and the
    graph never writes to the pointers of an earlier attachment."""
    import torch
    from cam_nor_physics_b200.device import DeviceTend
    monkeypatch.setenv("ZM_DEV_SUBBATCHES", subbatches)
    Z = init_cuda(16, 32)
    ch = S.make_chunks(16 * 300 - 5, 32, 16, p_conv=0.5)
    ref = Z.zm_conv_tend(ch.ncol, state_of(ch), ch.ztodt, hist=True)
    dev = DeviceTend(ch, hist=True)
    plain = DeviceTend(ch)
    L = Z.lib()

    def check(d, what):
        assert d.check() == 0
        for k in TEND_KEYS:
            assert np.array_equal(d.out[k].cpu().numpy(), ref[k]), (what, k)
        for k, v in d.hist.items():
            assert np.array_equal(v.cpu().numpy(), ref[k]), (what, k)

    L.zm_launch_count(1)
    plain.step()
    plain.check()
    n_plain = L.zm_launch_count(1)
    counts = []
    for it in range(4):
        for v in list(dev.out.values()) + list(dev.hist.values()):
            v.fill_(SENTINEL)
        dev.step()
        counts.append(L.zm_launch_count(1))
        check(dev, f"step {it}")
    assert len(set(counts)) == 1 and counts[0] > n_plain
    old = dev.hist
    dev.hist = {k: torch.full_like(v, SENTINEL) for k, v in old.items()}
    for v in old.values():
        v.fill_(SENTINEL)
    for it in range(3):
        dev.step()
        check(dev, f"new pointers, step {it}")
    for k, v in old.items():
        assert bool((v == SENTINEL).all()), f"{k}: a step wrote to a detached array"
    # the plain step after all this: same launches, same bits
    L.zm_launch_count(1)
    plain.step()
    plain.check()
    assert L.zm_launch_count(1) == n_plain
    for k in TEND_KEYS:
        assert np.array_equal(plain.out[k].cpu().numpy(), ref[k]), k
