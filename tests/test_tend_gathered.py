"""zm_conv_tend_batch_gathered: the host-pointer step with the (pcols,pver[p]) outputs returned as one record per
convective column, for the caller's own per-chunk scatter (the batched Fortran binding's gathered mode).

The contract rests on a premise that is asserted here first: in zm_conv_tend_batch's dense outputs the fourteen
column-indexed fields are exactly 0 outside the convective columns ideep(1:lengath), and the six pbuf fields are
exactly 0 in the rows above lengath.  Then the records, scattered, must give the dense step's arrays bit for bit,
in every configuration, pipeline schedule and attachment, and the bytes the step moves must be exactly the dense
bytes minus the arrays the records replace plus the records."""
import gc
import importlib.util
import os
import tempfile
import threading
import weakref

import numpy as np
import pytest

from cam_nor_physics_b200 import soundings as S
from cam_nor_physics_b200 import zm_conv as Z
from helpers import TEND_KEYS, assert_same, get_oracle, init_cuda, state_of

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
COL_FIELDS = Z.GATHERED_FIELDS
PBUF = Z.GATHERED_PBUF
PBUF_MIRROR = PBUF + ["dsubcld", "jt", "maxg"]        # what keep_pbuf_on_device leaves in the device mirror


def _cost_script():
    spec = importlib.util.spec_from_file_location("tend_gathered_cost",
                                                  os.path.join(ROOT, "scripts", "tend_gathered_cost.py"))
    m = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(m)
    return m


def same_bits(a, b):
    a, b = np.asarray(a), np.asarray(b)
    if a.dtype == np.float64:
        a, b = a.view(np.int64), b.view(np.int64)
    return a.shape == b.shape and np.array_equal(a, b)


def pack_records(dense, pver, with_pbuf):
    """numpy packer: the records zm_conv_tend_batch_gathered must return, from the dense outputs."""
    lay, rec_len = Z.gathered_layout(pver, with_pbuf)
    rows = []
    for c in range(dense["lengath"].shape[0]):
        for j in range(int(dense["lengath"][c])):
            i = int(dense["ideep"][c, j]) - 1
            r = np.empty(rec_len)
            for k, (o, n) in lay.items():
                r[o:o + n] = dense[k][c, :, j if k in PBUF else i]
            rows.append(r)
    return np.array(rows).reshape(len(rows), rec_len)


# ---- CPU: the C scatter of scripts/chunk_loop2.c equals scatter_gathered -------------------------------------------
@pytest.mark.parametrize("with_pbuf", [0, 1])
def test_chunk_loop2_scatter_matches_scatter_gathered(with_pbuf):
    """Synthetic records (random lengath including 0 and pcols, random distinct ideep): the gathered loop 2 of
    chunk_loop2.c, writing every chunk's buffer, equals scatter_gathered's dense arrays, and its dense loop 2 copies
    those arrays back into the same buffers.  Together with tests/test_fortran_binding.py this pins the record layout
    short of a Fortran compiler."""
    cost = _cost_script()
    rng = np.random.default_rng(11 + with_pbuf)
    nch, pc, L = 37, 13, 9
    lengath = rng.integers(0, pc + 1, nch).astype(np.int32)
    lengath[3], lengath[4] = 0, pc
    ideep = np.zeros((nch, pc), np.int32)
    for c in range(nch):
        ideep[c, :lengath[c]] = rng.permutation(pc)[:lengath[c]] + 1
    _, rec_len = Z.gathered_layout(L, bool(with_pbuf))
    res = dict(lengath=lengath, ideep=ideep, rec=rng.standard_normal((int(lengath.sum()), rec_len)),
               pbuf_in_records=with_pbuf)
    for k in Z.GATHERED_COL_OUT + ["jt", "maxg"]:
        res[k] = np.zeros((nch, pc))
    dense = Z.scatter_gathered(res)
    full_len = 20 * L + 4
    with tempfile.TemporaryDirectory() as tmp:
        lib = cost.load_loop2(tmp)
        got = np.full(nch * pc * full_len, np.nan)
        cost.run_gathered(lib, Z, 3, res, L, got, pc * full_len)
        back = np.full(nch * pc * full_len, np.nan)
        cost.run_dense(lib, Z, 3, dense, back, pc * full_len)
        scratch = np.zeros(4 * pc * full_len)          # per-thread chunk buffers (the timed form) must not fault
        cost.run_gathered(lib, Z, 4, res, L, scratch)
    got = got.reshape(nch, pc * full_len)
    assert same_bits(got, back.reshape(nch, pc * full_len))
    off = 0
    for k in cost.chunk_fields(Z):
        n = (L + 1 if k in Z.TEND_OUT_2DP else L) * pc
        assert same_bits(got[:, off:off + n].reshape(dense[k].shape), dense[k]), k
        off += n
    # scatter_gathered itself, against the packer: packing its arrays gives the records back
    assert same_bits(pack_records(dense, L, bool(with_pbuf)), res["rec"])
    if not with_pbuf:
        assert all(not dense[k].any() for k in PBUF)


class _StubLib:
    """Stands in for libzmconv_b200.so: remembers (weakly) every array an attachment call hands over as a raw pointer
    and, when the step is called, whether each of them is still alive."""

    def __init__(self):
        self.held, self.alive_at_step = [], None

    def _hold(self, *ptrs):
        self.held += [weakref.ref(p._arr) for p in ptrs if p is not None]
        return 0

    def zm_org_fields(self, org, orgt, org2d):
        return self._hold(org, orgt, org2d)

    def zm_convtran1_fields(self, pcnst, doconvtran, cnst_is_dry, q, fracis, ptend_q):
        return self._hold(q, fracis, ptend_q)

    def zm_conv_tend_hist_fields(self, *ptrs):
        return self._hold(*ptrs)

    def _step(self, *args):
        gc.collect()
        self.alive_at_step = [r() is not None for r in self.held]
        return 0

    zm_conv_tend_batch = zm_conv_tend_batch_gathered = _step


@pytest.mark.parametrize("entry", ["zm_conv_tend", "zm_conv_tend_gathered"])
def test_attached_copies_outlive_the_step(monkeypatch, entry):
    """org and the convtran1 q / fracis are attached as raw pointers before the step.  When they arrive as float32 or
    non-contiguous arrays the marshalling makes a float64 copy, and that copy must still exist when the step reads it."""
    stub = _StubLib()
    monkeypatch.setattr(Z, "_lib", stub)
    p = Z.ZmParams()
    p.pcols, p.pver = 16, 32
    monkeypatch.setattr(Z, "_params", p)
    ch = S.make_chunks(16 * 6, 32, 16, p_conv=0.6)
    st = state_of(ch)
    st["org"] = np.full(ch.t.shape, 0.25, np.float32)
    q, fracis, _ = S.make_tracers(ch, 4)
    t1 = dict(doconvtran=[0, 1, 1, 0], cnst_is_dry=None, q=np.asfortranarray(q), fracis=fracis.astype(np.float32))
    getattr(Z, entry)(ch.ncol, st, ch.ztodt, convtran1=t1, hist=["heat"])
    assert stub.alive_at_step is not None and len(stub.held) == 7
    assert all(stub.alive_at_step), stub.alive_at_step


# ---- GPU -----------------------------------------------------------------------------------------------------------
def _concat(a, b):
    import dataclasses
    kw = {f.name: (np.concatenate([getattr(a, f.name), getattr(b, f.name)])
                   if isinstance(getattr(a, f.name), np.ndarray) else getattr(a, f.name))
          for f in dataclasses.fields(a)}
    kw["nchunks"] = a.nchunks + b.nchunks
    return S.Chunks(**kw)


def make_case(name):
    """(pcols, pver, params, chunks, org)"""
    pc, L, over = {"p16_L32_1100": (16, 32, {}), "cam3": (16, 32, {"cam3": 1, "num_cin": 5}),
                   "zm_org": (16, 32, {"zm_org": 1}), "L58_parcel_pbl": (16, 58, {"lparcel_pbl": 1}),
                   "odd_13x29": (13, 29, {}), "pcols128": (128, 32, {}), "lengath_0_and_full": (16, 32, {}),
                   "ragged_ncol": (16, 32, {})}[name]
    if name == "p16_L32_1100":
        ch = S.make_chunks(16 * 1100 + 5, L, pc, p_conv=0.45)
    elif name == "L58_parcel_pbl":
        ch = S.make_chunks(16 * 40 - 3, L, pc, p_conv=0.6)
    elif name == "odd_13x29":
        ch = S.make_chunks(13 * 91 - 3, L, pc, p_conv=0.6)
    elif name == "pcols128":
        ch = S.make_chunks(128 * 20 - 7, L, pc, p_conv=0.5)
    elif name == "lengath_0_and_full":          # all-stable chunks (lengath 0) next to all-tropical ones
        ch = _concat(S.make_chunks(16 * 24, L, pc, p_conv=1.0), S.make_chunks(16 * 8, L, pc, p_conv=0.0, col0=10 ** 6))
    elif name == "ragged_ncol":
        ch = S.make_chunks(16 * 120, L, pc, p_conv=0.6)
        ch.ncol = np.random.default_rng(5).integers(1, pc + 1, ch.nchunks).astype(np.int32)
    else:
        ch = S.make_chunks(16 * 90 - 3, L, pc, p_conv=0.6)
    org = np.maximum(np.random.default_rng(3).uniform(-0.3, 1.0, ch.t.shape), 0.0) if over.get("zm_org") else None
    return pc, L, over, ch, org


CASES = ["p16_L32_1100", "cam3", "zm_org", "L58_parcel_pbl", "odd_13x29", "pcols128", "lengath_0_and_full",
         "ragged_ncol"]


def _state(ch, org):
    st = state_of(ch)
    if org is not None:
        st["org"] = org
    return st


def _dense_part(out):
    return {k: v for k, v in out.items() if k in TEND_KEYS}


@pytest.mark.gpu
@pytest.mark.parametrize("name", CASES)
def test_gathered_step(built, monkeypatch, name):
    pc, L, over, ch, org = make_case(name)
    Z_ = init_cuda(pc, L, **over)
    st = _state(ch, org)
    o, _, rc = get_oracle("pm", pc, L, **over)
    assert rc == 0
    ref = o.conv_tend_batch(ch, org=org)                   # (j) the oracle
    assert ref["rc"] == 0
    dense_full = Z_.zm_conv_tend(ch.ncol, st, ch.ztodt)
    b_full = Z_.last_transfer_bytes()
    dense_keep = Z_.zm_conv_tend(ch.ncol, st, ch.ztodt, keep_pbuf_on_device=True)
    b_keep = Z_.last_transfer_bytes()
    lg, ideep = dense_full["lengath"], dense_full["ideep"]
    nconv = int(lg.sum())
    assert nconv > 0
    if name == "lengath_0_and_full":
        assert (lg == 0).any() and ((lg == pc) & (ch.ncol == pc)).any(), lg
    # (a) the premise: zero outside the convective columns / above lengath
    incol = np.zeros((ch.nchunks, pc), bool)
    for c in range(ch.nchunks):
        incol[c, ideep[c, :lg[c]] - 1] = True
    inrow = np.arange(pc)[None, :] < lg[:, None]
    for k in COL_FIELDS:
        assert not dense_full[k][np.broadcast_to(~incol[:, None, :], dense_full[k].shape)].any(), f"{name}: {k}"
    for k in PBUF:
        assert not dense_full[k][np.broadcast_to(~inrow[:, None, :], dense_full[k].shape)].any(), f"{name}: {k}"

    # dense mirror consumers, for (e)
    ps = ch.pint[:, -1, :]
    q3, fracis, pdeldry = S.make_tracers(ch, 4)
    do, dry = [0, 1, 1, 1], [0, 0, 1, 0]
    Z_.zm_conv_tend(ch.ncol, st, ch.ztodt, keep_pbuf_on_device=True)
    mirror_ref = (Z_.zm_conv_tend_2(do, q3, pdeldry, fracis, ch.ztodt, dry), Z_.zm_conv_tend_diag(ch.ncol, ps, ch.pmid))

    for pbuf in (1, 0):
        keep = not pbuf
        dense = dense_keep if keep else dense_full
        res = Z_.zm_conv_tend_gathered(ch.ncol, st, ch.ztodt, keep_pbuf_on_device=keep)
        bg = Z_.last_transfer_bytes()
        _, rec_len = Z_.gathered_layout(L, bool(pbuf))
        assert res["rec"].shape == (nconv, rec_len)
        # (b) scattered records == dense outputs, per-column outputs identical
        back = Z_.scatter_gathered(res)
        for k in TEND_KEYS:
            assert same_bits(back[k], dense[k]), (name, pbuf, k)
        # (c) record order
        assert same_bits(res["rec"], pack_records(dense_full, L, bool(pbuf))), (name, pbuf)
        # (j) oracle, bit for bit (mu..dp / dsubcld / jt / maxg only where they travel)
        keys = [k for k in TEND_KEYS if not (keep and k in PBUF_MIRROR)]
        assert_same(back, ref, keys, pc, exact=True, what=f"{name} pbuf={pbuf}: gathered vs oracle")
        if org is not None:
            assert same_bits(res["orgt"], ref["orgt"]) and same_bits(res["org2d"], ref["org2d"])
        # (g) bytes: the dense step's, minus the arrays the records replace, plus the records
        replaced = sum(dense[k].nbytes for k in COL_FIELDS + (PBUF if pbuf else []))
        b_dense = b_keep if keep else b_full
        assert bg["h2d"] == b_dense["h2d"]
        assert bg["d2h"] == b_dense["d2h"] - replaced + nconv * rec_len * 8, (name, pbuf, bg, b_dense)
        # (d) pipeline schedules
        for var, val in (("ZM_TEND_SUBBATCHES", "1"), ("ZM_TEND_SUBBATCHES", "4"), ("ZM_TEND_SUBBATCHES", "8"),
                         ("ZM_TEND_SCHEDULE", "1,1,2,4,4,4")):
            monkeypatch.setenv(var, val)
            r2 = Z_.zm_conv_tend_gathered(ch.ncol, st, ch.ztodt, keep_pbuf_on_device=keep)
            monkeypatch.delenv(var)
            assert same_bits(r2["rec"], res["rec"]), (name, pbuf, var, val)
            for k in Z_.GATHERED_COL_OUT + ["jt", "maxg", "ideep", "lengath"]:
                assert same_bits(r2[k], res[k]), (name, pbuf, var, val, k)
        # (e) the device mirror the gathered step leaves
        Z_.zm_conv_tend_gathered(ch.ncol, st, ch.ztodt, keep_pbuf_on_device=keep)
        dq = Z_.zm_conv_tend_2(do, q3, pdeldry, fracis, ch.ztodt, dry)
        dg = Z_.zm_conv_tend_diag(ch.ncol, ps, ch.pmid)
        assert same_bits(dq, mirror_ref[0]), (name, pbuf)
        for k in dg:
            assert same_bits(dg[k], mirror_ref[1][k]), (name, pbuf, k)


@pytest.mark.gpu
@pytest.mark.parametrize("name", CASES)
def test_gathered_attachments(built, name):
    """(f) convtran1 and every history field attached: their arrays travel whole and equal the dense step's; the
    records do not change."""
    pc, L, over, ch, org = make_case(name)
    Z_ = init_cuda(pc, L, **over)
    st = _state(ch, org)
    pcnst = 5
    q, fracis, _ = S.make_tracers(ch, pcnst)
    t1 = dict(doconvtran=[1, 1, 0, 1, 1], cnst_is_dry=[0, 0, 0, 1, 0], q=q, fracis=fracis,
              ptend_q=np.full_like(q, 3.0))
    dense = Z_.zm_conv_tend(ch.ncol, st, ch.ztodt, convtran1=t1, hist=True)
    plain = Z_.zm_conv_tend_gathered(ch.ncol, st, ch.ztodt)
    plain = {k: (v.copy() if isinstance(v, np.ndarray) else v) for k, v in plain.items()}
    for pbuf in (1, 0):
        res = Z_.zm_conv_tend_gathered(ch.ncol, st, ch.ztodt, keep_pbuf_on_device=not pbuf, convtran1=t1, hist=True)
        for k in Z_.HIST_FIELDS + ["ptend_qc"] + (["orgt", "org2d"] if org is not None else []):
            assert same_bits(res[k], dense[k]), (name, pbuf, k)
        back = Z_.scatter_gathered(res)
        for k in TEND_KEYS:
            if pbuf or k not in PBUF_MIRROR:
                assert same_bits(back[k], dense[k]), (name, pbuf, k)
        if pbuf:
            assert same_bits(res["rec"], plain["rec"])
    # one-shot: the next call has nothing attached
    after = Z_.zm_conv_tend_gathered(ch.ncol, st, ch.ztodt)
    assert "heat" not in after and same_bits(after["rec"], plain["rec"])


@pytest.mark.gpu
def test_gathered_rec_cap_and_required_arguments(built):
    """(h) a record buffer below nchunks*pcols*rec_len is refused with a message before any work: nothing is written,
    the attachments stay for the next call, which succeeds.  NULL ideep / lengath are refused too."""
    Z_ = init_cuda(16, 32)
    ch = S.make_chunks(16 * 200 - 3, 32, 16, p_conv=0.5)
    st = state_of(ch)
    good = Z_.zm_conv_tend_gathered(ch.ncol, st, ch.ztodt, hist=["heat"])
    good = {k: (v.copy() if isinstance(v, np.ndarray) else v) for k, v in good.items()}
    _, rec_len = Z_.gathered_layout(32, True)
    cap = ch.nchunks * 16 * rec_len
    out = {k: np.full_like(good[k], 7 if good[k].dtype.kind == "i" else -5.5)
           for k in Z_.GATHERED_COL_OUT + ["jt", "maxg", "ideep", "lengath", "heat"]}
    out["rec_buf"] = np.full(cap - 1, -5.5)
    with pytest.raises(Z_.ZmError, match="rec_cap"):
        Z_.zm_conv_tend_gathered(ch.ncol, st, ch.ztodt, out=out, hist=["heat"])
    for k, v in out.items():
        assert np.all(v == (7 if v.dtype.kind == "i" else -5.5)), k
    out["rec_buf"] = np.full(cap, -5.5)
    res = Z_.zm_conv_tend_gathered(ch.ncol, st, ch.ztodt, out=out)   # the refused call's attachment is still there
    assert same_bits(res["heat"], good["heat"]) and same_bits(res["rec"], good["rec"])
    for k in Z_.GATHERED_COL_OUT + ["jt", "maxg", "ideep", "lengath"]:
        assert same_bits(res[k], good[k]), k
    assert np.all(out["rec_buf"][res["rec"].size:] == -5.5)          # only sum(lengath)*rec_len doubles written
    # required pointers
    L = Z_.lib()
    args = [ch.nchunks, Z_._ip(ch.ncol)] + [Z_._dp(np.ascontiguousarray(st[k])) for k in Z_.TEND_IN_ORDER]
    one = [Z_._dp(np.zeros((ch.nchunks, 16))) for _ in range(8)]
    ints = [Z_._ip(np.zeros((ch.nchunks, 16), np.int32)) for _ in range(3)]
    rc = L.zm_conv_tend_batch_gathered(*args, Z_.C.c_double(ch.ztodt), *one, ints[0], ints[1], None,
                                       Z_._ip(np.zeros(ch.nchunks, np.int32)), 1, Z_._dp(out["rec_buf"]),
                                       Z_.C.c_longlong(cap))
    assert rc < 0 and "ideep" in Z_.last_error()


@pytest.mark.gpu
def test_gathered_growth_and_threads(built):
    """(i) a small batch, then a larger one (the arenas grow), and two host threads with batches of their own: each
    result equals the serial dense step of the same batch."""
    Z_ = init_cuda(16, 32)
    big = S.make_chunks(16 * 1100, 32, 16, p_conv=0.5)
    small = S.make_chunks(16 * 30 - 5, 32, 16, p_conv=0.7, col0=5 * 10 ** 5)
    dense = {}
    for key, ch in (("small", small), ("big", big)):
        dense[key] = Z_.zm_conv_tend(ch.ncol, state_of(ch), ch.ztodt)

    def check(res, key):
        back = Z_.scatter_gathered(res)
        for k in TEND_KEYS:
            assert same_bits(back[k], dense[key][k]), (key, k)

    Z_.lib().zm_finalize()
    Z_ = init_cuda(16, 32)
    for key, ch in (("small", small), ("big", big)):
        check(Z_.zm_conv_tend_gathered(ch.ncol, state_of(ch), ch.ztodt), key)
    results, errors = {}, []

    def worker(key, ch):
        try:
            for _ in range(3):
                results[key] = Z_.zm_conv_tend_gathered(ch.ncol, state_of(ch), ch.ztodt)
        except Exception as e:      # noqa: BLE001 (reported below)
            errors.append(repr(e))

    th = [threading.Thread(target=worker, args=(k, c)) for k, c in (("small", small), ("big", big))]
    for t in th:
        t.start()
    for t in th:
        t.join()
    assert not errors, errors
    for key in ("small", "big"):
        check(results[key], key)


@pytest.mark.gpu
@pytest.mark.parametrize("entry", ["zm_conv_tend", "zm_conv_tend_gathered"])
def test_converted_attachments_give_the_same_step(built, entry):
    """A float32 org and non-contiguous / float32 convtran1 q and fracis are converted by the marshalling; the step
    must give what the same values give as contiguous float64 arrays."""
    Z_ = init_cuda(16, 32, zm_org=1)
    ch = S.make_chunks(16 * 200 - 3, 32, 16, p_conv=0.6)
    org32 = np.maximum(np.random.default_rng(3).uniform(-0.3, 1.0, ch.t.shape), 0.0).astype(np.float32)
    q, fracis, _ = S.make_tracers(ch, 5)
    f32 = fracis.astype(np.float32)
    do = [1, 1, 0, 1, 1]
    run = getattr(Z_, entry)
    ref = run(ch.ncol, {**state_of(ch), "org": org32.astype(np.float64)}, ch.ztodt,
              convtran1=dict(doconvtran=do, q=q.copy(), fracis=f32.astype(np.float64)))
    ref = {k: (v.copy() if isinstance(v, np.ndarray) else v) for k, v in ref.items()}
    got = run(ch.ncol, {**state_of(ch), "org": org32}, ch.ztodt,
              convtran1=dict(doconvtran=do, q=np.asfortranarray(q), fracis=f32))
    assert int(ref["lengath"].sum()) > 0
    for k, v in ref.items():
        if isinstance(v, np.ndarray):
            assert same_bits(got[k], v), (entry, k)
