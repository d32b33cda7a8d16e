"""zm_conv_tend_2 (convtran2) with its host loops, dense against gathered, on the f09 shard of BASELINE config 4:
55,296 columns x L32 in pcols=16 chunks, bench.py's soundings (p_conv 0.35), the 41-constituent stand-in with
doconvtran(4:41) set and every third of those dry (do2[3:] = 1, dry[3::3] = 1 in 0-based terms, as bench.py).

dense:    loop 1 copies each chunk's q, fracis, pdeldry whole into the rank-level arrays and zeroes ptend_q,
          zm_conv_tend_2_batch, loop 2 zeroes each chunk's ptend%q and copies the flagged slices;
gathered: loop 1 packs each chunk's convective columns of the flagged constituents (and their pdeldry),
          zm_conv_tend_2_batch_gathered, loop 2 zeroes each chunk's ptend%q and scatters the chunk's records.
The loops are scripts/tend2_loops.c, built here with gcc -O2 -fopenmp into a temporary directory, timed on 1 and on
min(16, cores) threads.  The mirror comes from one gathered zm_conv_tend step with keep_pbuf_on_device.  Every host
array is page-locked once before timing.  Before any timing the gathered records, scattered by tend2_loops.c and by
scatter_convtran2, are checked to equal the dense tendency bit for bit, and the C pack to equal convtran2_records.
The calls alternate dense / gathered; the host clock brackets each call (it returns synchronised) and each loop.
PCIe bytes come from zm_tend_2_transfer_bytes.  Writes one JSON record (GPU name and power limit included)."""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

NCOLS_F09, PVER, PCOLS, PCONV, PCNST = 55296, 32, 16, 0.35, 41
LOOPS_SRC = os.path.join(ROOT, "scripts", "tend2_loops.c")


def load_loops(tmpdir: str) -> C.CDLL:
    so = os.path.join(tmpdir, "libtend2_loops.so")
    subprocess.run(["gcc", "-O2", "-fopenmp", "-shared", "-fPIC", LOOPS_SRC, "-o", so], check=True)
    lib = C.CDLL(so)
    dp, ip, i, ll = C.POINTER(C.c_double), C.POINTER(C.c_int), C.c_int, C.c_longlong
    lib.loop1_dense.argtypes = [i, i, i, i, i, dp, dp, dp, dp, dp, dp, dp]
    lib.loop1_gathered.argtypes = [i, i, i, i, i, i, ip, ip, ip, dp, dp, dp, dp, dp, dp]
    lib.loop2_dense.argtypes = [i, i, i, i, i, i, ip, dp, dp, ll]
    lib.loop2_gathered.argtypes = [i, i, i, i, i, i, ip, ip, ip, dp, dp, ll]
    return lib


def gpu_info() -> dict:
    import torch
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    if q.returncode != 0:
        return {"gpu": torch.cuda.get_device_name(0), "power_limit": "unknown", "max_sm_clock": "unknown"}
    name, power, clk = [x.strip() for x in q.stdout.strip().splitlines()[0].split(",")]
    return {"gpu": name, "power_limit": power, "max_sm_clock": clk}


def stats(v):
    v = np.asarray(v)
    return {"median_ms": float(np.median(v)), "p10_ms": float(np.percentile(v, 10)),
            "p90_ms": float(np.percentile(v, 90)), "n": int(v.size)}


def main():
    import torch
    from cam_nor_physics_b200 import soundings as S, zm_conv as Z
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=100, help="timed calls per form (alternating)")
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--loop-reps", type=int, default=10, help="timed passes of each host loop per thread count")
    ap.add_argument("--ncols", type=int, default=NCOLS_F09)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "tend2_gathered_cost_f09.json"))
    a = ap.parse_args()
    assert torch.cuda.is_available(), "needs a CUDA device"
    torch.cuda.set_device(0)
    Z.zm_init(Z.default_params(PCOLS, PVER, S.limcnv_for(PVER)))
    ch = S.make_chunks(a.ncols, PVER, PCOLS, p_conv=PCONV)
    nch, L, pc = ch.nchunks, PVER, PCOLS
    pin = lambda x: torch.from_numpy(np.ascontiguousarray(x)).pin_memory().numpy()
    zeros = lambda shape, dt=torch.float64: torch.zeros(shape, dtype=dt).pin_memory().numpy()
    do = np.zeros(PCNST, np.int32); do[3:] = 1
    dry = np.zeros(PCNST, np.int32); dry[3::3] = 1
    act = Z.convtran2_active(do, PCNST)
    iact = np.ascontiguousarray(act, dtype=np.int32)
    nact = len(act)
    q, fracis, pdeldry = S.make_tracers(ch, PCNST)
    q, fracis, pdeldry = pin(q), pin(fracis), pin(pdeldry)              # the model's state%q, fracis, pdeldry

    # the mirror: one gathered tend step with the pbuf fields kept on the device
    g = Z.zm_conv_tend_gathered(ch.ncol, {k: getattr(ch, k) for k in Z.TEND_IN_ORDER}, ch.ztodt,
                                keep_pbuf_on_device=True)
    lengath, ideep = pin(g["lengath"]), pin(g["ideep"])
    ncv = int(lengath.astype(np.int64).sum())
    nrec = ncv * L * nact
    # dense form's rank-level arrays, gathered form's record buffers
    q_b, f_b, p_b, dq_b = zeros(q.shape), zeros(q.shape), zeros(pdeldry.shape), zeros(q.shape)
    q_r, f_r, p_r, dq_r = zeros(nrec), zeros(nrec), zeros(ncv * L), zeros(nrec)
    nth = min(16, os.cpu_count() or 1)
    lib2 = Z.lib()

    def call(form):
        if form == "dense":
            rc = lib2.zm_conv_tend_2_batch(C.c_int(nch), Z._ip(do), Z._dp(q_b), C.c_int(PCNST), Z._dp(p_b), Z._dp(f_b),
                                           Z._dp(dq_b), C.c_double(ch.ztodt), Z._ip(dry))
        else:
            rc = lib2.zm_conv_tend_2_batch_gathered(C.c_int(nch), Z._ip(lengath), Z._ip(do), C.c_int(PCNST), Z._ip(dry),
                                                    Z._dp(q_r), Z._dp(f_r), Z._dp(p_r), Z._dp(dq_r),
                                                    C.c_longlong(nrec), C.c_double(ch.ztodt))
        Z._check(rc, form)

    with tempfile.TemporaryDirectory() as tmp:
        lib = load_loops(tmp)
        ptend = zeros(nth * pc * L * PCNST)          # per-thread chunk ptend%q buffers

        def loop1(form, nt):
            if form == "dense":
                lib.loop1_dense(nt, nch, pc, L, PCNST, Z._dp(q), Z._dp(fracis), Z._dp(pdeldry), Z._dp(q_b), Z._dp(f_b),
                                Z._dp(p_b), Z._dp(dq_b))
            else:
                lib.loop1_gathered(nt, nch, pc, L, PCNST, nact, Z._ip(iact), Z._ip(lengath), Z._ip(ideep), Z._dp(q),
                                   Z._dp(fracis), Z._dp(pdeldry), Z._dp(q_r), Z._dp(f_r), Z._dp(p_r))

        def loop2(form, nt, dst=ptend, stride=0):
            if form == "dense":
                lib.loop2_dense(nt, nch, pc, L, PCNST, nact, Z._ip(iact), Z._dp(dq_b), Z._dp(dst), stride)
            else:
                lib.loop2_gathered(nt, nch, pc, L, PCNST, nact, Z._ip(iact), Z._ip(lengath), Z._ip(ideep), Z._dp(dq_r),
                                   Z._dp(dst), stride)

        # ---- correctness before timing ----
        moved = {}
        for form in ("dense", "gathered"):
            loop1(form, nth)
            call(form)
            moved[form] = Z.last_tend_2_transfer_bytes()
        qr, fr, pr = Z.convtran2_records(q, fracis, pdeldry, ideep, lengath, do, dry)
        for x, y in ((qr, q_r), (fr, f_r), (pr, p_r)):
            assert np.array_equal(x.view(np.int64), y.view(np.int64)), "tend2_loops.c pack differs from convtran2_records"
        back = Z.scatter_convtran2(dq_r, ideep, lengath, do, PCNST)
        assert np.array_equal(back.view(np.int64), dq_b.view(np.int64)), "scatter_convtran2(records) != dense tendency"
        full = {}
        for form in ("dense", "gathered"):
            full[form] = np.zeros(q.size)
            loop2(form, nth, full[form], pc * L * PCNST)
        assert np.array_equal(full["dense"].view(np.int64), full["gathered"].view(np.int64)), "loop 2 results differ"
        del full, back, qr, fr, pr

        # ---- timing: the calls alternate dense / gathered, each form with its loops ----
        t_call = {"dense": [], "gathered": []}
        for it in range(a.warmup + a.steps):
            for form in ("dense", "gathered"):
                t0 = time.perf_counter()
                call(form)
                if it >= a.warmup:
                    t_call[form].append((time.perf_counter() - t0) * 1e3)
        t_loop = {(form, which, nt): [] for form in ("dense", "gathered") for which in ("loop1", "loop2")
                  for nt in sorted({1, nth})}
        for nt in sorted({1, nth}):
            for it in range(1 + a.loop_reps):
                for form in ("dense", "gathered"):
                    for which, fn in (("loop1", loop1), ("loop2", loop2)):
                        t0 = time.perf_counter()
                        fn(form, nt)
                        if it:
                            t_loop[(form, which, nt)].append((time.perf_counter() - t0) * 1e3)

    forms = {}
    for form in ("dense", "gathered"):
        f = {"call": stats(t_call[form]), "h2d_bytes": moved[form]["h2d"], "d2h_bytes": moved[form]["d2h"]}
        for nt in sorted({1, nth}):
            l1, l2 = t_loop[(form, "loop1", nt)], t_loop[(form, "loop2", nt)]
            f[f"loop1_{nt}_threads"] = stats(l1)
            f[f"loop2_{nt}_threads"] = stats(l2)
            f[f"loop1_call_loop2_{nt}_threads_median_ms"] = float(np.median(l1) + np.median(t_call[form]) + np.median(l2))
        forms[form] = f
    rec = {"what": "zm_conv_tend_2 (convtran2) + the binding's loop 1 / loop 2: zm_conv_tend_2_batch with whole-array "
                   "copies against zm_conv_tend_2_batch_gathered with pack / zero-and-scatter",
           "workload": f"f09 shard: {a.ncols} columns x L{PVER}, pcols={PCOLS}, p_conv={PCONV}, bench soundings; "
                       f"{PCNST} constituents, {nact} flagged convtran2, {int(dry[act].sum())} of them dry; mirror from "
                       "zm_conv_tend_batch_gathered with keep_pbuf_on_device; page-locked host arrays",
           **gpu_info(), "host_cores": os.cpu_count(), "loop_threads": sorted({1, nth}), "convective_columns": ncv,
           "chunks": nch, "timed_calls_per_form": a.steps, "dense": forms["dense"], "gathered": forms["gathered"],
           "call_gathered_minus_dense_median_ms": forms["gathered"]["call"]["median_ms"] - forms["dense"]["call"]["median_ms"]}
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(rec, f, indent=1)
    print(json.dumps(rec))


if __name__ == "__main__":
    main()
