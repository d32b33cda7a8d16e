"""Host-pointer zm_conv_tend step plus the model's loop 2, dense against gathered return, on the f09 shard: 55,296
columns x L32 in pcols=16 chunks, bench.py's soundings (p_conv 0.35).

dense:    zm_conv_tend_batch into the twenty rank-level (pcols,pver[p]) arrays, then loop 2 copies each chunk's slices
          into a chunk buffer (zm_batch_scatter of fortran/zm_conv_intr_batched.F90);
gathered: zm_conv_tend_batch_gathered (pbuf fields in the records) into one record buffer, then loop 2 zeroes each
          chunk buffer and scatters the chunk's records into it (the binding's gathered mode).
Loop 2 is scripts/chunk_loop2.c, built here with gcc -O2 -fopenmp into a temporary directory; its chunk buffers are
per thread and stay in cache like the model's chunk-local ptend.  Every host array the step reads or writes is
page-locked once before timing.  Before any timing, the gathered step's records, scattered by scatter_gathered and by
chunk_loop2.c, are checked to equal the dense step's arrays bit for bit.  Steps alternate dense / gathered; the host
clock brackets each step (it returns synchronised) and each loop 2.  PCIe bytes come from zm_tend_transfer_bytes,
the sub-batch timeline of one step of each form from zm_tend_trace.  Writes one JSON record (GPU name and power limit included)."""
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

NCOLS_F09, PVER, PCOLS, PCONV = 55296, 32, 16, 0.35
LOOP2_SRC = os.path.join(ROOT, "scripts", "chunk_loop2.c")


def load_loop2(tmpdir: str) -> C.CDLL:
    so = os.path.join(tmpdir, "libchunk_loop2.so")
    subprocess.run(["gcc", "-O2", "-fopenmp", "-shared", "-fPIC", LOOP2_SRC, "-o", so], check=True)
    lib = C.CDLL(so)
    dp, ip = C.POINTER(C.c_double), C.POINTER(C.c_int)
    lib.loop2_dense.argtypes = [C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(dp), dp, C.c_longlong]
    lib.loop2_gathered.argtypes = [C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, ip, ip, dp, dp, C.c_longlong]
    return lib


def chunk_fields(Z):
    """The fields of chunk_loop2.c's chunk buffer, in order: the record order."""
    return Z.GATHERED_FIELDS + Z.GATHERED_PBUF


def run_dense(lib, Z, nthreads, out, dst, stride=0):
    arr = (C.POINTER(C.c_double) * 20)(*[Z._dp(out[k]) for k in chunk_fields(Z)])
    nch, L, pc = out["ptend_s"].shape
    lib.loop2_dense(nthreads, nch, pc, L, arr, Z._dp(dst), stride)


def run_gathered(lib, Z, nthreads, res, pver, dst, stride=0):
    nch, pc = res["ideep"].shape
    rec = np.ascontiguousarray(res["rec"])
    lib.loop2_gathered(nthreads, nch, pc, pver, int(res["pbuf_in_records"]), Z._ip(res["lengath"]), Z._ip(res["ideep"]),
                       Z._dp(rec), Z._dp(dst), stride)


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
    ap.add_argument("--steps", type=int, default=200, help="timed steps per form (alternating)")
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--single-thread-reps", type=int, default=20, help="timed 1-thread loop-2 passes per form")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "tend_gathered_cost_f09.json"))
    a = ap.parse_args()
    assert torch.cuda.is_available(), "needs a CUDA device"
    torch.cuda.set_device(0)
    Z.zm_init(Z.default_params(PCOLS, PVER, S.limcnv_for(PVER)))
    ch = S.make_chunks(NCOLS_F09, PVER, PCOLS, p_conv=PCONV)
    nch, L, pc = ch.nchunks, PVER, PCOLS
    pin = lambda x: torch.from_numpy(np.ascontiguousarray(x)).pin_memory().numpy()
    zeros = lambda shape, dt=torch.float64: torch.zeros(shape, dtype=dt).pin_memory().numpy()
    st = {k: pin(getattr(ch, k)) for k in Z.TEND_IN_ORDER}
    ncol = pin(ch.ncol.astype(np.int32))
    dense = {k: zeros((nch, L, pc)) for k in Z.TEND_OUT_2D}
    dense.update({k: zeros((nch, L + 1, pc)) for k in Z.TEND_OUT_2DP})
    dense.update({k: zeros((nch, pc)) for k in Z.TEND_OUT_1D})
    dense.update({k: zeros((nch, pc), torch.int32) for k in Z.TEND_OUT_INT})
    dense["lengath"] = zeros(nch, torch.int32)
    _, rec_len = Z.gathered_layout(L, True)
    gath = {k: zeros((nch, pc)) for k in Z.GATHERED_COL_OUT}
    gath.update({k: zeros((nch, pc), torch.int32) for k in ("jt", "maxg", "ideep")})
    gath["lengath"] = zeros(nch, torch.int32)
    gath["rec_buf"] = zeros(nch * pc * rec_len)

    nthreads = os.cpu_count() or 1
    with tempfile.TemporaryDirectory() as tmp:
        lib = load_loop2(tmp)
        bufs = zeros(nthreads * pc * rec_len)

        def step(form):
            if form == "dense":
                Z.zm_conv_tend(ncol, st, ch.ztodt, out=dense)
            else:
                Z.zm_conv_tend_gathered(ncol, st, ch.ztodt, out=gath)

        def loop2(form, nt):
            if form == "dense":
                run_dense(lib, Z, nt, dense, bufs)
            else:
                run_gathered(lib, Z, nt, gath, L, bufs)

        # ---- correctness before timing ----
        moved = {}
        for form in ("dense", "gathered"):
            step(form)
            moved[form] = Z.last_transfer_bytes()
        back = Z.scatter_gathered(gath)
        for k in Z.TEND_OUT_2D + Z.TEND_OUT_2DP + Z.TEND_OUT_1D + Z.TEND_OUT_INT + ["lengath"]:
            assert np.array_equal(back[k].view(np.int8), dense[k].view(np.int8)), f"scatter_gathered: {k} differs"
        full = {}
        for form in ("dense", "gathered"):
            full[form] = np.zeros(nch * pc * rec_len)
            if form == "dense":
                run_dense(lib, Z, nthreads, dense, full[form], pc * rec_len)
            else:
                run_gathered(lib, Z, nthreads, gath, L, full[form], pc * rec_len)
        assert np.array_equal(full["dense"].view(np.int64), full["gathered"].view(np.int64)), "loop 2 results differ"
        ncv = int(gath["lengath"].sum())

        # ---- timing: steps and loop 2 alternate dense / gathered ----
        t_step = {"dense": [], "gathered": []}
        t_loop = {"dense": [], "gathered": []}
        for it in range(a.warmup + a.steps):
            for form in ("dense", "gathered"):
                t0 = time.perf_counter()
                step(form)
                t1 = time.perf_counter()
                loop2(form, nthreads)
                t2 = time.perf_counter()
                if it >= a.warmup:
                    t_step[form].append((t1 - t0) * 1e3)
                    t_loop[form].append((t2 - t1) * 1e3)
        # pipeline timeline of one more step of each form (zm_tend_trace, ms from the first host->device copy): per
        # sub-batch, kernels done (column 3) and outputs -- for the gathered form its records -- on the host (column 5)
        trace = {}
        for form in ("dense", "gathered"):
            step(form)
            tr = Z.tend_trace()
            trace[form] = {"kernels_done_ms": [round(float(x), 3) for x in tr[:, 3]],
                           "outputs_on_host_ms": [round(float(x), 3) for x in tr[:, 5]]}
        t_single = {"dense": [], "gathered": []}
        for it in range(1 + a.single_thread_reps):
            for form in ("dense", "gathered"):
                t0 = time.perf_counter()
                loop2(form, 1)
                if it:
                    t_single[form].append((time.perf_counter() - t0) * 1e3)

    forms = {}
    for form in ("dense", "gathered"):
        tot = np.asarray(t_step[form]) + np.asarray(t_loop[form])
        forms[form] = {"step_plus_loop2": stats(tot), "step": stats(t_step[form]),
                       f"loop2_{nthreads}_threads": stats(t_loop[form]), "loop2_1_thread": stats(t_single[form]),
                       "h2d_bytes": moved[form]["h2d"], "d2h_bytes": moved[form]["d2h"], "sub_batch_trace": trace[form]}
    rec = {"what": "host-pointer zm_conv_tend step + loop 2 (chunk scatter): zm_conv_tend_batch + dense copy against "
                   "zm_conv_tend_batch_gathered (pbuf fields in the records) + zero-and-scatter",
           "workload": f"f09 shard: {NCOLS_F09} columns x L{PVER}, pcols={PCOLS}, p_conv={PCONV}, bench soundings; "
                       "page-locked host arrays",
           **gpu_info(), "host_cores": nthreads, "convective_columns": ncv, "rec_len": rec_len,
           "timed_steps_per_form": a.steps, "dense": forms["dense"], "gathered": forms["gathered"],
           "gathered_minus_dense_median_ms": forms["gathered"]["step_plus_loop2"]["median_ms"]
           - forms["dense"]["step_plus_loop2"]["median_ms"]}
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(rec, f, indent=1)
    print(json.dumps(rec))


if __name__ == "__main__":
    main()
