#!/usr/bin/env python
"""bench.py -- ZM deep-convection throughput (columns/s) on 1..N B200s.

Metric (BASELINE.json): "ZM convection columns/sec (f09 L32, r8)".  One step = one pass of the hot
path -- zm_conv_tend = zm_convr + physics_update + zm_conv_evap + momtran (BASELINE config 3;
reference physics/zm_conv_intr.F90:662-836) -- over synthetic soundings (pver=32, pcols=16, r8).
Columns shard with no hot-path communication; the only collective is one NCCL all-reduce of six
doubles per step for the global water/energy budget check.

  --scaling weak   (default) every rank owns its own f09 shard of --ncols columns (55,296)
  --scaling strong the ONE f09 grid of --ncols columns is cut into contiguous blocks of whole chunks,
                   one block per rank (what physpkg.F90:1147 gives a rank of a real run)

  value  : whole-job columns/s with physics_state resident in HBM (CUDA events, max over ranks)
  e2e    : the same step through the host-pointer C ABI (zm_conv_tend_batch) from pinned host
           buffers, H2D + kernels + D2H inside the timed region
  roofline: dominant kernel k_buoyan_dilute<1> (FP64-pipe bound), timed live with CUDA events;
           algorithmic flops = the CPU oracle's instrumented operation count of the first CAPE pass on
           the same soundings (profiles/flops_per_column.json), executed flops beside it
  configs: the default single-GPU run also times BASELINE config 2 (f19 grid, 13,824 columns) and
           config 4 (f09 + convtran over a 41-constituent stand-in for the OsloAero tracer set:
           convtran1 inside zm_conv_tend, convtran2 in zm_conv_tend_2) device-resident
  multi_gpu_parity (N > 1): rank 0 recomputes every rank's shard on its own GPU and compares
           per-field checksums of the bit patterns
  cpu_baseline / --impl reference: the CPU oracle port of the reference (OpenMP over chunks,
           glibc libm) timed on this box's host cores.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "ZM convection columns/sec (f09 L32, r8)"
UNIT = "columns/s"
NCOLS_F09 = 55296
NCOLS_F19 = 13824
NCNST_STANDIN = 41          # pcnst of the OsloAero configuration is not defined in the reference tree (SURVEY 8d)

# flop counts per column of one k_buoyan_dilute<1> launch on the default workload: algorithmic (oracle-instrumented,
# scripts/count_flops.py) and executed (ncu capture named inside)
FLOPS_FILE = os.path.join(ROOT, "profiles", "flops_per_column.json")
FP64_PEAK_FILE = os.path.join(ROOT, "profiles", "fp64_peak.json")


def _peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return json.load(f), "measured"
    except Exception:
        return {"hbm_gbs": 6650.0}, "fallback"


class ClockSampler:
    """Samples nvidia-smi clocks / throttle reasons during the timed region."""

    def __init__(self, index: int):
        self.index = index
        self.samples = []
        self.reasons = set()
        self._stop = threading.Event()
        self._t = None

    def _run(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        while not self._stop.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits",
                                      "-i", str(self.index)], capture_output=True, text=True, timeout=5).stdout
                parts = [p.strip() for p in out.strip().split(",")]
                if len(parts) >= 6:
                    self.samples.append((float(parts[0]), float(parts[1])))
                    for n, v in zip(names, parts[2:6]):
                        if v.lower().startswith("active"):
                            self.reasons.add(n)
            except Exception:
                pass
            self._stop.wait(0.1)

    def start(self):
        self._t = threading.Thread(target=self._run, daemon=True)
        self._t.start()

    def stop(self):
        self._stop.set()
        if self._t:
            self._t.join(timeout=10)
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": sorted(self.reasons), "samples": 0}
        return {"sm_mhz": statistics.median(s[0] for s in self.samples),
                "sm_max_mhz": max(s[1] for s in self.samples), "reasons": sorted(self.reasons),
                "samples": len(self.samples)}


def _oracle(pver, parcel_pbl):
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from oracle_lib import Oracle
    from cam_nor_physics_b200 import soundings as S
    o = Oracle("libm")
    op = o.default_params(16, pver, S.limcnv_for(pver))
    op.lparcel_pbl = int(parcel_pbl)
    o.convi(op)
    return o


def cpu_step(o, ch, cores, ncnst=0):
    """One pass of the hot path on the CPU port: zm_conv_tend (+ convtran1 and zm_conv_tend_2 for config 4)."""
    from cam_nor_physics_b200 import soundings as S
    if not ncnst:
        r = o.conv_tend_batch(ch, nthreads=cores)
    else:
        import numpy as np
        tr = getattr(ch, "_bench_tracers", None)
        if tr is None:
            tr = ch._bench_tracers = S.make_tracers(ch, ncnst)
        q3, fracis, pdeldry = tr
        do1 = np.zeros(ncnst, np.int32); do1[1:3] = 1
        do2 = np.zeros(ncnst, np.int32); do2[3:] = 1
        dry = np.zeros(ncnst, np.int32); dry[3::3] = 1
        r = o.conv_tend_batch(ch, nthreads=cores, convtran1=dict(doconvtran=do1, cnst_is_dry=dry, q=q3, fracis=fracis))
        r["ptend_qc"] = o.conv_tend_2_batch(do2, q3, pdeldry, fracis, ch.ztodt, dry, r, ptend_q=r["ptend_qc"],
                                            nthreads=cores)
    if r["rc"]:
        raise RuntimeError("oracle Brent failure")
    return r


def cpu_reference_rate(ncols, pver, pconv, reps, nthreads=0, parcel_pbl=False, ncnst=0):
    """Times the CPU port of the reference (oracle, glibc libm flavour, OpenMP over chunks)."""
    from cam_nor_physics_b200 import soundings as S
    o = _oracle(pver, parcel_pbl)
    ch = S.make_chunks(ncols, pver, 16, p_conv=pconv)
    cores = nthreads or (os.cpu_count() or 1)
    cpu_step(o, ch, cores, ncnst)          # warm-up
    best = 1e30
    for _ in range(reps):
        t0 = time.perf_counter()
        cpu_step(o, ch, cores, ncnst)
        best = min(best, time.perf_counter() - t0)
    return ncols / best, cores, best, o.backend()


def shard_of(rank, world, ncols, scaling):
    """(first global column, number of columns) of a rank: weak = its own grid of ncols columns; strong = a contiguous
    block of whole pcols=16 chunks of the one grid (chunk c -> rank floor(c*world/nchunks), SURVEY 8e)."""
    if scaling == "weak":
        return rank * ncols, ncols
    nch = (ncols + 15) // 16
    c0, c1 = (nch * rank) // world, (nch * (rank + 1)) // world
    return 16 * c0, min(ncols, 16 * c1) - 16 * c0


DUMP_BYTES = 60_000_000     # --dump-outputs stays under 64 MB in all, .npy headers included
DUMP_SEED = 20261020


def dump_outputs(path, chunked, totals=None):
    """Writes every output array as <path>/<name>.npy in float64 (integer fields convert exactly).  `chunked` arrays
    lead with the chunk dimension: when they exceed DUMP_BYTES in all, every one keeps the same sample of whole chunks,
    the first ones of a seeded permutation of all chunks, so two runs with the same arguments write the same elements
    and a smaller sample is a subset of a larger one.  The chosen chunks go to chunk_index.npy (0-based, ascending).
    `totals` are written whole."""
    import numpy as np
    nch = len(next(iter(chunked.values())))
    per_chunk = sum(np.asarray(a)[0].size for a in chunked.values()) * 8
    keep = min(nch, max(1, (DUMP_BYTES - 8 * nch) // per_chunk))
    idx = np.sort(np.random.default_rng(DUMP_SEED).permutation(nch)[:keep])
    os.makedirs(path, exist_ok=True)
    np.save(os.path.join(path, "chunk_index.npy"), idx.astype(np.float64))
    for k, a in chunked.items():
        np.save(os.path.join(path, k + ".npy"), np.asarray(a)[idx].astype(np.float64))
    for k, a in (totals or {}).items():
        np.save(os.path.join(path, k + ".npy"), np.asarray(a, dtype=np.float64))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--ncols", type=int, default=NCOLS_F09,
                    help="columns per GPU (--scaling weak) or of the whole grid (--scaling strong)")
    ap.add_argument("--pver", type=int, default=32)
    ap.add_argument("--pconv", type=float, default=0.35, help="convective fraction of the synthetic grid")
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"])
    ap.add_argument("--convtran", type=int, default=0, metavar="NCNST",
                    help="BASELINE config 4 as the main workload: zm_conv_tend incl. convtran1 + zm_conv_tend_2 over "
                         "NCNST constituents (41 = the stand-in for the OsloAero tracer set)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extra-configs", action="store_true", help="skip the config 2 / config 4 lines of the default run")
    ap.add_argument("--parcel-pbl", action="store_true", help="zmconv_parcel_pbl=.true. (CAM6 L58 default)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last timed step computed as DIR/<name>.npy (float64; "
                         "rank 0's shard; above 60 MB a fixed seeded sample of whole chunks)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3)
    # stdout carries the JSON line and nothing else: libraries that write to file descriptor 1 (NCCL prints its
    # version banner there) are sent to stderr for the whole run, the line goes to the saved descriptor
    sys.stdout.flush()
    json_out = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    L = args.pver
    col0, ncols_rank = shard_of(rank, world, args.ncols, args.scaling)
    ncols_job = args.ncols * world if args.scaling == "weak" else args.ncols
    per = "per GPU" if args.scaling == "weak" else f"in all, cut into {world} contiguous blocks of whole chunks (one per GPU)"
    if args.ncols == NCOLS_F09 and L == 32:
        grid = f"f09 FV grid{' shard' if args.scaling == 'weak' else ''}: {args.ncols} columns x L32 {per} (BASELINE config {4 if args.convtran else 3})"
    elif args.ncols == NCOLS_F19 and L == 32:
        grid = f"f19 FV grid: {args.ncols} columns x L32 {per} (BASELINE config 2)"
    else:
        grid = f"{args.ncols} columns x L{L} {per} (non-default size; BASELINE config 5 uses 131072 x L58 per GPU)"
    seq = "zm_conv_tend = zm_convr+physics_update+zm_conv_evap+momtran"
    if args.convtran:
        seq += f"+convtran1 (2 constituents), then zm_conv_tend_2 = convtran2 over {args.convtran - 3} of {args.convtran} constituents"
    workload = grid + ", pcols=16, " + seq
    step_gb = args.ncols * ((26 * L + 15) * 8 + 12 + (14 * L + 6) * 8 + 19 * L * 8 + 12) / 1e9
    config = {"workload": workload, "columns_per_gpu": ncols_rank if args.scaling == "strong" else args.ncols,
              "columns_total": ncols_job, "pver": L, "pcols": 16,
              "convective_fraction_target": args.pconv, "parcel_pbl": bool(args.parcel_pbl), "seed": 20261018,
              "parallelism": f"columns x{world} ({args.scaling})", "ncnst": args.convtran or None,
              "l2": f"per-step algorithmic inputs+outputs ({step_gb:.2f} GB per {args.ncols} columns) exceed the 126 MB L2; no explicit flush"}

    # ---------------- reference arm: CPU port of the reference on host cores ---------------------
    if args.impl == "reference":
        if rank != 0:
            return
        from cam_nor_physics_b200 import soundings as S
        o = _oracle(L, args.parcel_pbl)
        # weak: one rank's shard (the job is N such shards; the rate is per host); strong: the whole grid
        ch = S.make_chunks(args.ncols, L, 16, p_conv=args.pconv)
        cores = os.cpu_count() or 1
        backend = o.backend()
        times = []
        for i in range(args.warmup + args.steps):
            t0 = time.perf_counter()
            r = cpu_step(o, ch, cores, args.convtran)
            dt = time.perf_counter() - t0
            if i >= args.warmup:
                times.append(dt)
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, {k: v for k, v in r.items() if k != "rc"})
        t = statistics.mean(times)
        rate = args.ncols / t
        line = {"impl": "reference", "metric": METRIC, "value": rate, "unit": UNIT, "n_gpus": args.gpus,
                "steps": args.steps, "warmup": args.warmup, "ms_per_step": t * 1e3, "higher_is_better": True,
                "scaling": args.scaling, "vs_baseline": None, "dtype": "f64", "data": "synthetic", "config": config,
                "cpu_baseline": {"value": rate, "unit": UNIT, "cores": cores, "kind": "port",
                                 "sample": f"full step on {args.ncols} columns, CPU oracle ({backend}), "
                                           "OpenMP over pcols=16 chunks"},
                "e2e": {"value": rate, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
        json_out.write(json.dumps(line) + "\n"); json_out.flush()
        return

    # ---------------- B200 arm ---------------------------------------------------------------------
    import numpy as np
    import torch
    import torch.distributed as dist
    from cam_nor_physics_b200 import build, soundings as S, zm_conv as Z
    from cam_nor_physics_b200.device import DeviceTend

    if not torch.cuda.is_available():
        raise SystemExit("bench.py --impl b200 needs a CUDA device (there is no CPU fallback)")
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    build.build()
    zp = Z.default_params(16, L, S.limcnv_for(L))
    zp.lparcel_pbl = int(args.parcel_pbl)
    Z.zm_init(zp)
    stream = torch.cuda.current_stream()

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed_run(dev, steps, warmup, with_budget=True):
        """W warm-up + K timed steps of `dev` (device-resident), CUDA events on torch's stream, max over ranks."""
        def one_step():
            dev.step()
            if dev.ncnst:
                dev.step2()
            if not with_budget:
                return None
            cons = dev.conservation()
            if world > 1:
                dist.all_reduce(cons)
            return cons
        for _ in range(warmup):
            one_step()
        dev.check()
        barrier()
        Z.lib().zm_launch_count(1)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for _ in range(steps):
            cons = one_step()
        e1.record(stream)
        barrier()
        launches = int(Z.lib().zm_launch_count(1))
        nfail = dev.check()
        ms = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item()) / steps, launches, nfail, cons

    def kernel_profile(dev, nprof):
        """Per-kernel device times (events between the kernels; a loop of its own, not the timed one)."""
        Z.lib().zm_set_profiling(1)
        kt, gp = {}, {}
        for _ in range(nprof):
            dev.step()
            torch.cuda.synchronize()
            for n, t in Z.kernel_times():
                kt.setdefault(n, []).append(t)
            if dev.ncnst:
                dev.step2()
                torch.cuda.synchronize()
                for n, t in Z.kernel_times():
                    if n == "convtran2":
                        kt.setdefault(n, []).append(t)
        Z.lib().zm_set_profiling(0)
        return {n: statistics.mean(v) for n, v in kt.items()}

    ch = S.make_chunks(ncols_rank, L, 16, p_conv=args.pconv, col0=col0)
    dev = DeviceTend(ch, ncnst=args.convtran)
    sampler = ClockSampler(local_rank)
    sampler.start()
    ms_per_step, launches, nfail, cons = timed_run(dev, args.steps, args.warmup)
    value = ncols_job / (ms_per_step * 1e-3)
    cons_h = cons.cpu().numpy()
    if args.dump_outputs and rank == 0:
        outs = {k: v.cpu().numpy() for k, v in dev.out.items()}
        if dev.ncnst:
            outs["ptend_qc"] = dev.ptend_qc.cpu().numpy()
        dump_outputs(args.dump_outputs, outs, {"conservation": cons_h})
    kavg = kernel_profile(dev, min(args.steps, 10))
    gptl = Z.timers() if hasattr(Z, "timers") else {}

    # ---- multi-GPU parity: every rank's outputs against the same columns computed on rank 0's GPU -------------
    parity = None
    if world > 1:
        dev.step()
        if dev.ncnst:
            dev.step2()
        mine = dev.checksums()
        allsums = [torch.zeros_like(mine) for _ in range(world)]
        dist.all_gather(allsums, mine)
        if rank == 0:
            equal = []
            cons_parts = []          # per-shard budget terms, each reduced on rank 0's GPU (SURVEY section 4)
            for r in range(world):
                c0r, nr = shard_of(r, world, args.ncols, args.scaling)
                if r == 0:
                    ref = mine
                    dr = dev
                else:
                    dr = DeviceTend(S.make_chunks(nr, L, 16, p_conv=args.pconv, col0=c0r), ncnst=args.convtran)
                    dr.step()
                    if dr.ncnst:
                        dr.step2()
                    ref = dr.checksums()
                try:
                    cons_parts.append(dr.conservation().double().cpu().numpy().copy())
                except Exception as e:           # informational: never fatal for the bench line
                    cons_parts.append(repr(e))
                if r != 0:
                    del dr
                equal.append(bool(torch.equal(ref, allsums[r])))
            parity = {"ranks_checked": world, "fields": int(mine.numel()), "equal": all(equal), "per_rank": equal,
                      "how": "wrap-around 64-bit sums of the bit patterns of every zm_conv_tend output, rank r's shard "
                             "recomputed on rank 0's GPU"}
            try:
                import numpy as np
                tot = np.sum(np.stack(cons_parts), axis=0)
                rel = float(np.max(np.abs(tot - cons_h) / np.maximum(np.abs(cons_h), 1e-300)))
                parity["conservation_allreduce_rel_err"] = rel       # NCCL sum of the ranks' six budget terms against
                parity["conservation_within_1e-13"] = bool(rel <= 1e-13)   # the sum of the same shards reduced on rank 0
            except Exception as e:
                parity["conservation_check_error"] = repr(e)
        barrier()

    # ---- roofline of the dominant kernel ------------------------------------------------------------------------
    dom = "buoyan_dilute_pass1"
    t_dom = kavg.get(dom, float("nan")) * 1e-3
    peaks, peak_kind = _peaks()
    try:
        with open(FLOPS_FILE) as f:
            fl = json.load(f)
    except Exception:
        fl = {}
    fp64_live = Z.fp64_peak_flops(20000)
    try:
        with open(FP64_PEAK_FILE) as f:
            fp64_frozen = json.load(f)
    except Exception:
        fp64_frozen = {}
    fp64_peak = float(fp64_frozen.get("fp64_tflops", fp64_live / 1e12)) * 1e12
    # the committed flop counts belong to the default workload (they depend on the soundings), so the FP64 fraction is
    # only reported there; the counts are per column, so any shard of that grid may use them
    flops_valid = bool(fl) and (L == 32 and not args.parcel_pbl and abs(args.pconv - 0.35) < 1e-12
                                and args.ncols == int(fl.get("ncols", -1)) and (args.scaling == "weak" or world == 1))
    def _num(v):
        return float(v) if v is not None else float("nan")
    alg_fpc = _num(fl.get("algorithmic_flops_per_column")) if flops_valid else float("nan")
    exe_fpc = _num(fl.get("executed_flops_per_column")) if flops_valid else float("nan")
    if alg_fpc != alg_fpc:          # no oracle count on file: fall back to the executed count, and say so
        alg_fpc = exe_fpc
    achieved = alg_fpc * ncols_rank / t_dom / 1e12
    alg_bytes = (6 * L + 2 + 2 * L + 6) * 8 + 12      # inputs t,q,pap,zm (L) + paph,zi (L+1) + 3; outputs tp,qstp + 6 scalars
    import hashlib
    hsh = hashlib.sha256()
    for fn in ("zm_kernels.cuh", "zm_device.cuh", "zm_math.h", "zm_svp_table.h"):
        hsh.update(open(os.path.join(ROOT, "cam_nor_physics_b200", "csrc", fn), "rb").read())
    executed_stale = fl.get("executed_kernel_hash") != hsh.hexdigest()[:16]
    roofline = {"kernel": "k_buoyan_dilute<1> (dilute CAPE trigger, pass 1, all columns)",
                "bound": "fp64", "achieved": achieved if flops_valid else None, "peak": fp64_peak / 1e12,
                "unit": "TFLOP/s", "frac": achieved / (fp64_peak / 1e12) if flops_valid else None,
                "peak_source": (f"FP64 FMA-chain microbenchmark, frozen in profiles/fp64_peak.json with its clock record "
                                f"(live in this process: {fp64_live / 1e12:.2f} TFLOP/s); MEASURED_PEAKS.json has no FP64 entry"
                                if fp64_frozen else
                                "FP64 FMA-chain microbenchmark run live in this process (MEASURED_PEAKS.json has no FP64 entry)"),
                "algorithmic_flops_per_column": alg_fpc if flops_valid else None,
                "algorithmic_flops_source": fl.get("algorithmic_source"),
                "executed_flops_per_column": exe_fpc if flops_valid else None,
                "executed_tflops": exe_fpc * ncols_rank / t_dom / 1e12 if flops_valid else None,
                "executed_frac": exe_fpc * ncols_rank / t_dom / fp64_peak if flops_valid else None,
                "executed_flops_source": fl.get("executed_source"),
                "executed_flops_stale": bool(executed_stale) if flops_valid else None,   # kernel sources changed since the capture
                "algorithmic_calls_per_column": fl.get("algorithmic_calls_per_column") if flops_valid else None,
                "ms_per_launch": t_dom * 1e3,
                "traffic": fl.get("dram_bytes_per_launch") if flops_valid and ncols_rank == int(fl.get("ncols", -1)) else None,
                "hbm": {"achieved_gbs": alg_bytes * ncols_rank / t_dom / 1e9, "peak_gbs": peaks.get("hbm_gbs"),
                        "peak_kind": peak_kind, "alg_bytes_per_column": alg_bytes},
                "kernel_ms": kavg, "gptl_ms": gptl}

    # ---- e2e: host-pointer C ABI from pinned host buffers -----------------------------------------
    st = {k: v.numpy() for k, v in dev.host_in.items()}     # pinned host memory views
    nch, pc = ch.nchunks, 16
    out = {}
    for k in Z.TEND_OUT_2D:
        out[k] = torch.zeros((nch, L, pc), dtype=torch.float64).pin_memory().numpy()
    for k in Z.TEND_OUT_2DP:
        out[k] = torch.zeros((nch, L + 1, pc), dtype=torch.float64).pin_memory().numpy()
    for k in Z.TEND_OUT_1D:
        out[k] = torch.zeros((nch, pc), dtype=torch.float64).pin_memory().numpy()
    for k in Z.TEND_OUT_INT:
        out[k] = torch.zeros((nch, pc), dtype=torch.int32).pin_memory().numpy()
    out["lengath"] = torch.zeros(nch, dtype=torch.int32).pin_memory().numpy()
    h2d = sum(v.nbytes for v in st.values()) + ch.ncol.nbytes
    d2h = sum(v.nbytes for v in out.values())

    def e2e_rate(**kw):
        for _ in range(2):
            Z.zm_conv_tend(ch.ncol, st, ch.ztodt, out, **kw)
        barrier()
        t0 = time.perf_counter()
        n = max(3, min(args.steps, 10))
        for _ in range(n):
            Z.zm_conv_tend(ch.ncol, st, ch.ztodt, out, **kw)     # synchronous: returns after the D2H
        torch.cuda.synchronize()
        te = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(te, op=dist.ReduceOp.MAX)
        return ncols_job * n / float(te.item()), n

    e2e_value, nsteps_e2e = e2e_rate()
    tr_bytes = Z.last_transfer_bytes() if hasattr(Z, "last_transfer_bytes") else None
    # same call with the pbuf mass-flux fields (ZM_MU..ZM_MAXG) left in the library's device mirror for
    # zm_conv_tend_2_batch instead of being copied back -- informational, the headline e2e copies everything
    mirror_keys = ("mu", "md", "du", "eu", "ed", "dp", "dsubcld", "jt", "maxg")
    d2h_res = d2h - sum(out[k].nbytes for k in mirror_keys)
    e2e_resident, _ = e2e_rate(keep_pbuf_on_device=True)
    tr_bytes_res = Z.last_transfer_bytes() if hasattr(Z, "last_transfer_bytes") else None
    clocks = sampler.stop()       # sampled through the timed loop, the per-kernel loop and the e2e loop

    # ---- the other single-GPU BASELINE configs, device-resident (config 2: f19 grid; config 4: f09 + convtran) --
    extra = {}
    if world == 1 and not args.no_extra_configs and L == 32 and not args.parcel_pbl and not args.convtran \
            and args.ncols == NCOLS_F09:
        del dev
        torch.cuda.empty_cache()
        ksteps, kwarm = max(3, min(args.steps, 10)), 3
        d19 = DeviceTend(S.make_chunks(NCOLS_F19, L, 16, p_conv=args.pconv))
        ms19, l19, _, _ = timed_run(d19, ksteps, kwarm)
        k19 = kernel_profile(d19, 3)
        extra["config2_f19"] = {"workload": f"f19 FV grid: {NCOLS_F19} columns x L32 full-globe ZM step on 1 B200, " + seq,
                                "value": NCOLS_F19 / (ms19 * 1e-3), "unit": UNIT, "ms_per_step": ms19, "steps": ksteps,
                                "warmup": kwarm, "gpu_launches": l19, "kernel_ms": k19}
        del d19
        torch.cuda.empty_cache()
        d4 = DeviceTend(ch, ncnst=NCNST_STANDIN)
        ms4, l4, _, _ = timed_run(d4, ksteps, kwarm)
        k4 = kernel_profile(d4, 3)
        nact2 = NCNST_STANDIN - 3
        nconv = int(d4.out["lengath"].sum().item())
        # dense bytes the transport must move: q and fracis read at sector granularity (~ every 32-B sector of the
        # active slices holds a convective column at this convective fraction), dqdt written for every column
        dense = 3.0 * NCOLS_F09 * L * 8 * nact2
        useful = nconv * (7 * L * 8 + nact2 * 3 * L * 8)          # SURVEY 8d: per convective column
        t2 = k4.get("convtran2", float("nan")) * 1e-3
        extra["config4_convtran"] = {
            "workload": f"f09 L32 + convtran over a {NCNST_STANDIN}-constituent stand-in for the OsloAero tracer set "
                        f"(convtran1: 2 constituents inside zm_conv_tend; convtran2: {nact2} in zm_conv_tend_2, every third 'dry')",
            "value": NCOLS_F09 / (ms4 * 1e-3), "unit": UNIT, "ms_per_step": ms4, "steps": ksteps, "warmup": kwarm,
            "gpu_launches": l4, "kernel_ms": k4, "ncnst": NCNST_STANDIN,
            "convtran2_roofline": {"bound": "hbm", "ms_per_launch": t2 * 1e3,
                                   "algorithmic_bytes_dense": dense, "algorithmic_bytes_convective_columns": useful,
                                   "achieved_gbs_dense": dense / t2 / 1e9, "achieved_gbs_convective_columns": useful / t2 / 1e9,
                                   "peak_gbs": peaks.get("hbm_gbs"), "frac_dense": dense / t2 / 1e9 / peaks.get("hbm_gbs", float("nan"))}}
        del d4
        torch.cuda.empty_cache()

    if rank == 0:
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": args.scaling,
                "vs_baseline": None, "dtype": "f64", "data": "synthetic", "config": config, "clocks": clocks,
                "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": int(h2d),
                        "d2h_bytes_per_step": int(d2h), "steps": nsteps_e2e,
                        "api": "zm_conv_tend_batch (host pointers, pinned)", "pcie_bytes_moved": tr_bytes,
                        "pbuf_resident": {"value": e2e_resident, "d2h_bytes_per_step": int(d2h_res),
                                          "pcie_bytes_moved": tr_bytes_res,
                                          "note": "mu,md,du,eu,ed,dp,dsubcld,jt,maxg kept in the device mirror"}},
                "gpu_launches": launches, "roofline": roofline,
                "convective_columns_per_gpu": int(out["lengath"].sum()),
                "brent_failures": int(nfail),
                "conservation": {"sum_pdel_g_ptend_q": cons_h[0], "sum_1000_prec_plus_rliq": cons_h[1],
                                 "water_residual_rel": float((cons_h[0] + cons_h[1]) / max(abs(cons_h[1]), 1e-300)),
                                 "sum_pdel_g_ptend_s": cons_h[2], "sum_latent": cons_h[3],
                                 "convective_columns": cons_h[4], "columns": cons_h[5]}}
        if parity is not None:
            line["multi_gpu_parity"] = parity
        if extra:
            line["configs"] = extra
        if world == 1 and not args.no_cpu_baseline:
            rate, cores, best, backend = cpu_reference_rate(args.ncols, L, args.pconv, 3, parcel_pbl=args.parcel_pbl,
                                                            ncnst=args.convtran)
            line["cpu_baseline"] = {"value": rate, "unit": UNIT, "cores": cores, "kind": "port",
                                    "sample": f"full step on all {args.ncols} columns x3 (best), CPU oracle "
                                              f"({backend}) with OpenMP over pcols=16 chunks; {best*1e3:.1f} ms/step"}
        json_out.write(json.dumps(line) + "\n"); json_out.flush()
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
