"""Where a convective column's cycles go in the cloud-model kernels (k_cldprp_pass1_w, k_plume_w).

Builds the library with -DZM_PLUME_PHASE_CLOCKS into the output directory (never into the package: the macro is not
part of build.source_hash(), so an instrumented libzmconv_b200.so in the tree would pass for the default build), loads
that copy, runs one device-resident zm_conv_tend step on bench.py's f09 shard (55,296 columns x L32 in pcols=16
chunks, p_conv 0.35) to warm up and one more with the counters reset, and writes the mean clock64() cycles per column
of every phase (lane 0 of each warp, zm_plume_warp.cuh PlumePhase) with the GPU's name and power limit.

The timers add a few instructions per phase and cost registers, so the sum is a little more than the default build's
per-column time; compare the phases, not the kernels' wall time."""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from cam_nor_physics_b200 import build as B  # noqa: E402

NCOLS_F09, PVER, PCOLS, PCONV = 55296, 32, 16, 0.35
# PlumePhase in zm_plume_warp.cuh, in order
PHASES = ["gather", "init", "j0_search", "k1_prep", "k1_rec", "expdif_search", "f_taylor", "f_prefix_max", "mu_par",
          "hu_rec", "jt_search", "cloud_top_reset", "eu_scan", "suqu_prep", "suqu_rec", "sat_cu", "ql_prep", "ql_rec",
          "hd_prep", "hd_rec", "sd_prep", "sd_rec", "pflx", "closure", "q1q2", "scatter"]
KERNELS = ["k_cldprp_pass1_w", "k_plume_w"]


def build_instrumented(out_dir: str) -> str:
    lib = os.path.join(out_dir, "libzmconv_b200_phase_clocks.so")
    cmd = [B._nvcc()] + B.NVCC_FLAGS + ["-DZM_PLUME_PHASE_CLOCKS", "-o", lib, B.SRC]
    env = dict(os.environ)
    env.pop("CXX", None)
    env.pop("CC", None)
    res = subprocess.run(cmd, capture_output=True, text=True, env=env)
    if res.returncode != 0:
        raise SystemExit("nvcc failed:\n" + res.stdout + res.stderr)
    return lib


def gpu_info() -> dict:
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    if q.returncode != 0:
        raise SystemExit("nvidia-smi failed: " + q.stderr)
    name, power, clk = [x.strip() for x in q.stdout.strip().splitlines()[0].split(",")]
    return {"gpu": name, "power_limit": power, "max_sm_clock": clk}


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--out-dir", required=True, help="directory for the instrumented library and the JSON")
    ap.add_argument("--out", default="plume_phase_cycles.json", help="JSON file name inside --out-dir")
    ap.add_argument("--label", default="", help="free text stored with the result (e.g. the commit)")
    args = ap.parse_args()
    os.makedirs(args.out_dir, exist_ok=True)

    import torch
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    lib_path = build_instrumented(os.path.abspath(args.out_dir))

    from cam_nor_physics_b200 import soundings as S, zm_conv as Z
    from cam_nor_physics_b200.device import DeviceTend
    Z._LIBPATH = lib_path                  # load the instrumented copy instead of the package's library
    lib = Z.lib()
    lib.zm_plume_phase_cycles.restype = C.c_int
    lib.zm_plume_phase_cycles.argtypes = [C.POINTER(C.c_ulonglong), C.c_int]
    nph = len(PHASES)
    buf = (C.c_ulonglong * (2 * (nph + 1)))()

    Z.zm_init(Z.default_params(PCOLS, PVER, S.limcnv_for(PVER)))
    ch = S.make_chunks(NCOLS_F09, PVER, PCOLS, p_conv=PCONV)
    dev = DeviceTend(ch)
    dev.step()
    torch.cuda.synchronize()
    if lib.zm_plume_phase_cycles(None, 1) != nph:
        raise SystemExit("the library's phase list does not match PHASES")
    dev.step()
    torch.cuda.synchronize()
    if lib.zm_plume_phase_cycles(buf, 0) != nph:
        raise SystemExit("reading the phase counters failed")

    result = {"what": "mean clock64() cycles per convective column and phase, lane 0 of each warp",
              "workload": f"f09 shard {NCOLS_F09} columns x L{PVER}, pcols={PCOLS}, p_conv={PCONV}, one "
                          "device-resident zm_conv_tend step after one warm-up step",
              "label": args.label, **gpu_info(), "kernels": {}}
    for r, kname in enumerate(KERNELS):
        row = list(buf[r * (nph + 1):(r + 1) * (nph + 1)])
        ncol = row[nph]
        phases = {PHASES[p]: round(row[p] / ncol, 1) for p in range(nph) if row[p]} if ncol else {}
        result["kernels"][kname] = {"columns": ncol, "total": round(sum(phases.values()), 1), "phases": phases}
    path = os.path.join(args.out_dir, args.out)
    with open(path, "w") as f:
        json.dump(result, f, indent=1)
        f.write("\n")
    print(json.dumps({k: (v["columns"], v["total"]) for k, v in result["kernels"].items()}))
    print("wrote", path)


if __name__ == "__main__":
    main()
