"""Cost of zm_conv_tend's history fields (zm_conv_tend_hist_fields) on the f09 shard: 55,296 columns x L32 in pcols=16
chunks, bench.py's soundings (p_conv 0.35).

Device-resident step: a DeviceTend without and one with every history field attached run in alternating blocks in
one process (a block replays its own CUDA graph: the graph of a step is keyed on its pointers, so switching between
the two recaptures once per block, and the first steps of a block are not timed); CUDA events around each block.
Host-pointer step: plain and attached calls alternate one by one, host clock around each call (it synchronises);
PCIe bytes from zm_tend_transfer_bytes.  Before any timing the regular outputs of both forms are checked to be
bit-identical.  Writes one JSON record (GPU name and power limit included)."""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

from cam_nor_physics_b200 import soundings as S, zm_conv as Z  # noqa: E402
from cam_nor_physics_b200.device import DeviceTend  # noqa: E402

NCOLS_F09, PVER, PCOLS, PCONV = 55296, 32, 16, 0.35


def gpu_info() -> dict:
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    if q.returncode != 0:
        return {"gpu": torch.cuda.get_device_name(0), "power_limit": "unknown", "max_sm_clock": "unknown"}
    name, power, clk = [x.strip() for x in q.stdout.strip().splitlines()[0].split(",")]
    return {"gpu": name, "power_limit": power, "max_sm_clock": clk}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--blocks", type=int, default=5, help="alternating blocks per form (device-resident step)")
    ap.add_argument("--block-steps", type=int, default=50, help="timed steps per block")
    ap.add_argument("--block-warmup", type=int, default=3, help="untimed steps that open a block (run, capture)")
    ap.add_argument("--host-steps", type=int, default=200, help="timed host-pointer calls per form")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "tend_history_cost_f09.json"))
    a = ap.parse_args()
    assert torch.cuda.is_available(), "needs a CUDA device"
    torch.cuda.set_device(0)
    Z.zm_init(Z.default_params(PCOLS, PVER, S.limcnv_for(PVER)))
    ch = S.make_chunks(NCOLS_F09, PVER, PCOLS, p_conv=PCONV)
    lib = Z.lib()

    # ---- device-resident step ----
    dev = {"plain": DeviceTend(ch), "hist": DeviceTend(ch, hist=True)}
    launches = {}
    for k, d in dev.items():
        lib.zm_launch_count(1)
        d.step()
        assert d.check() == 0
        launches[k] = int(lib.zm_launch_count(1))
    for k in Z.TEND_ARG_ORDER:
        assert torch.equal(dev["plain"].out[k], dev["hist"].out[k]), f"device step: {k} differs with history attached"
    hist_bytes = sum(v.numel() * v.element_size() for v in dev["hist"].hist.values())
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    per_block = {"plain": [], "hist": []}
    for _ in range(a.blocks):
        for k, d in dev.items():
            for _ in range(a.block_warmup):
                d.step()
            torch.cuda.synchronize()
            ev0.record()
            for _ in range(a.block_steps):
                d.step()
            ev1.record()
            torch.cuda.synchronize()
            assert d.check() == 0
            per_block[k].append(ev0.elapsed_time(ev1) / a.block_steps)
    device = {k: {"ms_per_step_mean": float(np.mean(v)), "ms_per_step_blocks": [round(x, 4) for x in v],
                  "launches_per_step": launches[k]} for k, v in per_block.items()}
    device["overhead_ms"] = device["hist"]["ms_per_step_mean"] - device["plain"]["ms_per_step_mean"]
    device["timed_steps_per_form"] = a.blocks * a.block_steps
    device["history_bytes_written"] = hist_bytes

    # ---- host-pointer step ----
    st = {k: getattr(ch, k) for k in Z.TEND_IN_ORDER}
    outs = {"plain": Z.zm_conv_tend(ch.ncol, st, ch.ztodt), "hist": Z.zm_conv_tend(ch.ncol, st, ch.ztodt, hist=True)}
    for k in outs["plain"]:
        assert np.array_equal(outs["plain"][k], outs["hist"][k]), f"host step: {k} differs with history attached"
    moved = {}
    for k in outs:
        Z.zm_conv_tend(ch.ncol, st, ch.ztodt, out=outs[k], hist=(k == "hist"))
        moved[k] = Z.last_transfer_bytes()
    times = {"plain": [], "hist": []}
    for _ in range(a.host_steps):
        for k in ("plain", "hist"):
            t0 = time.perf_counter()
            Z.zm_conv_tend(ch.ncol, st, ch.ztodt, out=outs[k], hist=(k == "hist"))
            times[k].append((time.perf_counter() - t0) * 1e3)
    host = {k: {"ms_per_step_median": float(np.median(v)), "ms_per_step_mean": float(np.mean(v)),
                "h2d_bytes": moved[k]["h2d"], "d2h_bytes": moved[k]["d2h"]} for k, v in times.items()}
    host["overhead_ms_median"] = host["hist"]["ms_per_step_median"] - host["plain"]["ms_per_step_median"]
    host["timed_steps_per_form"] = a.host_steps

    rec = {"what": "zm_conv_tend with and without every history field attached (zm_conv_tend_hist_fields)",
           "workload": f"f09 shard: {NCOLS_F09} columns x L{PVER}, pcols={PCOLS}, p_conv={PCONV}, bench soundings",
           **gpu_info(), "device_resident": device, "host_pointer": host}
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(rec, f, indent=1)
    print(json.dumps(rec))


if __name__ == "__main__":
    main()
