"""Randomised pin of the CPU oracle to the reference's own source text (CPU only; reads the CAM-Nor source tree named by
$CAM_NOR_SRC, which is not part of this repository): random chunk widths, level counts, namelist values, zm_org / cam3 and
level-wise perturbed soundings go through the translated reference text (make_reference_fixtures.run_case) and through
the glibc-libm oracle; every output of zm_convr, zm_conv_evap, momtran, convtran and the zm_conv_tend glue must agree
bit for bit (the comparison is tests/test_oracle.py::test_oracle_equals_reference_source_text).
usage: python tests/golden/reference_text_fuzz.py [ncases] [seed]      (FUZZ_PVER=58 forces the level count)"""
import os, sys, json, time
HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "tests")); sys.path.insert(0, HERE)
import numpy as np
import make_reference_fixtures as M
import test_oracle as T

ncases = int(sys.argv[1]) if len(sys.argv) > 1 else 20
rng = np.random.default_rng(int(sys.argv[2]) if len(sys.argv) > 2 else 3)
noise_rng = [None]


def _st_noise(inp, c):
    r = noise_rng[0]
    inp["t"][:] = inp["t"] + r.normal(0.0, 2.5, inp["t"].shape)
    inp["q"][:] = np.maximum(inp["q"] * r.uniform(0.3, 1.7, inp["q"].shape), 1e-12)
    inp["pblh"][:] = r.uniform(20.0, 4000.0, inp["pblh"].shape)
    inp["tpert"][:] = r.uniform(0.0, 4.0, inp["tpert"].shape)
    inp["landfrac"][:] = r.choice([0.0, 1.0, 0.37], size=inp["landfrac"].shape)


M.STRESS["noise"] = _st_noise
report = []
t0 = time.time()
for case in range(ncases):
    pver = int(os.environ["FUZZ_PVER"]) if os.environ.get("FUZZ_PVER") else int(rng.choice([24, 26, 32, 32]))
    pcols = int(rng.choice([4, 8, 16, 24]))
    ncols = int(rng.integers(1, pcols + 1))
    cam3 = bool(rng.random() < 0.15)
    org = bool(rng.random() < 0.2) and not cam3
    nl = {}
    if rng.random() < 0.5: nl["num_cin"] = int(rng.choice([1, 3, 5]))
    if cam3: nl["num_cin"] = 5
    if rng.random() < 0.2: nl["no_deep_pbl"] = True
    if rng.random() < 0.3: nl["lparcel_pbl"] = True
    if rng.random() < 0.3: nl["tiedke_add"] = float(rng.choice([0.0, 0.25, 1.0]))
    if rng.random() < 0.3: nl["capelmt"] = float(rng.choice([20.0, 150.0, 400.0]))
    if rng.random() < 0.3: nl["dmpdz"] = float(rng.choice([-0.3e-3, -2.0e-3]))
    if rng.random() < 0.3: nl["tau"] = float(rng.choice([1200.0, 7200.0]))
    if rng.random() < 0.3: nl.update(c0_lnd=float(rng.uniform(0.001, 0.02)), c0_ocn=float(rng.uniform(0.005, 0.06)))
    if rng.random() < 0.3: nl.update(ke=float(rng.uniform(1e-6, 1e-5)), ke_lnd=float(rng.uniform(1e-6, 2e-5)))
    if rng.random() < 0.3: nl.update(momcu=float(rng.uniform(0.1, 1.0)), momcd=float(rng.uniform(0.1, 1.0)))
    if rng.random() < 0.15: nl["masterproc"] = False
    noisy = bool(rng.random() < 0.4)
    noise_rng[0] = np.random.default_rng(int(rng.integers(1, 2**31)))
    name = "fuzz_tmp_%d" % case
    cs = dict(name=name, ncols=ncols, pver=pver, p_conv=float(rng.choice([0.0, 0.3, 0.7, 1.0])), nl=nl, org=org, cam3=cam3,
              col0=int(rng.integers(0, 10**6)), pcols=pcols, transform="noise" if noisy else None,
              tracer_edge=bool(rng.random() < 0.3))
    path = os.path.join(HERE, "reftext_%s.npz" % name)
    try:
        M.run_case(**cs)
        T.test_oracle_equals_reference_source_text(name)
        g = np.load(path)
        rec = dict(case=case, pver=pver, pcols=pcols, ncol=ncols, cam3=cam3, org=org, noisy=noisy, nl=nl,
                   lengath=int(g["convr_lengath"]))
    finally:
        if os.path.exists(path):
            os.remove(path)
    report.append(rec)
    print(rec, flush=True)
print(json.dumps({"cases": len(report), "oracle_equals_reference_text_bit_for_bit": True,
                  "convective_columns": sum(r["lengath"] for r in report), "seconds": round(time.time() - t0, 1)}))
