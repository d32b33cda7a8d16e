"""CPU tests of the product's host side: the C-ABI library builds for sm_100a, loads without a GPU and
exports every symbol include/zmconv_b200.h declares; portable math accuracy; soundings generator."""
import ctypes
import math
import os
import re

import numpy as np
import pytest

from cam_nor_physics_b200 import soundings as S

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_exports_every_declared_symbol(built):
    from cam_nor_physics_b200 import zm_conv as Z
    hdr = open(os.path.join(ROOT, "include", "zmconv_b200.h")).read()
    hdr = re.sub(r"/\*.*?\*/", "", hdr, flags=re.S)
    names = set(re.findall(r"\b(?:int|void|double|long long|const char\*)\s+(zm_[a-z0-9_]+)\s*\(", hdr))
    assert len(names) >= 20
    lib = Z.lib()
    missing = [n for n in sorted(names) if not hasattr(lib, n)]
    assert not missing, missing
    assert set(Z.EXPORTS) <= names | {"zm_params_default"}


def test_library_is_built_from_the_sources_in_the_tree(built):
    """The hash of the sources and compiler flags is compiled into the library: a stale binary cannot be tested."""
    from cam_nor_physics_b200 import build, zm_conv as Z
    info = Z.lib().zm_build_info().decode()
    assert info.startswith("ZMSRCHASH:") and build.source_hash() in info
    assert build.built_hash() == build.source_hash() and not build.needs_build()


def test_sm100a_code_is_embedded(built):
    import subprocess
    from cam_nor_physics_b200 import build
    cuobjdump = os.path.join(os.path.dirname(os.path.realpath(build._nvcc())), "cuobjdump")   # nvcc's own toolkit
    out = subprocess.run([cuobjdump, "-lelf", build.LIB], capture_output=True, text=True).stdout
    assert "sm_100a" in out


def test_uninitialised_call_fails_loudly(built):
    from cam_nor_physics_b200 import zm_conv as Z
    Z.lib().zm_finalize()
    rc = Z.lib().zm_sync_check(None)
    assert rc == 0
    buf = np.zeros(4)
    rc = Z.lib().zm_thermo_eval_dev(0, 1, *(buf.ctypes.data_as(ctypes.c_void_p),) * 7)
    assert rc == -1 and "zm_init" in Z.last_error()


def test_portable_math_accuracy_host(built):
    """zm_math.h (host build inside the library) is < 1 ulp against mpmath."""
    import mpmath as mp
    from cam_nor_physics_b200 import zm_conv as Z
    mp.mp.prec = 120
    rng = np.random.default_rng(11)
    n = 3000
    cases = [(0, np.exp(rng.uniform(-20, 20, n)), None, lambda x, y: mp.log(x)),
             (1, rng.uniform(1.0, 3.0, n), None, lambda x, y: mp.log10(x)),
             (2, rng.uniform(-30, 30, n), None, lambda x, y: mp.exp(x)),
             (3, rng.uniform(-8, 8, n), None, lambda x, y: mp.power(10, x)),
             (4, rng.uniform(0.9, 30, n), np.full(n, 287.04 / 1004.64), lambda x, y: mp.power(x, y))]
    for fid, x, y, f in cases:
        got = Z.math_eval(fid, x, y, device=False)
        yy = x if y is None else y
        worst = 0.0
        for g, a, b in zip(got, x, yy):
            e = f(mp.mpf(float(a)), mp.mpf(float(b)))
            worst = max(worst, float(abs(mp.mpf(float(g)) - e) / math.ulp(float(e))))
        assert worst < 1.0, (fid, worst)


def test_saturation_vapour_pressure_table_host(built):
    """es(T) over water comes from per-kelvin polynomials of the Goff-Gratch formula (zm_svp_table.h): against the
    formula in 200-bit arithmetic the table is within 2 ulp over 139.5..349.5 K -- the formula evaluated in double
    (what the reference runs) is itself tens of ulp off at the cold end -- and the two agree to 2e-14 relative;
    outside the table the formula is used."""
    import mpmath as mp
    from cam_nor_physics_b200 import zm_conv as Z
    mp.mp.prec = 200
    c = {k: mp.mpf(float(v)) for k, v in dict(ts="373.16", a="7.90298", b="5.02808", c="1.3816e-7", d="11.344",
                                               e="8.1328e-3", f="3.49149").items()}

    def svp(t):
        u = c["ts"] / t
        ex = (-c["a"] * (u - 1) + c["b"] * mp.log10(u) - c["c"] * (mp.power(10, c["d"] * (1 - t / c["ts"])) - 1)
              + c["e"] * (mp.power(10, -c["f"] * (u - 1)) - 1) + mp.mpf(3.0057148979490314))
        return mp.power(10, ex) * 100

    rng = np.random.default_rng(3)
    T = np.concatenate([rng.uniform(139.5, 349.5, 1500), np.arange(140, 349) + 0.5 + 1e-13, np.arange(140, 349) + 0.5 - 1e-13,
                        np.arange(140, 349) + 0.5, np.arange(140, 350).astype(float)])      # incl. the cell edges
    tab, frm = Z.math_eval(10, T, device=False), Z.math_eval(11, T, device=False)
    worst = 0.0
    for t, a in zip(T, tab):
        e = svp(mp.mpf(float(t)))
        worst = max(worst, float(abs(mp.mpf(float(a)) - e)) / math.ulp(float(e)))
    assert worst < 2.0, worst
    assert np.max(np.abs(tab - frm) / frm) < 2e-14
    warm = T > 200.0
    assert np.max(np.abs(tab - frm)[warm] / frm[warm]) < 8e-15
    out = np.array([60.0, 89.499, 349.5, 360.0, 420.0])
    assert np.array_equal(Z.math_eval(10, out, device=False), Z.math_eval(11, out, device=False))
    assert np.all(np.diff(Z.math_eval(10, np.linspace(139.0, 350.5, 40001), device=False)) > 0)   # monotone across cells
    # the cells below 140 K (parcels of cold columns lifted to 40 hPa) follow a function that collapses
    # super-exponentially: relative accuracy degrades (3e-13 at 125 K, 4e-5 at 100 K), the absolute error stays
    # below 1e-23 Pa (an ulp at 139 K) -- nothing the state function can resolve against pressures of 4e3 Pa and more
    cold = np.concatenate([rng.uniform(89.5, 139.5, 1500), np.arange(90, 140) + 0.5, np.arange(90, 140).astype(float)])
    tabc, frmc = Z.math_eval(10, cold, device=False), Z.math_eval(11, cold, device=False)
    exact = np.array([float(svp(mp.mpf(float(t)))) for t in cold])
    assert np.all(tabc > 0) and np.max(np.abs(tabc - exact)) < 1e-23
    assert np.max(np.abs(tabc - frmc)) < 1e-21          # the formula in double is itself 1e-14 relative off here
    near = cold >= 125.0
    assert np.max(np.abs(tabc - exact)[near] / exact[near]) < 1e-12
    assert np.all(np.diff(Z.math_eval(10, np.linspace(95.0, 139.6, 20001), device=False)) > 0)
    # below 95 K (es < 1e-50 Pa) neighbouring cells meet with steps of the size of their own error
    low = Z.math_eval(10, np.linspace(89.6, 95.0, 5001), device=False)
    assert np.all(low > 0) and np.min(np.diff(low)) > -1e-50


def test_hot_math_variants_equal_general_ones_host(built):
    """The state function uses trimmed transcendentals (no special-case selects) and constant-reciprocal
    divisions; inside their stated domains they must return the same bits as the general ones."""
    from cam_nor_physics_b200 import zm_conv as Z
    rng = np.random.default_rng(5)
    n = 400_000
    xs = np.concatenate([np.exp(rng.uniform(-700, 700, n)), rng.uniform(0.5, 2.0, n), [1.0, 2.0, 0.5, 1e-300, 1e300]])
    assert np.array_equal(Z.math_eval(5, xs, device=False), Z.math_eval(0, xs, device=False))      # log
    assert np.array_equal(Z.math_eval(6, xs, device=False), Z.math_eval(1, xs, device=False))      # log10
    assert Z.math_eval(0, np.array([1.0]), device=False)[0] == 0.0 and not np.signbit(Z.math_eval(0, np.array([1.0]), device=False)[0])
    xp = np.concatenate([rng.uniform(-300, 300, n), rng.uniform(-3, 8, n), [0.0, -0.0]])
    assert np.array_equal(Z.math_eval(7, xp, device=False), Z.math_eval(3, xp, device=False))      # 10**x
    # a/b through RN(1/b) + one residual correction == IEEE division (divisors used by the state function)
    for b in (373.16, 1000.0, 273.15, 273.16):
        a = np.concatenate([rng.uniform(50, 1000, n), np.exp(rng.uniform(-50, 50, n))])
        bb = np.full_like(a, b)
        assert np.array_equal(Z.math_eval(8, a, bb, device=False), a / bb), b


def test_soundings_are_shard_independent():
    a = S.make_chunks(64, 32, 16, p_conv=0.5)
    b = S.make_chunks(32, 32, 16, p_conv=0.5, col0=32)
    for k in ["t", "q", "pmid", "pint", "zm", "zi", "u", "cld"]:
        assert np.array_equal(getattr(a, k)[2:], getattr(b, k)), k
    assert np.array_equal(a.phis[2:], b.phis)
    assert S.limcnv_for(32) == 3
    # hydrostatic and monotone
    assert np.all(np.diff(a.pint, axis=1) > 0) and np.all(np.diff(a.zi, axis=1) < 0)
    assert np.all(a.q >= 1e-12)
    # ragged last chunk
    c = S.make_chunks(40, 32, 16)
    assert list(c.ncol) == [16, 16, 8]
