"""Pin the oracle against the reference: its outputs stored in tests/golden (written by the UNMODIFIED reference,
tests/golden/make_golden.py) at the tolerances of the live comparison; the `reference`-marked tests run the reference
itself (an ImpDAR checkout at IMPDAR_REFERENCE_SRC, default /root/reference/src) and skip without it."""
import contextlib
import io

import numpy as np
import pytest

from conftest import load_golden, rel_l2
from oracle import filtering as of
from oracle import migration as om


def _ref():
    from oracle._refimport import import_reference
    return import_reference()


def _quiet(f, *a, **k):
    with contextlib.redirect_stdout(io.StringIO()):
        return f(*a, **k)


def _mk(RD, S, T, seed, tt0=0.0, dtype=np.float64):
    rng = np.random.default_rng(seed)
    d = RD(None)
    d.data = rng.standard_normal((S, T)).astype(dtype)
    d.snum, d.tnum, d.dt = S, T, 1e-8
    d.travel_time = tt0 + np.arange(S) * 0.01
    d.dist = np.arange(T) * 0.005
    d.trace_int = np.ones(T) * 5.0
    return d


# every stored shape with all four migrations: even and odd snum, first sample at t = 0 and after it (r65x50)
@pytest.mark.parametrize("shape", ["nu48x40", "r64x128", "r65x50", "r128x200"])
def test_migrations(shape):
    for nf in ("far", "near"):
        g = load_golden("%s_kirch_%s" % (shape, nf))
        out = om.kirchhoff(g["data"], g["travel_time"], g["dist"], float(g["vel"]), bool(g["nearfield"]))
        assert rel_l2(out, g["out"]) < 1e-13
    g = load_golden(shape + "_stolt")
    out = om.stolt(g["data"], float(g["dt"]), g["trace_int"], g["dist"], float(g["vel"]), float(g["htaper"]),
                   float(g["vtaper"]))[1]
    assert rel_l2(out, g["out"]) < 1e-13
    g = load_golden(shape + "_phsh_const")
    out = om.phase_shift(g["data"], float(g["dt"]), g["travel_time"], g["trace_int"], g["dist"], float(g["vel"]),
                         float(g["htaper"]), float(g["vtaper"]))[1]
    assert rel_l2(out, g["out"]) < 1e-13
    g = load_golden(shape + "_tk")
    assert np.array_equal(om.time_wavenumber(g["data"], float(g["htaper"]), float(g["vtaper"])), g["out"])


@pytest.mark.reference
def test_stolt_int_dtype_truncation():
    mp, RD, _ = _ref()
    d = _mk(RD, 32, 24, 5)
    d.data = (d.data * 10).astype(int); x = d.data.copy()
    _quiet(mp.migrationStolt, d, vel=1.68e8, htaper=4, vtaper=6)
    assert rel_l2(om.stolt(x, d.dt, d.trace_int, d.dist, 1.68e8, 4, 6)[1], d.data) < 1e-13


def test_filters_and_known_answer():
    g = load_golden("noinit_hfilt")        # NoInitRadarDataFiltering's data and hfilt_target_output
    assert np.all(of.horizontalfilt(g["data"], g["travel_time"], 0, 100) == g["target"])
    for w in (2, 10, 103, 192):            # first sample after t = 0
        g = load_golden("r256x96_ahfilt_w%d" % w)
        assert rel_l2(of.adaptivehfilt(g["data"], g["travel_time"], w), g["out"]) < 1e-13
    g = load_golden("r256x96_vbp_butter")  # the reference's defaults: 5th-order Butterworth
    assert np.array_equal(of.vertical_band_pass(g["data"], float(g["dt"]), float(g["low"]), float(g["high"])), g["out"])


@pytest.mark.reference
def test_reference_own_hot_path_tests_pass_here():
    """The reference's own test modules for the path run green with this environment (SURVEY.md 8c)."""
    import os
    import subprocess
    import sys
    import tempfile
    from oracle._refimport import REFERENCE_SRC
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    tests = [os.path.join(os.path.dirname(REFERENCE_SRC), "test", f)
             for f in ("test_migrationlib.py", "test_RadarDataFiltering.py")]
    env = dict(os.environ)
    code = ("import sys, types; sys.path.insert(0, %r);"
            "from oracle._refimport import import_reference; import_reference();"
            "import pytest; sys.exit(pytest.main(['-q', '-x', '-p', 'no:cacheprovider', %r, %r]))" % (root, tests[0], tests[1]))
    r = subprocess.run([sys.executable, "-c", code], env=env, stdout=subprocess.PIPE, stderr=subprocess.STDOUT,
                       text=True, cwd=tempfile.gettempdir())
    assert r.returncode == 0, r.stdout[-2000:]
