"""Parity of the CUDA path (through the host mirrors -> C ABI) against the golden vectors produced by the
unmodified reference and against the oracle.  Tolerance (BASELINE.json north_star): relative L2 <= 1e-5 for
the fp32 device path against the reference's float64 output, max-abs reported; shapes, dtypes-on-return
and flags exact."""
import numpy as np
import pytest

from conftest import golden_names, load_golden, max_abs, rel_l2
from util import dat_from_golden, synthetic_dat

pytestmark = pytest.mark.gpu

TOL = 1e-5


def _report(name, got, want):
    r, m = rel_l2(got, want), max_abs(got, want)
    print("%-28s rel-L2 %.3e  max-abs %.3e" % (name, r, m))
    return r


@pytest.mark.parametrize("mode", ["auto", "general", "table"])
@pytest.mark.parametrize("name", golden_names(contains="_kirch_"))
def test_kirchhoff_golden(name, mode):
    from impdar_b200 import migrationlib as ml
    g = load_golden(name)
    d = dat_from_golden(g)
    uniform = not name.startswith("nu")
    ml.set_kirchhoff_mode({"auto": ml.KIRCHHOFF_AUTO, "general": ml.KIRCHHOFF_GENERAL, "table": ml.KIRCHHOFF_TABLE}[mode])
    try:
        if mode == "table" and not uniform:
            with pytest.raises(ValueError):
                d.migrate(mtype='kirch', vel=float(g["vel"]), nearfield=bool(g["nearfield"]))
            return
        d.migrate(mtype='kirch', vel=float(g["vel"]), nearfield=bool(g["nearfield"]))
        path = ml.kirchhoff_last_path()
    finally:
        ml.set_kirchhoff_mode(ml.KIRCHHOFF_AUTO)
    assert path == ("general" if (mode == "general" or not uniform) else "table")
    assert d.data.dtype == np.float64 and d.data.shape == g["out"].shape
    assert d.flags.mig == 'kirch'
    assert _report(name + "[" + path + "]", d.data, g["out"]) < TOL


@pytest.mark.parametrize("mode", ["general", "table"])
@pytest.mark.parametrize("S,T,tt0,nearfield", [(300, 257, 0.0, False), (257, 300, 0.37, True), (64, 1100, 0.0, False)])
def test_kirchhoff_vs_oracle(S, T, tt0, nearfield, mode):
    """Rough (white-noise) data at sizes beyond the golden vectors: every nearest-sample pick must be the
    oracle's, otherwise rel-L2 jumps to ~1e-2.  The shard [x_begin, x_end) entry is exercised too."""
    from impdar_b200 import migrationlib as ml
    from oracle import migration as om
    import torch
    d = synthetic_dat(S, T, seed=S + T, tt0_us=tt0)
    x64 = d.data.astype(np.float64)
    xb, xe = T // 3, T // 3 + 61
    want = om.kirchhoff(x64, d.travel_time, d.dist, 1.69e8, nearfield, xb, xe)
    ml.set_kirchhoff_mode(ml.KIRCHHOFF_GENERAL if mode == "general" else ml.KIRCHHOFF_TABLE)
    try:
        ml.enable_kirchhoff_stats(True)
        got = ml.kirchhoff_device(torch.from_numpy(d.data).cuda(), d.travel_time, d.dist, 1.69e8, nearfield, xb, xe)
        torch.cuda.synchronize()
        pairs, exact = ml.kirchhoff_stats()
    finally:
        ml.enable_kirchhoff_stats(False)
        ml.set_kirchhoff_mode(ml.KIRCHHOFF_AUTO)
    assert got.shape == (S, xe - xb)
    assert pairs > 0
    assert _report("kirch %dx%d %s" % (S, T, mode), got.cpu().numpy(), want) < TOL


@pytest.mark.parametrize("mode", ["general", "table"])
@pytest.mark.parametrize("S,T,nearfield,nchunks", [(1100, 1030, False, 8), (257, 300, True, 5), (96, 4100, False, 32),
                                                   (64, 50, False, 1)])
def test_kirchhoff_host_pipeline_equals_device_path(S, T, nearfield, nchunks, mode):
    """The host-to-host entry (row chunks processed bottom-up with upload / kernels / download overlapped) returns
    bit for bit what the device-resident call returns: the chunking only reorders independent output rows.  The
    input carries NaNs in a few rows of its top chunk, which the bottom chunks (processed first) never read: the nansum
    variant and the tile kernel's stand-down are decided per output row from the deepest non-finite input row, so the
    chunks that run before the NaN rows are seen decide as the one-launch call does."""
    from impdar_b200 import migrationlib as ml
    import torch
    d = synthetic_dat(S, T, seed=7 * S + T, tt0_us=0.0 if not nearfield else 0.11)
    top = S // nchunks
    d.data[sorted({1, max(1, top // 2), top - 1}), T // 3:T // 3 + 5] = np.nan
    if mode == "general":
        d.dist = np.cumsum(0.004 + 0.002 * np.random.default_rng(1).random(T))      # irregular spacing
    ml.set_kirchhoff_mode(ml.KIRCHHOFF_GENERAL if mode == "general" else ml.KIRCHHOFF_AUTO)
    try:
        want = ml.kirchhoff_device(torch.from_numpy(d.data).cuda(), d.travel_time, d.dist, 1.69e8, nearfield)
        want = want.double().cpu().numpy()
        got = ml.kirchhoff_host(d.data, d.travel_time, d.dist, 1.69e8, nearfield, nchunks=nchunks)
        pinned = torch.from_numpy(d.data).pin_memory()
        got_pinned = ml.kirchhoff_host(pinned.numpy(), d.travel_time, d.dist, 1.69e8, nearfield, nchunks=nchunks)
        assert ml.kirchhoff_last_path() == mode
    finally:
        ml.set_kirchhoff_mode(ml.KIRCHHOFF_AUTO)
    assert got.dtype == np.float64 and got.shape == (S, T)
    assert np.isfinite(want).all()           # nansum: the NaN terms are skipped
    assert np.array_equal(got, want) and np.array_equal(got_pinned, want)


@pytest.mark.parametrize("pipeline", ["auto", "generic"])
@pytest.mark.parametrize("name", golden_names(contains="_stolt"))
def test_stolt_golden(name, pipeline):
    """auto = paired-trace C2C pipeline for even shapes; generic = R2C/C2R pipeline (odd shapes always use it)."""
    from impdar_b200 import migrationlib as ml
    g = load_golden(name)
    d = dat_from_golden(g)
    ml.stolt_force_generic(pipeline == "generic")
    try:
        d.migrate(mtype='stolt', vel=float(g["vel"]), htaper=float(g["htaper"]), vtaper=float(g["vtaper"]))
    finally:
        ml.stolt_force_generic(False)
    name = name + "[" + pipeline + "]"
    assert d.data.shape == g["out"].shape
    assert d.data.dtype == (np.float32 if g["data"].dtype == np.float32 else np.float64)
    assert _report(name, d.data, g["out"]) < TOL


@pytest.mark.parametrize("name", golden_names(contains="_phsh_"))
def test_phase_shift_golden(name):
    g = load_golden(name)
    d = dat_from_golden(g, dtype=np.float64)
    vel = g["vel"] if g["vel"].ndim else float(g["vel"])
    from impdar_b200 import migrationlib
    migrationlib.migrationPhaseShift(d, vel=vel, htaper=float(g["htaper"]), vtaper=float(g["vtaper"]))
    assert d.data.dtype == np.float64 and d.data.shape == g["out"].shape
    assert _report(name, d.data, g["out"]) < TOL


@pytest.mark.parametrize("name", golden_names(contains="_tk"))
def test_tk_golden(name):
    g = load_golden(name)
    d = dat_from_golden(g)
    d.migrate(mtype='tk', htaper=float(g["htaper"]), vtaper=float(g["vtaper"]))
    assert d.flags.mig == 'tk'
    assert _report(name, d.data, g["out"]) < 1e-6


@pytest.mark.parametrize("name", golden_names(contains="_hfilt"))
def test_hfilt_golden(name):
    g = load_golden(name)
    d = dat_from_golden(g)
    d.hfilt(ftype='hfilt', bounds=(int(g["ntr1"]), int(g["ntr2"])))
    assert d.data.dtype == g["out"].dtype
    assert np.all(d.flags.hfilt == 1)
    assert _report(name, d.data, g["out"]) < 1e-14
    if "target" in g:  # the reference's exact known-answer test, test_RadarDataFiltering.py:53-57
        assert np.all(d.data == g["target"])
    d32 = dat_from_golden(g, dtype=np.float32)
    d32.horizontalfilt(int(g["ntr1"]), int(g["ntr2"]))
    assert d32.data.dtype == np.float32
    assert rel_l2(d32.data, g["out"]) < TOL


@pytest.mark.parametrize("name", golden_names(contains="_ahfilt_"))
def test_ahfilt_golden(name):
    g = load_golden(name)
    d = dat_from_golden(g)
    d.hfilt(ftype='adaptive', window_size=int(g["window_size"]))
    assert d.flags.hfilt[0] == 1 and d.flags.hfilt[1] == 4
    assert _report(name, d.data, g["out"]) < 1e-13
    d32 = dat_from_golden(g, dtype=np.float32)
    d32.adaptivehfilt(int(g["window_size"]))
    assert d32.data.dtype == np.float32
    assert rel_l2(d32.data, g["out"]) < TOL


@pytest.mark.parametrize("S,T,w", [(300, 5000, 7), (300, 5000, 100), (130, 5000, 1001), (130, 5000, 4000),
                                   (70, 3000, 6000), (200, 8192, 1000), (64, 2500, 2), (40, 700, 1), (40, 700, 0),
                                   (33, 130, 129), (33, 130, 130), (33, 130, 131), (50, 65, 3), (20, 2049, 64)])
def test_ahfilt_strip_vs_oracle(S, T, w):
    """The default path (prefix-sum strip kernel with a rolling 7-row ring; warp-sliding kernel for windows wider than
    its buffer) against the float64 oracle on shapes with several strips, odd / even / oversized windows and a DC
    offset; the warp-sliding kernel and the one-row-per-CTA kernel forced through the testing hook, same oracle."""
    import torch
    from oracle import filtering as of
    from impdar_b200 import _lib, filtering as fl
    rng = np.random.default_rng(S + T + w)
    x = (rng.standard_normal((S, T)) + 25.0).astype(np.float32)
    tt = np.arange(S) * 0.01
    want = of.adaptivehfilt(x.astype(np.float64), tt, w)
    tp = np.exp(-tt * 0.05) / np.exp(-tt[0] * 0.05)
    xd = torch.from_numpy(x).cuda()
    got = fl.adaptivehfilt_device(xd, 'f32', tp, w).cpu().numpy()
    lib = _lib.load()
    others = []
    for mode in (1, 2, 3):                  # 1 = one-row-per-CTA kernel, 2 = first strip kernel, 3 = warp-sliding kernel
        lib.impdar_ahfilt_force_rowwise(mode)
        try:
            others.append(fl.adaptivehfilt_device(xd, 'f32', tp, w).cpu().numpy())
        finally:
            lib.impdar_ahfilt_force_rowwise(0)
    m = np.isfinite(want)
    assert np.array_equal(np.isfinite(got), m)
    assert _report("ahfilt %dx%d w%d" % (S, T, w), got[m], want[m]) < TOL
    for o in others:
        assert np.array_equal(np.isfinite(o), m) and rel_l2(o[m], want[m]) < TOL
    # batch of two profiles == the profiles one by one
    xb = torch.stack([xd, xd.flip(0).contiguous()])
    gb = fl.adaptivehfilt_device(xb, 'f32', tp, w)
    assert torch.equal(gb[0].nan_to_num(), torch.from_numpy(got).cuda().nan_to_num())


@pytest.mark.parametrize("name", golden_names(contains="_vbp_"))
def test_vbp_golden(name):
    g = load_golden(name)
    d = dat_from_golden(g)
    d.vertical_band_pass(float(g["low"]), float(g["high"]), order=int(g["order"]), filttype=str(g["filttype"]))
    assert d.flags.bpass[0] == 1 and d.flags.bpass[1] == float(g["low"]) and d.flags.bpass[2] == float(g["high"])
    assert _report(name, d.data, g["out"]) < 1e-6   # the recurrence itself differs ~1e-9 between fp64 orderings
    d32 = dat_from_golden(g, dtype=np.float32)
    d32.vertical_band_pass(float(g["low"]), float(g["high"]), order=int(g["order"]), filttype=str(g["filttype"]))
    assert d32.data.dtype == np.float32
    assert _report(name + "[f32]", d32.data, g["out"]) < TOL


@pytest.mark.parametrize("S,T", [(512, 768), (500, 1026), (333, 200)])
def test_stolt_vs_oracle(S, T):
    from oracle import migration as om
    d = synthetic_dat(S, T, seed=S * 3 + T)
    x64 = d.data.astype(np.float64)
    _, want = om.stolt(x64, d.dt, d.trace_int, d.dist, 1.68e8, 10, 20)
    d.migrate(mtype='stolt', vel=1.68e8, htaper=10, vtaper=20)
    assert d.data.shape == want.shape and d.data.dtype == np.float32
    assert _report("stolt %dx%d" % (S, T), d.data, want) < TOL


def test_noinit_fixtures():
    """The reference's own fixtures: zeros(10, 20) through every migration (test_migrationlib.py:103-135)."""
    import impdar_b200
    from impdar_b200 import migrationlib

    def big():
        d = impdar_b200.RadarData(np.zeros((10, 20)), dt=1, travel_time=np.arange(10), dist=np.arange(20),
                                  trace_int=1)
        return d
    for fn in (migrationlib.migrationStolt, migrationlib.migrationKirchhoff,
               migrationlib.migrationTimeWavenumber, migrationlib.migrationPhaseShift):
        d = fn(big())
        assert np.all(d.data == 0)
    d = big()
    d.data = d.data.astype(int)
    d = migrationlib.migrationStolt(d)
    assert np.all(d.data == 0) and d.data.dtype == np.float64
    d = big()
    d.data = np.ones((1, 1))
    with pytest.raises(ValueError):
        migrationlib.migrationStolt(d)
    with pytest.raises(TypeError):
        migrationlib.migrationPhaseShift(big(), vel_fn='notafile.txt')


def test_bad_mtype_and_ftype():
    d = synthetic_dat(32, 16)
    with pytest.raises(ValueError):
        d.migrate(mtype='dummy')
    with pytest.raises(ValueError):
        d.hfilt(ftype='dummy')
    with pytest.raises(ValueError):
        d.vertical_band_pass(0.1, 100., filttype='dummy')


# ------------------------------------------------------------------ sibling filters (SURVEY.md 8f rank 2)
@pytest.mark.parametrize("name", golden_names(contains="_winavg_"))
def test_winavg_golden(name):
    g = load_golden(name)
    d = dat_from_golden(g)
    d.winavg_hfilt(int(g["avg_win"]), taper=str(g["taper"]), filtdepth=int(g["filtdepth"]))
    assert d.flags.hfilt[0] == 0 and d.flags.hfilt[1] == 2
    assert d.data.dtype == g["out"].dtype
    assert _report(name, d.data, g["out"]) < 1e-13       # rel_l2 also checks the NaN pattern (avg_win = 1)
    d32 = dat_from_golden(g, dtype=np.float32)
    d32.winavg_hfilt(int(g["avg_win"]), taper=str(g["taper"]), filtdepth=int(g["filtdepth"]))
    assert d32.data.dtype == np.float32
    assert rel_l2(d32.data, g["out"]) < TOL
    with pytest.raises(ValueError):
        d.winavg_hfilt(5, taper='dummy')


@pytest.mark.parametrize("name", ["r96x160_highpass", "r96x160_lowpass", "r96x160_horizontal_band_pass"])
def test_horizontal_iir_golden(name):
    from impdar_b200.filtering import ImpdarError
    g = load_golden(name)
    meth = name[len("r96x160_"):]
    args = [float(a) for a in g["args"]]
    d = dat_from_golden(g)
    with pytest.raises(ImpdarError):            # not constantly spaced yet (flags.interp), :170 / :240 / :298
        getattr(d, meth)(*args)
    d.flags.interp = np.array([1., float(g["tracespace"])])
    getattr(d, meth)(*args)
    assert d.data.dtype == np.float64 and d.flags.hfilt[0] == 1 and d.flags.hfilt[1] == 3
    assert _report(name, d.data, g["out"]) < 1e-6    # the recurrence itself differs ~1e-9 between fp64 orderings
    d32 = dat_from_golden(g, dtype=np.float32)
    d32.flags.interp = np.array([1., float(g["tracespace"])])
    getattr(d32, meth)(*args)
    assert d32.data.dtype == np.float64              # filtfilt returns float64 whatever the input (:203)
    assert _report(name + "[f32]", d32.data, g["out"]) < TOL
    d.flags.elev = 1
    with pytest.raises(ImpdarError):
        getattr(d, meth)(*args)


@pytest.mark.parametrize("S,T", [(70, 1000), (33, 257), (200, 64)])
def test_horizontal_iir_vs_oracle(S, T):
    """Row counts that are not multiples of 32, trace counts that are not multiples of the 32-sample chunk."""
    from oracle import filtering as of
    d = synthetic_dat(S, T, seed=S + T, dtype=np.float64)
    d.flags.interp = np.array([1., 5.])
    want = of.highpass(d.data, 100., 5., d.dt)
    d.highpass(100.)
    assert _report("highpass %dx%d" % (S, T), d.data, want) < 1e-6
    d = synthetic_dat(S, T, seed=S + T, dtype=np.float64)
    d.flags.interp = np.array([1., 5.])
    want = of.horizontal_band_pass(d.data, 40., 200., 5.) if T > 40 else None
    if want is not None:
        d.horizontal_band_pass(40., 200.)
        assert _report("hbp %dx%d" % (S, T), d.data, want) < 1e-6


@pytest.mark.parametrize("name", golden_names(contains="_rangegain_") + golden_names(contains="_agc"))
def test_gains_golden(name):
    g = load_golden(name)
    for dtype in (np.float64, np.float32):
        d = dat_from_golden(g, dtype=dtype)
        if "_agc" in name:
            d.agc(window=int(g["window"]), scaling_factor=int(g["scaling_factor"]))
            assert d.flags.agc is True
        else:
            d.trig = g["trig"] if g["trig"].ndim else int(g["trig"])
            d.rangegain(float(g["slope"]))
            assert d.flags.rgain is True
        assert d.data.dtype == dtype
        if dtype == np.float64:
            assert np.array_equal(d.data, g["out"])          # one rounding per element: bit-exact
        else:
            assert _report(name + "[f32]", d.data, g["out"]) < TOL
    d = dat_from_golden(g, dtype=np.int32)
    with pytest.raises(TypeError):
        d.trig = 0
        d.rangegain(1.0)


def test_winavg_long_rows_vs_oracle():
    """Rows longer than the shared-memory prefix buffer take the global-scratch path."""
    from oracle import filtering as of
    d = synthetic_dat(16, 30000, seed=5, dtype=np.float64)
    d.data += 10.0
    want = of.winavg_hfilt(d.data[:, :], d.travel_time, 201)
    d.winavg_hfilt(201)
    assert _report("winavg 16x30000", d.data, want) < 1e-12


@pytest.mark.parametrize("name", golden_names(contains="_denoise_"))
def test_denoise_golden(name):
    g = load_golden(name)
    noise = None if np.isnan(g["noise"]) else float(g["noise"])
    d = dat_from_golden(g)
    d.denoise(vert_win=int(g["vert_win"]), hor_win=int(g["hor_win"]), noise=noise)
    assert isinstance(d.data, np.ndarray) and d.data.dtype == np.float64 and d.data.shape == g["out"].shape
    assert _report(name, d.data, g["out"]) < (1e-6 if g["data"].dtype == np.float32 else 1e-12)


def test_denoise_large_vs_oracle_and_errors():
    from oracle import filtering as of
    import torch
    d = synthetic_dat(700, 1300, seed=41)
    want = of.wiener(d.data, 5, 9)
    x = d.data.copy()
    d.denoise(vert_win=5, hor_win=9)
    assert _report("denoise 700x1300 f32", d.data, want) < 1e-12
    d = synthetic_dat(64, 96, seed=42)
    d.data = torch.from_numpy(d.data).cuda()                     # device lane: stays on the GPU, float32 in -> float32 out
    d.denoise(noise=0.3)
    assert isinstance(d.data, torch.Tensor) and d.data.is_cuda and d.data.dtype == torch.float32
    d = synthetic_dat(32, 64, seed=43)
    d.data[:] = 1.0
    d.data[:, 40:] = np.arange(32, dtype=np.float32)[:, None]    # zero local variance in the left half, not overall
    with pytest.raises(ValueError):
        d.denoise(vert_win=1, hor_win=3)
    with pytest.raises(ValueError):
        d.denoise(ftype='dummy')


@pytest.mark.parametrize("name", golden_names(contains="_median_"))
def test_denoise_median_golden(name):
    """Pure selection: bit-exact, dtype kept (float64, float32, int16)."""
    g = load_golden(name)
    d = dat_from_golden(g)
    d.denoise(vert_win=int(g["vert_win"]), hor_win=int(g["hor_win"]), ftype='median')
    assert d.data.dtype == g["out"].dtype and np.array_equal(d.data, g["out"])


def test_denoise_median_large_vs_oracle():
    from oracle import filtering as of
    d = synthetic_dat(257, 1031, seed=51)
    d.data = np.round(d.data * 4) / 4                      # many ties: the stable rank must still pick the right value
    want = of.median_filter(d.data, 7, 9)
    d.denoise(vert_win=7, hor_win=9, ftype='median')
    assert np.array_equal(d.data, want)
    d = synthetic_dat(5, 6, seed=52)                       # window wider than the radargram: repeated reflection
    want = of.median_filter(d.data, 3, 15)
    d.denoise(vert_win=3, hor_win=15, ftype='median')
    assert np.array_equal(d.data, want)
    with pytest.raises(ValueError):
        d.denoise(vert_win=17, hor_win=16, ftype='median')  # 272 samples > the 256 the kernel holds


def test_tk_float64_is_exact_and_device_dtypes_never_narrow():
    """The time-wavenumber stub is `data *= H * V` (mig_python.py:330-335): a float64 radargram is tapered in float64,
    bit for bit numpy's result, on the host lane and on the device lane; a float64 CUDA tensor comes back float64 from
    every migration (values float32-accurate where the path computes in float32 - the documented dtype policy)."""
    import torch
    from oracle import migration as om
    d = synthetic_dat(70, 90, seed=4, dtype=np.float64)
    want = om.time_wavenumber(d.data, 13, 9)
    d.migrate(mtype='tk', htaper=13, vtaper=9)
    assert d.data.dtype == np.float64 and np.array_equal(d.data, want)
    d = synthetic_dat(70, 90, seed=4, dtype=np.float64)
    d.data = torch.from_numpy(d.data).cuda()
    d.migrate(mtype='tk', htaper=13, vtaper=9)
    assert d.data.dtype == torch.float64 and np.array_equal(d.data.cpu().numpy(), want)
    for mtype in ('stolt', 'kirch', 'phsh'):
        d = synthetic_dat(64, 96, seed=5, dtype=np.float64)
        d.data = torch.from_numpy(d.data).cuda()
        d.migrate(mtype=mtype)
        assert d.data.is_cuda and d.data.dtype == torch.float64, mtype
        d = synthetic_dat(64, 96, seed=5, dtype=np.float32)
        d.data = torch.from_numpy(d.data).cuda()
        d.migrate(mtype=mtype)
        assert d.data.is_cuda and d.data.dtype == torch.float32, mtype


def test_rangegain_negative_per_trace_triggers():
    """Per-trace triggers below -1 (they occur after crop(..., zero_trig=False)): the reference slices
    data[int(trig) + 1:, i] with Python's negative-index rules (_RadarDataProcessing.py:466-469), so only the last rows
    get the gain."""
    d = synthetic_dat(40, 12, seed=9, dtype=np.float64)
    trig = np.array([3, -1, -2, -5, 0, -40, -41, -100, 38, 39, 45, -3])
    d.trig = trig.copy()
    want = d.data.copy()
    for i, t in enumerate(trig):                                   # the reference's own loop
        gain = d.travel_time[int(t) + 1:] * 0.3
        want[int(t) + 1:, i] *= gain
    d.rangegain(0.3)
    assert np.array_equal(d.data, want)
