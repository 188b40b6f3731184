"""Migration velocity scan: Stolt images over a velocity grid, a per-window focus measure, picks, and the RMS field they
give Kirchhoff.

CPU part: closed forms of a numpy float64 restatement of the focus measure; recovery of the diffractors' velocities
through the float64 Stolt oracle (constant velocity: the exact grid velocity; a layered RMS profile: within one grid
step of V(t_apex)); scan_rms_field's masking, interpolation, fill, merging and trace map; argument errors of the Python
and C entries.
GPU part: every image of a scan equals stolt_device at its velocity bit for bit on each lane; the focus panel against
the restatement, across calls, with and without images, host and device lanes; recovery at config-2 size; and the scan
-> scan_rms_field -> kirchhoff_lateral_device chain focusing a layered synthetic better than one velocity does.
"""
import ctypes

import numpy as np
import pytest

from util import synthetic_dat
from test_kirchhoff_lateral import _diffractors

GRID = np.arange(1.4e8, 2.0e8 + 1.0, 0.1e8)     # steps of 5-7 %
LAYERED_GRID = np.arange(1.6e8, 2.4e8 + 1.0, 0.1e8)
F0 = 25e6     # 4 samples a period at dt = 10 ns; with 1 m traces the steepest limb moves < 1/4 period per trace


def focus_np(img, ws, wt):
    """The focus measure restated in float64: n E4 / E2^2 per window, 0 where E2 == 0."""
    m = np.asarray(img, dtype=np.float32).astype(np.float64)
    S2, T = m.shape
    rs, cs = np.arange(0, S2, ws), np.arange(0, T, wt)
    e2 = np.add.reduceat(np.add.reduceat(m ** 2, rs, axis=0), cs, axis=1)
    e4 = np.add.reduceat(np.add.reduceat(m ** 4, rs, axis=0), cs, axis=1)
    n = (np.minimum(rs + ws, S2) - rs)[:, None] * (np.minimum(cs + wt, T) - cs)[None, :]
    with np.errstate(invalid='ignore', divide='ignore'):
        return np.where(e2 == 0, 0.0, n * e4 / e2 ** 2)


def ricker_dat(S, T, points, vel, seed=0, noise=0.01):
    """Diffractors rendered like synthetic.diffractor_radargram (Ricker wavelets of support 1.5 / f0 along
    t = sqrt(t0^2 + (2 x / v)^2), plus white noise) on 1 m traces."""
    d = synthetic_dat(S, T, seed=seed, dx=1.0)
    t = np.arange(S) * d.dt
    x = np.arange(T) * 1.0
    img = noise * np.random.default_rng(seed).standard_normal((S, T))
    for s0, x0 in points:
        th = np.sqrt(t[s0] ** 2 + (2.0 * (x - x[x0]) / vel) ** 2)
        dtt = t[:, None] - th[None, :]
        a = (np.pi * F0 * dtt) ** 2
        img += np.where(np.abs(dtt) < 1.5 / F0, (1 - 2 * a) * np.exp(-a), 0.0)
    d.data = img.astype(np.float32)
    return d


def layered_dat(S, T, points):
    """Diffractors along the layered RMS profile's hyperbolas (test_kirchhoff_lateral._diffractors), and that profile."""
    from impdar_b200 import migrationlib as ml, synthetic
    d = synthetic_dat(S, T, seed=1, dx=1.0)
    V = ml.rms_velocity(d.travel_time, ml.getVelocityProfile(d, synthetic.layered_velocity(d.travel_time)))
    d.data = _diffractors(d, np.repeat(V[:, None], T, 1), points, f0=F0)
    return d, V


def oracle_scan(d, vels, window, htaper=4, vtaper=4):
    from oracle import migration as om
    from impdar_b200 import migrationlib as ml
    F = np.array([focus_np(om.stolt(np.asarray(d.data, dtype=np.float64), d.dt, d.trace_int, d.dist, v, htaper,
                                    vtaper)[1].astype(np.float32), *window) for v in vels])
    return ml.velocity_scan_result(F, vels, window, d.snum, d.tnum)


def apex_points(nws, nwt, ws, wt, rows, cols):
    """Apexes at window centres, in every other window row and column: two windows apart, half a window from edges."""
    return [(i * ws + ws // 2, j * wt + wt // 2) for i in rows for j in cols if i < nws and j < nwt]


# ------------------------------------------------------------------------------------------------------ CPU
def test_focus_closed_forms():
    ws, wt = 4, 5
    img = np.zeros((10, 12), np.float32)      # windows: rows 4, 4, 2; columns 5, 5, 2
    img[1, 2] = 3.0                            # spike
    img[4:8, 5:10] = -2.5                      # constant
    img[8:10, 10:12] = 7.0                     # constant, partial in both directions
    img[8, 0] = 1.0                            # spike in a partial window (2 x 5)
    f = focus_np(img, ws, wt)
    assert f.shape == (3, 3)
    assert f[0, 0] == 20.0 and f[1, 1] == 1.0 and f[2, 2] == 1.0 and f[2, 0] == 10.0
    assert f[0, 1] == 0.0 and f[1, 0] == 0.0 and f[2, 1] == 0.0
    one = np.zeros((7, 3), np.float32)
    one[6, 2] = 1e-30                          # float64 accumulation: tiny values keep their measure
    assert focus_np(one, 4, 2)[1, 1] == 3.0


@pytest.mark.parametrize("v0", [1.5e8, 1.7e8, 1.9e8])
def test_oracle_recovery_constant(v0):
    S, T, w = 512, 256, (64, 64)
    pts = apex_points(8, 4, 64, 64, (1, 3), (1, 3))
    d = ricker_dat(S, T, pts, v0)
    scan = oracle_scan(d, GRID, w)
    for s0, x0 in pts:
        assert scan.vrms[s0 // 64, x0 // 64] == v0, (s0, x0, scan.focus[:, s0 // 64, x0 // 64])


def test_oracle_recovery_layered():
    S, T, w = 512, 256, (64, 64)
    pts = [(96, 96), (224, 224), (352, 96)]
    d, V = layered_dat(S, T, pts)
    scan = oracle_scan(d, LAYERED_GRID, w)
    step = LAYERED_GRID[1] - LAYERED_GRID[0]
    for s0, x0 in pts:
        assert abs(scan.vrms[s0 // 64, x0 // 64] - V[s0]) <= step, (s0, x0, V[s0])


def _scan(focus, vels, window, snum, tnum):
    from impdar_b200 import migrationlib as ml
    return ml.velocity_scan_result(np.asarray(focus, dtype=np.float64), np.asarray(vels, dtype=np.float64), window,
                                   snum, tnum)


def test_scan_result_picks():
    vels = [1.5e8, 1.6e8, 1.7e8]
    F = np.zeros((3, 3, 2))
    F[:, 0, 0] = [1.0, 3.0, 3.0]               # tie: the first maximum
    F[:, 1, 0] = [5.0, 1.0, 2.0]
    F[:, 2, 1] = [0.0, 0.0, 2.0]
    s = _scan(F, vels, (4, 8), 11, 13)        # S2 = 10: window rows of 4, 4, 2
    assert np.array_equal(s.center_rows, [1.5, 5.5, 8.5])
    assert s.vrms[0, 0] == 1.6e8 and s.vrms[1, 0] == 1.5e8 and s.vrms[2, 1] == 1.7e8
    assert np.isnan(s.vrms[2, 0]) and np.isnan(s.vrms[0, 1]) and np.isnan(s.vrms[1, 1])


def test_scan_rms_field_interpolation_and_masking():
    from impdar_b200 import migrationlib as ml
    vels = [1.5e8, 1.6e8, 1.7e8, 1.8e8]
    F = np.ones((4, 3, 1))
    F[3, 0, 0] = 9.0     # row 0: 1.8e8, strong
    F[0, 1, 0] = 1.5     # row 1: 1.5e8, weak
    F[1, 2, 0] = 4.0     # row 2: 1.6e8
    s = _scan(F, vels, (10, 100), 31, 40)     # odd snum: S2 = 30, the last row lies beyond the image
    prof, colp = ml.scan_rms_field(s)
    rows = np.arange(31)
    assert prof.shape == (1, 31) and np.array_equal(colp, np.zeros(40, dtype=int))
    assert np.array_equal(prof[0], np.interp(rows, [4.5, 14.5, 24.5], [1.8e8, 1.5e8, 1.6e8]))
    assert prof[0, 0] == 1.8e8 and prof[0, 30] == 1.6e8 and prof[0, 25] == 1.6e8
    prof2, _ = ml.scan_rms_field(s, min_focus=2.0)    # row 1 (best 1.5) dropped
    assert np.array_equal(prof2[0], np.interp(rows, [4.5, 24.5], [1.8e8, 1.6e8]))
    with pytest.raises(ValueError):
        ml.scan_rms_field(s, min_focus=10.0)
    Z = np.zeros((4, 3, 1))
    with pytest.raises(ValueError):
        ml.scan_rms_field(_scan(Z, vels, (10, 100), 31, 40))


def test_scan_rms_field_fill_merge_and_trace_map():
    from impdar_b200 import migrationlib as ml
    vels = [1.5e8, 1.6e8, 1.7e8]
    nwt = 6
    F = np.zeros((3, 2, nwt))
    F[0, :, 1] = 2.0          # column 1: 1.5e8 everywhere
    F[2, :, 3] = 2.0          # column 3: 1.7e8 everywhere
    F[0, :, 5] = 2.0          # column 5: 1.5e8, bit-identical to column 1
    # columns 0, 2, 4 have no pick: 0 -> 1; 2 -> 1 (tie between 1 and 3 goes left); 4 -> 3 (tie between 3 and 5)
    s = _scan(F, vels, (8, 7), 16, 40)        # 40 traces over 6 columns of 7, the last partial
    prof, colp = ml.scan_rms_field(s)
    assert prof.shape == (2, 16)
    assert np.all(prof[0] == 1.5e8) and np.all(prof[1] == 1.7e8)
    win = np.array([0, 0, 0, 1, 1, 0])
    assert np.array_equal(colp, win[np.arange(40) // 7])
    one = _scan(F[:, :, 3:4], vels, (8, 64), 16, 40)
    prof1, colp1 = ml.scan_rms_field(one)
    assert prof1.shape == (1, 16) and np.array_equal(colp1, np.zeros(40, dtype=int))


def test_python_argument_errors():
    import torch
    import impdar_b200
    from impdar_b200 import migrationlib as ml
    d = synthetic_dat(32, 24)
    x = torch.zeros((32, 24))
    for v in ([], [[1.7e8, 1.8e8]], [1.7e8, np.nan], [1.7e8, np.inf], [1.7e8, 0.0], [-1.7e8], ["fast"]):
        with pytest.raises(ValueError):
            impdar_b200.migrationVelocityScan(d, v)
        with pytest.raises(ValueError):
            ml.stolt_scan_device(x, 1e-8, 5.0, v, 10, 10, (8, 8))
    for w in ((0, 8), (8, 0), (8,), (8, 8, 8), 8, (8.0, 8), (True, 8), (-1, 4)):
        with pytest.raises(ValueError):
            impdar_b200.migrationVelocityScan(d, [1.7e8], window=w)
        with pytest.raises(ValueError):
            ml.stolt_scan_device(x, 1e-8, 5.0, [1.7e8], 10, 10, w)
    with pytest.raises(ValueError):
        ml.stolt_scan_device(x, 1e-8, 5.0, [1.7e8], 10, 10, (8, 8))     # a host tensor
    bad = synthetic_dat(32, 24)
    bad.data = bad.data[:, :20]
    with pytest.raises(ValueError):
        impdar_b200.migrationVelocityScan(bad, [1.7e8])


def test_c_entry_rejects_bad_input():
    from impdar_b200 import _lib
    lib = _lib.load()
    S, T = 64, 32
    fake = ctypes.c_void_p(8)
    ws = lib.impdar_stolt_scan_workspace_bytes(S, T, 3)
    assert ws == lib.impdar_stolt_scan_workspace_bytes(S, T, 1)
    assert ws >= 3 * S * T * 4 and lib.impdar_stolt_scan_workspace_bytes(1, T, 1) == 0
    good = np.array([1.5e8, 1.6e8, 1.7e8])

    def call(data=fake, snum=S, dt=1e-8, dx=5.0, vels=good, nvel=3, ws_s=8, ws_t=8, focus=fake, ws_bytes=ws):
        vp = vels.ctypes.data_as(ctypes.c_void_p) if vels is not None else None
        return lib.impdar_stolt_scan_f32(data, snum, T, dt, dx, vp, nvel, 10., 10., 0, ws_s, ws_t, focus, None, fake,
                                         ws_bytes, None)
    assert call(data=None) == 1
    assert call(focus=None) == 1
    assert call(snum=1) == 1
    assert call(dt=0.0) == 1 and call(dt=-1e-8) == 1 and call(dt=float('nan')) == 1
    assert call(dx=0.0) == 1
    assert call(nvel=0) == 1 and call(vels=None) == 1
    for badval in (0.0, -1.0, np.nan, np.inf):
        b = good.copy()
        b[2] = badval
        assert call(vels=b) == 1
    assert call(ws_s=0) == 1 and call(ws_t=0) == 1
    assert call(ws_bytes=ws - 1) == 1
    assert "workspace" in _lib.last_error()


def test_symbols_exported():
    import impdar_b200
    from impdar_b200 import _lib
    lib = ctypes.CDLL(_lib.LIB_PATH)
    for s in ("impdar_stolt_scan_f32", "impdar_stolt_scan_workspace_bytes"):
        assert hasattr(lib, s) and s in _lib.PROTOTYPES
    assert callable(impdar_b200.migrationVelocityScan) and callable(impdar_b200.scan_rms_field)


# ------------------------------------------------------------------------------------------------------ GPU
LANES = {  # name: (snum, tnum, pipeline, expected lane)
    "five_pass": (1024, 8192, 0, "five_pass"),
    "cufft_paired": (2048, 4096, 0, "cufft_paired"),
    "cufft_r2c": (65, 50, 1, "cufft_r2c"),
}


def _with_pipeline(mode, fn):
    from impdar_b200 import migrationlib as ml
    ml.set_stolt_pipeline(mode)
    try:
        return fn()
    finally:
        ml.set_stolt_pipeline(ml.STOLT_AUTO)


@pytest.mark.gpu
@pytest.mark.parametrize("lane", list(LANES))
@pytest.mark.parametrize("dtype", ["float32", "int16"])
def test_scan_images_equal_stolt_device(lane, dtype):
    import torch
    from impdar_b200 import migrationlib as ml
    S, T, mode, want = LANES[lane]
    vels = np.array([1.45e8, 1.69e8, 2.1e8])
    rng = np.random.default_rng(S + T)
    host = rng.standard_normal((S, T)).astype(np.float32)
    trunc = dtype == "int16"
    if trunc:
        host = (host * 3000).astype(np.int16)
    x = torch.from_numpy(host.astype(np.float32)).cuda()
    S2, w = 2 * (S // 2), (16, 24)
    for htaper, vtaper in ((100, 1000), (7, 3)):
        imgs = torch.empty((len(vels), S2, T), dtype=torch.float32, device="cuda")
        focus = _with_pipeline(mode, lambda: ml.stolt_scan_device(x, 1e-8, 5.0, vels, htaper, vtaper, w, trunc, imgs))
        assert ml.stolt_last_pipeline() == want
        for k, v in enumerate(vels):
            ref = _with_pipeline(mode, lambda: ml.stolt_device(x, 1e-8, 5.0, v, htaper, vtaper, trunc))
            assert ml.stolt_last_pipeline() == want
            assert torch.equal(imgs[k], ref), (lane, dtype, htaper, k)
        got = focus.cpu().numpy()
        want_f = np.array([focus_np(im, *w) for im in imgs.cpu().numpy()])
        assert got.shape == want_f.shape
        assert np.max(np.abs(got - want_f) / np.maximum(np.abs(want_f), 1e-300)) <= 1e-12


@pytest.mark.gpu
@pytest.mark.parametrize("lane", list(LANES))
def test_focus_panel_deterministic_and_lane_independent(lane):
    import torch
    import impdar_b200
    from impdar_b200 import migrationlib as ml
    S, T, mode, _ = LANES[lane]
    vels = np.array([1.5e8, 1.7e8])
    d = synthetic_dat(S, T, seed=3)
    keep = d.data.copy()
    x = torch.from_numpy(d.data).cuda()
    w = (64, 48)
    a = _with_pipeline(mode, lambda: ml.stolt_scan_device(x, d.dt, 5.0, vels, 100, 1000, w))
    b = _with_pipeline(mode, lambda: ml.stolt_scan_device(x, d.dt, 5.0, vels, 100, 1000, w))
    imgs = torch.empty((2, 2 * (S // 2), T), dtype=torch.float32, device="cuda")
    c = _with_pipeline(mode, lambda: ml.stolt_scan_device(x, d.dt, 5.0, vels, 100, 1000, w, images=imgs))
    assert torch.equal(a, b) and torch.equal(a, c)
    host = _with_pipeline(mode, lambda: impdar_b200.migrationVelocityScan(d, vels, window=w))
    assert np.array_equal(d.data, keep)          # dat is not modified
    dev = synthetic_dat(S, T, seed=3)
    dev.data = torch.from_numpy(dev.data).cuda()
    before = dev.data.clone()
    devscan = _with_pipeline(mode, lambda: impdar_b200.migrationVelocityScan(dev, vels, window=w))
    assert torch.equal(dev.data, before)
    assert np.array_equal(host.focus, a.cpu().numpy()) and np.array_equal(devscan.focus, host.focus)
    assert np.array_equal(host.vrms, devscan.vrms, equal_nan=True)
    assert host.snum == S and host.tnum == T and host.window == w


@pytest.mark.gpu
def test_gpu_recovery_config2():
    import impdar_b200
    S, T, ws, wt = 2048, 4096, 128, 128
    pts = apex_points(S // ws, T // wt, ws, wt, (1, 5, 9), (2, 10, 18, 26))
    for v0 in (1.5e8, 1.8e8):
        d = ricker_dat(S, T, pts, v0, seed=4)
        scan = impdar_b200.migrationVelocityScan(d, GRID, window=(ws, wt), htaper=4, vtaper=4)
        for s0, x0 in pts:
            assert scan.vrms[s0 // ws, x0 // wt] == v0, (v0, s0, x0, scan.focus[:, s0 // ws, x0 // wt])
    d, V = layered_dat(S, T, pts)
    scan = impdar_b200.migrationVelocityScan(d, LAYERED_GRID, window=(ws, wt), htaper=4, vtaper=4)
    step = LAYERED_GRID[1] - LAYERED_GRID[0]
    for s0, x0 in pts:
        assert abs(scan.vrms[s0 // ws, x0 // wt] - V[s0]) <= step, (s0, x0, V[s0], scan.vrms[s0 // ws, x0 // wt])


@pytest.mark.gpu
def test_scan_field_focuses_kirchhoff_better():
    """Layered synthetic: scan -> scan_rms_field -> kirchhoff_lateral_device concentrates more of each diffractor's
    energy near its apex than kirchhoff_device at 1.69e8 (the energy share of test_oracle_lateral_focuses_better)."""
    import torch
    import impdar_b200
    from impdar_b200 import migrationlib as ml
    S, T = 512, 256
    pts = [(96, 96), (224, 224), (352, 96)]
    d, V = layered_dat(S, T, pts)
    scan = impdar_b200.migrationVelocityScan(d, LAYERED_GRID, window=(64, 64), htaper=4, vtaper=4)
    prof, colp = impdar_b200.scan_rms_field(scan)
    x = torch.from_numpy(d.data).cuda()
    lat = ml.kirchhoff_lateral_device(x, d.travel_time, d.dist, prof, colp, False).cpu().numpy()
    one = ml.kirchhoff_device(x, d.travel_time, d.dist, 1.69e8, False).cpu().numpy()

    def share(out, s0, x0):
        e = out.astype(np.float64) ** 2
        return e[s0 - 8:s0 + 9, x0 - 2:x0 + 3].sum() / e[max(s0 - 40, 0):s0 + 41, max(x0 - 40, 0):x0 + 41].sum()
    res = [(share(lat, s0, x0), share(one, s0, x0)) for s0, x0 in pts]
    assert res[0][0] > 1.3 * res[0][1], res           # the shallow (fast) diffractor, far from 1.69e8
    assert all(a >= 0.98 * b for a, b in res), res
    assert sum(a for a, _ in res) > sum(b for _, b in res), res
