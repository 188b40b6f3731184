"""Interval velocities and depth sections: depth_curves, the bounded Dix inversion of a velocity scan
(scan_interval_field), (v, z) table export (interval_table) and the time-to-depth conversion kernel (depthConvert).

CPU part: depth curves against closed forms and a per-element loop (tests/depth_conversion_oracle.py); the batched
active-set Dix solve against scipy's bvls; recovery from exact and noisy picks; the field semantics shared with
scan_rms_field; interval_table through getVelocityProfile; argument errors of the Python and C entries.
GPU part: depth_convert_device against the float64 reference bit for bit (float64 and float32, one profile, a scan-like
field, one profile per trace, pre-trigger samples, NaN samples, exact node hits, rows outside a column); repeatability;
depthConvert's host and device lanes; a layered synthetic through scan, Dix, lateral Kirchhoff and depth conversion;
an interval_table through migrationPhaseShift.
"""
import ctypes

import numpy as np
import pytest

import depth_conversion_oracle as do
from util import synthetic_dat

C = 2.99792458e8


def firn(t):
    """Interval velocity of the Dix experiments: a firn gradient from 2.29e8 to 1.69e8 with a slow 1.55e8 layer."""
    v = 1.69e8 + 0.6e8 * np.exp(-t / 0.6e-6)
    return np.where((t > 2.5e-6) & (t < 3.2e-6), 1.55e8, v)


def make_scan(vrms, snum, tnum, window, travel_time, focus=None, vels=None):
    """A VelocityScan with the given (nws, nwt) picks (focus 1 everywhere unless given)."""
    from impdar_b200 import migrationlib as ml
    vrms = np.asarray(vrms, dtype=np.float64)
    ws = window[0]
    S2 = 2 * (snum // 2)
    starts = np.arange(vrms.shape[0]) * ws
    n_i = np.minimum(starts + ws, S2) - starts
    if focus is None:
        focus = np.ones((1,) + vrms.shape)
    return ml.VelocityScan(vels=np.array([1.4e8, 2.4e8]) if vels is None else vels, window=tuple(window), snum=snum,
                           tnum=tnum, center_rows=starts + (n_i - 1) / 2.0, focus=focus, vrms=vrms,
                           travel_time=np.asarray(travel_time, dtype=np.float64))


def dix_rms(tk, u):
    """Exact RMS picks of the Dix model: u = v_int^2 linear between picks, u_1 on [0, t_1]."""
    D = np.empty(len(tk))
    acc = tk[0] * u[0]
    D[0] = acc
    for k in range(1, len(tk)):
        acc += (tk[k] - tk[k - 1]) / 2 * (u[k - 1] + u[k])
        D[k] = acc
    return np.sqrt(D / tk)


# ------------------------------------------------------------------------------------------------------ CPU
def test_depth_curves_constant_profile():
    from impdar_b200 import migrationlib as ml
    for tt in (np.arange(300) * 0.01, (np.arange(300) - 17) * 0.01, np.arange(300) * 0.01 + 0.01):
        t = tt / 1e6
        for v in (2.0 ** 27, 2.0 ** 28):     # exact products and differences: the sum telescopes to v t / 2 exactly
            z = ml.depth_curves(tt, np.full((1, len(tt)), v))[0]
            assert np.array_equal(z, v * t / 2)
        z = ml.depth_curves(tt, np.full((2, len(tt)), 1.69e8))
        assert np.allclose(z, 1.69e8 * t / 2, rtol=1e-13, atol=1e-12)


def test_depth_curves_monotone_and_loop():
    from impdar_b200 import migrationlib as ml
    rng = np.random.default_rng(1)
    for tt in (np.arange(200) * 0.01, (np.arange(200) - 23) * 0.01 + 0.003, np.sort(rng.uniform(-0.5, 3.0, 200))):
        v = rng.uniform(0.8e8, 2.9e8, (5, 200))
        z = ml.depth_curves(tt, v)
        assert np.all(np.diff(z, axis=1) > 0)
        for p in range(5):
            assert np.array_equal(z[p], do.depth_curve_loop(tt, v[p]))
    neg = -np.arange(10)[::-1] * 0.01 - 0.01           # no sample at t >= 0: anchored at the last one
    vn = rng.uniform(1e8, 2e8, (1, 10))
    z = ml.depth_curves(neg, vn)
    assert np.all(np.diff(z) > 0) and np.array_equal(z[0], do.depth_curve_loop(neg, vn[0]))


def test_dix_exact_picks_recover_model():
    from impdar_b200 import migrationlib as ml
    dt, ws, nws = 1e-8, 64, 64
    S = ws * nws
    tt = np.arange(S) * dt * 1e6
    t = tt / 1e6
    tk = (np.arange(nws) * ws + (ws - 1) / 2.0) * dt
    u = firn(tk) ** 2
    V = dix_rms(tk, u)
    vrms = np.stack([V, V * 1.0], 1)
    scan = make_scan(vrms, S, 100, (ws, 64), tt)
    prof, colp = ml.scan_interval_field(scan, smooth=0.0)
    assert prof.shape == (1, S) and np.array_equal(colp, np.zeros(100, dtype=int))
    want = np.sqrt(np.interp(t, tk, u))
    assert np.max(np.abs(prof[0] / want - 1)) < 1e-9


def _dense_dix(tk, V, s):
    K = len(tk)
    A = np.zeros((K, K))
    A[:, 0] += tk[0]
    for k in range(1, K):
        A[k:, k - 1] += (tk[k] - tk[k - 1]) / 2
        A[k:, k] += (tk[k] - tk[k - 1]) / 2
    ub = np.mean(V ** 2)
    M = A * ub / (tk * V ** 2)[:, None]
    b = np.ones(K)
    if K > 1:
        M = np.vstack([M, s * np.diff(np.eye(K), axis=0)])
        b = np.concatenate([b, np.zeros(K - 1)])
    return M, b, ub


def test_batched_active_set_matches_bvls():
    from scipy.optimize import lsq_linear
    from impdar_b200 import migrationlib as ml
    rng = np.random.default_rng(2)
    active = 0
    for K in (1, 2, 7, 33):
        for s in (0.0, 0.3, 1.0):
            n = 6
            tk = np.sort(rng.uniform(5e-8, 6e-6, (n, K)), axis=1)
            V = rng.uniform(1.5e8, 2.3e8, (n, K))
            vmin, vmax = 1.6e8, 2.1e8                     # narrow: noisy picks push many unknowns onto a bound
            H, g, ub = ml._dix_normal(tk, V)
            for c in range(n):
                M, b, ub_c = _dense_dix(tk[c], V[c], s)
                Hs = H[c] + (s ** 2 * np.diff(np.eye(K), axis=0).T @ np.diff(np.eye(K), axis=0) if K > 1 else 0)
                assert np.allclose(Hs, M.T @ M, rtol=1e-12, atol=1e-12 * np.abs(Hs).max())
            us = ml._dix_columns(list(tk), list(V), vmin, vmax, s)
            for c in range(n):
                M, b, ub_c = _dense_dix(tk[c], V[c], s)
                ref = lsq_linear(M, b, bounds=(vmin ** 2 / ub_c, vmax ** 2 / ub_c), method='bvls', tol=1e-14).x
                got = us[c] / ub_c
                assert np.max(np.abs(got / ref - 1)) <= 1e-8, (K, s, c)
                active += int(np.sum((ref <= vmin ** 2 / ub_c * (1 + 1e-12)) | (ref >= vmax ** 2 / ub_c * (1 - 1e-12))))
    assert active > 20


def test_dix_noisy_picks_bounded():
    from impdar_b200 import migrationlib as ml
    rng = np.random.default_rng(3)
    dt, ws, nws, nwt, wt = 1e-8, 64, 64, 16, 8
    S = ws * nws
    tt = np.arange(S) * dt * 1e6
    tk = (np.arange(nws) * ws + (ws - 1) / 2.0) * dt
    V = dix_rms(tk, firn(tk) ** 2)
    vrms = V[:, None] * (1 + 0.01 * rng.standard_normal((nws, nwt)))
    vels = np.linspace(1.4e8, 2.6e8, 32)
    scan = make_scan(vrms, S, nwt * wt, (ws, wt), tt, vels=vels)
    prof, colp = ml.scan_interval_field(scan)
    vmin = 0.5 * vels.min()
    assert prof.shape == (nwt, S) and np.all(prof >= vmin * (1 - 1e-12)) and np.all(prof <= C * (1 + 1e-12))
    rows = (np.arange(nws) * ws + ws // 2)
    err = np.abs(prof[:, rows] / firn(tt[rows] / 1e6)[None, :] - 1)
    assert np.median(err) < 0.03, np.median(err)
    tight = ml.scan_interval_field(scan, vmin=1.6e8, vmax=2.0e8)[0]
    assert tight.min() >= 1.6e8 * (1 - 1e-12) and tight.max() <= 2.0e8 * (1 + 1e-12)


def test_field_semantics_match_scan_rms_field():
    from impdar_b200 import migrationlib as ml
    S, ws, wt, nwt = 64, 16, 7, 6
    tt = np.arange(S) * 0.01
    vrms = np.full((4, nwt), np.nan)
    vrms[:, 1] = 1.6e8                   # columns 1 and 5 equal, 3 differs; 0, 2, 4 empty
    vrms[:, 3] = [1.9e8, 1.8e8, 1.7e8, 1.7e8]
    vrms[:, 5] = 1.6e8
    focus = np.ones((1, 4, nwt))
    focus[0, 2, 3] = 0.5                 # masked by min_focus = 1
    scan = make_scan(vrms, S, 40, (ws, wt), tt, focus=focus)
    for mf in (0.0, 1.0):
        rp, rc = ml.scan_rms_field(scan, min_focus=mf)
        ip, ic = ml.scan_interval_field(scan, min_focus=mf)
        assert ip.shape == rp.shape == (2, S) and np.array_equal(ic, rc)
        assert np.array_equal(ic, np.array([0, 0, 0, 1, 1, 0])[np.arange(40) // wt])
        assert np.allclose(ip[0], 1.6e8, rtol=1e-12)
    masked = ml.scan_interval_field(scan, min_focus=1.0)[0][1]
    full = ml.scan_interval_field(scan, min_focus=0.0)[0][1]
    assert not np.array_equal(masked, full)
    early = make_scan(vrms, S, 40, (ws, wt), tt - 0.2, focus=focus)   # the first window centre lies before time zero
    assert ml.scan_interval_field(early)[0].shape == (2, S)
    with pytest.raises(ValueError):
        ml.scan_interval_field(make_scan(np.full((4, nwt), np.nan), S, 40, (ws, wt), tt))


def test_interval_table_round_trip():
    from impdar_b200 import migrationlib as ml
    S = 4096
    d = synthetic_dat(S, 4)
    t = d.travel_time / 1e6
    tk = (np.arange(64) * 64 + 31.5) * 1e-8
    v = np.sqrt(np.interp(t, tk, firn(tk) ** 2))            # a Dix-produced profile: continuous, decreasing (firn)
    tab = ml.interval_table(d.travel_time, v)
    assert tab.shape[1] == 2 and np.all(np.diff(tab[:, 1]) > 0)
    err = np.abs(ml.getVelocityProfile(d, tab) / v - 1)
    # getVelocityProfile resamples z(t) linearly on its own depth grid and differentiates with np.gradient: exact where
    # z(t) is linear, a little off where the shallow gradient curves it and where the slope changes at the picks
    assert np.median(err) < 1e-9 and np.max(err) < 1e-3
    steps = np.select([t < 1e-6, t < 2.5e-6, t < 3.2e-6], [2.2e8, 1.9e8, 1.55e8], 1.69e8)    # layers: z(t) piecewise linear
    err = np.abs(ml.getVelocityProfile(d, ml.interval_table(d.travel_time, steps)) / steps - 1)
    edge = np.zeros(S, bool)
    for k in np.nonzero(np.diff(steps))[0]:
        edge[k - 1:k + 3] = True
    assert np.max(err[~edge]) < 1e-9
    inc = np.linspace(1.7e8, 2.2e8, S)                       # increasing with depth
    assert np.max(np.abs(ml.getVelocityProfile(d, ml.interval_table(d.travel_time, inc)) / inc - 1)) < 1e-4
    pre = synthetic_dat(300, 4, tt0_us=-0.2)
    vp = np.where(np.arange(300) < 150, 2.2e8, 1.7e8)        # firn over ice, 20 samples before time zero
    got = ml.getVelocityProfile(pre, ml.interval_table(pre.travel_time, vp))
    ok = np.r_[np.arange(22, 148), np.arange(152, 300)]
    assert np.max(np.abs(got[ok] / vp[ok] - 1)) < 1e-9


def test_interval_table_file_runs_through_vel_fn(tmp_path):
    from impdar_b200 import migrationlib as ml
    d = synthetic_dat(500, 4)
    v = np.linspace(2.3e8, 1.69e8, 500)
    fn = str(tmp_path / "vint.txt")
    np.savetxt(fn, ml.interval_table(d.travel_time, v))
    back = ml.getVelocityProfile(d, np.genfromtxt(fn))
    assert np.array_equal(back, ml.getVelocityProfile(d, ml.interval_table(d.travel_time, v)))
    assert np.max(np.abs(back / v - 1)) < 1e-3   # a steep gradient over 500 samples: getVelocityProfile's own resampling


def test_python_argument_errors():
    import torch
    import impdar_b200
    from impdar_b200 import migrationlib as ml
    tt = np.arange(32) * 0.01
    with pytest.raises(ValueError):
        ml.depth_curves(tt, np.ones((2, 31)))
    with pytest.raises(ValueError):
        ml.interval_table(tt, np.ones(31))
    with pytest.raises(ValueError):
        ml.interval_table(tt, -np.ones(32))
    with pytest.raises(ValueError):
        ml.interval_table(tt[::-1], np.ones(32))
    scan = make_scan(np.full((2, 2), 1.7e8), 32, 8, (16, 4), tt)
    for kw in ({'vmin': 2e8, 'vmax': 1e8}, {'vmin': 0.0}, {'vmax': np.inf}, {'smooth': -1.0}, {'smooth': np.nan}):
        with pytest.raises(ValueError):
            ml.scan_interval_field(scan, **kw)
    scan.travel_time = None
    with pytest.raises(ValueError):
        ml.scan_interval_field(scan)
    d = synthetic_dat(32, 8)
    field = (np.full((1, 32), 1.7e8), np.zeros(8, dtype=int))
    with pytest.raises(ValueError):
        impdar_b200.depthConvert(d, vel=1.8e8, field=field)
    with pytest.raises(ValueError):
        impdar_b200.depthConvert(d, field=(np.full((1, 31), 1.7e8), np.zeros(8, dtype=int)))
    with pytest.raises(ValueError):
        impdar_b200.depthConvert(d, field=(np.full((1, 32), 1.7e8), np.ones(8, dtype=int)))
    with pytest.raises(ValueError):
        impdar_b200.depthConvert(d, field=(np.full((1, 32), -1.7e8), np.zeros(8, dtype=int)))
    with pytest.raises(ValueError):
        impdar_b200.depthConvert(d, vel=[[1.7e8, 0.0]])
    with pytest.raises(ValueError):
        impdar_b200.depthConvert(d, dz=0.0)
    with pytest.raises(TypeError):
        impdar_b200.depthConvert(d, vel_fn="/nonexistent/velocity.txt")
    x = torch.zeros((32, 8))
    with pytest.raises(ValueError):          # a host tensor
        ml.depth_convert_device(x, tt, *field, np.arange(4.0))


def test_c_entry_rejects_bad_input():
    from impdar_b200 import _lib
    lib = _lib.load()
    S, T, nz, P = 16, 6, 5, 2
    fake = ctypes.c_void_p(8)
    ws = lib.impdar_depth_workspace_bytes(S, T, nz, P)
    assert ws >= 2 * P * S * 8 + S * 8 + nz * 8 + T * 4
    assert lib.impdar_depth_workspace_bytes(1, T, nz, P) == 0 and lib.impdar_depth_workspace_bytes(S, T, 0, P) == 0
    good_tt = np.arange(S) * 0.01
    good_prof = np.full((P, S), 1.7e8)
    good_colp = np.array([0, 0, 1, 1, 0, 1], dtype=np.int32)
    good_zg = np.arange(nz) * 0.5

    def call(x=fake, snum=S, nzz=nz, tt=good_tt, prof=good_prof, nprof=P, colp=good_colp, zg=good_zg, wsb=ws,
             entry="impdar_depth_convert_f32"):
        def p(a):
            return None if a is None else a.ctypes.data_as(ctypes.c_void_p)
        return getattr(lib, entry)(x, fake, snum, T, nzz, p(tt), p(prof), nprof, p(colp), p(zg), fake, wsb, None)
    for entry in ("impdar_depth_convert_f32", "impdar_depth_convert_f32_f64", "impdar_depth_convert_f64"):
        assert call(x=None, entry=entry) == 1 and "null" in _lib.last_error()
        assert call(snum=1, entry=entry) == 1
    assert call(nzz=0) == 1
    assert call(tt=None) == 1 and call(prof=None) == 1 and call(colp=None) == 1 and call(zg=None) == 1
    for bad in (0.0, -1.0, np.nan, np.inf):
        b = good_prof.copy()
        b[1, 7] = bad
        assert call(prof=b) == 1 and "velocity" in _lib.last_error()
    bt = good_tt.copy()
    bt[5] = bt[4]
    assert call(tt=bt) == 1 and "ascending" in _lib.last_error()
    bt[5] = np.nan
    assert call(tt=bt) == 1
    for bad in (-1, 2):
        c = good_colp.copy()
        c[3] = bad
        assert call(colp=c) == 1 and "col_profile" in _lib.last_error()
    bz = good_zg.copy()
    bz[2] = bz[1]
    assert call(zg=bz) == 1 and "zgrid" in _lib.last_error()
    bz[2] = np.inf
    assert call(zg=bz) == 1
    assert call(wsb=ws - 1) == 1 and "workspace" in _lib.last_error()


def test_symbols_exported():
    import impdar_b200
    from impdar_b200 import _lib
    lib = ctypes.CDLL(_lib.LIB_PATH)
    for s in ("impdar_depth_workspace_bytes", "impdar_depth_convert_f32", "impdar_depth_convert_f32_f64",
              "impdar_depth_convert_f64"):
        assert hasattr(lib, s) and s in _lib.PROTOTYPES
    for name in ("depthConvert", "scan_interval_field", "depth_curves", "interval_table"):
        assert callable(getattr(impdar_b200, name))
    assert "depthConvert" not in impdar_b200._MIGRATION_NAMES + impdar_b200._FILTER_NAMES + impdar_b200._PROCESSING_NAMES


# ------------------------------------------------------------------------------------------------------ GPU
def _case(S, T, P, seed, tt0=0.0, runs=None):
    """Image with NaN samples, pre-trigger times, interval profiles and a trace map; a depth grid that includes node
    depths of profile 0 exactly and rows above and below every column."""
    from impdar_b200 import migrationlib as ml
    rng = np.random.default_rng(seed)
    tt = tt0 + np.arange(S) * 0.01
    img = rng.standard_normal((S, T))
    img[rng.integers(0, S, 40), rng.integers(0, T, 40)] = np.nan
    base = np.linspace(2.3e8, 1.69e8, S)
    prof = base[None, :] * (1 + 0.05 * rng.uniform(-1, 1, (P, 1))) * (1 + 0.01 * rng.standard_normal((P, S)))
    if runs:
        colp = np.minimum(np.arange(T) // runs, P - 1)
    else:
        colp = rng.permutation(T) % P
    z = ml.depth_curves(tt, prof)
    dz = prof.min() * 1e-8 / 2
    zg = np.arange(z[:, 0].min() - 3 * dz, z[:, -1].max() + 3 * dz, dz)
    zg = np.unique(np.concatenate([zg, z[0, ::7]]))
    return img, tt, prof, colp, zg, z


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["one", "scan", "per_trace"])
@pytest.mark.parametrize("tt0", [0.0, -0.13])
def test_device_equals_reference_bit_for_bit(kind, tt0):
    import torch
    from impdar_b200 import migrationlib as ml
    S, T = 300, 257
    P, runs = {"one": (1, None), "scan": (5, 64), "per_trace": (T, None)}[kind]
    img, tt, prof, colp, zg, z = _case(S, T, P, seed=S + P, tt0=tt0, runs=runs)
    ref = do.depth_convert(img, tt, prof, colp, zg, curves=z)
    assert np.isnan(ref[0]).all() and np.isnan(ref[-1]).all() and np.isfinite(ref).mean() > 0.8
    x64 = torch.from_numpy(img).cuda()
    got = ml.depth_convert_device(x64, tt, prof, colp, zg).cpu().numpy()
    assert got.dtype == np.float64 and np.array_equal(got, ref, equal_nan=True)
    x32 = torch.from_numpy(img.astype(np.float32)).cuda()
    ref32 = do.depth_convert(img.astype(np.float32), tt, prof, colp, zg, curves=z)
    got32 = ml.depth_convert_device(x32, tt, prof, colp, zg).cpu().numpy()
    assert got32.dtype == np.float32 and np.array_equal(got32, ref32.astype(np.float32), equal_nan=True)
    out = torch.empty((len(zg), T), dtype=torch.float64, device="cuda")
    ml.depth_convert_device(x32, tt, prof, colp, zg, out=out)
    assert np.array_equal(out.cpu().numpy(), ref32, equal_nan=True)


@pytest.mark.gpu
def test_device_repeatable_and_dtype_checks():
    import torch
    from impdar_b200 import migrationlib as ml
    img, tt, prof, colp, zg, _ = _case(512, 1000, 16, seed=7, runs=64)
    x = torch.from_numpy(img.astype(np.float32)).cuda()
    a = ml.depth_convert_device(x, tt, prof, colp, zg)
    b = ml.depth_convert_device(x, tt, prof, colp, zg)
    assert torch.equal(torch.nan_to_num(a, nan=7.0), torch.nan_to_num(b, nan=7.0))
    with pytest.raises(ValueError):
        ml.depth_convert_device(x.double(), tt, prof, colp, zg, out=torch.empty_like(a))
    with pytest.raises(ValueError):
        ml.depth_convert_device(x, tt, prof, colp, zg, out=torch.empty((3, 1000), device="cuda"))
    with pytest.raises(ValueError):
        ml.depth_convert_device(x.half(), tt, prof, colp, zg)
    with pytest.raises(ValueError):
        ml.depth_convert_device(x, tt, prof, colp, zg[::-1])


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", ["float32", "float64", "int16"])
def test_depthConvert_lanes(dtype):
    import torch
    import impdar_b200
    from impdar_b200 import migrationlib as ml
    S, T, v = 200, 40, 1.69e8
    d = synthetic_dat(S, T, seed=5, tt0_us=0.05)
    if dtype == "int16":
        d.data = (d.data * 1000).astype(np.int16)
    else:
        d.data = d.data.astype(dtype)
    tt = d.travel_time.copy()
    host = synthetic_dat(S, T)
    host.data, host.travel_time = d.data.copy(), tt.copy()
    dev = synthetic_dat(S, T)
    dev.data, dev.travel_time = torch.from_numpy(d.data.copy()).cuda(), tt.copy()
    impdar_b200.depthConvert(host, vel=v)
    impdar_b200.depthConvert(dev, vel=v)
    z = v * (tt / 1e6) / 2                        # constant velocity: resampling at z = v t / 2
    zg = z[0] + v * 1e-8 / 2 * np.arange(host.snum)
    assert np.array_equal(host.nmo_depth, zg) and host.snum == len(zg) == host.data.shape[0]
    zc = ml.depth_curves(tt, np.full((1, S), v))[0]
    assert zg[-1] <= zc[-1] < zg[-1] + v * 1e-8 / 2
    want = do.depth_convert(d.data, tt, np.full((1, S), v), np.zeros(T, dtype=int), zg,
                            curves=ml.depth_curves(tt, np.full((1, S), v)))
    assert np.max(np.abs(ml.depth_curves(tt, np.full((1, S), v))[0] - z)) < 1e-9
    assert host.data.dtype == np.float64 and np.array_equal(host.data, want, equal_nan=True)
    want_dt = {"float32": torch.float32, "float64": torch.float64, "int16": torch.float64}[dtype]
    assert dev.data.dtype == want_dt and dev.snum == host.snum and np.array_equal(dev.nmo_depth, zg)
    ref_dev = want.astype(np.float32) if dtype == "float32" else want
    assert np.array_equal(dev.data.cpu().numpy(), ref_dev, equal_nan=True)
    assert np.allclose(host.travel_time, 2 * zg / v * 1e6, rtol=1e-12, atol=1e-9)
    assert np.array_equal(host.travel_time, dev.travel_time)


@pytest.mark.gpu
def test_depthConvert_tables_and_most_used_profile(tmp_path):
    import impdar_b200
    from impdar_b200 import migrationlib as ml, synthetic
    S, T = 300, 30
    d = synthetic_dat(S, T, seed=2)
    tab = synthetic.layered_velocity(d.travel_time)
    a = synthetic_dat(S, T, seed=2)
    impdar_b200.depthConvert(a, vel=tab)
    fn = str(tmp_path / "v.txt")
    np.savetxt(fn, tab)
    b = synthetic_dat(S, T, seed=2)
    impdar_b200.depthConvert(b, vel_fn=fn)
    vint = ml.getVelocityProfile(d, tab)
    c = synthetic_dat(S, T, seed=2)
    impdar_b200.depthConvert(c, field=(vint[None, :], np.zeros(T, dtype=int)))
    for o in (b, c):
        assert np.array_equal(a.data, o.data, equal_nan=True) and np.array_equal(a.nmo_depth, o.nmo_depth)
    # lateral: two profiles, the second on more traces; travel_time follows it, extended past its last sample
    slow = np.full(S, 1.6e8)
    fast = np.full(S, 2.0e8)
    colp = (np.arange(T) >= 10).astype(int)
    e = synthetic_dat(S, T, seed=2)
    impdar_b200.depthConvert(e, field=(np.stack([slow, fast]), colp))
    zend = ml.depth_curves(d.travel_time, fast[None, :])[0, -1]
    assert e.nmo_depth[0] == 0.0 and e.nmo_depth[-1] <= zend < e.nmo_depth[-1] + 1.6e8 * 1e-8 / 2
    assert np.allclose(e.travel_time, 2 * e.nmo_depth / 2.0e8 * 1e6, rtol=1e-12, atol=1e-9)
    assert np.isnan(e.data[-1, 0]) and np.isfinite(e.data[-1, -1])


@pytest.mark.gpu
def test_end_to_end_layered_diffractor_depths():
    """Layered synthetic -> velocity scan -> Dix field -> lateral Kirchhoff with its RMS field -> depth section.  Each
    diffractor focuses within two samples of its apex time, its peak in the depth section lies within two depth rows
    of the depth the field gives that peak time, and that depth is within 8 % of the true one (the scan's 0.1e8 grid
    and the hyperbola tails in neighbouring windows limit the picks on this small synthetic)."""
    import torch
    import impdar_b200
    from impdar_b200 import migrationlib as ml, synthetic
    from test_velocity_scan import layered_dat, LAYERED_GRID
    S, T = 512, 256
    pts = [(96, 96), (224, 224), (352, 96)]
    d, V = layered_dat(S, T, pts)
    vint = ml.getVelocityProfile(d, synthetic.layered_velocity(d.travel_time))
    ztrue = ml.depth_curves(d.travel_time, vint[None, :])[0]
    scan = impdar_b200.migrationVelocityScan(d, LAYERED_GRID, window=(64, 64), htaper=4, vtaper=4)
    prof, colp = impdar_b200.scan_interval_field(scan, min_focus=50.0)
    assert prof.shape[1] == S and len(colp) == T
    x = torch.from_numpy(d.data).cuda()
    mig = ml.kirchhoff_lateral_device(x, d.travel_time, d.dist, ml.rms_velocity_profiles(d.travel_time, prof), colp,
                                      False).cpu().numpy()
    zfield = ml.depth_curves(d.travel_time, prof)
    d.data = mig
    impdar_b200.depthConvert(d, field=(prof, colp))
    zg = d.nmo_depth
    dz = zg[1] - zg[0]
    for s0, x0 in pts:
        tpk = s0 - 8 + int(np.argmax(np.abs(mig[s0 - 8:s0 + 9, x0])))
        assert abs(tpk - s0) <= 2, (s0, tpk)
        zf = zfield[colp[x0]][tpk]
        k0 = int(np.searchsorted(zg, zf))
        win = slice(max(k0 - 30, 0), k0 + 30)
        k = win.start + int(np.argmax(np.abs(np.nan_to_num(d.data[win, x0]))))
        assert abs(zg[k] - zf) <= 2 * dz, (s0, zg[k], zf, dz)
        assert abs(zfield[colp[x0]][s0] / ztrue[s0] - 1) < 0.08, (s0, zfield[colp[x0]][s0], ztrue[s0])


@pytest.mark.gpu
def test_interval_table_of_scan_column_through_phase_shift():
    import impdar_b200
    from impdar_b200 import migrationlib as ml
    from test_velocity_scan import layered_dat
    S, T = 512, 128
    d, _ = layered_dat(S, T, [(160, 64)])
    scan = impdar_b200.migrationVelocityScan(d, np.arange(1.6e8, 2.4e8 + 1.0, 0.05e8), window=(64, 64), htaper=4,
                                             vtaper=4)
    prof, _ = impdar_b200.scan_interval_field(scan)
    tab = ml.interval_table(d.travel_time, prof[0])
    back = ml.getVelocityProfile(d, tab)
    assert np.median(np.abs(back / prof[0] - 1)) < 1e-3 and np.max(np.abs(back[1:] / prof[0][1:] - 1)) < 1e-2
    impdar_b200.migrationPhaseShift(d, vel=tab, htaper=4, vtaper=4)
    assert d.data.shape == (S, T) and np.all(np.isfinite(d.data))
