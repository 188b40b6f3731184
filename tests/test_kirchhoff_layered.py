"""Kirchhoff migration with a depth-varying (per-sample RMS) velocity.

CPU part: rms_velocity, the per-row float64 reference (tests/kirchhoff_layered_oracle.py) against the scalar oracle,
row locality, focusing of a layered profile against a constant one, the tile schedule with per-row velocities (which
kernel each GPU case must run), the host-side window / range helpers and the argument errors.
GPU part: a constant vector reproduces the scalar call bit for bit on every kernel and entry; layered profiles match
the float64 reference on the table (tile / gather) and general kernels, far and near field; bottom-up row chunks,
column windows and the host pipeline each equal one call bit for bit.
"""
import numpy as np
import pytest

from conftest import rel_l2
from util import synthetic_dat
import kirchhoff_layered_oracle as lo
from test_geometry_regimes import KirchTable, KT_SPAN, _pick

TOL = 1e-5


def layered_rms(d):
    """RMS velocity of synthetic.layered_velocity (the C3 firn profile: 2.3e8 at the top, 1.69e8 at depth)."""
    from impdar_b200 import synthetic, migrationlib as ml
    vmig = ml.getVelocityProfile(d, synthetic.layered_velocity(d.travel_time))
    return ml.rms_velocity(d.travel_time, vmig)


class KirchTableVZ(KirchTable):
    """KirchTable (kirch_table_build_kernel restated) with one velocity per output row: zs and t use v[ti], the table
    width uses max v, the ambiguity margin eps_t uses min v."""

    def __init__(self, travel_time_us, dist_km, v):
        tt = np.asarray(travel_time_us, dtype=np.float64) / 1.0e6
        dist = np.asarray(dist_km, dtype=np.float64) * 1.0e3
        S, T = len(tt), len(dist)
        self.S, self.T = S, T
        v = np.asarray(v, dtype=np.float64)
        tmax, tt0 = tt.max(), tt[0]
        dxm = (dist[T - 1] - dist[0]) / (T - 1)
        maxdev_d = float(np.max(np.abs(dist - (dist[0] + np.arange(T) * dxm))))
        eps_t = (2.0 / v.min()) * (2.0 * maxdev_d) + 1e-15 * (abs(tmax) + abs(tt0))
        amax = int(min(float(T - 1), np.floor(v.max() * tmax / 2.0 / dxm) + 2.0))
        A1 = max(amax, 0) + 1
        zs = v * tt / 2.0
        zs2 = zs * zs
        d = np.arange(A1) * dxm
        self.A1 = A1
        self.k = np.empty((S, A1), dtype=np.int32)
        for r0 in range(0, S, 256):
            r1 = min(S, r0 + 256)
            rs = np.sqrt(d[None, :] * d[None, :] + zs2[r0:r1, None])
            t = 2.0 * rs / v[r0:r1, None]
            in_lo = ~((t - eps_t) > tmax)
            in_hi = ~((t + eps_t) > tmax)
            k = _pick(tt, t)
            amb = in_lo & (~in_hi | (_pick(tt, t - eps_t) != _pick(tt, t + eps_t)))
            apex = (rs == 0.0) & (zs[r0:r1, None] == 0.0)
            k = np.where(amb, -2, k)
            k = np.where(~in_lo | apex, -1, k)
            self.k[r0:r1] = k


def predicted_kernel(d, v):
    """Far-field, finite input, uniform spacing: 'table_tile' unless an aligned 28-row block has an offset interval
    wider than the tile kernel's staged span (then the gather kernel does the work)."""
    return 'table_tile' if KirchTableVZ(d.travel_time, d.dist, v).widest(aligned=True) <= KT_SPAN else 'table_gather'


# ------------------------------------------------------------------------------------------------------ CPU
def test_rms_velocity_constant():
    from impdar_b200 import migrationlib as ml
    tt = np.arange(500) * 0.01
    v = ml.rms_velocity(tt, np.full(500, 1.69e8))
    # The sum is sequential by definition, so its rounding grows with the sample count: <= n * 2^-53 relative on I after
    # n additions, half that on v = sqrt(I / t).  A short profile meets 1e-15; 500 samples are bounded by 500 * 2^-54.
    assert np.max(np.abs(ml.rms_velocity(tt[:8], np.full(8, 1.69e8)) / 1.69e8 - 1.0)) <= 1e-15
    assert np.max(np.abs(v / 1.69e8 - 1.0)) <= 500 * 2.0 ** -54
    assert np.array_equal(v, lo.rms_velocity(tt, np.full(500, 1.69e8)))


def test_rms_velocity_two_layers():
    """Step from v1 to v2 between samples k-1 and k: closed form sqrt((v1^2 t1 + v2^2 (t - t1)) / t) with the step at
    t1 = (t[k-1] + t[k]) / 2; the trapezoid over the step interval is exact for that t1."""
    from impdar_b200 import migrationlib as ml
    S, k, v1, v2 = 400, 150, 2.3e8, 1.69e8
    tt = np.arange(S) * 0.01
    t = tt / 1e6
    vmig = np.where(np.arange(S) < k, v1, v2)
    got = ml.rms_velocity(tt, vmig)
    t1 = (t[k - 1] + t[k]) / 2.
    want = np.where(t < t1, v1, np.sqrt((v1 ** 2 * t1 + v2 ** 2 * (t - t1)) / np.where(t > 0, t, 1.0)))
    want[0] = v1
    assert np.max(np.abs(got / want - 1.0)) < 1e-12
    assert np.array_equal(got, lo.rms_velocity(tt, vmig))
    assert got[0] == v1 and np.all(np.diff(got[k:]) < 0)


def test_rms_velocity_pretrigger():
    from impdar_b200 import migrationlib as ml
    tt = (np.arange(300) - 20) * 0.01          # 20 pre-trigger samples, sample 20 at t == 0
    rng = np.random.default_rng(3)
    vmig = 1.6e8 + 0.7e8 * rng.random(300)
    got = ml.rms_velocity(tt, vmig)
    assert np.array_equal(got[:21], vmig[:21])
    t = tt / 1e6
    assert got[21] == np.sqrt((vmig[20] ** 2 * t[20] + (vmig[21] ** 2 + vmig[20] ** 2) / 2 * (t[21] - t[20])) / t[21])
    assert np.array_equal(got, lo.rms_velocity(tt, vmig))


@pytest.mark.parametrize("S,T", [(48, 48), (40, 56)])
@pytest.mark.parametrize("nearfield", [False, True])
def test_oracle_constant_vector_is_scalar(S, T, nearfield):
    from oracle import migration as om
    d = synthetic_dat(S, T, seed=S + T)
    want = om.kirchhoff(d.data, d.travel_time, d.dist, 1.69e8, nearfield)
    got = lo.kirchhoff(d.data, d.travel_time, d.dist, np.full(S, 1.69e8), nearfield)
    assert np.array_equal(got, want)
    tr = (0, T // 3, T - 1)
    assert np.array_equal(lo.kirchhoff_sparse(d.data, d.travel_time, d.dist, np.full(S, 1.69e8), nearfield, tr),
                          om.kirchhoff_sparse(d.data, d.travel_time, d.dist, 1.69e8, nearfield, tr))
    assert lo.kirchhoff_pair_count(d.travel_time, d.dist, np.full(S, 1.69e8)) == \
        om.kirchhoff_pair_count(d.travel_time, d.dist, 1.69e8)


def test_oracle_row_locality():
    S, T = 64, 64     # S == T: a mis-broadcast velocity would pair v with the trace axis
    d = synthetic_dat(S, T, seed=5)
    v = layered_rms(d)
    full = lo.kirchhoff(d.data, d.travel_time, d.dist, v, True)
    for ti in (0, 1, 17, 40, 63):
        row = lo.kirchhoff(d.data, d.travel_time, d.dist, np.full(S, v[ti]), True)[ti]
        assert np.array_equal(full[ti], row)


def _diffractor_image(d, v, points, f0=50e6):
    """Ricker wavelets along t = sqrt(t0^2 + (2 x / v(t0))^2) (straight rays at the RMS velocity of the apex)."""
    t = np.asarray(d.travel_time, dtype=np.float64) / 1e6
    x = np.asarray(d.dist, dtype=np.float64) * 1e3
    img = np.zeros((len(t), len(x)))
    for s0, x0 in points:
        th = np.sqrt(t[s0] ** 2 + (2.0 * (x - x[x0]) / v[s0]) ** 2)
        a = (np.pi * f0 * (t[:, None] - th[None, :])) ** 2
        img += (1 - 2 * a) * np.exp(-a)
    return img.astype(np.float32)


def test_oracle_layered_focuses_better():
    """A shallow and a deep diffractor through the firn profile: the layered migration concentrates more of the output
    energy next to each apex than constant 1.69e8 does, clearly so for the shallow one."""
    S, T = 400, 160
    d = synthetic_dat(S, T, seed=0)
    v = layered_rms(d)
    pts = [(60, 50), (330, 110)]
    img = _diffractor_image(d, v, pts)

    def share(out, s0, x0):
        e = out ** 2
        return e[s0 - 8:s0 + 9, x0 - 2:x0 + 3].sum() / e[max(s0 - 40, 0):s0 + 41, max(x0 - 40, 0):x0 + 41].sum()
    tr = sorted(set(range(pts[0][1] - 40, pts[0][1] + 41)) | set(range(pts[1][1] - 40, min(pts[1][1] + 41, T))))
    lay = np.zeros((S, T))
    con = np.zeros((S, T))
    lay[:, tr] = lo.kirchhoff_sparse(img, d.travel_time, d.dist, v, False, tr)
    con[:, tr] = lo.kirchhoff_sparse(img, d.travel_time, d.dist, 1.69e8, False, tr)
    (s_lay, s_con), (d_lay, d_con) = [(share(lay, s0, x0), share(con, s0, x0)) for s0, x0 in pts]
    assert s_lay > 1.5 * s_con, (s_lay, s_con)
    assert d_lay > d_con, (d_lay, d_con)


def test_table_schedule_vz_constant_matches_scalar():
    from test_geometry_regimes import GEOMETRIES
    g = GEOMETRIES["G0"]
    S, T = 256, 512
    d = synthetic_dat(S, T, dt=g.dt, dx=g.dx)
    a = KirchTable(S, T, g)
    b = KirchTableVZ(d.travel_time, d.dist, np.full(S, g.vel))
    assert np.array_equal(a.k, b.k)


@pytest.mark.parametrize("S,T,dx,want", [(2048, 4096, 5.0, 'table_tile'), (512, 1024, 1.0, 'table_gather')])
def test_table_schedule_vz_predictions(S, T, dx, want):
    """The layered cases the GPU part runs: the config-2 shape keeps the tile kernel (the issue's 56-trace interval),
    the dense 1 m geometry makes it stand down."""
    d = synthetic_dat(S, T, dx=dx)
    assert predicted_kernel(d, layered_rms(d)) == want


def test_windows_and_ranges_vector():
    from impdar_b200 import migrationlib as ml, parallel
    S, T = 256, 1024
    d = synthetic_dat(S, T)
    v = layered_rms(d)
    for xb, xe in ((0, 100), (300, 600), (900, 1024)):
        assert ml.kirchhoff_input_window(S, d.travel_time, d.dist, np.full(S, 1.69e8), xb, xe) == \
            ml.kirchhoff_input_window(S, d.travel_time, d.dist, 1.69e8, xb, xe)
        c0, c1 = ml.kirchhoff_input_window(S, d.travel_time, d.dist, v, xb, xe)
        # every input trace the reference can read: 2 r / v[ti] <= max(tt) for some row
        x = d.dist * 1e3
        tmax = d.travel_time.max() / 1e6
        reach = np.max(v * tmax / 2.0)
        need0 = int(np.searchsorted(x, x[xb] - reach, side='left'))
        need1 = int(np.searchsorted(x, x[xe - 1] + reach, side='right'))
        assert c0 <= need0 and c1 >= need1
    for world in (2, 3):
        assert parallel.kirchhoff_output_ranges(T, world, d.travel_time, d.dist, np.full(S, 1.69e8)) == \
            parallel.kirchhoff_output_ranges(T, world, d.travel_time, d.dist, 1.69e8)
        irr = np.cumsum(np.r_[0, 5 + np.random.default_rng(world).random(T - 1)]) / 1e3
        assert parallel.kirchhoff_output_ranges(T, world, d.travel_time, irr, np.full(S, 1.69e8)) == \
            parallel.kirchhoff_output_ranges(T, world, d.travel_time, irr, 1.69e8)
        assert np.array_equal(parallel.kirchhoff_trace_cost(d.travel_time, irr, np.full(S, 1.69e8)),
                              parallel.kirchhoff_trace_cost(d.travel_time, irr, 1.69e8))
    assert parallel._spacing_is_uniform(d.travel_time, d.dist, v)


def test_argument_errors(tmp_path):
    from impdar_b200 import migrationlib as ml
    S, T = 64, 32
    d = synthetic_dat(S, T)
    with pytest.raises(ValueError):
        ml.migrationKirchhoffLayered(d, vel=np.array([[1.7e8, 0., 0.], [1.7e8, 1e3, 10.]]))
    for bad in (np.full(S - 1, 1.7e8), np.r_[np.full(S - 1, 1.7e8), 0.0], np.r_[np.full(S - 1, 1.7e8), np.nan],
                np.r_[np.full(S - 1, 1.7e8), -1.0], np.r_[np.full(S - 1, 1.7e8), np.inf]):
        with pytest.raises(ValueError):
            ml.kirchhoff_input_window(S, d.travel_time, d.dist, bad, 0, T)
    with pytest.raises(TypeError):
        ml.migrationKirchhoffLayered(d, vel_fn=str(tmp_path / "missing_velocity.txt"))


def test_c_entries_reject_bad_vectors():
    import ctypes
    from impdar_b200 import _lib
    lib = _lib.load()
    S, T = 16, 8
    tt = np.arange(S) * 1e-8
    dist = np.arange(T) * 5.0
    c0, c1 = ctypes.c_int(0), ctypes.c_int(0)
    ptr = lambda a: a.ctypes.data_as(ctypes.c_void_p)   # noqa: E731
    good = np.full(S, 1.7e8)
    assert lib.impdar_kirchhoff_input_window_vz(S, T, ptr(dist), ptr(tt), ptr(good), 0, T, ctypes.byref(c0),
                                                ctypes.byref(c1)) == 0
    for badval in (0.0, -1.0, np.nan, np.inf):
        bad = good.copy()
        bad[5] = badval
        assert lib.impdar_kirchhoff_input_window_vz(S, T, ptr(dist), ptr(tt), ptr(bad), 0, T, ctypes.byref(c0),
                                                    ctypes.byref(c1)) == 1
        assert lib.impdar_kirchhoff_window_vz_f32(ctypes.c_void_p(8), 0, T, T, ctypes.c_void_p(8), T, S, T, ptr(dist),
                                                  ptr(tt), ptr(np.zeros(3 * S)), ptr(bad), 0, 0, T, 0, S, S,
                                                  ctypes.c_void_p(8), 1 << 30, None) == 1
        assert lib.impdar_kirchhoff_host_pipelined_vz_f64(ctypes.c_void_p(8), ctypes.c_void_p(8), S, T, ptr(dist),
                                                          ptr(tt), ptr(np.zeros(3 * S)), ptr(bad), 0, 1,
                                                          ctypes.c_void_p(8), 1 << 30, None) == 1


# ------------------------------------------------------------------------------------------------------ GPU
def _run(fn, mode=0):
    from impdar_b200 import migrationlib as ml
    ml.set_kirchhoff_mode(mode)
    try:
        out = fn()
        return out, ml.kirchhoff_last_kernel()
    finally:
        ml.set_kirchhoff_mode(0)


MODES = {'auto': 0, 'general': 1, 'table_gather': 3}


@pytest.mark.gpu
@pytest.mark.parametrize("mode", list(MODES))
@pytest.mark.parametrize("nearfield", [False, True])
@pytest.mark.parametrize("nan", [False, True])
def test_constant_vector_bit_for_bit_kernels(mode, nearfield, nan):
    import torch
    from impdar_b200 import migrationlib as ml
    S, T = 300, 700
    d = synthetic_dat(S, T, seed=11)
    if nan:
        d.data[40, 100:140] = np.nan
    x = torch.from_numpy(d.data).cuda()
    for vel in (1.69e8, 2.1e8):
        a, ka = _run(lambda: ml.kirchhoff_device(x, d.travel_time, d.dist, vel, nearfield).cpu().numpy(), MODES[mode])
        b, kb = _run(lambda: ml.kirchhoff_device(x, d.travel_time, d.dist, np.full(S, vel), nearfield).cpu().numpy(),
                     MODES[mode])
        assert ka == kb
        assert np.array_equal(a, b, equal_nan=True), (mode, nearfield, nan, vel)
    if mode == 'auto' and not nearfield and not nan:
        assert ka == 'table_tile'


@pytest.mark.gpu
def test_device_entries_reject_bad_vectors():
    import torch
    from impdar_b200 import migrationlib as ml
    S, T = 64, 32
    d = synthetic_dat(S, T)
    x = torch.from_numpy(d.data).cuda()
    for bad in (np.full(S + 1, 1.7e8), np.r_[np.full(S - 1, 1.7e8), np.nan], np.r_[np.full(S - 1, 1.7e8), 0.0]):
        with pytest.raises(ValueError):
            ml.kirchhoff_host(d.data, d.travel_time, d.dist, bad, False)
        with pytest.raises(ValueError):
            ml.kirchhoff_device(x, d.travel_time, d.dist, bad, False)


@pytest.mark.gpu
def test_constant_vector_bit_for_bit_entries():
    import torch
    from impdar_b200 import migrationlib as ml
    S, T = 512, 1024
    d = synthetic_dat(S, T, seed=12)
    x = torch.from_numpy(d.data).cuda()
    vel, vec = 1.69e8, np.full(S, 1.69e8)
    whole = ml.kirchhoff_device(x, d.travel_time, d.dist, vel, False).cpu().numpy()
    assert np.array_equal(whole, ml.kirchhoff_device(x, d.travel_time, d.dist, vec, False).cpu().numpy())
    for v in (vel, vec):
        out = torch.empty((S, T), dtype=torch.float32, device='cuda')
        g_hi = S
        for r0, r1 in reversed([(0, 100), (100, 333), (333, S)]):
            ml.kirchhoff_rows_device(x, d.travel_time, d.dist, v, False, 0, T, r0, r1, g_hi, out)
            g_hi = r0
        assert np.array_equal(out.cpu().numpy(), whole)
        img = torch.empty((S, T), dtype=torch.float32, device='cuda')
        for xb, xe in ((0, 300), (300, 700), (700, T)):
            c0, c1 = ml.kirchhoff_input_window(S, d.travel_time, d.dist, v, xb, xe)
            ml.kirchhoff_window_device(x[:, c0:c1], c0, T, d.travel_time, d.dist, v, False, xb, xe, out=img[:, xb:xe])
        assert np.array_equal(img.cpu().numpy(), whole)
        host = ml.kirchhoff_host(d.data, d.travel_time, d.dist, v, False, nchunks=4)
        assert np.array_equal(host, whole.astype(np.float64))


def _layered_case(S, T, dx=5.0, irregular=False, seed=0):
    d = synthetic_dat(S, T, seed=seed, dx=dx)
    if irregular:
        d.dist = np.cumsum(np.r_[0.0, dx * (0.6 + 0.8 * np.random.default_rng(seed).random(T - 1))]) / 1e3
    return d, layered_rms(d)


@pytest.mark.gpu
@pytest.mark.parametrize("S,T,irregular,nearfield,want", [
    (200, 300, False, False, None),
    (333, 257, False, True, 'table_gather'),
    (256, 256, False, False, None),
    (300, 400, True, False, 'general'),
    (300, 400, True, True, 'general'),
])
def test_layered_against_oracle(S, T, irregular, nearfield, want):
    import torch
    from impdar_b200 import migrationlib as ml
    d, v = _layered_case(S, T, irregular=irregular, seed=S)
    ref = lo.kirchhoff(d.data, d.travel_time, d.dist, v, nearfield)
    got = ml.kirchhoff_device(torch.from_numpy(d.data).cuda(), d.travel_time, d.dist, v, nearfield).cpu().numpy()
    assert rel_l2(got, ref) <= TOL
    kern = ml.kirchhoff_last_kernel()
    assert kern == (want or predicted_kernel(d, v))
    if not irregular:   # the general kernel on the same geometry (its sigma-scaled fast path)
        g, kg = _run(lambda: ml.kirchhoff_device(torch.from_numpy(d.data).cuda(), d.travel_time, d.dist, v,
                                                 nearfield).cpu().numpy(), 1)
        assert kg == 'general' and rel_l2(g, ref) <= TOL


@pytest.mark.gpu
@pytest.mark.parametrize("S,T,dx", [(2048, 4096, 5.0), (512, 1024, 1.0)])
def test_layered_config_shapes(S, T, dx):
    """Config 2 (tile kernel) and a dense geometry where the tile kernel stands down, on sampled output traces."""
    import torch
    from impdar_b200 import migrationlib as ml
    d, v = _layered_case(S, T, dx=dx, seed=7)
    got = ml.kirchhoff_device(torch.from_numpy(d.data).cuda(), d.travel_time, d.dist, v, False).cpu().numpy()
    assert ml.kirchhoff_last_kernel() == predicted_kernel(d, v)
    tr = list(np.unique(np.r_[0, 1, np.linspace(0, T - 1, 9).astype(int), T - 1]))
    ref = lo.kirchhoff_sparse(d.data, d.travel_time, d.dist, v, False, tr)
    assert rel_l2(got[:, tr], ref) <= TOL


@pytest.mark.gpu
def test_layered_velocity_file_host_and_device(tmp_path):
    import torch
    import impdar_b200
    from impdar_b200 import synthetic
    S, T = 256, 200
    d, v = _layered_case(S, T, seed=3)
    fn = tmp_path / "firn_velocity.txt"
    np.savetxt(fn, synthetic.layered_velocity(d.travel_time))
    ref = lo.kirchhoff(d.data, d.travel_time, d.dist, v, False)
    host = synthetic_dat(S, T, seed=3)
    impdar_b200.migrationKirchhoffLayered(host, vel_fn=str(fn))
    assert isinstance(host.data, np.ndarray) and host.data.dtype == np.float64
    assert rel_l2(host.data, ref) <= TOL
    dev = synthetic_dat(S, T, seed=3)
    dev.data = torch.from_numpy(dev.data).cuda()
    impdar_b200.migrationKirchhoffLayered(dev, vel_fn=str(fn))
    assert torch.is_tensor(dev.data) and dev.data.is_cuda
    assert np.array_equal(dev.data.cpu().numpy().astype(np.float64), host.data)
    # a scalar is exactly migrationKirchhoff
    a, b = synthetic_dat(S, T, seed=4), synthetic_dat(S, T, seed=4)
    impdar_b200.migrationKirchhoffLayered(a, vel=1.8e8)
    impdar_b200.migrationKirchhoff(b, vel=1.8e8)
    assert np.array_equal(a.data, b.data)


@pytest.mark.gpu
@pytest.mark.parametrize("nan", [False, True])
def test_layered_cut_invariance(nan):
    import torch
    from impdar_b200 import migrationlib as ml
    S, T = 700, 900
    d, v = _layered_case(S, T, seed=9)
    if nan:
        d.data[30, 10:20] = np.nan
    x = torch.from_numpy(d.data).cuda()
    whole = ml.kirchhoff_device(x, d.travel_time, d.dist, v, False).cpu().numpy()
    out = torch.empty((S, T), dtype=torch.float32, device='cuda')
    g_hi = S
    for r0, r1 in reversed([(0, 150), (150, 401), (401, S)]):
        ml.kirchhoff_rows_device(x, d.travel_time, d.dist, v, False, 0, T, r0, r1, g_hi, out)
        g_hi = r0
    assert np.array_equal(out.cpu().numpy(), whole, equal_nan=True)
    img = torch.empty((S, T), dtype=torch.float32, device='cuda')
    for xb, xe in ((0, 256), (256, 512), (512, T)):
        c0, c1 = ml.kirchhoff_input_window(S, d.travel_time, d.dist, v, xb, xe)
        ml.kirchhoff_window_device(x[:, c0:c1].contiguous(), c0, T, d.travel_time, d.dist, v, False, xb, xe,
                                   out=img[:, xb:xe])
    if not nan:
        assert np.array_equal(img.cpu().numpy(), whole)
    else:   # NaNs that lie in one window only: that window runs the nansum variant, the others do not (no bit-for-bit
        # promise, DESIGN.md), so the assembled image is checked against the float64 reference instead
        assert rel_l2(img.cpu().numpy(), lo.kirchhoff(d.data, d.travel_time, d.dist, v, False)) <= TOL
    host = ml.kirchhoff_host(d.data, d.travel_time, d.dist, v, False, nchunks=5)
    assert np.array_equal(host, whole.astype(np.float64), equal_nan=True)
