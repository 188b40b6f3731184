"""Kirchhoff migration with a laterally varying velocity (a (v, z, x) table: one RMS profile per output trace).

CPU part: getVelocityProfile's lateral branch computes each distinct griddata column once and still returns exactly what
the per-trace loop returned (golden vmig arrays, a verbatim restatement of that loop, the same ValueErrors); the
per-profile RMS velocities; argument errors of the Python and C entries; the routing of migrationKirchhoffLateral; and a
float64 focusing check through the per-column reference (column xi = the layered reference with profile V[:, xi]).
GPU part: the lateral general kernel gives, column by column, the single-profile general kernel's bits; the per-run
table path gives each run the single-profile table path's bits; both match the per-column float64 reference; windows,
sub-ranges and the pair counters.
"""
import ctypes
import time

import numpy as np
import pytest

from conftest import golden_names, load_golden, rel_l2
from util import dat_from_golden, synthetic_dat
import kirchhoff_layered_oracle as lo

TOL = 1e-5


def old_lateral_vmig(dat, vels_in):
    """getVelocityProfile's (v, z, x) branch as it was: the per-trace loop (mig_python.py's), kept verbatim."""
    from scipy.interpolate import griddata, interp1d
    vel_v = vels_in[:, 0]
    vel_z = vels_in[:, 1]
    twtt = np.asarray(dat.travel_time, dtype=np.float64).copy() / 1.0e6
    vel_x = vels_in[:, 2]
    zs = np.linspace(np.min(vel_v) * twtt[0], np.max(vel_v) * twtt[-1], dat.snum) / 2.
    if dat.dist is None or all(dat.dist == 0):
        raise ValueError('The distance vector was never set.')
    XS, ZS = np.meshgrid(dat.dist, zs)
    VS = griddata(np.transpose([vel_x, vel_z]), vel_v,
                  np.transpose([XS.flatten(), ZS.flatten()]), method='nearest')
    VS = np.reshape(VS, np.shape(XS))
    vmig = np.zeros_like(VS)
    trapz = getattr(np, 'trapezoid', None) or np.trapz
    for i in range(dat.tnum):
        vz = ZS[:, i]
        vv = VS[:, i]
        vel_t = 2 * np.array([trapz(1. / vv[:j], vz[:j]) for j in range(dat.snum)])
        tofz = interp1d(ZS[:, i], vel_t)(zs)
        zinterp = interp1d(tofz, zs)
        if twtt[-1] > tofz[-1]:
            raise ValueError('Two-way travel time array extends outside of interpolation range')
        vmig[:, i] = 2. * np.gradient(zinterp(twtt), twtt)
    return vmig


def grid_table(d, nx=5, v_top=2.2e8, v_bottom=1.7e8, spread=0.06):
    """Rectangular (v, z, x) node grid: nx x strips across the profile, each a firn-like column (fast on top) scaled by
    its own factor, three depth nodes."""
    x = np.asarray(d.dist, dtype=np.float64)
    xs = np.linspace(x[0], x[-1], nx)
    zmax = v_top * d.travel_time[-1] / 1e6 / 2.
    rows = []
    for j, xj in enumerate(xs):
        f = 1.0 + spread * (j / max(nx - 1, 1) - 0.5)
        for z, v in ((0.0, v_top), (0.3 * zmax, v_top), (0.5 * zmax, v_bottom), (1.2 * zmax, v_bottom)):
            rows.append((v * f, z, xj))
    return np.array(rows)


def scattered_table(d, n=40, seed=0):
    """Randomly placed nodes: many distinct griddata columns."""
    rng = np.random.default_rng(seed)
    x = np.asarray(d.dist, dtype=np.float64)
    zmax = 2.2e8 * d.travel_time[-1] / 1e6 / 2.
    z = rng.random(n) * 1.2 * zmax
    v = np.where(z < 0.4 * zmax, 2.2e8, 1.7e8) * (1 + 0.05 * rng.random(n))
    return np.column_stack([v, z, x[0] + (x[-1] - x[0]) * rng.random(n)])


# ------------------------------------------------------------------------------------------------------ CPU
@pytest.mark.parametrize("name", [n for n in golden_names(contains="_phsh_lateral") if "vmig" in load_golden(n)])
def test_getVelocityProfile_lateral_golden(name):
    from impdar_b200 import migrationlib as ml
    g = load_golden(name)
    d = dat_from_golden(g)
    assert np.array_equal(ml.getVelocityProfile(d, g["vel"]), g["vmig"])


@pytest.mark.parametrize("kind", ["grid", "scattered"])
def test_getVelocityProfile_lateral_equals_old_loop(kind):
    from impdar_b200 import migrationlib as ml
    d = synthetic_dat(48, 64, seed=1)
    if kind == "scattered":
        d.dist = np.arange(64) * 5.0    # positions on the depth axis' scale: griddata's nearest node varies along x too
    table = grid_table(d) if kind == "grid" else scattered_table(d)
    new = ml.getVelocityProfile(d, table)
    old = old_lateral_vmig(d, table)
    assert new.dtype == old.dtype and new.shape == old.shape
    assert np.array_equal(new, old)
    profiles, colp = ml.lateral_velocity_profiles(d, table)
    assert np.array_equal(profiles[colp].T, old)
    if kind == "scattered":
        assert profiles.shape[0] > 10


def test_getVelocityProfile_lateral_same_errors():
    from impdar_b200 import migrationlib as ml
    d = synthetic_dat(32, 40, seed=2)
    x = d.dist
    const = np.array([[1.7e8, 0., x[0]], [1.7e8, 1e4, x[0]], [1.7e8, 0., x[-1]], [1.7e8, 1e4, x[-1]]])
    msgs = []
    for fn in (old_lateral_vmig, ml.getVelocityProfile):
        with pytest.raises(ValueError) as e:
            fn(d, const)    # a column at the table's largest velocity everywhere ends short of the last sample
        msgs.append(str(e.value))
    d0 = synthetic_dat(32, 40, seed=2)
    d0.dist = np.zeros(40)
    for fn in (old_lateral_vmig, ml.getVelocityProfile):
        with pytest.raises(ValueError) as e:
            fn(d0, grid_table(d))
        msgs.append(str(e.value))
    assert msgs[0] == msgs[1] and msgs[2] == msgs[3]


def test_getVelocityProfile_lateral_cost_is_per_distinct_column():
    """1024 x 1024 with a 5-strip grid table: the per-trace loop took about 15 s; five columns cost a fraction."""
    from impdar_b200 import migrationlib as ml
    d = synthetic_dat(1024, 1024, seed=3)
    table = grid_table(d, nx=5)
    t0 = time.perf_counter()
    profiles, colp = ml.lateral_velocity_profiles(d, table)
    elapsed = time.perf_counter() - t0
    assert profiles.shape == (5, 1024)
    assert elapsed < 4.0, elapsed


@pytest.mark.parametrize("nx", [2, 3, 7])
def test_grid_table_profile_count(nx):
    from impdar_b200 import migrationlib as ml
    d = synthetic_dat(40, 90, seed=4)
    profiles, colp = ml.lateral_velocity_profiles(d, grid_table(d, nx=nx))
    assert profiles.shape[0] == nx
    assert np.all(np.diff(colp) >= 0) and colp[0] == 0 and colp[-1] == nx - 1   # strips in order along the profile


def test_rms_velocity_profiles_rows():
    from impdar_b200 import migrationlib as ml
    rng = np.random.default_rng(5)
    for tt in (np.arange(300) * 0.01, (np.arange(300) - 20) * 0.01):
        prof = 1.6e8 + 0.7e8 * rng.random((6, 300))
        got = ml.rms_velocity_profiles(tt, prof)
        for i in range(6):
            assert np.array_equal(got[i], ml.rms_velocity(tt, prof[i]))
    with pytest.raises(ValueError):
        ml.rms_velocity_profiles(np.arange(10) * 0.01, np.ones((2, 9)))


def test_argument_errors(tmp_path):
    import torch
    from impdar_b200 import migrationlib as ml
    S, T = 16, 12
    d = synthetic_dat(S, T)
    x = torch.zeros((S, T))      # validation happens before anything touches the device
    good = np.full((2, S), 1.7e8)
    colp = np.zeros(T, dtype=np.int64)
    bad_profiles = [np.full((2, S - 1), 1.7e8), np.full(S, 1.7e8), np.full((0, S), 1.7e8)]
    for badval in (0.0, -1.0, np.nan, np.inf):
        b = good.copy()
        b[1, 3] = badval
        bad_profiles.append(b)
    for b in bad_profiles:
        with pytest.raises(ValueError):
            ml.kirchhoff_lateral_device(x, d.travel_time, d.dist, b, colp, False)
    for c in (np.full(T, 2), np.full(T, -1), np.zeros(T - 1, dtype=int), np.zeros(T) + 0.5):
        with pytest.raises(ValueError):
            ml.kirchhoff_lateral_device(x, d.travel_time, d.dist, good, c, False)
    with pytest.raises(TypeError):
        ml.migrationKirchhoffLateral(d, vel_fn=str(tmp_path / "missing_velocity.txt"))


def test_c_entry_rejects_bad_input():
    from impdar_b200 import _lib
    lib = _lib.load()
    S, T, P = 16, 8, 3
    tt = np.arange(S) * 1e-8
    dist = np.arange(T) * 5.0
    coef = np.zeros(3 * S)
    ptr = lambda a: a.ctypes.data_as(ctypes.c_void_p)   # noqa: E731
    fake = ctypes.c_void_p(8)
    good = np.full((P, S), 1.7e8)
    colp = np.zeros(T, dtype=np.int32)
    ws = lib.impdar_kirchhoff_lateral_workspace_bytes(S, T, P, 0)
    assert ws >= lib.impdar_kirchhoff_workspace_bytes(S, T, 0) + P * S * 8 * 3
    assert lib.impdar_kirchhoff_lateral_workspace_bytes(S, T, 0, 0) == 0

    def call(profiles, nprof, cp, ws_bytes=1 << 40, x_begin=0, x_end=T):
        return lib.impdar_kirchhoff_window_vxz_f32(fake, 0, T, T, fake, T, S, T, ptr(dist), ptr(tt), ptr(coef),
                                                   ptr(profiles), nprof, ptr(cp), 0, x_begin, x_end, fake, ws_bytes,
                                                   None)
    for badval in (0.0, -1.0, np.nan, np.inf):
        b = good.copy()
        b[2, 5] = badval
        assert call(b, P, colp) == 1
    for c in (np.full(T, P, dtype=np.int32), np.full(T, -1, dtype=np.int32)):
        assert call(good, P, c) == 1
    assert call(good, 0, colp) == 1
    assert call(good, P, colp, ws_bytes=ws - 1) == 1
    assert call(good, P, colp, x_begin=3, x_end=3) == 1
    assert lib.impdar_kirchhoff_window_vxz_f32(fake, 0, T, T, fake, T, S, T, ptr(dist), ptr(tt), ptr(coef), None, P,
                                               ptr(colp), 0, 0, T, fake, 1 << 40, None) == 1


def test_symbols_exported():
    from impdar_b200 import _lib
    lib = ctypes.CDLL(_lib.LIB_PATH)
    for s in ("impdar_kirchhoff_window_vxz_f32", "impdar_kirchhoff_lateral_workspace_bytes"):
        assert hasattr(lib, s) and s in _lib.PROTOTYPES


def test_routing(monkeypatch):
    """A recording stand-in for the library's Kirchhoff entries: a single-profile field goes to the layered (vz) entry
    with that RMS vector, a (v, z) table or a scalar to migrationKirchhoffLayered, a lateral field to the vxz entry."""
    from impdar_b200 import migrationlib as ml
    calls = []
    monkeypatch.setattr(ml, "kirchhoff_host", lambda data, tt, dist, v, nf, nchunks=None: calls.append(
        ("vz", np.array(v), nf)) or np.zeros(np.shape(data)))
    monkeypatch.setattr(ml, "kirchhoff_lateral_device", lambda *a, **k: calls.append(("vxz",)))
    monkeypatch.setattr(ml, "migrationKirchhoffLayered", lambda dat, vel=None, nearfield=False: calls.append(
        ("layered", vel, nearfield)) or dat)
    S, T = 40, 30
    d = synthetic_dat(S, T, seed=6)
    one = grid_table(d, nx=2)
    one[:, 2] = d.dist[0]          # every node at one x: a single profile
    ml.migrationKirchhoffLateral(d, vel=one, nearfield=True)
    assert len(calls) == 1 and calls[0][0] == "vz" and calls[0][2] is True
    prof, _ = ml.lateral_velocity_profiles(synthetic_dat(S, T, seed=6), one)
    assert prof.shape[0] == 1
    assert np.array_equal(calls[0][1], ml.rms_velocity(d.travel_time, prof[0]))
    assert isinstance(d.data, np.ndarray) and d.data.dtype == np.float64
    calls.clear()
    layered = np.array([[2.2e8, 0.], [1.7e8, 50.], [1.7e8, 1e4]])
    for vel in (1.8e8, layered):
        ml.migrationKirchhoffLateral(synthetic_dat(S, T), vel=vel)
    assert [c[0] for c in calls] == ["layered", "layered"]
    assert calls[0][1] == 1.8e8 and np.array_equal(calls[1][1], layered)


def _diffractors(d, V, points, f0=50e6):
    """Ricker wavelets along t = sqrt(t0^2 + (2 x / V[t0, x0])^2)."""
    t = np.asarray(d.travel_time, dtype=np.float64) / 1e6
    x = np.asarray(d.dist, dtype=np.float64) * 1e3
    img = np.zeros((len(t), len(x)))
    for s0, x0 in points:
        th = np.sqrt(t[s0] ** 2 + (2.0 * (x - x[x0]) / V[s0, x0]) ** 2)
        a = (np.pi * f0 * (t[:, None] - th[None, :])) ** 2
        img += (1 - 2 * a) * np.exp(-a)
    return img.astype(np.float32)


def lateral_oracle(data, tt, dist, V, nearfield, traces):
    """Per-column float64 reference: column xi is the layered reference with the profile V[:, xi]."""
    return np.column_stack([lo.kirchhoff_sparse(data, tt, dist, V[:, xi], nearfield, [xi])[:, 0] for xi in traces])


def test_oracle_lateral_focuses_better():
    """A slow (1.69e8) and a fast (firn, 2.2e8 on top) half: a diffractor in each half.  The lateral field focuses the
    fast-side one better than the slow profile alone and as well as the fast one, and the slow-side one better than the
    fast profile alone: only the lateral field focuses both."""
    S, T = 300, 200
    d = synthetic_dat(S, T, seed=0)
    from impdar_b200 import migrationlib as ml, synthetic
    fast = ml.rms_velocity(d.travel_time, ml.getVelocityProfile(d, synthetic.layered_velocity(d.travel_time)))
    slow = np.full(S, 1.69e8)
    V = np.where(np.arange(T)[None, :] >= T // 2, fast[:, None], slow[:, None])
    pts = [(50, 150), (60, 50)]     # fast side (shallow, where the two differ most), slow side
    img = _diffractors(d, V, pts)

    def share(out, cols, s0, x0):
        e = np.zeros((S, T))
        e[:, cols] = out ** 2
        return e[s0 - 8:s0 + 9, x0 - 2:x0 + 3].sum() / e[max(s0 - 40, 0):s0 + 41, max(x0 - 40, 0):x0 + 41].sum()
    res = {}
    for s0, x0 in pts:
        cols = list(range(max(x0 - 40, 0), min(x0 + 41, T)))
        res[x0] = {k: share(lateral_oracle(img, d.travel_time, d.dist, W, False, cols), cols, s0, x0)
                   for k, W in (("lateral", V), ("fast", np.repeat(fast[:, None], T, 1)),
                                ("slow", np.repeat(slow[:, None], T, 1)))}
    f, s = res[150], res[50]
    assert f["lateral"] > 1.3 * f["slow"] and f["lateral"] >= 0.999 * f["fast"], f
    assert s["lateral"] > 1.3 * s["fast"] and s["lateral"] >= 0.999 * s["slow"], s


# ------------------------------------------------------------------------------------------------------ GPU
def _run(fn, mode=0):
    from impdar_b200 import migrationlib as ml
    ml.set_kirchhoff_mode(mode)
    try:
        out = fn()
        return out, ml.kirchhoff_last_kernel()
    finally:
        ml.set_kirchhoff_mode(0)


def _field(d, kind, seed=0):
    """(profiles, col_profile, V) of a test field: 'grid' (5-strip table), 'per_trace' (the firn profile scaled by
    1 + 0.03 x / T), 'mixed' (four profiles scattered over the traces)."""
    from impdar_b200 import migrationlib as ml, synthetic
    S, T = d.snum, d.tnum
    if kind == "grid":
        prof, colp = ml.lateral_rms_field(d, grid_table(d))
    else:
        base = ml.rms_velocity(d.travel_time, ml.getVelocityProfile(d, synthetic.layered_velocity(d.travel_time)))
        if kind == "per_trace":
            prof = base[None, :] * (1 + 0.03 * np.arange(T) / T)[:, None]
            colp = np.arange(T)
        else:
            prof = base[None, :] * np.array([1.0, 0.93, 1.05, 0.97])[:, None]
            colp = np.random.default_rng(seed).integers(0, 4, T)
    return prof, colp, prof[colp].T


def _geometry(d, geom, seed=0):
    T = d.tnum
    if geom == "irregular":
        d.dist = np.cumsum(np.r_[0.0, 5.0 * (0.6 + 0.8 * np.random.default_rng(seed).random(T - 1))]) / 1e3
    elif geom == "nonmonotone":
        d.dist = np.random.default_rng(seed).permutation(T) * 5.0 / 1e3
    return d


@pytest.mark.gpu
@pytest.mark.parametrize("S,T,geom,kind", [
    (200, 200, "uniform", "mixed"),          # S == T
    (160, 90, "uniform", "per_trace"),
    (180, 120, "irregular", "mixed"),
    (150, 70, "nonmonotone", "mixed"),
    (120, 1, "uniform", "per_trace"),        # tnum == 1
])
@pytest.mark.parametrize("nearfield", [False, True])
@pytest.mark.parametrize("nan", [False, True])
def test_lateral_kernel_columns_equal_vz_general(S, T, geom, kind, nearfield, nan):
    import torch
    from impdar_b200 import migrationlib as ml
    d = _geometry(synthetic_dat(S, T, seed=S + T), geom, seed=S)
    if nan:
        d.data[S // 5, :max(T // 4, 1)] = np.nan
    prof, colp, _ = _field(d, kind, seed=T)
    x = torch.from_numpy(d.data).cuda()
    got, k = _run(lambda: ml.kirchhoff_lateral_device(x, d.travel_time, d.dist, prof, colp, nearfield).cpu().numpy(),
                  ml.KIRCHHOFF_GENERAL)
    assert k == 'general_lateral'
    for p in np.unique(colp):
        want, kw = _run(lambda: ml.kirchhoff_device(x, d.travel_time, d.dist, prof[p], nearfield).cpu().numpy(),
                        ml.KIRCHHOFF_GENERAL)
        assert kw == 'general'
        cols = colp == p
        assert np.array_equal(got[:, cols], want[:, cols], equal_nan=True), (p, np.flatnonzero(cols)[:5])


@pytest.mark.gpu
@pytest.mark.parametrize("mode,nearfield,want", [("auto", False, "table_tile"), ("auto", True, "table_gather"),
                                                 ("table", False, "table_tile"), ("table_gather", False, "table_gather")])
def test_per_run_columns_equal_layered_table_call(mode, nearfield, want):
    import torch
    from impdar_b200 import migrationlib as ml
    m = {"auto": ml.KIRCHHOFF_AUTO, "table": ml.KIRCHHOFF_TABLE, "table_gather": ml.KIRCHHOFF_TABLE_GATHER}[mode]
    S, T = 400, 1000     # 5 runs: tnum >= 192 x runs, the automatic rule takes the per-run path
    d = synthetic_dat(S, T, seed=21)
    prof, colp, _ = _field(d, "grid")
    assert prof.shape[0] == 5
    x = torch.from_numpy(d.data).cuda()
    got, k = _run(lambda: ml.kirchhoff_lateral_device(x, d.travel_time, d.dist, prof, colp, nearfield).cpu().numpy(), m)
    assert k == want
    for p in range(prof.shape[0]):
        ref, kr = _run(lambda: ml.kirchhoff_device(x, d.travel_time, d.dist, prof[p], nearfield).cpu().numpy(), m)
        assert kr == want
        cols = colp == p
        assert np.array_equal(got[:, cols], ref[:, cols]), p


@pytest.mark.gpu
def test_per_run_path_irregular_spacing_raises_when_forced():
    import torch
    from impdar_b200 import migrationlib as ml
    d = _geometry(synthetic_dat(100, 80, seed=1), "irregular")
    prof, colp, _ = _field(d, "mixed")
    x = torch.from_numpy(d.data).cuda()
    for m in (ml.KIRCHHOFF_TABLE, ml.KIRCHHOFF_TABLE_GATHER):
        with pytest.raises(ValueError):
            _run(lambda: ml.kirchhoff_lateral_device(x, d.travel_time, d.dist, prof, colp, False), m)
    _, k = _run(lambda: ml.kirchhoff_lateral_device(x, d.travel_time, d.dist, prof, colp, False))
    assert k == 'general_lateral'


@pytest.mark.gpu
def test_constant_field_equals_scalar_call():
    import torch
    from impdar_b200 import migrationlib as ml
    S, T = 256, 600
    d = synthetic_dat(S, T, seed=22)
    x = torch.from_numpy(d.data).cuda()
    prof = np.full((3, S), 1.69e8)
    for colp in (np.repeat([0, 1, 2], 200), np.arange(T) % 3):   # wide runs (per-run path), narrow runs
        for m in (ml.KIRCHHOFF_AUTO, ml.KIRCHHOFF_GENERAL):
            a, ka = _run(lambda: ml.kirchhoff_lateral_device(x, d.travel_time, d.dist, prof, colp,
                                                             False).cpu().numpy(), m)
            # the scalar call on the same kernel: the general kernel when the lateral field took the lateral kernel
            b, kb = _run(lambda: ml.kirchhoff_device(x, d.travel_time, d.dist, 1.69e8, False).cpu().numpy(),
                         ml.KIRCHHOFF_GENERAL if ka == 'general_lateral' else m)
            assert ka == ('table_tile' if m == ml.KIRCHHOFF_AUTO and len(np.unique(colp[:3])) == 1
                          else 'general_lateral')
            assert kb == ('general' if ka == 'general_lateral' else ka)
            assert np.array_equal(a, b)


@pytest.mark.gpu
def test_single_profile_equals_layered_both_lanes():
    import torch
    import impdar_b200
    from impdar_b200 import migrationlib as ml
    S, T = 256, 200
    d = synthetic_dat(S, T, seed=23)
    one = grid_table(d, nx=2)
    one[:, 2] = d.dist[T // 2]
    prof, _ = ml.lateral_rms_field(d, one)
    assert prof.shape[0] == 1
    host = synthetic_dat(S, T, seed=23)
    impdar_b200.migrationKirchhoffLateral(host, vel=one)
    assert host.data.dtype == np.float64
    assert np.array_equal(host.data, ml.kirchhoff_host(synthetic_dat(S, T, seed=23).data, d.travel_time, d.dist,
                                                       prof[0], False))
    dev = synthetic_dat(S, T, seed=23)
    dev.data = torch.from_numpy(dev.data).cuda()
    impdar_b200.migrationKirchhoffLateral(dev, vel=one)
    assert torch.is_tensor(dev.data) and dev.data.is_cuda
    want = ml.kirchhoff_device(torch.from_numpy(synthetic_dat(S, T, seed=23).data).cuda(), d.travel_time, d.dist,
                               prof[0], False)
    assert torch.equal(dev.data, want)


@pytest.mark.gpu
@pytest.mark.parametrize("S,T,kind,geom,nearfield", [
    (300, 400, "grid", "uniform", False),
    (257, 333, "grid", "uniform", True),
    (300, 400, "per_trace", "uniform", False),
    (220, 260, "mixed", "irregular", True),
])
def test_lateral_against_oracle(S, T, kind, geom, nearfield):
    import torch
    from impdar_b200 import migrationlib as ml
    d = _geometry(synthetic_dat(S, T, seed=S), geom, seed=T)
    prof, colp, V = _field(d, kind, seed=S)
    got = ml.kirchhoff_lateral_device(torch.from_numpy(d.data).cuda(), d.travel_time, d.dist, prof, colp,
                                      nearfield).cpu().numpy()
    ref = lateral_oracle(d.data, d.travel_time, d.dist, V, nearfield, range(T))
    assert rel_l2(got, ref) <= TOL


@pytest.mark.gpu
def test_lateral_velocity_file_host_and_device(tmp_path):
    import torch
    import impdar_b200
    from impdar_b200 import migrationlib as ml
    S, T = 256, 300
    d = synthetic_dat(S, T, seed=24)
    fn = tmp_path / "velocity_lateral.txt"
    np.savetxt(fn, grid_table(d))
    prof, colp, V = _field(d, "grid")
    ref = lateral_oracle(d.data, d.travel_time, d.dist, V, False, range(T))
    host = synthetic_dat(S, T, seed=24)
    impdar_b200.migrationKirchhoffLateral(host, vel_fn=str(fn))
    assert isinstance(host.data, np.ndarray) and host.data.dtype == np.float64
    assert rel_l2(host.data, ref) <= TOL
    dev = synthetic_dat(S, T, seed=24)
    dev.data = torch.from_numpy(dev.data).cuda()
    impdar_b200.migrationKirchhoffLateral(dev, vel_fn=str(fn))
    assert torch.is_tensor(dev.data) and dev.data.is_cuda
    assert np.array_equal(dev.data.cpu().numpy().astype(np.float64), host.data)


@pytest.mark.gpu
@pytest.mark.parametrize("S,T,dx,kind,want", [(2048, 4096, 5.0, "grid", "table_tile"),
                                              (2048, 4096, 5.0, "per_trace", "general_lateral"),
                                              (512, 1024, 1.0, "grid", "table_gather")])
def test_lateral_config_shapes(S, T, dx, kind, want):
    """Config 2 on both sides of the dispatch, and a dense geometry where the tile kernel stands down, on sampled
    output traces (run edges included)."""
    import torch
    from impdar_b200 import migrationlib as ml
    d = synthetic_dat(S, T, seed=7, dx=dx)
    prof, colp, V = _field(d, kind)
    got = ml.kirchhoff_lateral_device(torch.from_numpy(d.data).cuda(), d.travel_time, d.dist, prof, colp,
                                      False).cpu().numpy()
    assert ml.kirchhoff_last_kernel() == want
    edges = np.flatnonzero(np.diff(colp))[:3]
    tr = list(np.unique(np.r_[0, 1, np.linspace(0, T - 1, 7).astype(int), edges, edges + 1, T - 1]))
    ref = lateral_oracle(d.data, d.travel_time, d.dist, V, False, tr)
    assert rel_l2(got[:, tr], ref) <= TOL


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["auto", "general"])
@pytest.mark.parametrize("kind", ["grid", "mixed"])
def test_windows_and_ranges(mode, kind):
    import torch
    from impdar_b200 import _lib, migrationlib as ml
    m = ml.KIRCHHOFF_GENERAL if mode == "general" else ml.KIRCHHOFF_AUTO
    S, T = 300, 1000
    d = synthetic_dat(S, T, seed=25)
    prof, colp, _ = _field(d, kind, seed=3)
    x = torch.from_numpy(d.data).cuda()
    whole, _ = _run(lambda: ml.kirchhoff_lateral_device(x, d.travel_time, d.dist, prof, colp, False).cpu().numpy(), m)
    for xb, xe in ((0, 1), (5, 333), (333, 640), (640, T), (100, 101)):
        part, _ = _run(lambda: ml.kirchhoff_lateral_device(x, d.travel_time, d.dist, prof, colp, False, xb,
                                                           xe).cpu().numpy(), m)
        assert np.array_equal(part, whole[:, xb:xe]), (xb, xe)
    # column windows: the window of each range for the row-wise largest velocity
    tt_sec = d.travel_time / 1e6
    dist_m = np.ascontiguousarray(d.dist * 1e3)
    coef = ml.gradient_coefficients(tt_sec)
    v, cp = ml._kirch_lateral_args(prof, colp, S, T)
    img = torch.empty((S, T), dtype=torch.float32, device='cuda')
    for xb, xe in ((0, 300), (300, 640), (640, T)):
        c0, c1 = ml.kirchhoff_input_window(S, d.travel_time, d.dist, prof.max(axis=0), xb, xe)
        win = x[:, c0:c1].contiguous()
        _run(lambda: ml._kirch_window_vxz(_lib.load(), win.data_ptr(), c0, c1 - c0, win.stride(0), img[:, xb:xe], S, T,
                                          dist_m, tt_sec, coef, v, cp, False, xb, xe), m)
    assert np.array_equal(img.cpu().numpy(), whole)


def lateral_pair_count(travel_time_us, dist_km, prof, colp):
    """Pairs with 2 r / V[ti, xi] <= max(tt) (kirchhoff_layered_oracle.kirchhoff_pair_count per profile and column)."""
    tt = np.asarray(travel_time_us, dtype=np.float64) / 1e6
    dist = np.asarray(dist_km, dtype=np.float64) * 1e3
    tmax = tt.max()
    total = 0
    for p in np.unique(colp):
        v = prof[p]
        zs = v * tt / 2.
        ap2 = (v * tmax / 2.) ** 2 - zs ** 2
        xs = dist[colp == p]
        for a2 in ap2:
            if a2 < 0:
                continue
            a = np.sqrt(a2)
            total += int(np.sum(np.searchsorted(dist, xs + a, side='right') - np.searchsorted(dist, xs - a,
                                                                                               side='left')))
    return total


def _pairs(fn, mode):
    from impdar_b200 import migrationlib as ml
    ml.enable_kirchhoff_stats(True)
    try:
        _, k = _run(fn, mode)
        return ml.kirchhoff_stats()[0], k
    finally:
        ml.enable_kirchhoff_stats(False)


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["grid", "mixed", "per_trace"])
def test_pair_counters(kind):
    """The lateral kernel counts the per-column reference's pairs.  The per-run path reports the sum of its runs'
    single-profile table-path counters (which, as for one profile, leave out the pairs of entries sent to the exact
    float64 pass)."""
    import torch
    from impdar_b200 import migrationlib as ml
    S, T = 256, 1000
    d = synthetic_dat(S, T, seed=26)
    x = torch.from_numpy(d.data).cuda()
    prof, colp, _ = _field(d, kind, seed=5)
    pairs, k = _pairs(lambda: ml.kirchhoff_lateral_device(x, d.travel_time, d.dist, prof, colp, False),
                      ml.KIRCHHOFF_GENERAL)
    assert k == 'general_lateral'
    assert pairs == lateral_pair_count(d.travel_time, d.dist, prof, colp)
    if kind == "grid":
        runs, k = _pairs(lambda: ml.kirchhoff_lateral_device(x, d.travel_time, d.dist, prof, colp, False),
                         ml.KIRCHHOFF_AUTO)
        assert k == 'table_tile'
        edges = np.r_[0, np.flatnonzero(np.diff(colp)) + 1, T]
        want = sum(_pairs(lambda: ml.kirchhoff_device(x, d.travel_time, d.dist, prof[colp[a]], False, a, b),
                          ml.KIRCHHOFF_AUTO)[0] for a, b in zip(edges[:-1], edges[1:]))
        assert runs == want
