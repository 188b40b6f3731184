"""The migrations across acquisition geometries.

Most parity tests run one geometry (dt = 10 ns, dx = 5 m, v = 1.69e8 m/s).  The kernel branches that depend on
geometry are governed by one number, rho = v dt / (2 dx):

* phase shift: a kx column propagates only the frequencies with |w| > v |kx| / 2.  For rho > 1 the highest kx columns
  hold no propagating bin at all, near the cut-off a column holds one partial tensor-core stage or only the Nyquist bin,
  and on power-of-two geometries the propagating test `vkx2 < w2` has exact ties;
* Stolt: the query w' = v/2 sqrt(kz^2 + kx^2) is clamped to the last node; for rho > 1 whole kx columns are clamped;
* Kirchhoff: a block of KT_Q = 28 output rows starting at sample i0 reads each source row over an offset interval about
  rho sqrt(54 i0 + 729) traces wide; above KT_SPAN = 120 the tile kernel stands down and the gather kernel runs.  A
  small rho gives an aperture of a few traces.

The CPU part proves, in plain float64 numpy with the kernels' operation order, that each named geometry really is in
the regime it is named for, so the GPU part cannot pass vacuously if a constant moves.  The GPU part checks every kernel
against the float64 oracle in those regimes, and that the Kirchhoff tile kernel's stand-down decisions do not depend on
how an image is cut into row chunks, host pipeline chunks or column windows.
"""
import functools
from collections import namedtuple

import numpy as np
import pytest

from conftest import max_abs, rel_l2
from util import synthetic_dat

TOL = 1e-5          # float32 paths against the float64 oracle
TOL_FFD = 1e-10     # the laterally varying branch is float64 end to end

KT_Q = 28           # output rows per tile-kernel block (kirchhoff_tile.cuh)
KT_SPAN = 120       # widest offset interval the tile kernel stages
TC_KC = 32          # frequencies per tensor-core phase-shift stage (phaseshift_tc.cu)
NUM_SMS = 148       # B200

Geo = namedtuple("Geo", "dt dx vel")
GEOMETRIES = {
    "G0": Geo(1e-8, 5.0, 1.69e8),           # control, rho 0.169
    "G1": Geo(1e-8, 1.0, 1.69e8),           # dense traces, rho 0.845
    "G2": Geo(1e-8, 0.5, 1.69e8),           # evanescent kx columns, rho 1.69
    "G3": Geo(2.0 ** -27, 0.5, 2.0 ** 27),  # every factor a power of two, rho = 1 exactly: exact ties
    "G4": Geo(1e-8, 50.0, 1.69e8),          # sparse traces, rho 0.0169
}


def rho(geo):
    return geo.vel * geo.dt / (2.0 * geo.dx)


def _dat(S, T, geo, seed):
    return synthetic_dat(S, T, seed=seed, dt=geo.dt, dx=geo.dx)


def _report(name, got, want):
    r, m = rel_l2(got, want), max_abs(got, want)
    print("%-52s rel-L2 %.3e  max-abs %.3e" % (name, r, m))
    return r


# ------------------------------------------------------------------------------------- CPU restatements of the regimes
def phsh_column_census(S, T, geo):
    """Propagating-bin census of the kx columns the constant-velocity kernels process (k = 0 .. T // 2), with numpy's
    float64 operation sequence (mig_python.py:405-412, phsh_tc_phase_kernel).  Returns a dict: columns with no
    propagating bin, with 1-31 listed bins (one partial stage), with only the Nyquist bin, and the number of exact ties
    vkx2 == w2 over all (w, kx) bins."""
    nt = 2 ** int(np.ceil(np.log(S) / np.log(2)))
    K = T // 2 + 1
    kx = 2. * np.pi * (np.arange(K) * (1.0 / (T * geo.dx)))
    vkx2 = (geo.vel * kx / 2.) ** 2.
    w = 2. * np.pi * np.fft.fftfreq(nt, d=geo.dt)
    w[w == 0.0] = 1e-10 / geo.dt
    w2 = w ** 2.
    prop = vkx2[None, :] < w2[:, None]
    nh = nt // 2
    n_list = prop[:nh].sum(axis=0) + prop[nh + 1:].sum(axis=0)   # the Nyquist bin has its own kernel
    nyq = prop[nh]
    return {
        "nt": nt, "K": K,
        "evanescent": int(np.sum(~prop.any(axis=0))),
        "partial": int(np.sum((n_list >= 1) & (n_list < TC_KC))),
        "nyquist_only": int(np.sum((n_list == 0) & nyq)),
        "ties": int(np.sum(vkx2[None, :] == w2[:, None])),
        "min_fraction": float((prop.sum(axis=0) / nt).min()),
    }


def stolt_clamped_columns(S, T, geo):
    """kx columns in which every kz query w' lies at or beyond the last w node (oracle.migration.stolt, :229-238)."""
    ws = 2. * np.pi * np.fft.rfftfreq(S, d=geo.dt)
    kx = 2. * np.pi * np.fft.fftfreq(T, d=geo.dx)
    kz = ws[:S // 2] * 2. / geo.vel
    wsj = geo.vel / 2. * np.sqrt(kz[:, None] ** 2. + kx[None, :] ** 2.)
    return int(np.sum((wsj >= ws[-1]).all(axis=0)))


def _pick(tt, t):
    """argmin_k |tt[k] - t|, first minimum (mig_python.py:49)."""
    from oracle.migration import nearest_sample_index
    return nearest_sample_index(tt, t)


class KirchTable:
    """The uniform-geometry pick table of kirch_table_build_kernel, restated in float64 numpy: entry (ti, m) is the
    nearest-sample pick k of offset m from output row ti, -1 past the aperture cut 2r/v > max(tt) (or at the 0/0 apex of
    a zero-depth sample), -2 when the pick or the cut is ambiguous within eps_t (those pairs go through the exact
    fix-up pass and are not part of the tile schedule)."""

    def __init__(self, S, T, geo):
        self.S, self.T = S, T
        tt = (np.arange(S) * geo.dt * 1e6) / 1.0e6          # migrationlib: travel_time [us] / 1e6
        dist = (np.arange(T) * geo.dx / 1e3) * 1.0e3        # dist [km] * 1e3
        vel = geo.vel
        tmax, tt0 = tt.max(), tt[0]
        dxm = (dist[T - 1] - dist[0]) / (T - 1)
        maxdev_d = float(np.max(np.abs(dist - (dist[0] + np.arange(T) * dxm))))
        eps_t = (2.0 / vel) * (2.0 * maxdev_d) + 1e-15 * (abs(tmax) + abs(tt0))
        amax = int(min(float(T - 1), np.floor(vel * tmax / 2.0 / dxm) + 2.0))
        A1 = max(amax, 0) + 1
        zs = vel * tt / 2.0
        zs2 = zs * zs
        d = np.arange(A1) * dxm
        self.A1 = A1
        self.k = np.empty((S, A1), dtype=np.int32)
        for r0 in range(0, S, 256):
            r1 = min(S, r0 + 256)
            rs = np.sqrt(d[None, :] * d[None, :] + zs2[r0:r1, None])
            t = 2.0 * rs / vel
            in_lo = ~((t - eps_t) > tmax)
            in_hi = ~((t + eps_t) > tmax)
            k = _pick(tt, t)
            amb = in_lo & (~in_hi | (_pick(tt, t - eps_t) != _pick(tt, t + eps_t)))
            apex = (rs == 0.0) & (zs[r0:r1, None] == 0.0)
            k = np.where(amb, -2, k)
            k = np.where(~in_lo | apex, -1, k)
            self.k[r0:r1] = k

    def ambiguous(self):
        return int(np.sum(self.k == -2))

    def intervals(self, s_begin, s_end, aligned=False):
        """kirch_tile_sched_kernel: widest [mlo, mhi] interval (mhi - mlo) of every block of KT_Q output rows of
        [s_begin, s_end); blocks start at s_begin, or at absolute multiples of KT_Q clipped to the range (aligned)."""
        starts = list(range((s_begin // KT_Q) * KT_Q if aligned else s_begin, s_end, KT_Q))
        m = np.broadcast_to(np.arange(self.A1), (KT_Q, self.A1))
        widths = []
        for t0 in starts:
            a, b = max(t0, s_begin), min(t0 + KT_Q, s_end)
            k = self.k[a:b]
            ok = k >= 0
            kk, mm = k[ok], m[:b - a][ok]
            if kk.size == 0:
                widths.append(-1)
                continue
            lo = np.full(self.S, np.iinfo(np.int32).max, dtype=np.int64)
            hi = np.full(self.S, -1, dtype=np.int64)
            np.minimum.at(lo, kk, mm)
            np.maximum.at(hi, kk, mm)
            used = hi >= 0
            widths.append(int(np.max(hi[used] - lo[used])))
        return np.array(widths)

    def widest(self, s_begin=0, s_end=None, aligned=False):
        return int(self.intervals(s_begin, self.S if s_end is None else s_end, aligned).max())


@functools.lru_cache(maxsize=None)
def kirch_table(S, T, name):
    return KirchTable(S, T, GEOMETRIES[name] if isinstance(name, str) else name)


def stand_in_items(rows, ntr):
    """Work items of the gather kernel standing in for the tile kernel (kirchhoff.cu: rows x blocks of 512 traces)."""
    return rows * -(-ntr // 512)


BOUNDARY_S, BOUNDARY_T = 2048, 4096


@functools.lru_cache(maxsize=None)
def boundary_geometry():
    """A trace spacing at which the widest interval of the one-launch partition (blocks from row 0) and that of the
    bottom chunk of a row chunking (blocks from r0) sit on different sides of KT_SPAN.  The bottom chunk runs first in a
    bottom-up sequence, so a stand-down decision taken per launch from the chunk's own blocks would differ between the
    two decompositions.  Bisects dx between 5 m (widest 56) and 1 m (widest 282) for the crossing of the one-launch
    partition, then looks for a chunk boundary r0 = S (n - 1) / n (the bottom chunk of an n-chunk host pipeline) whose
    partition lies on the other side.  Returns (dx, r0, n, widest from 0, widest from r0)."""
    S, T = BOUNDARY_S, BOUNDARY_T

    def widths(dx):
        tab = KirchTable(S, T, Geo(1e-8, dx, 1.69e8))
        return tab, tab.widest(0, S)

    lo, hi = 1.0, 5.0        # widest(lo) > KT_SPAN >= widest(hi)
    for _ in range(40):
        mid = 0.5 * (lo + hi)
        if widths(mid)[1] > KT_SPAN:
            lo = mid
        else:
            hi = mid
        if hi - lo < 1e-9:
            break
    for dx in (lo, hi):
        tab, w0 = widths(dx)
        for n in range(2, 33):
            r0 = S * (n - 1) // n
            if r0 % KT_Q == 0:
                continue
            wr = tab.widest(r0, S)
            if (w0 > KT_SPAN) != (wr > KT_SPAN):
                return dx, r0, n, w0, wr
    raise AssertionError("no chunk boundary separates the two partitions near dx = %.6f" % lo)


# ------------------------------------------------------------------------------------------------------ CPU: regimes
def test_geometry_rho():
    assert abs(rho(GEOMETRIES["G0"]) - 0.169) < 1e-12
    assert abs(rho(GEOMETRIES["G1"]) - 0.845) < 1e-12
    assert abs(rho(GEOMETRIES["G2"]) - 1.69) < 1e-12
    assert rho(GEOMETRIES["G3"]) == 1.0
    assert abs(rho(GEOMETRIES["G4"]) - 0.0169) < 1e-12


def test_phase_shift_regimes():
    """G0 keeps most bins of every column; G1 keeps at least ~15 %; G2 has fully evanescent columns, columns with one
    partial stage and a Nyquist-only column; G3 has an exact tie at every k / T == |f| / nt."""
    c0 = phsh_column_census(512, 512, GEOMETRIES["G0"])
    assert c0["min_fraction"] > 0.8 and c0["evanescent"] == c0["partial"] == c0["nyquist_only"] == 0
    c1 = phsh_column_census(512, 512, GEOMETRIES["G1"])
    assert 0.1 < c1["min_fraction"] < 0.5 and c1["evanescent"] == 0
    c2 = phsh_column_census(512, 512, GEOMETRIES["G2"])
    print("G2 512x512:", c2)
    assert c2["evanescent"] == 105 and c2["partial"] == 8 and c2["nyquist_only"] == 1
    for S, T in ((512, 256), (300, 257), (1024, 130), (70, 33), (5000, 40)):
        c = phsh_column_census(S, T, GEOMETRIES["G2"])
        assert c["evanescent"] > 0, (S, T, c)
    c3 = phsh_column_census(512, 512, GEOMETRIES["G3"])
    assert c3["ties"] >= c3["nt"] - 1 == 511
    assert phsh_column_census(256, 256, GEOMETRIES["G3"])["ties"] == 255
    assert c3["evanescent"] == 1       # the Nyquist kx column: its one candidate, the Nyquist frequency, is a tie


def test_stolt_regimes():
    """Whole kx columns are clamped to the last w node at G2 (and none at G0)."""
    assert stolt_clamped_columns(512, 768, GEOMETRIES["G0"]) == 0
    for S, T in ((512, 768), (333, 200), (500, 1026), (1024, 8192)):
        assert stolt_clamped_columns(S, T, GEOMETRIES["G2"]) > 0, (S, T)


def test_kirchhoff_tile_regimes():
    """At 2048 x 4096 the widest offset interval of a tile block stays within KT_SPAN at G0 and G4 and exceeds it at G1
    and G2, where the gather kernel's stand-in grid (16 CTAs per SM) strides over more items than it holds."""
    S, T = 2048, 4096
    widest = {n: kirch_table(S, T, n).widest() for n in ("G0", "G1", "G2", "G3", "G4")}
    print("widest tile interval at %dx%d:" % (S, T), widest)
    assert widest["G0"] <= KT_SPAN and widest["G4"] <= KT_SPAN
    assert widest["G1"] > KT_SPAN and widest["G2"] > KT_SPAN
    assert 50 <= widest["G0"] <= 60 and widest["G1"] > 250
    assert stand_in_items(S, T) > 16 * NUM_SMS
    # sparse traces: at 300 samples the aperture is a few traces, a table row much narrower than a warp
    assert kirch_table(300, 257, "G4").A1 <= 8 and kirch_table(S, T, "G4").A1 < 64
    # exact half-sample ties of the nearest-sample pick at G3 go through the ambiguous-entry list
    assert kirch_table(S, T, "G3").ambiguous() > 0


def test_kirchhoff_boundary_geometry():
    """The boundary geometry exists: the one-launch partition and the bottom chunk's own partition disagree about the
    stand-down, while the partition into aligned blocks (absolute multiples of KT_Q, clipped to a chunk) of any chunk
    never has a wider interval than the whole image's."""
    dx, r0, n, w0, wr = boundary_geometry()
    print("boundary geometry: dx %.9f m, bottom chunk from row %d (%d chunks): widest %d from 0, %d from r0"
          % (dx, r0, n, w0, wr))
    assert max(w0, wr) > KT_SPAN >= min(w0, wr)
    tab = KirchTable(BOUNDARY_S, BOUNDARY_T, Geo(1e-8, dx, 1.69e8))
    whole = tab.widest(0, BOUNDARY_S, aligned=True)
    for a, b in ((r0, BOUNDARY_S), (700, 1500), (3, 700)):
        assert tab.widest(a, b, aligned=True) <= whole


# ----------------------------------------------------------------------------------------------- GPU: oracle parity
PHSH_GEOS = ("G0", "G1", "G2", "G3")


@pytest.mark.gpu
@pytest.mark.parametrize("S,T", [(512, 256), (512, 512), (256, 256), (300, 257), (1024, 130), (70, 33), (5000, 40)])
@pytest.mark.parametrize("geo", PHSH_GEOS)
def test_phase_shift_const_geometry(geo, S, T):
    """Constant velocity through the tensor-core kernel (0), the SIMT pair kernel (3) and the first-generation kernel
    (1) against the float64 oracle."""
    import torch
    from impdar_b200 import migrationlib as ml, _lib
    from oracle import migration as om
    g = GEOMETRIES[geo]
    lib = _lib.load()
    d = _dat(S, T, g, seed=S * 7 + T)
    _, want = om.phase_shift(d.data.astype(np.float64), g.dt, d.travel_time, d.trace_int, d.dist, g.vel, 10, 10)
    xd = torch.from_numpy(d.data).cuda()
    for mode, name in ((0, "tensor-core"), (3, "simt pair"), (1, "first gen")):
        lib.impdar_phsh_set_legacy(mode)
        try:
            got = ml.phase_shift_device(xd, g.dt, g.dx, d.travel_time, g.vel, 10, 10).double().cpu().numpy()
        finally:
            lib.impdar_phsh_set_legacy(0)
        assert _report("phsh const %s %dx%d %s" % (geo, S, T, name), got, want) < TOL, name


def _layered_table(travel_time_us, geo):
    from impdar_b200 import synthetic
    return synthetic.layered_velocity(travel_time_us, v0=geo.vel, v1=geo.vel * (2.3 / 1.69))


@pytest.mark.gpu
@pytest.mark.parametrize("S,T", [(256, 96), (300, 257), (512, 512)])
@pytest.mark.parametrize("geo", PHSH_GEOS)
def test_phase_shift_layered_geometry(geo, S, T):
    """Layered v(z): pair kernel + Nyquist kernel (mode 0) and the first-generation kernel (mode 1)."""
    import torch
    from impdar_b200 import migrationlib as ml, _lib
    from oracle import migration as om
    g = GEOMETRIES[geo]
    lib = _lib.load()
    d = _dat(S, T, g, seed=S * 11 + T)
    table = _layered_table(d.travel_time, g)
    _, want = om.phase_shift(d.data.astype(np.float64), g.dt, d.travel_time, d.trace_int, d.dist, table, 10, 10)
    vmig = ml.getVelocityProfile(d, table)
    xd = torch.from_numpy(d.data).cuda()
    for mode, name in ((0, "pair"), (1, "first gen")):
        lib.impdar_phsh_set_legacy(mode)
        try:
            got = ml.phase_shift_device(xd, g.dt, g.dx, d.travel_time, vmig, 10, 10).double().cpu().numpy()
        finally:
            lib.impdar_phsh_set_legacy(0)
        assert _report("phsh layered %s %dx%d %s" % (geo, S, T, name), got, want) < TOL, name


def _stolt_case(geo, S, T, pipeline, expect):
    import torch
    from impdar_b200 import migrationlib as ml
    from oracle import migration as om
    g = GEOMETRIES[geo]
    d = _dat(S, T, g, seed=S * 3 + T)
    _, want = om.stolt(d.data.astype(np.float64), g.dt, d.trace_int, d.dist, g.vel, 10, 12)
    ml.set_stolt_pipeline(pipeline)
    try:
        got = ml.stolt_device(torch.from_numpy(d.data).cuda(), g.dt, g.dx, g.vel, 10, 12).double().cpu().numpy()
        assert ml.stolt_last_pipeline() == expect
    finally:
        ml.set_stolt_pipeline(ml.STOLT_AUTO)
    assert _report("stolt %s %dx%d %s" % (geo, S, T, expect), got, want) < TOL


@pytest.mark.gpu
@pytest.mark.parametrize("S,T", [(512, 768), (333, 200), (500, 1026)])
@pytest.mark.parametrize("geo", PHSH_GEOS)
def test_stolt_cufft_geometry(geo, S, T):
    from impdar_b200 import migrationlib as ml
    _stolt_case(geo, S, T, ml.STOLT_CUFFT_R2C, "cufft_r2c")
    paired = S % 2 == 0 and T % 2 == 0        # the paired-trace pipeline covers even shapes; odd ones stay on R2C
    _stolt_case(geo, S, T, ml.STOLT_CUFFT_PAIRED, "cufft_paired" if paired else "cufft_r2c")


@pytest.mark.gpu
@pytest.mark.parametrize("geo", PHSH_GEOS)
def test_stolt_five_pass_geometry(geo):
    """1024 x 8192: the smallest shape the hand-written five-pass transform covers."""
    from impdar_b200 import migrationlib as ml
    _stolt_case(geo, 1024, 8192, ml.STOLT_FIVE_PASS, "five_pass")


def _lateral_table(d, geo):
    """(v, z, x) table: the layered profile, 2 % faster on one side of the profile than on the other in its deepest
    fifth.  (The reference's explicit finite-difference term grows without bound at w ~ 0 wherever v varies laterally:
    confined to the deep rows it stays finite.)"""
    tt = d.travel_time
    zmax = geo.vel * (2.3 / 1.69) * tt[-1] * 1e-6 / 2
    z = np.linspace(0, 1.05 * zmax, 24)
    v = geo.vel + (geo.vel * (2.3 / 1.69) - geo.vel) * np.exp(-z / (0.15 * zmax))
    x0, x1 = float(d.dist.min()), float(d.dist.max())
    rows = []
    for i, x in enumerate((x0 - 0.01, 0.5 * (x0 + x1), x1 + 0.01)):
        rows.append(np.stack([v * (1.0 + 0.01 * (i - 1) * (z >= 0.8 * zmax)), z, np.full_like(z, x)], 1))
    return np.concatenate(rows)


@pytest.mark.gpu
@pytest.mark.parametrize("S,T", [(33, 1), (64, 33), (64, 1100), (40, 2049)])
@pytest.mark.parametrize("geo", ("G0", "G2"))
def test_phase_shift_lateral_geometry(geo, S, T):
    """Laterally varying v(x, z) (Fourier finite difference), float64 end to end: one trace (its own branch of the chain
    kernel), and tnum > 1024 (several traces per thread)."""
    from impdar_b200 import migrationlib as ml
    from oracle import migration as om
    g = GEOMETRIES[geo]
    d = _dat(S, T, g, seed=S * 5 + T)
    d.dist = d.dist + 0.1                      # a one-trace profile at 0 km reads as "distance never set"
    table = _lateral_table(d, g)
    x64 = d.data.astype(np.float64)
    _, want = om.phase_shift(x64, g.dt, d.travel_time, d.trace_int, d.dist, table, 5, 7)
    ml.migrationPhaseShift(d, vel=table, htaper=5, vtaper=7)
    assert d.data.dtype == np.float64 and d.data.shape == want.shape
    assert np.isfinite(want).all() and (T == 1 or np.abs(want).max() > 0)   # one trace: the edge taper zeroes it
    assert _report("phsh lateral %s %dx%d" % (geo, S, T), d.data, want) < TOL_FFD


KIRCH_MODES = (("auto", 0), ("general", 1), ("table_gather", 3))


def _expected_kernel(mode, nearfield, S, T, geo):
    if mode == "general":
        return "general"
    if mode == "table_gather" or nearfield:
        return "table_gather"
    return "table_gather" if kirch_table(S, T, geo).widest() > KT_SPAN else "table_tile"


@pytest.mark.gpu
@pytest.mark.parametrize("S,T", [(300, 257), (257, 300)])
@pytest.mark.parametrize("nearfield", [False, True])
@pytest.mark.parametrize("geo", tuple(GEOMETRIES))
def test_kirchhoff_full_geometry(geo, nearfield, S, T):
    import torch
    from impdar_b200 import migrationlib as ml
    from oracle import migration as om
    g = GEOMETRIES[geo]
    d = _dat(S, T, g, seed=S + 13 * T)
    want = om.kirchhoff(d.data.astype(np.float64), d.travel_time, d.dist, g.vel, nearfield)
    xd = torch.from_numpy(d.data).cuda()
    for name, mode in KIRCH_MODES:
        ml.set_kirchhoff_mode(mode)
        try:
            got = ml.kirchhoff_device(xd, d.travel_time, d.dist, g.vel, nearfield)
            kernel = ml.kirchhoff_last_kernel()
        finally:
            ml.set_kirchhoff_mode(ml.KIRCHHOFF_AUTO)
        assert kernel == _expected_kernel(name, nearfield, S, T, geo)
        assert _report("kirch %s %dx%d nf=%d %s" % (geo, S, T, nearfield, kernel), got.cpu().numpy(), want) < TOL


@pytest.mark.gpu
@pytest.mark.parametrize("nearfield", [False, True])
@pytest.mark.parametrize("geo", tuple(GEOMETRIES))
def test_kirchhoff_config2_geometry(geo, nearfield):
    """The config-2 shape (2048 x 4096): first / interior / last output-trace blocks, all rows, against the sparse
    oracle; the far-field kernel is the one the CPU restatement of the schedule predicts (tile at G0 and G4, the gather
    stand-in at G1 and G2)."""
    import torch
    from impdar_b200 import migrationlib as ml
    from oracle import migration as om
    S, T = 2048, 4096
    g = GEOMETRIES[geo]
    d = _dat(S, T, g, seed=71)
    xd = torch.from_numpy(d.data).cuda()
    blocks = [(0, 3), (2046, 2050), (T - 3, T)] if not nearfield else [(1000, 1003)]
    if geo in ("G0", "G4", "G1", "G2"):
        assert _expected_kernel("auto", False, S, T, geo) == ("table_tile" if geo in ("G0", "G4") else "table_gather")
    for xb, xe in blocks:
        want = om.kirchhoff_sparse(d.data, d.travel_time, d.dist, g.vel, nearfield, range(xb, xe))
        for name, mode in KIRCH_MODES:
            ml.set_kirchhoff_mode(mode)
            try:
                got = ml.kirchhoff_device(xd, d.travel_time, d.dist, g.vel, nearfield, xb, xe)
                kernel = ml.kirchhoff_last_kernel()
            finally:
                ml.set_kirchhoff_mode(ml.KIRCHHOFF_AUTO)
            assert kernel == _expected_kernel(name, nearfield, S, T, geo)
            assert _report("kirch %s 2048x4096 nf=%d [%d,%d) %s" % (geo, nearfield, xb, xe, kernel),
                           got.cpu().numpy(), want) < TOL


# ------------------------------------------------------------------- GPU: the same image gives the same bits however cut
def _rows_image(ml, x, tt, dist, vel, chunks, xb=0, xe=None):
    import torch
    S, T = x.shape
    xe = T if xe is None else xe
    out = torch.empty((S, xe - xb), dtype=torch.float32, device="cuda")
    g_hi = S
    for r0, r1 in sorted(chunks, reverse=True):
        ml.kirchhoff_rows_device(x, tt, dist, vel, False, xb, xe, r0, r1, g_hi, out)
        g_hi = r0
    return out


def _window_image(ml, parallel, x, tt, dist, vel, chunks, world=4):
    import torch
    S, T = x.shape
    image = torch.full((S, T), float('nan'), dtype=torch.float32, device="cuda")
    for xb, xe in parallel.kirchhoff_output_ranges(T, world, tt, dist, vel):
        c0, c1 = ml.kirchhoff_input_window(S, tt, dist, vel, xb, xe)
        win = x[:, c0:c1].contiguous()
        g_hi = S
        for r0, r1 in sorted(chunks, reverse=True):
            ml.kirchhoff_window_device(win, c0, T, tt, dist, vel, False, xb, xe, image[:, xb:xe], (r0, r1, g_hi))
            g_hi = r0
    return image


def _assert_cut_invariant(x_np, tt, dist, vel, chunkings, host_chunks, label):
    import torch
    from impdar_b200 import migrationlib as ml, parallel
    x = torch.from_numpy(x_np).cuda()
    whole = ml.kirchhoff_device(x, tt, dist, vel, False)
    kernel = ml.kirchhoff_last_kernel()
    for chunks in chunkings:
        assert torch.equal(_rows_image(ml, x, tt, dist, vel, chunks), whole), "%s: row chunks %s" % (label, chunks)
    for n in host_chunks:
        got = ml.kirchhoff_host(x_np, tt, dist, vel, False, nchunks=n)
        assert np.array_equal(got, whole.double().cpu().numpy()), "%s: host pipeline, %d chunks" % (label, n)
    assert torch.equal(_window_image(ml, parallel, x, tt, dist, vel, chunkings[0]), whole), "%s: column windows" % label
    return whole, kernel


def _chunkings(S):
    from impdar_b200 import parallel
    return [[(1500, S), (700, 1500), (3, 700), (0, 3)], parallel.row_chunks(S, 4), parallel.row_chunks(S, (1, 2, 3, 3, 2, 1))]


@pytest.mark.gpu
@pytest.mark.parametrize("geo", ("G1", "G2"))
def test_kirchhoff_wide_intervals_cut_invariant(geo):
    """Wide intervals (the tile kernel stands down): row chunks with boundaries off the 28-row grid, the host pipeline and
    four column windows all equal the one-launch image bit for bit."""
    S, T = 2048, 4096
    g = GEOMETRIES[geo]
    d = _dat(S, T, g, seed=81)
    _, kernel = _assert_cut_invariant(d.data, d.travel_time, d.dist, g.vel, _chunkings(S), (8, 5), geo)
    assert kernel == "table_gather"


@pytest.mark.gpu
def test_kirchhoff_standdown_boundary_cut_invariant():
    """The boundary geometry: the one-launch partition and the bottom chunk's own partition lie on different sides of
    KT_SPAN.  The stand-down is decided once per image, so every decomposition still gives the same bits."""
    S, T = BOUNDARY_S, BOUNDARY_T
    dx, r0, n, w0, wr = boundary_geometry()
    d = synthetic_dat(S, T, seed=83, dx=dx)
    chunkings = [[(r0, S), (1000, r0), (0, 1000)]] + _chunkings(S)
    _, kernel = _assert_cut_invariant(d.data, d.travel_time, d.dist, 1.69e8, chunkings, (n,), "boundary dx %.6f" % dx)
    assert kernel == ("table_gather" if w0 > KT_SPAN else "table_tile")


@pytest.mark.gpu
def test_kirchhoff_nonfinite_rows_cut_invariant():
    """NaN in a few rows of the top chunk: the nansum variant and the tile stand-down are decided per output row from
    the deepest non-finite input row, which every decomposition sees the same - so row chunks, the host pipeline and
    column windows (NaN columns in every window) equal the one-launch image bit for bit, and match the oracle."""
    from oracle import migration as om
    S, T = 2048, 4096
    g = GEOMETRIES["G0"]
    d = _dat(S, T, g, seed=85)
    x = d.data.copy()
    x[[2, 3, 200], :] = np.nan
    x[101, 17:19] = np.nan
    whole, kernel = _assert_cut_invariant(x, d.travel_time, d.dist, g.vel, _chunkings(S), (8, 4), "G0 NaN rows")
    assert np.isfinite(whole.cpu().numpy()).all()
    assert kernel == "table_gather"             # the gather kernel did the rows that read non-finite input
    want = om.kirchhoff_sparse(x, d.travel_time, d.dist, g.vel, False, [0, 1000, T - 1])
    assert _report("kirch G0 NaN rows", whole[:, [0, 1000, T - 1]].cpu().numpy(), want) < TOL


@pytest.mark.gpu
def test_kirchhoff_nonfinite_one_window_vs_oracle():
    """NaN confined to one rank's column window: ranks see different non-finite rows, so the sharded image is not
    promised bit for bit (DESIGN.md); it matches the float64 oracle."""
    import torch
    from impdar_b200 import migrationlib as ml, parallel
    from oracle import migration as om
    S, T = 2048, 4096
    g = GEOMETRIES["G0"]
    d = _dat(S, T, g, seed=87)
    x = d.data.copy()
    x[[5, 6], 10:13] = np.nan
    ranges = parallel.kirchhoff_output_ranges(T, 4, d.travel_time, d.dist, g.vel)
    assert ml.kirchhoff_input_window(S, d.travel_time, d.dist, g.vel, *ranges[1])[0] > 12
    image = _window_image(ml, parallel, torch.from_numpy(x).cuda(), d.travel_time, d.dist, g.vel,
                          parallel.row_chunks(S, 4))
    cols = [0, 11, ranges[0][1] - 1, ranges[1][0], T - 1]
    want = om.kirchhoff_sparse(x, d.travel_time, d.dist, g.vel, False, cols)
    assert _report("kirch G0 NaN in one window", image[:, cols].cpu().numpy(), want) < TOL
