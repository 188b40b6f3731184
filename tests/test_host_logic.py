"""Host-side logic of the product (no GPU): argument preparation, dispatch, error behaviour, the seam."""
import sys
from unittest.mock import MagicMock, patch

import numpy as np
import pytest

import impdar_b200
from impdar_b200 import filtering, migrationlib, parallel
from oracle import filtering as of
from oracle import migration as om


def test_gradient_coefficients_match_numpy():
    rng = np.random.default_rng(0)
    f = rng.standard_normal((17, 5))
    for x in (np.arange(17) * 0.01 / 1e6,                    # arange*dt: numpy's non-uniform branch
              np.arange(17) * 0.5,                           # exactly uniform branch
              np.cumsum(0.5 + rng.random(17)),               # irregular
              np.array([0.0, 1.0])):                         # two samples
        ff = f[:len(x)]
        c = migrationlib.gradient_coefficients(x)
        g = np.zeros_like(ff)
        for s in range(len(x)):
            if s > 0:
                g[s] += c[0, s] * ff[s - 1]
            g[s] += c[1, s] * ff[s]
            if s < len(x) - 1:
                g[s] += c[2, s] * ff[s + 1]
        assert np.allclose(g, np.gradient(ff, x, axis=0), rtol=1e-13, atol=0)
    c = migrationlib.gradient_coefficients(np.arange(9) * 0.5)
    assert np.all(c[1, 1:-1] == 0)                           # uniform branch never reads f[s]
    with pytest.raises(ValueError):
        migrationlib.gradient_coefficients(np.array([1.0]))


def test_iir_prepare_matches_scipy_filtfilt():
    from scipy.signal import butter, filtfilt
    b, a = butter(5, [0.04, 0.2], 'bandpass')
    bb, aa, zi, padlen = filtering.iir_prepare(b, a)
    assert padlen == 33 and len(bb) == 11 and aa[0] == 1.0 and len(zi) == 10
    x = np.random.default_rng(1).standard_normal((120, 3))
    assert np.allclose(of.filtfilt_explicit(bb, aa, x, padlen), filtfilt(b, a, x, axis=0), rtol=0, atol=1e-6)
    bb, aa, zi, padlen = filtering.iir_prepare([.25, .25, .25, .25], 1)
    assert padlen == 12 and np.allclose(aa, [1, 0, 0, 0])


def test_hfilt_bounds_like_reference():
    for n1, n2, T in [(0, 100, 400), (-5, 10, 50), (60, 10, 50), (3, 1000, 50), (49, 49, 50)]:
        assert of.hfilt_bounds(n1, n2, T) == (int(max(0, min(n1, T - 1))), int(max(int(max(0, min(n1, T - 1))) + 1, min(n2, T))))


def test_velocity_profile_matches_oracle_and_errors():
    d = impdar_b200.RadarData(np.zeros((10, 20)), dt=1, travel_time=np.arange(10) / 10., dist=np.arange(20), trace_int=1)
    assert migrationlib.getVelocityProfile(d, 1.68e8) == 1.68e8
    layers = np.array([[1.677e8, 0], [1.677e8, 50], [1.2e8, 51], [2.2e8, 100]])
    v = migrationlib.getVelocityProfile(d, layers)
    assert np.allclose(v, om.get_velocity_profile_layered(d.travel_time, layers), rtol=1e-14)
    twod = 1.68e8 * np.ones((10, 2)); twod[:, 1] = 0.
    for bad in (twod, 1.68e8 * np.ones((8,)), 1.68e8 * np.ones((8, 1)), 1.68e8 * np.ones((1, 2)), 1.68e8 * np.ones((8, 4))):
        with pytest.raises(ValueError):
            migrationlib.getVelocityProfile(d, bad)
    d.dist = None
    with pytest.raises(ValueError):
        migrationlib.getVelocityProfile(d, np.ones((5, 3)))


def test_check_data_shape():
    d = impdar_b200.RadarData(np.zeros((10, 20)), dt=1, travel_time=np.arange(10), dist=np.arange(20), trace_int=1)
    migrationlib._check_data_shape(d)
    d.data = np.ones((1, 1))
    with pytest.raises(ValueError):
        migrationlib._check_data_shape(d)


def _dat():
    return impdar_b200.RadarData(np.ones((50, 40)), dt=1e-9, travel_time=0.001 * np.arange(50) + 0.001,
                                 dist=np.arange(40) * 1e-3, trace_int=np.ones(40))


def test_migrate_forwards_exact_kwargs():
    """Mirror of the reference's seam contract, test_RadarDataFiltering.py:291-331."""
    with patch('impdar_b200.migrationlib.migrationKirchhoff') as m:
        d = _dat(); d.migrate(mtype='kirch', vel=10., nearfield=False)
        m.assert_called_with(d, vel=10., nearfield=False)
        assert d.flags.mig == 'kirch'
    with patch('impdar_b200.migrationlib.migrationStolt') as m:
        d = _dat(); d.migrate(mtype='stolt', htaper=1, vtaper=2, vel=999.)
        m.assert_called_with(d, htaper=1, vtaper=2, vel=999.)
    with patch('impdar_b200.migrationlib.migrationPhaseShift') as m:
        d = _dat(); d.migrate(mtype='phsh', vel=1., vel_fn='dummy', htaper=1, vtaper=2)
        m.assert_called_with(d, vel=1., vel_fn='dummy', htaper=1, vtaper=2)
    with patch('impdar_b200.migrationlib.migrationTimeWavenumber') as m:
        d = _dat(); d.migrate(mtype='tk', vel=1., vel_fn='dummy', htaper=1, vtaper=2)
        m.assert_called_with(d, vel=1., vel_fn='dummy', htaper=1, vtaper=2)
    with pytest.raises(ValueError):
        _dat().migrate(mtype='dummy')
    with pytest.raises(Exception):
        _dat().migrate(mtype='su_dummy')


def test_hfilt_wrapper_dispatch():
    """test_RadarDataFiltering.py:249-266."""
    d = _dat(); d.adaptivehfilt = MagicMock()
    d.hfilt(ftype='adaptive', window_size=1000)
    d.adaptivehfilt.assert_called_with(window_size=1000)
    d = _dat(); d.horizontalfilt = MagicMock()
    d.hfilt(ftype='hfilt', bounds=(0, 100))
    d.horizontalfilt.assert_called_with(0, 100)
    with pytest.raises(ValueError):
        _dat().hfilt(ftype='dummy')
    with pytest.raises(ValueError):
        _dat().vertical_band_pass(0.1, 100., filttype='dummy')


def test_no_gpu_means_error_not_fallback():
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        _dat().migrate(mtype='stolt')
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        _dat().horizontalfilt(0, 10)
    # every radargram pass of the index / resampling operations, the denoising filters and the host-to-host Kirchhoff
    # call need the device as well: nothing computes on the CPU
    for call in (lambda d: d.migrate(mtype='kirch'), lambda d: d.reverse(), lambda d: d.crop(2, 'top', 'snum'),
                 lambda d: d.hcrop(3, 'left'), lambda d: d.restack(3), lambda d: d.nmo(0.),
                 lambda d: d.denoise(noise=0.1), lambda d: d.denoise(ftype='median')):
        d = _dat()
        d.trig = np.zeros(d.tnum)
        with pytest.raises(RuntimeError, match="no CPU fallback"):
            call(d)


def test_kirchhoff_ranges_cover_and_balance():
    tt = np.arange(512) * 0.01
    dist = np.arange(4096) * 0.005
    for world in (1, 2, 3, 4, 8):
        r = parallel.kirchhoff_output_ranges(4096, world, tt, dist, 1.69e8)
        assert r[0][0] == 0 and r[-1][1] == 4096
        assert all(r[i][1] == r[i + 1][0] for i in range(world - 1))
        assert all(b % 8 == 0 for b, _ in r)
        cost = parallel.kirchhoff_trace_cost(tt, dist, 1.69e8)
        shares = [cost[b:e].sum() for b, e in r]
        assert max(shares) / (sum(shares) / world) < 1.1
    assert parallel.profiles_for_rank(10, 1, 4) == [1, 5, 9]


@pytest.mark.reference
def test_install_rebinds_reference_seam():
    from oracle._refimport import import_reference
    mig_python, RefRadarData, NoInit = import_reference()
    import impdar.lib.migrationlib as ref_mig
    orig = ref_mig.migrationStolt
    impdar_b200.install()
    try:
        assert ref_mig.migrationStolt is migrationlib.migrationStolt
        assert ref_mig.migrationKirchhoff is migrationlib.migrationKirchhoff
        assert RefRadarData.vertical_band_pass is filtering.vertical_band_pass
        # the reference's own wrapper tests still hold with the backend installed
        with patch('impdar.lib.migrationlib.migrationKirchhoff') as m:
            rd = NoInit.NoInitRadarDataFiltering()
            rd.migrate(mtype='kirch', vel=10., nearfield=False)
            assert m.call_args.kwargs == dict(vel=10., nearfield=False)
        rd = NoInit.NoInitRadarDataFiltering()
        rd.horizontalfilt = MagicMock()
        rd.hfilt(ftype='hfilt', bounds=(0, 100))
        rd.horizontalfilt.assert_called_with(0, 100)
    finally:
        impdar_b200.uninstall()
    assert ref_mig.migrationStolt is orig


def test_peer_image_and_window_address_arithmetic(monkeypatch):
    """The peer-mapped image / window helpers (impdar_b200/parallel.py) hand raw addresses to impdar_copy2d_f32 and to
    the column-window entry: byte offsets, row strides and plain-int conversion (range bounds arrive as numpy integers)
    checked against a recording stand-in of the C library - no GPU involved."""
    import ctypes
    import numpy as np
    import torch
    from impdar_b200 import parallel, device, _lib

    calls = []

    class Lib(object):
        def impdar_copy2d_f32(self, src, lds, dst, ldd, rows, cols, stream):
            for v in (lds, ldd, rows, cols):
                assert type(v) is int
            calls.append((src.value, lds, dst.value, ldd, rows, cols))
            return 0

    monkeypatch.setattr(device, "current_stream_ptr", lambda: ctypes.c_void_p(0))
    monkeypatch.setattr(_lib, "check", lambda rc, *a: None)
    S, T = 16, 40
    img = object.__new__(parallel._PeerImage)
    img.S, img.T, img.src, img.is_src, img.lib, img.address = S, T, 0, True, Lib(), 1 << 20
    out = torch.zeros((S, T), dtype=torch.float32)
    img.copy_rows_to(out, np.int64(2), np.int64(5), np.int64(8), np.int64(24))
    assert calls[-1] == ((1 << 20) + 4 * (2 * T + 8), T, out.data_ptr() + 4 * (2 * T + 8), T, 3, 16)
    view = out[:, 4:]                                        # a column slice of the final image keeps the row stride
    img.copy_rows_to(view, 0, S, 0, 4)
    assert calls[-1] == (1 << 20, T, view.data_ptr(), T, S, 4)
    n = len(calls)
    img.copy_rows_to(out, 3, 3, 0, 4)                        # empty blocks are not issued
    img.copy_rows_to(out, 0, 4, 7, 7)
    assert len(calls) == n
    blk = img.block(np.int64(8), np.int64(24))
    assert blk.data_ptr() == (1 << 20) + 32 and blk.shape == (S, 16) and blk.stride(0) == T and blk.stride(1) == 1
    assert device.ptr(blk).value == blk.data_ptr()

    win = object.__new__(parallel._PeerWindows)
    win.S, win.widths, win.rank, win.src, win.is_src, win.lib = S, [0, 12, 20], 0, 0, True, Lib()
    win.address, win.mapped = 0, {1: 1 << 24, 2: 1 << 25}
    x = torch.zeros((S, T), dtype=torch.float32)
    win.push(x, np.int64(3), np.int64(9), np.int64(4), np.int64(16), 1)
    assert calls[-1] == (x.data_ptr() + 4 * (3 * T + 4), T, (1 << 24) + 4 * 3 * 12, 12, 6, 12)
    try:
        win.push(x, 0, 4, 0, 16, 1)                          # not rank 1's window width
    except AssertionError:
        pass
    else:
        raise AssertionError("push must check the window width")
    win.rank, win.is_src, win.address = 2, False, 1 << 26
    w = win.window()
    assert w.data_ptr() == 1 << 26 and w.shape == (S, 20) and w.stride(0) == 20


def _bench_module():
    import importlib.util
    import os
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    spec = importlib.util.spec_from_file_location("bench_module", os.path.join(root, "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    return bench


def test_bench_config_is_the_same_object_for_both_arms():
    """`bench.py --impl reference` must print the `config` of our arm's line at the same --gpus (the driver compares
    them): both come from Workload.config(), which depends on the workload and the GPU count only."""
    import argparse
    bench = _bench_module()
    args = argparse.Namespace(gpus=1, steps=1, warmup=0, profiles=8, workload='kirchhoff_c5', cpu_samples=0)
    for name, cls in bench.WORKLOADS.items():
        for world in (1, 2, 8):
            ours = cls(args, 0, world).config()                 # what measure() prints on rank 0 of `world` ranks
            ref = cls(args, 0, 1).config(world=world)           # what run_reference() prints with --gpus world
            assert ours == ref and set(ours) == {"workload", "snum", "tnum", "l2", "parallelism"}, (name, world)
    c5 = bench.WORKLOADS["kirchhoff_c5"]
    assert c5(args, 0, 1).config()["parallelism"] != c5(args, 0, 8).config()["parallelism"]
    assert "65536" in c5.name and (c5.S, c5.T) == (8192, 65536)


def test_bench_output_sample_is_bounded_and_the_same_every_run():
    """`bench.py --dump-outputs`: an output larger than its byte share keeps every row at a sorted, seeded choice of
    output traces, the same in every run; an output that fits is written whole; integer outputs become float32."""
    import torch
    bench = _bench_module()
    x = torch.arange(2 * 3 * 1000, dtype=torch.float32).reshape(2, 3, 1000)    # value = row * 1000 + trace
    s = bench.output_sample(x, 2 * 3 * 100 * 4)
    assert s.shape == (2, 3, 100) and s.dtype == np.float32
    cols = s[0, 0].astype(int)
    assert np.all(np.diff(cols) > 0) and np.array_equal(s, x.numpy()[..., cols])
    assert np.array_equal(bench.output_sample(x, 2 * 3 * 100 * 4), s)
    assert np.array_equal(bench.output_sample(x, x.numel() * 4), x.numpy())
    assert bench.output_sample(x.double(), 10 ** 9).dtype == np.float64
    assert bench.output_sample(x.int(), 10 ** 9).dtype == np.float32
    with pytest.raises(ValueError):
        bench.output_sample(x, 2 * 3 * 4 - 1)


def test_bench_dump_of_every_record_line_stays_below_64mb(tmp_path):
    """The records each line carries and the files --dump-outputs writes for them at the real output shapes (zero-stride
    stand-ins of the device outputs): together below 64 MB for every record list."""
    import argparse
    import os
    import torch
    bench = _bench_module()
    for workload, no_records, world, keys in (("kirchhoff_c5", False, 1, ["stolt_65536x8192", "kirchhoff_4096x2048_per_gpu"]),
                                              ("kirchhoff_c5", False, 2, ["kirchhoff_4096x2048_per_gpu"]),
                                              ("kirchhoff_c5", True, 1, []), ("pipeline", False, 1, [])):
        args = argparse.Namespace(workload=workload, no_records=no_records)
        subs = bench.sub_records(args, world)
        assert [k for k, _ in subs] == keys
        budget = bench.dump_budget(1 + len(subs))
        total = 0
        for name, cls in [(workload, bench.WORKLOADS[workload])] + subs:
            shape = (cls.S, cls.T) if workload != "pipeline" else (8, 2 * (cls.S // 2), cls.T)
            fn = os.path.join(str(tmp_path), name + ".npy")
            np.save(fn, bench.output_sample(torch.zeros(()).expand(*shape), budget))
            total += os.path.getsize(fn)
        assert total <= 64 * 1000 * 1000, (workload, world, total)


@pytest.mark.gpu
def test_bench_main_dumps_the_last_timed_step_of_every_record(tmp_path, monkeypatch, capsys):
    """bench.main() with a stand-in workload in every record: the line and every record time --steps steps, and
    --dump-outputs writes the output of the last timed step (3 warm-up steps + 12 timed ones) under each record's name."""
    import json
    import os
    import torch
    bench = _bench_module()

    class Stub(bench.Workload):
        name, S, T = "stub", 64, 48

        def l2_note(self):
            return "inputs in L2; no flush needed"

        def setup(self):
            self.x = torch.arange(self.S * self.T, dtype=torch.float32, device="cuda").reshape(self.S, self.T)
            self.units, self.calls = self.S * self.T, 0

        def step(self):
            self.calls += 1
            self.out = self.x * self.calls

        def roofline(self, ms, hbm_gbs, src):
            return {}

    monkeypatch.setitem(bench.WORKLOADS, "kirchhoff_c5", Stub)
    monkeypatch.setattr(bench, "StoltC5", Stub)
    monkeypatch.setattr(bench, "KirchhoffC2", Stub)
    for k in ("RANK", "LOCAL_RANK", "WORLD_SIZE"):
        monkeypatch.delenv(k, raising=False)
    monkeypatch.setattr(sys, "argv", ["bench.py", "--gpus", "1", "--steps", "12", "--warmup", "0", "--no-cpu-baseline",
                                      "--no-e2e", "--dump-outputs", str(tmp_path)])
    bench.main()
    line = json.loads(capsys.readouterr().out.strip().splitlines()[-1])
    assert line["steps"] == 12 and sorted(line["records"]) == ["kirchhoff_4096x2048_per_gpu", "stolt_65536x8192"]
    assert all(r["steps"] == 12 for r in line["records"].values())
    want = np.arange(64 * 48, dtype=np.float32).reshape(64, 48) * 15
    for name in ("kirchhoff_c5", "stolt_65536x8192", "kirchhoff_4096x2048_per_gpu"):
        got = np.load(os.path.join(str(tmp_path), name + ".npy"))
        assert got.dtype == np.float32 and np.array_equal(got, want), name


def test_kirchhoff_input_window_covers_the_aperture():
    """impdar_kirchhoff_input_window (host arithmetic of the C library; what the multi-GPU exchange sends a rank): the
    window must contain every input column an output trace of the range can read - by distance on any monotone geometry
    (mig_python.py:46-50: 2 r / v <= max(tt)) and by trace count on the fitted uniform grid (the table path reads
    x +- m for m up to the grid aperture) - start on a multiple of four columns and stay inside the radargram."""
    import numpy as np
    from impdar_b200 import migrationlib as ml
    vel = 1.69e8
    rng = np.random.default_rng(4)
    for S, T, dx_m, jitter in [(256, 4000, 0.5, 0.0), (256, 4001, 0.5, 0.3), (512, 3000, 2.0, 0.0), (128, 50, 5.0, 0.2),
                               (300, 2050, 0.25, 0.0)]:
        tt_us = np.arange(S) * 0.01 + 0.003
        d_m = np.arange(T) * dx_m + (jitter * dx_m * (rng.random(T) - 0.5) if jitter else 0.0)
        d_m = np.sort(d_m)
        reach = vel * tt_us.max() * 1e-6 / 2.0
        dxm = (d_m[-1] - d_m[0]) / (T - 1)
        amax = int(min(T - 1, np.floor(reach / dxm) + 2))
        for xb, xe in [(0, 1), (0, T), (T // 3, T // 2), (T - 7, T), (5, 6), (T // 2, min(T // 2 + 257, T))]:
            c0, c1 = ml.kirchhoff_input_window(S, tt_us, d_m / 1e3, vel, xb, xe)
            assert 0 <= c0 <= xb and xe <= c1 <= T and c0 % 4 == 0 and (c1 % 4 == 0 or c1 == T)
            near = np.nonzero((d_m >= d_m[xb] - reach) & (d_m <= d_m[xe - 1] + reach))[0]     # by distance
            assert c0 <= near.min() and near.max() < c1, (S, T, xb, xe)
            assert c0 <= max(xb - amax, 0) and min(xe - 1 + amax, T - 1) < c1, (S, T, xb, xe)  # by trace count
            # and it is a window, not the image, whenever the aperture is short against the profile
            if xe - xb + 2 * amax + 16 < T:
                assert c1 - c0 < T


def test_sharding_partitions_are_exact():
    """Output-trace ranges and row chunks of the multi-GPU Kirchhoff (impdar_b200/parallel.py): contiguous, disjoint,
    covering - whatever the world size, the geometry and the chunk pattern - and the uniform-geometry ranges are equal
    to within one CTA tile."""
    import numpy as np
    from impdar_b200 import parallel
    rng = np.random.default_rng(8)
    for T in (7, 40, 4096, 6002, 65536):
        tt = np.arange(64) * 0.01
        for jitter in (0.0, 0.4):
            d = np.arange(T) * 0.005 + (jitter * 0.005 * (rng.random(T) - 0.5) if jitter else 0.0)
            d = np.sort(d)
            for world in (1, 2, 3, 4, 8):
                r = parallel.kirchhoff_output_ranges(T, world, tt, d, 1.69e8)
                assert len(r) == world and r[0][0] == 0 and r[-1][1] == T
                assert all(type(v) is int for be in r for v in be)
                assert all(r[i][1] == r[i + 1][0] and r[i][0] <= r[i][1] for i in range(world - 1))
                if not jitter and T >= 8 * 256 * world:
                    w = [e - b for b, e in r]
                    assert max(w) - min(w) <= 256 and all(b % 256 == 0 for b, _ in r)
    for S in (1, 5, 24, 1024, 8192):
        for pattern in (1, 2, 4, 7, 5000, (1, 2, 3, 3, 2, 1), (1, 2, 1), (3.5, 0.25, 1), parallel.DEFAULT_CHUNKS):
            c = parallel.row_chunks(S, pattern)
            assert c[0][0] == 0 and c[-1][1] == S and all(c[i][1] == c[i + 1][0] for i in range(len(c) - 1))
            assert all(b < e for b, e in c) and all(type(v) is int for be in c for v in be)
    assert parallel.default_chunks(8192, 65536) == parallel.DEFAULT_CHUNKS
    assert parallel.default_chunks(4096, 16384) == 1
