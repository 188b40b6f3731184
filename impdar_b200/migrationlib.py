"""Host side of the migration hot path: drop-in mirrors of impdar.lib.migrationlib's callables.

Same names, signatures, mutation of ``dat`` and exception types as the reference
(migrationlib/mig_python.py :63 migrationKirchhoff, :126 migrationStolt, :211 migrationPhaseShift,
:290 migrationTimeWavenumber, :543 getVelocityProfile, :646 _check_data_shape).  The arithmetic runs in
libimpdar_b200.so on the current CUDA device; this module only validates, prepares O(snum)/O(tnum)
vectors in float64 numpy and moves buffers.  There is no CPU fallback.
"""
import ctypes
import dataclasses
import time

import numpy as np

from . import _lib, device


# ------------------------------------------------------------------------------------------ helpers
def _check_data_shape(dat):
    """mig_python.py:646-648."""
    shape = tuple(dat.data.shape)
    if len(shape) != 2 or shape[1] != dat.tnum or shape[0] != dat.snum:
        raise ValueError('The input array must be of size (snum, tnum)')


def _np_dtype(data):
    if device.is_device_array(data):
        return None
    return np.asarray(data).dtype


def gradient_coefficients(x):
    """Rows a, b, c (shape (3, n)) of np.gradient(f, x, axis=0)'s stencil g[i] = a f[i-1] + b f[i] + c f[i+1]
    (edge_order=1).  numpy switches to the uniform central difference - which never reads f[i] - when all
    spacings are bit-identical; b == 0 everywhere encodes that branch for the kernel."""
    x = np.asarray(x, dtype=np.float64)
    n = len(x)
    if n < 2:
        raise ValueError("Shape of array too small to calculate a numerical gradient, "
                         "at least (edge_order + 1) elements are required.")
    coef = np.zeros((3, n))
    dx = np.diff(x)
    if n > 2:
        if (dx == dx[0]).all():
            coef[0, 1:-1] = -1.0 / (2. * dx[0])
            coef[2, 1:-1] = 1.0 / (2. * dx[0])
        else:
            dx1 = dx[0:-1]
            dx2 = dx[1:]
            coef[0, 1:-1] = -(dx2) / (dx1 * (dx1 + dx2))
            coef[1, 1:-1] = (dx2 - dx1) / (dx1 * dx2)
            coef[2, 1:-1] = dx1 / (dx2 * (dx1 + dx2))
    coef[1, 0] = -1.0 / dx[0]
    coef[2, 0] = 1.0 / dx[0]
    coef[0, -1] = -1.0 / dx[-1]
    coef[1, -1] = 1.0 / dx[-1]
    return np.ascontiguousarray(coef)


def _mean_trace_spacing(dat):
    """mig_python.py:163-168 (and :262-267, :337-342), quirks included."""
    if np.mean(dat.trace_int) <= 0:
        trace_int = np.gradient(np.asarray(dat.dist, dtype=np.float64))
    else:
        trace_int = dat.trace_int
    return float(np.mean(trace_int))


def _finish(dat, out_dev, np_dtype, was_device, in_torch_dtype=None):
    """Hand the result back the way the input came: a host array of the reference's dtype, or - device-resident lane -
    a CUDA tensor of the INPUT tensor's dtype (a float64 tensor stays float64; the migrations compute in float32, so its
    values are float32-accurate - the documented dtype policy - but the dtype never narrows silently)."""
    if was_device:
        dat.data = out_dev if in_torch_dtype is None or out_dev.dtype == in_torch_dtype else out_dev.to(in_torch_dtype)
    else:
        dat.data = device.to_host(out_dev, np_dtype)
    return dat


def _torch_dtype(data):
    return data.dtype if device.is_device_array(data) else None


# ---------------------------------------------------------------------------------------- Kirchhoff
# Every Kirchhoff entry below takes `vel` as a scalar (the reference's single velocity) or as a length-snum vector of
# RMS velocities, one per output sample (rms_velocity; straight rays: row ti migrates with vel[ti] wherever the
# reference's formula uses vel).  A scalar runs the single-velocity C entries exactly as before.
def _kirch_vel_vector(vel, snum):
    """None for a scalar velocity; otherwise the validated contiguous float64 per-sample vector."""
    if np.ndim(vel) == 0:
        return None
    v = np.ascontiguousarray(device.host_f64(vel))
    if v.shape != (int(snum),):
        raise ValueError('Kirchhoff velocity vector must have one value per sample (%d), got shape %s'
                         % (int(snum), str(v.shape)))
    if not (np.all(np.isfinite(v)) and np.all(v > 0)):
        raise ValueError('Kirchhoff velocity vector must be finite and positive')
    return v


def _kirch_window_vz(lib, win_ptr, col0, ncols, ld, out, S, T, dist_m, tt_sec, coef, v, nearfield, x_begin, x_end,
                     rows):
    s_begin, s_end, g_hi = (0, S, S) if rows is None else rows
    ws = device.workspace(lib.impdar_kirchhoff_workspace_bytes(S, int(T), int(bool(nearfield))))
    rc = lib.impdar_kirchhoff_window_vz_f32(win_ptr, int(col0), int(ncols), int(ld), device.ptr(out), int(out.stride(0)),
                                            S, int(T), device.ptr(dist_m), device.ptr(tt_sec), device.ptr(coef),
                                            device.ptr(v), int(bool(nearfield)), int(x_begin), int(x_end),
                                            int(s_begin), int(s_end), int(g_hi), device.ptr(ws), ws.numel(),
                                            device.current_stream_ptr())
    _lib.check(rc)
    return out


def kirchhoff_device(data_dev, travel_time_us, dist_km, vel, nearfield, x_begin=0, x_end=None, out=None):
    """Run the Kirchhoff kernel on a (snum, tnum) float32 CUDA tensor; returns the (snum, x_end-x_begin)
    float32 block of migrated output traces (the unit of multi-GPU sharding)."""
    import torch
    lib = _lib.load()
    S, T = data_dev.shape
    x_end = T if x_end is None else x_end
    v = _kirch_vel_vector(vel, S)
    tt_sec = device.host_f64(travel_time_us) / 1.0e6                     # mig_python.py:98
    dist_m = np.ascontiguousarray(device.host_f64(dist_km) * 1.0e3)      # :108
    if not np.all(np.diff(tt_sec) > 0):
        raise ValueError('travel_time must be strictly ascending for Kirchhoff migration')
    coef = gradient_coefficients(tt_sec)                                 # np.gradient of :93
    if out is None:
        out = torch.empty((S, x_end - x_begin), dtype=torch.float32, device=data_dev.device)
    if v is not None:   # the whole-image window: any trace order, like impdar_kirchhoff_f32
        return _kirch_window_vz(lib, device.ptr(data_dev), 0, T, T, out, S, T, dist_m, tt_sec, coef, v, nearfield,
                                x_begin, x_end, None)
    nbytes = lib.impdar_kirchhoff_workspace_bytes(S, T, int(bool(nearfield)))
    ws = device.workspace(nbytes)
    rc = lib.impdar_kirchhoff_f32(device.ptr(data_dev), device.ptr(out), S, T, device.ptr(dist_m),
                                  device.ptr(tt_sec), device.ptr(coef), float(vel), int(bool(nearfield)),
                                  int(x_begin), int(x_end), device.ptr(ws), ws.numel(),
                                  device.current_stream_ptr())
    _lib.check(rc)
    return out


def kirchhoff_rows_device(data_dev, travel_time_us, dist_km, vel, nearfield, x_begin, x_end, s_begin, s_end, g_hi, out):
    """Output rows [s_begin, s_end) of the trace range [x_begin, x_end) into the (snum, x_end - x_begin) tensor `out`
    (impdar_kirchhoff_rows_f32).  Only input rows >= s_begin - 1 of `data_dev` need to be valid.  Calls of one image
    go bottom-up on the same stream; g_hi = snum for the first, the previous call's s_begin afterwards.  Raises
    ValueError for irregular trace spacing (use kirchhoff_device)."""
    lib = _lib.load()
    S, T = data_dev.shape
    v = _kirch_vel_vector(vel, S)
    tt_sec = device.host_f64(travel_time_us) / 1.0e6
    dist_m = np.ascontiguousarray(device.host_f64(dist_km) * 1.0e3)
    coef = gradient_coefficients(tt_sec)
    if v is not None:
        return _kirch_window_vz(lib, device.ptr(data_dev), 0, T, T, out, S, T, dist_m, tt_sec, coef, v, nearfield,
                                x_begin, x_end, (s_begin, s_end, g_hi))
    ws = device.workspace(lib.impdar_kirchhoff_workspace_bytes(S, T, int(bool(nearfield))))
    rc = lib.impdar_kirchhoff_rows_f32(device.ptr(data_dev), device.ptr(out), S, T, device.ptr(dist_m),
                                       device.ptr(tt_sec), device.ptr(coef), float(vel), int(bool(nearfield)),
                                       int(x_begin), int(x_end), int(s_begin), int(s_end), int(g_hi),
                                       device.ptr(ws), ws.numel(), device.current_stream_ptr())
    _lib.check(rc)
    return out


def kirchhoff_input_window(snum, travel_time_us, dist_km, vel, x_begin, x_end):
    """[col0, col1): the input columns the output traces [x_begin, x_end) can read (the range plus one aperture each
    side; impdar_kirchhoff_input_window).  Host arithmetic only."""
    lib = _lib.load()
    tt_sec = device.host_f64(travel_time_us) / 1.0e6
    dist_m = np.ascontiguousarray(device.host_f64(dist_km) * 1.0e3)
    c0, c1 = ctypes.c_int(0), ctypes.c_int(0)
    v = _kirch_vel_vector(vel, snum)
    if v is not None:
        _lib.check(lib.impdar_kirchhoff_input_window_vz(int(snum), len(dist_m), device.ptr(dist_m), device.ptr(tt_sec),
                                                        device.ptr(v), int(x_begin), int(x_end), ctypes.byref(c0),
                                                        ctypes.byref(c1)))
        return c0.value, c1.value
    _lib.check(lib.impdar_kirchhoff_input_window(int(snum), len(dist_m), device.ptr(dist_m), device.ptr(tt_sec), float(vel),
                                                 int(x_begin), int(x_end), ctypes.byref(c0), ctypes.byref(c1)))
    return c0.value, c1.value


def kirchhoff_window_device(win_dev, col0, tnum, travel_time_us, dist_km, vel, nearfield, x_begin, x_end, out=None,
                            rows=None):
    """Kirchhoff on a COLUMN WINDOW of the radargram (impdar_kirchhoff_window_f32, the unit of the multi-GPU halo
    exchange): `win_dev` is a (snum, ncols) float32 CUDA tensor (last stride 1, any row stride) holding columns
    [col0, col0 + ncols) of a tnum-trace radargram whose full geometry is given; returns / fills the
    (snum, x_end - x_begin) block `out` (last stride 1, any row stride: a column slice of the final image works).
    rows = (s_begin, s_end, g_hi) runs one chunk of a bottom-up row sequence (see kirchhoff_rows_device).  The result
    equals kirchhoff_device on the whole image bit for bit."""
    import torch
    lib = _lib.load()
    S, ncols = win_dev.shape
    assert win_dev.stride(1) == 1
    tt_sec = device.host_f64(travel_time_us) / 1.0e6
    dist_m = np.ascontiguousarray(device.host_f64(dist_km) * 1.0e3)
    if not np.all(np.diff(tt_sec) > 0):
        raise ValueError('travel_time must be strictly ascending for Kirchhoff migration')
    coef = gradient_coefficients(tt_sec)
    if out is None:
        out = torch.empty((S, x_end - x_begin), dtype=torch.float32, device=win_dev.device)
    assert out.stride(1) == 1 and out.shape == (S, x_end - x_begin)
    v = _kirch_vel_vector(vel, S)
    if v is not None:
        return _kirch_window_vz(lib, device.ptr(win_dev), col0, ncols, win_dev.stride(0), out, S, tnum, dist_m, tt_sec,
                                coef, v, nearfield, x_begin, x_end, rows)
    s_begin, s_end, g_hi = (0, S, S) if rows is None else rows
    ws = device.workspace(lib.impdar_kirchhoff_workspace_bytes(S, int(tnum), int(bool(nearfield))))
    rc = lib.impdar_kirchhoff_window_f32(device.ptr(win_dev), int(col0), int(ncols), int(win_dev.stride(0)),
                                         device.ptr(out), int(out.stride(0)), S, int(tnum), device.ptr(dist_m),
                                         device.ptr(tt_sec), device.ptr(coef), float(vel), int(bool(nearfield)),
                                         int(x_begin), int(x_end), int(s_begin), int(s_end), int(g_hi),
                                         device.ptr(ws), ws.numel(), device.current_stream_ptr())
    _lib.check(rc)
    return out


def kirchhoff_host(data, travel_time_us, dist_km, vel, nearfield, nchunks=None):
    """Host numpy radargram -> host float64 migrated image with upload, kernels and download overlapped in row
    chunks (impdar_kirchhoff_host_pipelined_f64).  The result lives in page-locked memory owned by the array."""
    import torch
    device.require_cuda()
    lib = _lib.load()
    a = np.asarray(data)
    if a.dtype != np.float32 or not a.flags.c_contiguous:
        a = np.ascontiguousarray(a, dtype=np.float32)         # the device path computes in float32
    S, T = a.shape
    v = _kirch_vel_vector(vel, S)
    tt_sec = device.host_f64(travel_time_us) / 1.0e6
    dist_m = np.ascontiguousarray(device.host_f64(dist_km) * 1.0e3)
    if not np.all(np.diff(tt_sec) > 0):
        raise ValueError('travel_time must be strictly ascending for Kirchhoff migration')
    coef = gradient_coefficients(tt_sec)
    if nchunks is None:
        nchunks = 8 if S * T >= (1 << 20) and S >= 64 else 1
    host_out = torch.empty((S, T), dtype=torch.float64, pin_memory=True)
    ws = device.workspace(lib.impdar_kirchhoff_host_workspace_bytes(S, T, int(bool(nearfield))))
    if v is None:
        rc = lib.impdar_kirchhoff_host_pipelined_f64(device.ptr(a), device.ptr(host_out), S, T, device.ptr(dist_m),
                                                     device.ptr(tt_sec), device.ptr(coef), float(vel),
                                                     int(bool(nearfield)), int(nchunks), device.ptr(ws), ws.numel(),
                                                     device.current_stream_ptr())
    else:
        rc = lib.impdar_kirchhoff_host_pipelined_vz_f64(device.ptr(a), device.ptr(host_out), S, T, device.ptr(dist_m),
                                                        device.ptr(tt_sec), device.ptr(coef), device.ptr(v),
                                                        int(bool(nearfield)), int(nchunks), device.ptr(ws), ws.numel(),
                                                        device.current_stream_ptr())
    torch.cuda.current_stream().synchronize()                 # `a` and the vectors stay alive until here
    _lib.check(rc)
    return host_out.numpy()


def migrationKirchhoff(dat, vel=1.69e8, nearfield=False):
    """Kirchhoff diffraction summation; mirrors mig_python.py:63-123 (dat.data becomes float64)."""
    print('Kirchhoff Migration (diffraction summation) of %.0fx%.0f matrix' % (dat.snum, dat.tnum))
    _check_data_shape(dat)
    start = time.time()
    if device.is_device_array(dat.data):
        in_dt = dat.data.dtype
        out = kirchhoff_device(device.to_device(dat.data), dat.travel_time, dat.dist, vel, nearfield)
        dat.data = out if out.dtype == in_dt or not in_dt.is_floating_point else out.to(in_dt)
    else:
        dat.data = kirchhoff_host(dat.data, dat.travel_time, dat.dist, vel, nearfield)
    print('Kirchhoff Migration of %.0fx%.0f matrix complete in %.2f seconds'
          % (dat.snum, dat.tnum, time.time() - start))
    return dat


def rms_velocity(travel_time_us, vmig):
    """RMS velocity per sample from the interval velocity `vmig` (getVelocityProfile's (v, z) result) against two-way
    time: v[i] = sqrt(I[i] / t[i]) with I the trapezoid integral of vmig^2 dt from the first sample at t >= 0 (whose
    own term is vmig^2 t), summed sequentially in float64; samples with t <= 0 (pre-trigger, time zero) keep vmig."""
    t = np.asarray(travel_time_us, dtype=np.float64) / 1.0e6
    vm = np.asarray(vmig, dtype=np.float64)
    if vm.shape != t.shape:
        raise ValueError('vmig must have one value per sample (%d), got shape %s' % (len(t), str(vm.shape)))
    v = vm.copy()
    nonneg = np.nonzero(t >= 0)[0]
    if len(nonneg):
        j0 = nonneg[0]
        v2 = vm[j0:] ** 2
        steps = (v2[1:] + v2[:-1]) / 2. * np.diff(t[j0:])
        integral = np.cumsum(np.concatenate([[v2[0] * t[j0]], steps]))   # sequential, left to right
        pos = t[j0:] > 0
        v[j0:][pos] = np.sqrt(integral[pos] / t[j0:][pos])
    return v


def migrationKirchhoffLayered(dat, vel=1.69e8, vel_fn=None, nearfield=False, **genfromtxt_kwargs):
    """Kirchhoff migration with a depth-varying velocity: `vel` (or the file `vel_fn`, loaded like
    migrationPhaseShift does) is a scalar or a (v, z) table; the table becomes the interval velocity per sample
    (getVelocityProfile) and then the RMS velocity per sample (rms_velocity), and output sample ti migrates with its
    own v[ti] along straight rays.  A scalar is exactly migrationKirchhoff.  dat.data becomes float64 on the host
    lane, a tensor on the device lane.  A lateral (v, z, x) table raises ValueError."""
    if vel_fn is not None:
        try:
            vel = np.genfromtxt(vel_fn, **genfromtxt_kwargs)
            print('Velocities loaded from %s.' % vel_fn)
        except Exception:
            raise TypeError('File %s was given for input velocity array, but cannot be loaded. Please reformat to txt file.' % vel_fn)
    if np.ndim(vel) == 0:
        return migrationKirchhoff(dat, vel=vel, nearfield=nearfield)
    if len(np.shape(vel)) == 2 and np.shape(vel)[1] == 3:
        raise ValueError('Kirchhoff migration takes a (v, z) velocity table; lateral (v, z, x) tables are not supported')
    print('Kirchhoff Migration (diffraction summation, layered velocity) of %.0fx%.0f matrix' % (dat.snum, dat.tnum))
    _check_data_shape(dat)
    start = time.time()
    v = rms_velocity(dat.travel_time, getVelocityProfile(dat, np.asarray(vel, dtype=np.float64)))
    if device.is_device_array(dat.data):
        in_dt = dat.data.dtype
        out = kirchhoff_device(device.to_device(dat.data), dat.travel_time, dat.dist, v, nearfield)
        dat.data = out if out.dtype == in_dt or not in_dt.is_floating_point else out.to(in_dt)
    else:
        dat.data = kirchhoff_host(dat.data, dat.travel_time, dat.dist, v, nearfield)
    print('Kirchhoff Migration of %.0fx%.0f matrix complete in %.2f seconds'
          % (dat.snum, dat.tnum, time.time() - start))
    return dat


def rms_velocity_profiles(travel_time_us, profiles):
    """rms_velocity of each row of a (P, snum) array of interval-velocity profiles.  The same operations along axis 1
    (the cumulative sum runs left to right within each row), so row i equals rms_velocity(travel_time_us, profiles[i])
    bit for bit."""
    t = np.asarray(travel_time_us, dtype=np.float64) / 1.0e6
    vm = np.asarray(profiles, dtype=np.float64)
    if vm.ndim != 2 or vm.shape[1] != t.shape[0]:
        raise ValueError('profiles must have shape (P, %d), got %s' % (len(t), str(vm.shape)))
    v = vm.copy()
    nonneg = np.nonzero(t >= 0)[0]
    if len(nonneg):
        j0 = nonneg[0]
        v2 = vm[:, j0:] ** 2
        steps = (v2[:, 1:] + v2[:, :-1]) / 2. * np.diff(t[j0:])
        integral = np.cumsum(np.concatenate([v2[:, :1] * t[j0], steps], axis=1), axis=1)
        pos = t[j0:] > 0
        v[:, j0:][:, pos] = np.sqrt(integral[:, pos] / t[j0:][pos])
    return v


def _kirch_lateral_args(profiles, col_profile, snum, tnum):
    """Validated contiguous (P, snum) float64 profiles and (tnum,) int32 trace -> profile map."""
    v = np.ascontiguousarray(device.host_f64(profiles))
    if v.ndim != 2 or v.shape[1] != int(snum) or v.shape[0] < 1:
        raise ValueError('Kirchhoff lateral profiles must have shape (P, %d), got %s' % (int(snum), str(v.shape)))
    if not (np.all(np.isfinite(v)) and np.all(v > 0)):
        raise ValueError('Kirchhoff lateral profiles must be finite and positive')
    c = np.asarray(col_profile)
    if c.shape != (int(tnum),) or not (np.issubdtype(c.dtype, np.integer) or c.dtype == bool):
        raise ValueError('col_profile must be an integer array of shape (%d,), got %s %s' % (int(tnum), c.dtype, c.shape))
    if c.size and (c.min() < 0 or c.max() >= v.shape[0]):
        raise ValueError('col_profile values must lie in [0, %d)' % v.shape[0])
    return v, np.ascontiguousarray(c, dtype=np.int32)


def _kirch_window_vxz(lib, win_ptr, col0, ncols, ld, out, S, T, dist_m, tt_sec, coef, profiles, colp, nearfield,
                      x_begin, x_end):
    ws = device.workspace(lib.impdar_kirchhoff_lateral_workspace_bytes(S, int(T), profiles.shape[0],
                                                                       int(bool(nearfield))))
    rc = lib.impdar_kirchhoff_window_vxz_f32(win_ptr, int(col0), int(ncols), int(ld), device.ptr(out),
                                             int(out.stride(0)), S, int(T), device.ptr(dist_m), device.ptr(tt_sec),
                                             device.ptr(coef), device.ptr(profiles), int(profiles.shape[0]),
                                             device.ptr(colp), int(bool(nearfield)), int(x_begin), int(x_end),
                                             device.ptr(ws), ws.numel(), device.current_stream_ptr())
    _lib.check(rc)
    return out


def kirchhoff_lateral_device(data_dev, travel_time_us, dist_km, profiles, col_profile, nearfield, x_begin=0,
                             x_end=None, out=None):
    """Kirchhoff with a laterally varying velocity on a (snum, tnum) float32 CUDA tensor: output trace xi migrates with
    the RMS profile profiles[col_profile[xi]] ((P, snum) velocities, finite and positive); returns the
    (snum, x_end - x_begin) float32 block.  Column xi equals kirchhoff_device's column xi with that profile
    (impdar_kirchhoff_window_vxz_f32)."""
    import torch
    lib = _lib.load()
    S, T = data_dev.shape
    x_end = T if x_end is None else x_end
    v, colp = _kirch_lateral_args(profiles, col_profile, S, T)
    tt_sec = device.host_f64(travel_time_us) / 1.0e6
    dist_m = np.ascontiguousarray(device.host_f64(dist_km) * 1.0e3)
    if not np.all(np.diff(tt_sec) > 0):
        raise ValueError('travel_time must be strictly ascending for Kirchhoff migration')
    coef = gradient_coefficients(tt_sec)
    if out is None:
        out = torch.empty((S, x_end - x_begin), dtype=torch.float32, device=data_dev.device)
    return _kirch_window_vxz(lib, device.ptr(data_dev), 0, T, T, out, S, T, dist_m, tt_sec, coef, v, colp, nearfield,
                             x_begin, x_end)


def lateral_rms_field(dat, vel):
    """(P, snum) RMS profiles and the (tnum,) trace -> profile map of a (v, z, x) table: lateral_velocity_profiles
    then rms_velocity_profiles."""
    profiles, col_profile = lateral_velocity_profiles(dat, np.asarray(vel, dtype=np.float64))
    return rms_velocity_profiles(dat.travel_time, profiles), col_profile


def migrationKirchhoffLateral(dat, vel=1.69e8, vel_fn=None, nearfield=False, **genfromtxt_kwargs):
    """Kirchhoff migration with a laterally varying velocity: a (v, z, x) table (or the file `vel_fn`, loaded like
    migrationKirchhoffLayered does) gives each trace the RMS velocity of its column of getVelocityProfile, and output
    sample (ti, xi) migrates with V[ti, xi] along straight rays.  A scalar or a (v, z) table is exactly
    migrationKirchhoffLayered; a field with a single profile runs the layered path with that vector.  dat.data becomes
    float64 on the host lane, a tensor on the device lane."""
    if vel_fn is not None:
        try:
            vel = np.genfromtxt(vel_fn, **genfromtxt_kwargs)
            print('Velocities loaded from %s.' % vel_fn)
        except Exception:
            raise TypeError('File %s was given for input velocity array, but cannot be loaded. Please reformat to txt file.' % vel_fn)
    if not (len(np.shape(vel)) == 2 and np.shape(vel)[1] == 3):
        return migrationKirchhoffLayered(dat, vel=vel, nearfield=nearfield)
    print('Kirchhoff Migration (diffraction summation, lateral velocity) of %.0fx%.0f matrix' % (dat.snum, dat.tnum))
    _check_data_shape(dat)
    start = time.time()
    profiles, col_profile = lateral_rms_field(dat, vel)
    on_device = device.is_device_array(dat.data)
    if profiles.shape[0] == 1:
        v = profiles[0]
        if on_device:
            in_dt = dat.data.dtype
            out = kirchhoff_device(device.to_device(dat.data), dat.travel_time, dat.dist, v, nearfield)
            dat.data = out if out.dtype == in_dt or not in_dt.is_floating_point else out.to(in_dt)
        else:
            dat.data = kirchhoff_host(dat.data, dat.travel_time, dat.dist, v, nearfield)
    elif on_device:
        in_dt = dat.data.dtype
        out = kirchhoff_lateral_device(device.to_device(dat.data), dat.travel_time, dat.dist, profiles, col_profile,
                                       nearfield)
        dat.data = out if out.dtype == in_dt or not in_dt.is_floating_point else out.to(in_dt)
    else:   # upload, migrate, download back to back; float32 results widened like kirchhoff_host's
        device.require_cuda()
        x = device.to_device(np.asarray(dat.data))
        out = kirchhoff_lateral_device(x, dat.travel_time, dat.dist, profiles, col_profile, nearfield)
        dat.data = out.cpu().numpy().astype(np.float64)
    print('Kirchhoff Migration of %.0fx%.0f matrix complete in %.2f seconds'
          % (dat.snum, dat.tnum, time.time() - start))
    return dat


def kirchhoff_stats():
    """(pairs, exact_pairs) of the last Kirchhoff call (needs enable_kirchhoff_stats(True) beforehand)."""
    lib = _lib.load()
    a = ctypes.c_ulonglong(0)
    b = ctypes.c_ulonglong(0)
    _lib.check(lib.impdar_kirchhoff_last_stats(ctypes.byref(a), ctypes.byref(b)), RuntimeError)
    return a.value, b.value


def enable_kirchhoff_stats(on=True):
    _lib.check(_lib.load().impdar_kirchhoff_enable_stats(int(bool(on))))


KIRCHHOFF_AUTO, KIRCHHOFF_GENERAL, KIRCHHOFF_TABLE, KIRCHHOFF_TABLE_GATHER = 0, 1, 2, 3


def set_kirchhoff_mode(mode=KIRCHHOFF_AUTO):
    """Kernel selection: AUTO picks the uniform-geometry table path when the trace spacing is uniform and the
    general-geometry kernel otherwise; GENERAL / TABLE force one (TABLE raises ValueError on irregular spacing).  On the
    table path the far-field sum runs in the shared-memory tile kernel (kirchhoff_tile.cuh); TABLE_GATHER keeps the
    global-gather table kernel for everything (A/B runs, and what near field / non-finite input use anyway)."""
    _lib.check(_lib.load().impdar_kirchhoff_set_mode(int(mode)))


def kirchhoff_last_path():
    """'general' or 'table': which path the last Kirchhoff call ran."""
    return {1: 'general', 2: 'table', 3: 'table', 4: 'general'}.get(_lib.load().impdar_kirchhoff_last_path(), 'none')


def kirchhoff_last_kernel():
    """'general', 'general_lateral', 'table_gather' or 'table_tile' - the kernel that did the far-field sum of the last
    call ('table_tile' only if the tile kernel did all of it - for a lateral field, in every run; it stands down for
    hyperbola intervals wider than its staged segments, and leaves the rows that read non-finite input to the gather
    kernel).  Synchronises the call's stream."""
    lib = _lib.load()
    path = lib.impdar_kirchhoff_last_path()
    if path != 3:
        return {1: 'general', 2: 'table_gather', 4: 'general_lateral'}.get(path, 'none')
    v = ctypes.c_int(0)
    _lib.check(lib.impdar_kirchhoff_last_tile_standdown(ctypes.byref(v)), RuntimeError)
    return 'table_gather' if v.value else 'table_tile'


# -------------------------------------------------------------------------------------------- Stolt
def stolt_device(data_dev, dt, dx, vel, htaper, vtaper, trunc_int=False, out=None):
    """(batch, snum, tnum) or (snum, tnum) float32 CUDA tensor -> migrated (.., 2*(snum//2), tnum)."""
    import torch
    lib = _lib.load()
    squeeze = data_dev.dim() == 2
    x = data_dev.unsqueeze(0) if squeeze else data_dev
    B, S, T = x.shape
    S2 = 2 * (S // 2)
    if out is None:
        out = torch.empty((B, S2, T), dtype=torch.float32, device=x.device)
    ws = device.workspace(lib.impdar_stolt_workspace_bytes(S, T, B))
    rc = lib.impdar_stolt_f32(device.ptr(x), device.ptr(out), S, T, B, float(dt), float(dx), float(vel),
                              float(htaper) if htaper != 0 else 0.0, float(vtaper) if vtaper != 0 else 0.0,
                              int(bool(trunc_int)), device.ptr(ws), ws.numel(), device.current_stream_ptr())
    _lib.check(rc)
    return out[0] if squeeze else out


def stolt_force_generic(on=True):
    """Testing hook: force the generic R2C/C2R Stolt pipeline even where the paired-trace C2C pipeline applies."""
    _lib.check(_lib.load().impdar_stolt_force_r2c(int(bool(on))))


STOLT_AUTO, STOLT_CUFFT_R2C, STOLT_CUFFT_PAIRED, STOLT_FIVE_PASS = 0, 1, 2, 3


def set_stolt_pipeline(mode=STOLT_AUTO):
    """Pipeline selection (testing / benchmarking): AUTO runs the five-pass hand-written transform kernels for the
    power-of-two shapes they cover and the cuFFT pipelines otherwise."""
    _lib.check(_lib.load().impdar_stolt_set_pipeline(int(mode)))


def stolt_last_pipeline():
    return {1: 'cufft_r2c', 2: 'cufft_paired', 3: 'five_pass'}.get(_lib.load().impdar_stolt_last_pipeline(), 'none')


def migrationStolt(dat, vel=1.68e8, htaper=100, vtaper=1000):
    """Stolt f-k migration; mirrors mig_python.py:126-208 (output has 2*(snum//2) rows, :202)."""
    print('Stolt Migration (f-k migration) of %.0fx%.0f matrix' % (dat.snum, dat.tnum))
    _check_data_shape(dat)
    start = time.time()
    was_device = device.is_device_array(dat.data)
    in_dtype = _np_dtype(dat.data)
    trunc_int = in_dtype is not None and np.issubdtype(in_dtype, np.integer)  # .astype(dat.data.dtype), :157
    out_dtype = np.float32 if in_dtype == np.float32 else np.float64         # dtype of np.fft.irfft2
    in_tdt = _torch_dtype(dat.data)
    x = device.to_device(dat.data)
    out = stolt_device(x, dat.dt, _mean_trace_spacing(dat), vel, htaper, vtaper, trunc_int)
    _finish(dat, out, out_dtype, was_device, in_tdt)
    print('Stolt Migration of %.0fx%.0f matrix complete in %.2f seconds'
          % (dat.snum, dat.tnum, time.time() - start))
    return dat


# -------------------------------------------------------------------------------- migration velocity scan
# Constant-velocity Stolt images over a velocity grid, one focus measure per image window (n E4 / E2^2, the varimax),
# and the best velocity per window.  Constant-velocity time migration focuses a diffraction with apex time t0 when the
# velocity equals the hyperbola's straight-ray RMS velocity at t0, the model the layered and lateral Kirchhoff kernels
# take, so the picks feed kirchhoff_device / kirchhoff_lateral_device directly (scan_rms_field).
def _scan_vels(vels):
    try:
        v = np.array(vels, dtype=np.float64)
    except (TypeError, ValueError):
        raise ValueError('scan velocities must be a 1-D array of numbers')
    if v.ndim != 1 or v.size == 0:
        raise ValueError('scan velocities must be a non-empty 1-D array, got shape %s' % (v.shape,))
    if not (np.all(np.isfinite(v)) and np.all(v > 0)):
        raise ValueError('scan velocities must be finite and positive')
    return np.ascontiguousarray(v)


def _scan_window(window):
    try:
        ws, wt = window
    except (TypeError, ValueError):
        raise ValueError('window must be a pair (rows, traces), got %r' % (window,))
    out = []
    for w in (ws, wt):
        if isinstance(w, (bool, np.bool_)) or not isinstance(w, (int, np.integer)) or w < 1:
            raise ValueError('window sizes must be integers >= 1, got %r' % (window,))
        out.append(int(w))
    return tuple(out)


def stolt_scan_device(data_dev, dt, dx, vels, htaper, vtaper, window, trunc_int=False, images=None):
    """Focus panel of a Stolt velocity scan of a (snum, tnum) float32 CUDA tensor: returns the (nv, nws, nwt) float64
    focus tensor (impdar_stolt_scan_f32).  `images`, a (nv, 2*(snum//2), tnum) float32 CUDA tensor, receives each
    velocity's image, equal to stolt_device at that velocity; without it no image-sized buffer is allocated per velocity."""
    import torch
    v = _scan_vels(vels)
    ws, wt = _scan_window(window)
    if not (device.is_device_array(data_dev) and data_dev.dim() == 2 and data_dev.dtype == torch.float32):
        raise ValueError('stolt_scan_device needs a 2-D float32 CUDA tensor')
    lib = _lib.load()
    x = data_dev.contiguous()
    S, T = x.shape
    S2 = 2 * (S // 2)
    if images is not None and not (device.is_device_array(images) and images.dtype == torch.float32
                                   and tuple(images.shape) == (len(v), S2, T) and images.is_contiguous()):
        raise ValueError('images must be a contiguous float32 CUDA tensor of shape %s' % ((len(v), S2, T),))
    focus = torch.empty((len(v), -(-S2 // ws), -(-T // wt)), dtype=torch.float64, device=x.device)
    wsb = device.workspace(lib.impdar_stolt_scan_workspace_bytes(S, T, len(v)))
    rc = lib.impdar_stolt_scan_f32(device.ptr(x), S, T, float(dt), float(dx), v.ctypes.data_as(ctypes.c_void_p), len(v),
                                   float(htaper) if htaper != 0 else 0.0, float(vtaper) if vtaper != 0 else 0.0,
                                   int(bool(trunc_int)), ws, wt, device.ptr(focus), device.ptr(images),
                                   device.ptr(wsb), wsb.numel(), device.current_stream_ptr())
    _lib.check(rc)
    return focus


@dataclasses.dataclass
class VelocityScan:
    """Result of migrationVelocityScan.  focus[k, i, j] is the focus of window (i, j) of the image at vels[k];
    vrms[i, j] the velocity of its largest focus (the first on ties), NaN where every focus is 0; center_rows[i] the
    centre row of window row i."""
    vels: np.ndarray
    window: tuple
    snum: int
    tnum: int
    center_rows: np.ndarray
    focus: np.ndarray
    vrms: np.ndarray
    travel_time: np.ndarray = None    # us, snum: what scan_interval_field places the picks by


def velocity_scan_result(focus, vels, window, snum, tnum, travel_time=None):
    """VelocityScan from a (nv, nws, nwt) focus panel: the per-window picks and the window-row centres."""
    focus = np.asarray(focus, dtype=np.float64)
    v = np.asarray(vels, dtype=np.float64)
    ws, wt = window
    S2 = 2 * (int(snum) // 2)
    starts = np.arange(focus.shape[1]) * ws
    n_i = np.minimum(starts + ws, S2) - starts
    vrms = v[np.argmax(focus, axis=0)]
    vrms[np.all(focus == 0, axis=0)] = np.nan
    return VelocityScan(vels=v, window=(int(ws), int(wt)), snum=int(snum), tnum=int(tnum),
                        center_rows=starts + (n_i - 1) / 2.0, focus=focus, vrms=vrms,
                        travel_time=None if travel_time is None else np.array(travel_time, dtype=np.float64))


def migrationVelocityScan(dat, vels, window=(64, 64), htaper=100, vtaper=1000):
    """Migration velocity scan: Stolt-migrate dat at every constant velocity of `vels` (one shared forward transform),
    measure the focus of every window (rows x traces) of every image, and pick the best velocity per window.
    dat is not modified.  Returns a VelocityScan; scan_rms_field turns it into Kirchhoff's lateral RMS field."""
    print('Stolt velocity scan of %.0fx%.0f matrix over %d velocities' % (dat.snum, dat.tnum, np.size(vels)))
    _check_data_shape(dat)
    v = _scan_vels(vels)
    window = _scan_window(window)
    start = time.time()
    in_dtype = _np_dtype(dat.data)
    trunc_int = in_dtype is not None and np.issubdtype(in_dtype, np.integer)  # as migrationStolt
    x = device.to_device(dat.data)
    focus = stolt_scan_device(x, dat.dt, _mean_trace_spacing(dat), v, htaper, vtaper, window, trunc_int)
    scan = velocity_scan_result(focus.cpu().numpy(), v, window, dat.snum, dat.tnum, dat.travel_time)
    print('Stolt velocity scan of %.0fx%.0f matrix complete in %.2f seconds'
          % (dat.snum, dat.tnum, time.time() - start))
    return scan


def scan_rms_field(scan, min_focus=0.0):
    """(profiles (P, snum), col_profile (tnum,)) from a VelocityScan, the compact field kirchhoff_lateral_device takes:
    picks whose best focus is below min_focus are dropped; each window column's picks are interpolated linearly over
    the rows (np.interp: constant beyond the first and last window centre); a column without picks takes the nearest
    column that has some (the left one on ties); trace x takes window column x // wt; identical profiles (bit for bit)
    are merged in order of first appearance.  With one window column P == 1 and profiles[0] suits kirchhoff_device."""
    vrms = _scan_picks(scan, min_focus)
    rows = np.arange(scan.snum, dtype=np.float64)
    cols = []
    for j in range(vrms.shape[1]):
        ok = np.isfinite(vrms[:, j])
        cols.append(np.interp(rows, scan.center_rows[ok], vrms[ok, j]) if ok.any() else None)
    return _scan_field(scan, cols, min_focus)


def _scan_picks(scan, min_focus):
    """The (nws, nwt) picks of a VelocityScan, NaN where the best focus is below min_focus."""
    vrms = np.array(scan.vrms, dtype=np.float64)
    best = np.max(scan.focus, axis=0)
    vrms[best < min_focus] = np.nan
    return vrms


def _scan_field(scan, cols, min_focus):
    """(profiles, col_profile) from one profile per window column (None: no pick there): an empty column takes the
    nearest column that has one (the left one on ties), identical profiles (bit for bit) merge in order of first
    appearance, and trace x takes window column x // wt."""
    nwt = len(cols)
    have = [j for j in range(nwt) if cols[j] is not None]
    if not have:
        raise ValueError('velocity scan: no window has a pick (min_focus = %g)' % min_focus)
    for j in range(nwt):
        if cols[j] is None:
            cols[j] = cols[min(have, key=lambda k: (abs(k - j), k))]
    index, profiles, win_profile = {}, [], []
    for c in cols:
        key = c.tobytes()
        if key not in index:
            index[key] = len(profiles)
            profiles.append(c)
        win_profile.append(index[key])
    col_profile = np.asarray(win_profile, dtype=np.intp)[np.arange(scan.tnum) // scan.window[1]]
    return np.array(profiles), col_profile


# ---------------------------------------------------------------------- interval velocities (Dix) and depth
# RMS picks -> interval velocities by a bounded, smoothed least-squares Dix inversion (closed-form Dix takes differences
# of noisy picks and turns negative), and a time section -> depth section with interval profiles (csrc/depth.cu).
def depth_curves(travel_time_us, profiles):
    """(P, snum) float64 one-way depth of every sample for (P, snum) interval velocities: with t = tt / 1e6 and j0 the
    first sample with t >= 0 (the last sample if there is none), z[j0] = v[j0] t[j0] / 2, then the trapezoid
    (v[i-1] + v[i]) / 2 (t[i] - t[i-1]) / 2 summed sequentially left to right for the samples after j0 and subtracted
    right to left for those before it - rms_velocity's trapezoid and anchor, so a constant profile gives v t / 2 (to rounding; exactly when v
    is a power of two and neighbouring sample times differ exactly).  Strictly increasing for
    positive velocities and strictly ascending times.  impdar_depth_convert_* computes the same bits on the GPU."""
    t = np.asarray(travel_time_us, dtype=np.float64) / 1.0e6
    v = np.asarray(profiles, dtype=np.float64)
    if v.ndim != 2 or v.shape[1] != t.shape[0] or t.shape[0] < 1:
        raise ValueError('profiles must have shape (P, %d), got %s' % (len(t), str(v.shape)))
    nonneg = np.nonzero(t >= 0)[0]
    j0 = nonneg[0] if len(nonneg) else len(t) - 1
    z = np.empty_like(v)
    z0 = v[:, j0:j0 + 1] * t[j0] / 2.
    steps = (v[:, j0:-1] + v[:, j0 + 1:]) / 2. * np.diff(t[j0:]) / 2.
    z[:, j0:] = np.cumsum(np.concatenate([z0, steps], axis=1), axis=1)          # sequential, left to right
    if j0 > 0:
        back = (v[:, :j0] + v[:, 1:j0 + 1]) / 2. * np.diff(t[:j0 + 1]) / 2.
        z[:, :j0 + 1] = np.cumsum(np.concatenate([z0, -back[:, ::-1]], axis=1), axis=1)[:, ::-1]   # right to left
    return z


def _dix_normal(tk, Vk):
    """Normal equations H w = g (n, K, K), (n, K) of the Dix least squares of n columns of K picks (t_k > 0 ascending,
    RMS V_k) in normalised unknowns w = u / mean(V^2), u = v_int^2 at the pick times, without the smoothing term.
    D = A u with A = C B: C the lower-triangular ones (a running sum), B bidiagonal (b_m = B[m, m]: t_1, then
    (t_m - t_{m-1}) / 2; s_m = B[m + 1, m] = (t_{m+1} - t_m) / 2, s_{K-1} = 0).  With W = (ub / D)^2 and
    R_i = sum_{k >= i} W_k (R_K = 0), A^T W A = B^T G B with G[i, j] = R_max(i, j), which is
      H[a, b] = (b_a + s_a) (b_b R_b + s_b R_{b+1})                        for a < b (and symmetric),
      H[a, a] = b_a^2 R_a + (2 b_a s_a + s_a^2) R_{a+1},
    so H costs O(K^2) per column, not O(K^3)."""
    n, K = tk.shape
    ub = np.mean(Vk ** 2, axis=1)
    r = ub[:, None] / (tk * Vk ** 2)
    R = np.zeros((n, K + 1))
    R[:, :K] = np.cumsum((r ** 2)[:, ::-1], axis=1)[:, ::-1]
    half = np.diff(tk, axis=1) / 2.
    bd = np.concatenate([tk[:, :1], half], axis=1)
    bs = np.concatenate([half, np.zeros((n, 1))], axis=1)
    c = bd + bs
    e = bd * R[:, :K] + bs * R[:, 1:]
    O = c[:, :, None] * e[:, None, :]
    H = np.where(np.triu(np.ones((K, K), dtype=bool), 1), O, O.transpose(0, 2, 1))
    di = np.arange(K)
    H[:, di, di] = bd ** 2 * R[:, :K] + (2. * bd * bs + bs ** 2) * R[:, 1:]
    y = np.zeros((n, K + 1))
    y[:, :K] = np.cumsum(r[:, ::-1], axis=1)[:, ::-1]               # C^T (ub / D)
    g = bd * y[:, :K] + bs * y[:, 1:]
    return H, g, ub


def _solve_free(H, g, pinned, wfix):
    """Minimise 1/2 w H w - g w over the free variables with the pinned ones held at wfix (batched)."""
    if not pinned.any():
        return np.linalg.solve(H, g[..., None])[..., 0]
    free = ~pinned
    Hf = np.where(free[:, :, None] & free[:, None, :], H, np.eye(H.shape[1]))
    fix = np.where(pinned, wfix, 0.0)
    rhs = np.where(free, g - np.einsum('nij,nj->ni', H, fix), fix)
    return np.linalg.solve(Hf, rhs[..., None])[..., 0]


def box_qp(H, g, lo, hi):
    """argmin 1/2 w H w - g w subject to lo <= w <= hi for a batch of positive definite H (n, K, K), by a primal active
    set: from a feasible point, solve for the free variables with the pinned ones at their bounds; if that leaves the box,
    step towards it up to the first bound and pin the variable there; otherwise take it, and release every pinned
    variable whose gradient points into the box.  Stops when no free variable violates and every pinned gradient points
    out of the box (the KKT conditions).  Each full step lowers the objective, so no active set repeats."""
    n, K = g.shape
    lo = np.broadcast_to(lo, (n, K))
    hi = np.broadcast_to(hi, (n, K))
    w = np.clip(np.linalg.solve(H, g[..., None])[..., 0], lo, hi)
    at_lo, at_hi = w <= lo, w >= hi
    tol = 1e-12 * (1.0 + np.abs(g).max(axis=1))
    todo = np.nonzero((at_lo | at_hi).any(axis=1))[0]     # the others hold the unconstrained minimum
    for _ in range(10 * K + 50):
        if todo.size == 0:
            break
        Ht, gt, lt, ht, wt = H[todo], g[todo], lo[todo], hi[todo], w[todo]
        al, ah = at_lo[todo], at_hi[todo]
        pinned = al | ah
        ws = _solve_free(Ht, gt, pinned, np.where(al, lt, ht))
        viol = ~pinned & ((ws < lt) | (ws > ht))
        stepped = viol.any(axis=1)
        # columns that leave the box: move to the first bound on the way
        d = ws - wt
        with np.errstate(divide='ignore', invalid='ignore'):
            ratio = np.where(viol & (d < 0), (lt - wt) / d, np.where(viol & (d > 0), (ht - wt) / d, np.inf))
        alpha = np.clip(ratio.min(axis=1), 0.0, 1.0)
        first = viol & (ratio <= alpha[:, None])
        wn = np.where(stepped[:, None], np.clip(wt + alpha[:, None] * d, lt, ht), ws)
        wn = np.where(first & (d < 0), lt, np.where(first & (d > 0), ht, wn))
        al = al | (first & (d < 0))
        ah = ah | (first & (d > 0))
        # columns that stay inside: release the pinned variables whose gradient points into the box
        grad = np.einsum('nij,nj->ni', Ht, wn) - gt
        rel = ~stepped[:, None] & ((al & (grad < -tol[todo, None])) | (ah & (grad > tol[todo, None])))
        al, ah = al & ~rel, ah & ~rel
        w[todo], at_lo[todo], at_hi[todo] = wn, al, ah
        todo = todo[stepped | rel.any(axis=1)]
    return w


def _dix_columns(tk_list, V_list, vmin, vmax, smooth):
    """u = v_int^2 at the picks of every column (lists of 1-D arrays), columns with the same pick count solved together."""
    out = [None] * len(tk_list)
    by_k = {}
    for i, tk in enumerate(tk_list):
        by_k.setdefault(len(tk), []).append(i)
    for K, cols in by_k.items():
        tk = np.array([tk_list[i] for i in cols])
        Vk = np.array([V_list[i] for i in cols])
        H, g, ub = _dix_normal(tk, Vk)
        if K > 1 and smooth > 0:    # + smooth^2 L^T L, L the first difference
            di = np.arange(K)
            H[:, di, di] += smooth ** 2 * np.r_[1., 2. * np.ones(K - 2), 1.]
            H[:, di[:-1], di[1:]] -= smooth ** 2
            H[:, di[1:], di[:-1]] -= smooth ** 2
        w = box_qp(H, g, (vmin ** 2 / ub)[:, None], (vmax ** 2 / ub)[:, None])
        for c, i in enumerate(cols):
            out[i] = w[c] * ub[c]
    return out


def scan_interval_field(scan, min_focus=0.0, vmin=None, vmax=2.99792458e8, smooth=0.3, travel_time=None):
    """(profiles (P, snum), col_profile (tnum,)) of INTERVAL velocities from a VelocityScan, the field depthConvert and
    interval_table take.  Masking, empty-column fill, merging and the trace map are scan_rms_field's.  Per window column
    the picks (t_k > 0, V_k) sit at the window-centre times; the unknowns u_k = v_int^2 at those times are linear in t
    between picks and constant (u_1) on [0, t_1], so D_k = t_k V_k^2 = (A u)_k.  The fit minimises
    sum_k ((A u)_k / D_k - 1)^2 + smooth^2 sum_k ((u_{k+1} - u_k) / mean(V^2))^2 with vmin^2 <= u <= vmax^2 (vmin
    defaults to half the slowest scan velocity, vmax to the speed of light), all columns at once (box_qp).  Sample i
    gets sqrt(np.interp(t_i, t_k, u)): constant beyond the first and last pick.  `travel_time` (us, snum) defaults to
    the scan's own."""
    tt = scan.travel_time if travel_time is None else travel_time
    if tt is None:
        raise ValueError('scan_interval_field needs the travel times of the scanned radargram')
    t = np.asarray(tt, dtype=np.float64) / 1.0e6
    if t.shape != (scan.snum,) or not np.all(np.isfinite(t)) or not np.all(np.diff(t) > 0):
        raise ValueError('travel_time must be %d finite, strictly ascending values' % scan.snum)
    vmin = 0.5 * float(np.min(scan.vels)) if vmin is None else float(vmin)
    vmax = float(vmax)
    if not (np.isfinite(vmin) and np.isfinite(vmax) and 0 < vmin < vmax):
        raise ValueError('need finite bounds 0 < vmin < vmax, got vmin = %g, vmax = %g' % (vmin, vmax))
    smooth = float(smooth)
    if not (np.isfinite(smooth) and smooth >= 0):
        raise ValueError('smooth must be finite and >= 0, got %g' % smooth)
    vrms = _scan_picks(scan, min_focus)
    tc = np.interp(scan.center_rows, np.arange(scan.snum, dtype=np.float64), t)
    have = [j for j in range(vrms.shape[1]) if np.any(np.isfinite(vrms[:, j]) & (tc > 0))]
    oks = [np.isfinite(vrms[:, j]) & (tc > 0) for j in have]
    tks = [tc[ok] for ok in oks]
    us = _dix_columns(tks, [vrms[ok, j] for ok, j in zip(oks, have)], vmin, vmax, smooth)
    cols = [None] * vrms.shape[1]
    for j, tk, u in zip(have, tks, us):
        cols[j] = np.sqrt(np.interp(t, tk, u))
    return _scan_field(scan, cols, min_focus)


def interval_table(travel_time_us, vint):
    """A (v, z) table of the interval profile `vint` (snum) that getVelocityProfile maps back onto these travel times,
    for migrationPhaseShift / migrationKirchhoffLayered or as a vel_fn file (np.savetxt).  getVelocityProfile reads
    the v column as the AVERAGE velocity down to z (t = 2 z / v), so the rows are (2 z_i / t_i, z_i) with z =
    depth_curves for every sample with t_i > 0, after a row (v, 0) at the surface, and a last row that continues the
    deepest interval velocity to max(v) t_end / 2 or deeper, which getVelocityProfile's coverage check asks for when the
    velocity decreases with depth (firn)."""
    t = np.asarray(travel_time_us, dtype=np.float64) / 1.0e6
    v = np.asarray(vint, dtype=np.float64)
    if v.shape != t.shape or v.ndim != 1:
        raise ValueError('vint must have one value per sample (%d), got shape %s' % (len(t), str(v.shape)))
    if not (np.all(np.isfinite(v)) and np.all(v > 0)):
        raise ValueError('interval velocities must be finite and positive')
    if not (np.all(np.isfinite(t)) and np.all(np.diff(t) > 0)):
        raise ValueError('travel_time must be finite and strictly ascending')
    pos = t > 0
    if not pos.any():
        raise ValueError('no sample after time zero')
    z = depth_curves(travel_time_us, v[None, :])[0][pos]
    tp = t[pos]
    va = 2. * z / tp
    rows = [(va[0], 0.0)] + list(zip(va, z))
    z_end = max(va.max(), v[-1]) * tp[-1] / 2.
    if z_end > z[-1]:
        te = tp[-1] + 2. * (z_end - z[-1]) / v[-1]
        rows.append((2. * z_end / te, z_end))
    return np.array(rows, dtype=np.float64)


def _depth_args(profiles, col_profile, snum, tnum, zgrid):
    v, colp = _kirch_lateral_args(profiles, col_profile, snum, tnum)
    zg = np.ascontiguousarray(np.asarray(zgrid, dtype=np.float64))
    if zg.ndim != 1 or zg.size < 1 or not np.all(np.isfinite(zg)) or not np.all(np.diff(zg) > 0):
        raise ValueError('zgrid must be a non-empty 1-D array of finite, strictly ascending depths')
    return v, colp, zg


_DEPTH_ENTRIES = {('float32', 'float32'): 'impdar_depth_convert_f32', ('float32', 'float64'): 'impdar_depth_convert_f32_f64',
                  ('float64', 'float64'): 'impdar_depth_convert_f64'}


def depth_convert_device(data_dev, travel_time_us, profiles, col_profile, zgrid, out=None):
    """Depth section (nz, tnum) of a (snum, tnum) float32 or float64 CUDA tensor: out[k, x] = np.interp(zgrid[k], z_p,
    data[:, x], left=nan, right=nan) with z_p = depth_curves(travel_time_us, profiles)[col_profile[x]] ((P, snum) interval
    velocities), computed in float64 bit for bit (impdar_depth_convert_*).  `out` (default: the input dtype) may be
    float64 for float32 input."""
    import torch
    if not (device.is_device_array(data_dev) and data_dev.dim() == 2
            and data_dev.dtype in (torch.float32, torch.float64)):
        raise ValueError('depth_convert_device needs a 2-D float32 or float64 CUDA tensor')
    x = data_dev.contiguous()
    S, T = x.shape
    if S < 2:
        raise ValueError('depth conversion needs at least two samples per trace')
    tt = np.ascontiguousarray(device.host_f64(travel_time_us))
    if tt.shape != (S,) or not np.all(np.isfinite(tt)) or not np.all(np.diff(tt / 1.0e6) > 0):
        raise ValueError('travel_time must be %d finite, strictly ascending values' % S)
    v, colp, zg = _depth_args(profiles, col_profile, S, T, zgrid)
    nz = zg.size
    if out is None:
        out = torch.empty((nz, T), dtype=x.dtype, device=x.device)
    if not (device.is_device_array(out) and tuple(out.shape) == (nz, T) and out.is_contiguous()):
        raise ValueError('out must be a contiguous CUDA tensor of shape %s' % ((nz, T),))
    name = _DEPTH_ENTRIES.get((str(x.dtype).split('.')[-1], str(out.dtype).split('.')[-1]))
    if name is None:
        raise ValueError('depth conversion runs float32 -> float32, float32 -> float64 or float64 -> float64, got %s -> %s'
                         % (x.dtype, out.dtype))
    lib = _lib.load()
    ws = device.workspace(lib.impdar_depth_workspace_bytes(S, T, nz, v.shape[0]))
    rc = getattr(lib, name)(device.ptr(x), device.ptr(out), S, T, nz, device.ptr(tt), device.ptr(v), v.shape[0],
                            device.ptr(colp), device.ptr(zg), device.ptr(ws), ws.numel(), device.current_stream_ptr())
    _lib.check(rc)
    return out


def _depth_field(dat, vel, vel_fn, field, genfromtxt_kwargs):
    """(P, snum) interval profiles and the (tnum,) trace map of depthConvert's velocity argument."""
    if field is not None:
        if vel_fn is not None or not (np.ndim(vel) == 0 and vel == 1.69e8):
            raise ValueError('give the velocity as vel / vel_fn or as field, not both')
        try:
            profiles, col_profile = field
        except (TypeError, ValueError):
            raise ValueError('field must be a pair (profiles, col_profile)')
        return _kirch_lateral_args(profiles, col_profile, dat.snum, dat.tnum)
    if vel_fn is not None:
        try:
            vel = np.genfromtxt(vel_fn, **genfromtxt_kwargs)
            print('Velocities loaded from %s.' % vel_fn)
        except Exception:
            raise TypeError('File %s was given for input velocity array, but cannot be loaded. Please reformat to txt file.' % vel_fn)
    if np.ndim(vel) == 0:
        profiles = np.full((1, dat.snum), float(vel))
    elif len(np.shape(vel)) == 2 and np.shape(vel)[1] == 3:
        profiles, col_profile = lateral_velocity_profiles(dat, np.asarray(vel, dtype=np.float64))
        return _kirch_lateral_args(profiles, col_profile, dat.snum, dat.tnum)
    else:
        profiles = np.asarray(getVelocityProfile(dat, np.asarray(vel, dtype=np.float64)), dtype=np.float64)[None, :]
    return _kirch_lateral_args(profiles, np.zeros(dat.tnum, dtype=np.int32), dat.snum, dat.tnum)


def depthConvert(dat, vel=1.69e8, vel_fn=None, field=None, dz=None, **genfromtxt_kwargs):
    """Convert a (migrated) time section to depth with a velocity that may vary with depth and laterally.  The velocity
    is a scalar, a (v, z) table (getVelocityProfile), a (v, z, x) table (lateral_velocity_profiles), a file `vel_fn`
    loaded like migrationKirchhoffLateral loads one, or field=(profiles, col_profile) of interval velocities
    (scan_interval_field).  Depth rows are zgrid = z0 + dz * arange(nz), z0 the shallowest first-sample depth of any
    profile, and the last row the deepest last-sample depth of any profile does not pass; dz defaults to min(v) dt / 2, so no depth row is coarser than the
    finest sample.  Each trace is resampled with np.interp on its own depth curve (NaN outside it; depth_convert_device).
    dat.data becomes the (nz, tnum) section (float64 on the host lane, the tensor's dtype on the device lane, integer
    input widened to float64), dat.snum = nz, dat.nmo_depth = zgrid, and dat.travel_time the two-way time of each depth
    row in a trace of the most-used profile (the lowest index on ties), continued linearly beyond its first and last
    samples with its first and last interval velocities."""
    import torch
    print('Depth conversion of %.0fx%.0f matrix' % (dat.snum, dat.tnum))
    _check_data_shape(dat)
    start = time.time()
    profiles, col_profile = _depth_field(dat, vel, vel_fn, field, genfromtxt_kwargs)
    z = depth_curves(dat.travel_time, profiles)
    if dz is None:
        dz = float(np.min(profiles)) * float(dat.dt) / 2.
    dz = float(dz)
    if not (np.isfinite(dz) and dz > 0):
        raise ValueError('dz must be finite and positive, got %g' % dz)
    z0, z1 = float(np.min(z[:, 0])), float(np.max(z[:, -1]))
    nz = int(np.floor((z1 - z0) / dz)) + 1            # the last row no deeper than the deepest sample
    while z0 + dz * nz <= z1:
        nz += 1
    while nz > 1 and z0 + dz * (nz - 1) > z1:
        nz -= 1
    zgrid = z0 + dz * np.arange(nz)
    on_device = device.is_device_array(dat.data)
    if on_device:
        x = dat.data if dat.data.dtype in (torch.float32, torch.float64) else (
            dat.data.to(torch.float32) if dat.data.is_floating_point() else dat.data.to(torch.float64))
        out = depth_convert_device(x, dat.travel_time, profiles, col_profile, zgrid)
        dat.data = out if out.dtype == dat.data.dtype or not dat.data.is_floating_point() else out.to(dat.data.dtype)
    else:
        device.require_cuda()
        a = np.asarray(dat.data)
        x = device.to_device(a, torch.float32 if a.dtype == np.float32 else torch.float64)
        out = torch.empty((nz, dat.tnum), dtype=torch.float64, device=x.device)
        dat.data = device.to_host(depth_convert_device(x, dat.travel_time, profiles, col_profile, zgrid, out=out),
                                  np.float64)
    p = int(np.argmax(np.bincount(col_profile, minlength=profiles.shape[0])))
    tt = np.asarray(dat.travel_time, dtype=np.float64)
    zp, vp = z[p], profiles[p]
    newt = np.interp(zgrid, zp, tt)
    below, above = zgrid > zp[-1], zgrid < zp[0]
    newt[below] = tt[-1] + 2. * (zgrid[below] - zp[-1]) / vp[-1] * 1.0e6
    newt[above] = tt[0] - 2. * (zp[0] - zgrid[above]) / vp[0] * 1.0e6
    dat.travel_time = newt
    dat.nmo_depth = zgrid
    dat.snum = nz
    print('Depth conversion of %.0fx%.0f matrix complete in %.2f seconds' % (nz, dat.tnum, time.time() - start))
    return dat


# -------------------------------------------------------------------------------------- phase shift
def getVelocityProfile(dat, vels_in):
    """Map a (v, z) or (v, z, x) velocity table onto the data's travel-time axis; mirrors
    mig_python.py:543-643 including every ValueError.  O(snum) host work in float64."""
    from scipy.interpolate import griddata, interp1d
    if not hasattr(vels_in, "__len__"):
        return vels_in
    if len(np.shape(vels_in)) != 2 or np.shape(vels_in)[1] == 1:
        raise ValueError('If non-constant vel, inputs needs to be 2d (v, z) or (v, z, x)')
    nlay, dimension = np.shape(vels_in)
    vel_v = vels_in[:, 0]
    vel_z = vels_in[:, 1]
    twtt = np.asarray(dat.travel_time, dtype=np.float64).copy() / 1.0e6
    if nlay == 1:
        raise ValueError('It does not make sense to only give one layer of velocity--if you want constant velocity just input v')
    elif dimension == 2:
        zs = np.max(vel_v) / 2. * twtt
        zs[0] = twtt[0] * vel_v[0] / 2.
        if (vel_z[0] > 1.1 * np.nanmin(zs) and vel_z[0] / np.nanmax(zs) > 1.0e-3) or vel_z[-1] * 1.1 < np.nanmax(zs):
            raise ValueError('Your velocity data doesnt come close to covering the depths in the data')
        if vel_z[0] > np.nanmin(zs):
            vel_v = np.insert(vel_v, 0, vel_v[np.argmin(vel_z)])
            vel_z = np.insert(vel_z, 0, np.nanmin(zs))
        if vel_z[-1] < np.nanmax(zs):
            vel_v = np.append(vel_v, vel_v[np.argmax(vel_z)])
            vel_z = np.append(vel_z, np.nanmax(zs))
        vel_t = 2. * vel_z / vel_v
        tofz = interp1d(vel_z, vel_t)(zs)
        zoft = interp1d(tofz, zs)(twtt)
        vmig = 2. * np.gradient(zoft, twtt)
    elif dimension == 3:
        profiles, col_profile = lateral_velocity_profiles(dat, vels_in)
        vmig = np.zeros((dat.snum, dat.tnum), dtype=profiles.dtype)
        vmig[:] = profiles.T[:, col_profile]
    else:
        raise ValueError('Input must be 2d with 2 or 3 columns')
    return vmig


def lateral_velocity_profiles(dat, vels_in):
    """getVelocityProfile's (v, z, x) branch in compact form: (profiles, col_profile) with profiles[p] the interval
    velocity (P, snum) of the p-th distinct column and col_profile (tnum,) the profile of each trace, so that
    getVelocityProfile(dat, vels_in)[:, i] == profiles[col_profile[i]].  The reference's per-trace loop (O(snum^2)
    trapezoids per trace) depends on a trace only through its nearest-neighbour griddata column, so it runs once per
    distinct column - columns are compared bit for bit - in order of first appearance (the same first ValueError)."""
    from scipy.interpolate import griddata, interp1d
    vel_v, vel_z, vel_x = vels_in[:, 0], vels_in[:, 1], vels_in[:, 2]
    twtt = np.asarray(dat.travel_time, dtype=np.float64).copy() / 1.0e6
    zs = np.linspace(np.min(vel_v) * twtt[0], np.max(vel_v) * twtt[-1], dat.snum) / 2.
    if dat.dist is None or all(dat.dist == 0):
        raise ValueError('The distance vector was never set.')
    XS, ZS = np.meshgrid(dat.dist, zs)
    VS = griddata(np.transpose([vel_x, vel_z]), vel_v,
                  np.transpose([XS.flatten(), ZS.flatten()]), method='nearest')
    VS = np.reshape(VS, np.shape(XS))
    cols = np.ascontiguousarray(VS.T)
    keys = cols.view(np.dtype((np.void, cols.dtype.itemsize * cols.shape[1]))).ravel()
    _, first, inverse = np.unique(keys, return_index=True, return_inverse=True)
    order = np.argsort(first)                       # profiles in order of first appearance
    rank = np.empty_like(order)
    rank[order] = np.arange(len(order))
    col_profile = rank[inverse.ravel()]
    profiles = np.zeros((len(order), dat.snum), dtype=VS.dtype)
    trapz = getattr(np, 'trapezoid', None) or np.trapz
    for p, i in enumerate(first[order]):
        vz = ZS[:, i]
        vv = VS[:, i]
        vel_t = 2 * np.array([trapz(1. / vv[:j], vz[:j]) for j in range(dat.snum)])
        tofz = interp1d(ZS[:, i], vel_t)(zs)
        zinterp = interp1d(tofz, zs)
        if twtt[-1] > tofz[-1]:
            raise ValueError('Two-way travel time array extends outside of interpolation range')
        profiles[p] = 2. * np.gradient(zinterp(twtt), twtt)
    return profiles, col_profile


def phase_shift_device(data_dev, dt, dx, travel_time_us, vmig, htaper, vtaper, out=None):
    """(snum, tnum) float32 CUDA tensor -> phase-shift migrated (snum, tnum) float32; vmig a scalar or a
    length-snum float64 profile."""
    import torch
    lib = _lib.load()
    S, T = data_dev.shape
    if out is None:
        out = torch.empty((S, T), dtype=torch.float32, device=data_dev.device)
    ws = device.workspace(lib.impdar_phsh_workspace_bytes(S, T))
    if hasattr(vmig, "__len__"):
        tt = device.host_f64(travel_time_us)
        thr2 = ((tt / 1.0e6) / tt[-1] / 1e6) ** 2.                      # mig_python.py:484
        vm_dev = device.to_device(device.host_f64(vmig), torch.float64)
        th_dev = device.to_device(thr2, torch.float64)
        vconst = 0.0
    else:
        vm_dev = th_dev = None
        vconst = float(vmig)
    rc = lib.impdar_phsh_f32(device.ptr(data_dev), device.ptr(out), S, T, float(dt), float(dx), vconst,
                             device.ptr(vm_dev), device.ptr(th_dev), float(htaper), float(vtaper),
                             device.ptr(ws), ws.numel(), device.current_stream_ptr())
    _lib.check(rc)
    return out


def phase_shift_ffd_device(data_dev, dt, dx, dx_fd, travel_time_us, vmig, htaper, vtaper):
    """Laterally varying v(x, z) branch (Fourier finite difference, mig_python.py:428-432, 466-481, 496-540):
    (snum, tnum) float64 CUDA tensor + (snum, tnum) float64 vmig -> migrated (snum, tnum) float64."""
    import torch
    lib = _lib.load()
    S, T = data_dev.shape
    vm = np.ascontiguousarray(np.asarray(vmig, dtype=np.float64))
    if vm.shape != (S, T):
        raise ValueError('operands could not be broadcast together with shapes (%d,) %s' % (T, str(vm.shape[1:])))
    out = torch.empty((S, T), dtype=torch.float64, device=data_dev.device)
    ws = device.workspace(lib.impdar_phsh_ffd_workspace_bytes(S, T))
    tt = device.host_f64(travel_time_us)
    thr2 = ((tt / 1.0e6) / tt[-1] / 1e6) ** 2.                          # mig_python.py:484
    vm_dev = device.to_device(vm, torch.float64)
    th_dev = device.to_device(thr2, torch.float64)
    rc = lib.impdar_phsh_ffd_f64(device.ptr(data_dev), device.ptr(out), S, T, float(dt), float(dx), float(dx_fd),
                                 device.ptr(vm_dev), device.ptr(th_dev), float(htaper), float(vtaper),
                                 device.ptr(ws), ws.numel(), device.current_stream_ptr())
    _lib.check(rc)
    return out


def _reject_integer_inplace(dat):
    in_dtype = _np_dtype(dat.data)
    if in_dtype is not None and not np.issubdtype(in_dtype, np.floating):
        # the reference does ``dat.data *= H*V`` in place (mig_python.py:258/:335), which numpy refuses
        raise TypeError("Cannot cast ufunc 'multiply' output from dtype('float64') to dtype('%s') "
                        "with casting rule 'same_kind'" % in_dtype)
    return in_dtype


def migrationPhaseShift(dat, vel=1.69e8, vel_fn=None, htaper=100, vtaper=1000, **genfromtxt_kwargs):
    """Gazdag phase-shift migration, constant or layered velocity; mirrors mig_python.py:211-287."""
    print('Phase-Shift Migration of %.0fx%.0f matrix' % (dat.snum, dat.tnum))
    _check_data_shape(dat)
    start = time.time()
    was_device = device.is_device_array(dat.data)
    in_tdt = _torch_dtype(dat.data)
    _reject_integer_inplace(dat)
    dx = _mean_trace_spacing(dat)
    if vel_fn is not None:
        try:
            vel = np.genfromtxt(vel_fn, **genfromtxt_kwargs)
            print('Velocities loaded from %s.' % vel_fn)
        except Exception:
            raise TypeError('File %s was given for input velocity array, but cannot be loaded. Please reformat to txt file.' % vel_fn)
    vmig = getVelocityProfile(dat, vel)
    if hasattr(vmig, "__len__"):
        if not hasattr(vmig, 'shape'):
            raise ValueError('vmig needs to be an array or float')
        if len(vmig) != dat.snum:
            raise ValueError('Interpolated velocity profile is not the length of the number of samples in a trace.')
    if hasattr(vmig, "__len__") and hasattr(vmig[0], "__len__"):
        import torch
        print('2-D velocity structure, Fourier Finite-Difference Migration')
        x = device.to_device(dat.data, torch.float64)
        out = phase_shift_ffd_device(x, dat.dt, dx, float(np.mean(dat.trace_int)), dat.travel_time, vmig,
                                     htaper, vtaper)
    else:
        x = device.to_device(dat.data)
        out = phase_shift_device(x, dat.dt, dx, dat.travel_time, vmig, htaper, vtaper)
    _finish(dat, out, np.float64, was_device, in_tdt)
    print('Phase-Shift Migration of %.0fx%.0f matrix complete in %.2f seconds'
          % (dat.snum, dat.tnum, time.time() - start))
    return dat


def migrationTimeWavenumber(dat, vel=1.69e8, vel_fn=None, htaper=100, vtaper=1000):
    """The reference's T-K migration is a stub that only tapers the data in place (mig_python.py:290-355);
    this reproduces exactly that."""
    import torch
    print('Time-Wavenumber Migration of %.0fx%.0f matrix' % (dat.snum, dat.tnum))
    _check_data_shape(dat)
    start = time.time()
    was_device = device.is_device_array(dat.data)
    in_dtype = _reject_integer_inplace(dat)
    lib = _lib.load()
    # a pure elementwise product: float64 radargrams (host or device) are tapered in float64, exactly like numpy
    f64 = (in_dtype == np.float64) if in_dtype is not None else (dat.data.dtype == torch.float64)
    x = device.to_device(dat.data, torch.float64 if f64 else torch.float32)
    S, T = x.shape
    out = x if was_device else torch.empty_like(x)
    if f64:
        rc = lib.impdar_taper_f64(device.ptr(x), device.ptr(out), S, T, 1, float(htaper), float(vtaper),
                                  device.current_stream_ptr())
    else:
        rc = lib.impdar_taper_f32(device.ptr(x), device.ptr(out), S, T, 1, float(htaper), float(vtaper), 0,
                                  device.current_stream_ptr())
    _lib.check(rc)
    _finish(dat, out, in_dtype, was_device)
    print('Time-Wavenumber Migration of %.0fx%.0f matrix complete in %.2f seconds'
          % (dat.snum, dat.tnum, time.time() - start))
    return dat
