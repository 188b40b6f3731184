"""Float64 numpy restatement of Kirchhoff migration with one velocity per output sample (straight rays).

The arithmetic per (output sample, input trace) pair is that of oracle.migration.kirchhoff / kirchhoff_sparse /
kirchhoff_pair_count (mig_python.py:35-123) with `vel` replaced by v[ti] of the pair's output row.  The velocity is
reshaped to (S, 1) explicitly: a bare length-S vector would broadcast against the trace axis, silently so when S == T.
A constant vector performs exactly the scalar operations, so it reproduces the scalar oracle bit for bit.  The product
package keeps its own copy of rms_velocity (it never imports the test helpers or the oracle).
"""
import numpy as np

from oracle.migration import nearest_sample_index


def rms_velocity(travel_time_us, vmig):
    """RMS velocity per sample, an explicit sequential loop: I[j0] = vmig[j0]^2 t[j0] at the first sample with t >= 0,
    I[i] = I[i-1] + (vmig[i]^2 + vmig[i-1]^2) / 2 (t[i] - t[i-1]); v = sqrt(I / t) where t > 0, vmig where t <= 0."""
    t = np.asarray(travel_time_us, dtype=np.float64) / 1.0e6
    vm = np.asarray(vmig, dtype=np.float64)
    v = vm.copy()
    nonneg = np.nonzero(t >= 0)[0]
    if len(nonneg) == 0:
        return v
    j0 = int(nonneg[0])
    acc = vm[j0] ** 2 * t[j0]
    for i in range(j0, len(t)):
        if i > j0:
            acc = acc + (vm[i] ** 2 + vm[i - 1] ** 2) / 2. * (t[i] - t[i - 1])
        if t[i] > 0:
            v[i] = np.sqrt(acc / t[i])
    return v


def _rows(vel, S):
    """(S, 1) float64 column of per-row velocities (a scalar is broadcast)."""
    v = np.asarray(vel, dtype=np.float64)
    if v.ndim == 0:
        return np.full((S, 1), float(v))
    assert v.shape == (S,), v.shape
    return v.reshape(S, 1)


def kirchhoff(data, travel_time_us, dist_km, vel, nearfield=False, x_begin=0, x_end=None):
    """oracle.migration.kirchhoff with a per-row velocity."""
    data = np.asarray(data)
    tt_sec = np.asarray(travel_time_us, dtype=np.float64) / 1.0e6
    gradD = np.gradient(data.astype(np.float64), tt_sec, axis=0)
    data = data.astype(np.float64)
    max_tt = np.max(tt_sec)
    S, T = data.shape
    v = _rows(vel, S)
    zs = v[:, 0] * tt_sec / 2.0
    zs2 = zs ** 2.
    dist = np.ascontiguousarray(dist_km, dtype=np.float64) * 1.0e3
    x_end = T if x_end is None else x_end
    out = np.zeros((S, x_end - x_begin))
    ar = np.arange(T)[None, :]
    for xi in range(x_begin, x_end):
        with np.errstate(invalid='ignore', divide='ignore'):
            rs = np.sqrt(((dist - dist[xi]) ** 2.)[None, :] + zs2[:, None])
            costheta = zs[:, None] / rs
            t = 2. * rs / v
            Didx = nearest_sample_index(tt_sec, t)
            g = gradD[Didx, ar]
            g[t > max_tt] = 0.
            integral = np.nansum(g * costheta / v, axis=1)
            if nearfield:
                d = data[Didx, ar]
                d[t > max_tt] = 0.
                integral = integral + np.nansum(d * costheta / rs ** 2., axis=1)
        out[:, xi - x_begin] = 1. / (2. * np.pi) * integral
    return out


def kirchhoff_sparse(data, travel_time_us, dist_km, vel, nearfield=False, traces=(0,), rows=None):
    """oracle.migration.kirchhoff_sparse with a per-row velocity (the column window uses the largest velocity)."""
    tt_sec = np.asarray(travel_time_us, dtype=np.float64) / 1.0e6
    max_tt = np.max(tt_sec)
    S = len(tt_sec)
    vcol = _rows(vel, S)
    zs = vcol[:, 0] * tt_sec / 2.0
    zs2 = zs ** 2.
    dist = np.ascontiguousarray(dist_km, dtype=np.float64) * 1.0e3
    T = len(dist)
    rows = np.arange(S) if rows is None else np.asarray(rows, dtype=int)
    v = vcol[rows]
    out = np.zeros((len(rows), len(traces)))
    reach = float(vcol.max()) * max_tt / 2.0 * (1.0 + 1e-9) + 1e-6
    monotone = bool(np.all(np.diff(dist) >= 0))
    for j, xi in enumerate(traces):
        if monotone:
            c0 = int(np.searchsorted(dist, dist[xi] - reach, side='left'))
            c1 = int(np.searchsorted(dist, dist[xi] + reach, side='right'))
        else:
            c0, c1 = 0, T
        win = data[:, c0:c1]
        if hasattr(win, 'cpu'):
            win = win.cpu().numpy()
        win = np.asarray(win, dtype=np.float64)
        gradD = np.gradient(win, tt_sec, axis=0)
        ar = np.arange(c1 - c0)[None, :]
        with np.errstate(invalid='ignore', divide='ignore'):
            rs = np.sqrt(((dist[c0:c1] - dist[xi]) ** 2.)[None, :] + zs2[rows, None])
            costheta = zs[rows, None] / rs
            t = 2. * rs / v
            Didx = nearest_sample_index(tt_sec, t)
            g = gradD[Didx, ar]
            g[t > max_tt] = 0.
            integral = np.nansum(g * costheta / v, axis=1)
            if nearfield:
                d = win[Didx, ar]
                d[t > max_tt] = 0.
                integral = integral + np.nansum(d * costheta / rs ** 2., axis=1)
        out[:, j] = 1. / (2. * np.pi) * integral
    return out


def kirchhoff_pair_count(travel_time_us, dist_km, vel):
    """oracle.migration.kirchhoff_pair_count with a per-row velocity: pairs with 2 r / v[ti] <= max(tt)."""
    tt = np.asarray(travel_time_us, dtype=np.float64) / 1e6
    dist = np.asarray(dist_km, dtype=np.float64) * 1e3
    tmax = tt.max()
    v = _rows(vel, len(tt))[:, 0]
    zs = v * tt / 2.
    ap2 = (v * tmax / 2.) ** 2 - zs ** 2
    total = 0
    for a2 in ap2:
        if a2 < 0:
            continue
        a = np.sqrt(a2)
        lo = np.searchsorted(dist, dist - a, side='left')
        hi = np.searchsorted(dist, dist + a, side='right')
        total += int(np.sum(hi - lo))
    return total
