"""Float64 reference of the time-to-depth conversion: a per-element loop for the depth curves and numpy.interp per
trace for the resampling (what impdar_depth_convert_* must equal bit for bit)."""
import numpy as np


def depth_curve_loop(travel_time_us, v):
    """One profile's one-way depths, one sample at a time in the documented order."""
    t = [float(x) / 1.0e6 for x in travel_time_us]
    v = [float(x) for x in v]
    n = len(t)
    j0 = next((i for i in range(n) if t[i] >= 0), n - 1)
    z = [0.0] * n
    z[j0] = v[j0] * t[j0] / 2
    for i in range(j0 + 1, n):
        z[i] = z[i - 1] + (v[i - 1] + v[i]) / 2 * (t[i] - t[i - 1]) / 2
    for i in range(j0 - 1, -1, -1):
        z[i] = z[i + 1] - (v[i] + v[i + 1]) / 2 * (t[i + 1] - t[i]) / 2
    return np.array(z)


def depth_convert(image, travel_time_us, profiles, col_profile, zgrid, curves=None):
    """(nz, tnum) float64: column x is np.interp(zgrid, z_p, image[:, x], left=nan, right=nan), p = col_profile[x].
    `curves` (P, snum) may be passed in (impdar_b200.migrationlib.depth_curves, equal to the loop bit for bit)."""
    img = np.asarray(image).astype(np.float64)
    if curves is None:
        curves = np.array([depth_curve_loop(travel_time_us, p) for p in profiles])
    out = np.empty((len(zgrid), img.shape[1]))
    for x in range(img.shape[1]):
        out[:, x] = np.interp(zgrid, curves[col_profile[x]], img[:, x], left=np.nan, right=np.nan)
    return out
