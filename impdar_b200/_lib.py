"""ctypes binding of libimpdar_b200.so (declared in include/impdar_b200.h).

There is no CPU fallback: if the CUDA library is missing or a call fails, an exception is raised.
"""
import ctypes
import os
import threading

HERE = os.path.dirname(os.path.abspath(__file__))
# IMPDAR_B200_LIB selects another build of the same library (development A/B runs of kernel variants)
LIB_PATH = os.environ.get("IMPDAR_B200_LIB") or os.path.join(HERE, "libimpdar_b200.so")

_c_int = ctypes.c_int
_c_dbl = ctypes.c_double
_c_sz = ctypes.c_size_t
_vp = ctypes.c_void_p

# name -> (restype, argtypes); must list every symbol include/impdar_b200.h declares
PROTOTYPES = {
    "impdar_b200_version": (_c_int, []),
    "impdar_b200_last_error": (ctypes.c_char_p, []),
    "impdar_b200_launch_count": (ctypes.c_ulonglong, []),
    "impdar_b200_kernel_timer": (_c_int, [_c_int]),
    "impdar_b200_kernel_timer_read": (_c_int, [ctypes.c_char_p, _vp, _vp]),
    "impdar_taper_f32": (_c_int, [_vp, _vp, _c_int, _c_int, _c_int, _c_dbl, _c_dbl, _c_int, _vp]),
    "impdar_taper_f64": (_c_int, [_vp, _vp, _c_int, _c_int, _c_int, _c_dbl, _c_dbl, _vp]),
    "impdar_hfilt_f32": (_c_int, [_vp, _vp, _c_int, _c_int, _c_int, _c_int, _c_int, _vp, _c_int, _vp]),
    "impdar_hfilt_f64": (_c_int, [_vp, _vp, _c_int, _c_int, _c_int, _c_int, _c_int, _vp, _c_int, _vp]),
    "impdar_ahfilt_workspace_bytes": (_c_sz, [_c_int, _c_int, _c_int]),
    "impdar_ahfilt_force_rowwise": (_c_int, [_c_int]),
    "impdar_ahfilt_f32": (_c_int, [_vp, _vp, _c_int, _c_int, _c_int, _c_int, _vp, _vp, _c_sz, _vp]),
    "impdar_ahfilt_f64": (_c_int, [_vp, _vp, _c_int, _c_int, _c_int, _c_int, _vp, _vp, _c_sz, _vp]),
    "impdar_filtfilt_workspace_bytes": (_c_sz, [_c_int, _c_int, _c_int, _c_int, _c_int]),
    "impdar_filtfilt_f32": (_c_int, [_vp, _vp, _c_int, _c_int, _c_int, _vp, _vp, _c_int, _vp, _c_int, _vp, _c_sz, _vp]),
    "impdar_filtfilt_f64": (_c_int, [_vp, _vp, _c_int, _c_int, _c_int, _vp, _vp, _c_int, _vp, _c_int, _vp, _c_sz, _vp]),
    "impdar_fir_f32": (_c_int, [_vp, _vp, _c_int, _c_int, _c_int, _vp, _c_int, _vp]),
    "impdar_fir_f64": (_c_int, [_vp, _vp, _c_int, _c_int, _c_int, _vp, _c_int, _vp]),
    "impdar_winavg_workspace_bytes": (_c_sz, [_c_int, _c_int, _c_int]),
    "impdar_winavg_f32": (_c_int, [_vp, _vp, _c_int, _c_int, _c_int, _c_int, _vp, _vp, _c_sz, _vp]),
    "impdar_winavg_f64": (_c_int, [_vp, _vp, _c_int, _c_int, _c_int, _c_int, _vp, _vp, _c_sz, _vp]),
    "impdar_filtfilt_rows_workspace_bytes": (_c_sz, [_c_int, _c_int, _c_int, _c_int, _c_int]),
    "impdar_filtfilt_rows_f32": (_c_int, [_vp, _vp, _c_int, _c_int, _c_int, _vp, _vp, _c_int, _vp, _c_int, _vp, _c_sz, _vp]),
    "impdar_filtfilt_rows_f64": (_c_int, [_vp, _vp, _c_int, _c_int, _c_int, _vp, _vp, _c_int, _vp, _c_int, _vp, _c_sz, _vp]),
    "impdar_rowabsmax_f32": (_c_int, [_vp, _vp, _c_int, _c_int, _c_int, _vp]),
    "impdar_rowabsmax_f64": (_c_int, [_vp, _vp, _c_int, _c_int, _c_int, _vp]),
    "impdar_rowgain_f32": (_c_int, [_vp, _vp, _c_int, _c_int, _c_int, _vp, _vp, _c_int, _vp]),
    "impdar_rowgain_f64": (_c_int, [_vp, _vp, _c_int, _c_int, _c_int, _vp, _vp, _c_int, _vp]),
    "impdar_kirchhoff_workspace_bytes": (_c_sz, [_c_int, _c_int, _c_int]),
    "impdar_kirchhoff_f32": (_c_int, [_vp, _vp, _c_int, _c_int, _vp, _vp, _vp, _c_dbl, _c_int, _c_int, _c_int,
                                      _vp, _c_sz, _vp]),
    "impdar_kirchhoff_rows_f32": (_c_int, [_vp, _vp, _c_int, _c_int, _vp, _vp, _vp, _c_dbl, _c_int, _c_int, _c_int,
                                           _c_int, _c_int, _c_int, _vp, _c_sz, _vp]),
    "impdar_kirchhoff_input_window": (_c_int, [_c_int, _c_int, _vp, _vp, _c_dbl, _c_int, _c_int, _vp, _vp]),
    "impdar_kirchhoff_window_f32": (_c_int, [_vp, _c_int, _c_int, _c_int, _vp, _c_int, _c_int, _c_int, _vp, _vp, _vp,
                                             _c_dbl, _c_int, _c_int, _c_int, _c_int, _c_int, _c_int, _vp, _c_sz, _vp]),
    "impdar_kirchhoff_last_tile_standdown": (_c_int, [_vp]),
    "impdar_kirchhoff_host_workspace_bytes": (_c_sz, [_c_int, _c_int, _c_int]),
    "impdar_kirchhoff_host_pipelined_f64": (_c_int, [_vp, _vp, _c_int, _c_int, _vp, _vp, _vp, _c_dbl, _c_int, _c_int,
                                                     _vp, _c_sz, _vp]),
    "impdar_kirchhoff_window_vz_f32": (_c_int, [_vp, _c_int, _c_int, _c_int, _vp, _c_int, _c_int, _c_int, _vp, _vp,
                                                _vp, _vp, _c_int, _c_int, _c_int, _c_int, _c_int, _c_int, _vp, _c_sz,
                                                _vp]),
    "impdar_kirchhoff_input_window_vz": (_c_int, [_c_int, _c_int, _vp, _vp, _vp, _c_int, _c_int, _vp, _vp]),
    "impdar_kirchhoff_host_pipelined_vz_f64": (_c_int, [_vp, _vp, _c_int, _c_int, _vp, _vp, _vp, _vp, _c_int, _c_int,
                                                        _vp, _c_sz, _vp]),
    "impdar_kirchhoff_lateral_workspace_bytes": (_c_sz, [_c_int, _c_int, _c_int, _c_int]),
    "impdar_kirchhoff_window_vxz_f32": (_c_int, [_vp, _c_int, _c_int, _c_int, _vp, _c_int, _c_int, _c_int, _vp, _vp,
                                                 _vp, _vp, _c_int, _vp, _c_int, _c_int, _c_int, _vp, _c_sz, _vp]),
    "impdar_kirchhoff_enable_stats": (_c_int, [_c_int]),
    "impdar_kirchhoff_last_stats": (_c_int, [_vp, _vp]),
    "impdar_kirchhoff_set_mode": (_c_int, [_c_int]),
    "impdar_kirchhoff_last_path": (_c_int, []),
    "impdar_peer_alloc": (_c_int, [_c_sz, _vp, _vp]),
    "impdar_peer_free": (_c_int, [_vp]),
    "impdar_peer_open": (_c_int, [_vp, _vp]),
    "impdar_peer_close": (_c_int, [_vp]),
    "impdar_copy2d_f32": (_c_int, [_vp, _c_sz, _vp, _c_sz, _c_int, _c_int, _vp]),
    "mig_kirch_loop": (None, [_vp, _c_int, _c_int, _vp, _vp, _vp, _vp, _c_dbl, _vp, _c_dbl, _c_int]),
    "impdar_kirchhoff_host_f64": (_c_int, [_vp, _vp, _c_int, _c_int, _vp, _vp, _c_dbl, _c_int]),
    "impdar_stolt_workspace_bytes": (_c_sz, [_c_int, _c_int, _c_int]),
    "impdar_stolt_f32": (_c_int, [_vp, _vp, _c_int, _c_int, _c_int, _c_dbl, _c_dbl, _c_dbl, _c_dbl, _c_dbl, _c_int,
                                  _vp, _c_sz, _vp]),
    "impdar_stolt_force_r2c": (_c_int, [_c_int]),
    "impdar_stolt_set_pipeline": (_c_int, [_c_int]),
    "impdar_stolt_last_pipeline": (_c_int, []),
    "impdar_stolt_debug_stop_after": (_c_int, [_c_int]),
    "impdar_stolt_scan_workspace_bytes": (_c_sz, [_c_int, _c_int, _c_int]),
    "impdar_stolt_scan_f32": (_c_int, [_vp, _c_int, _c_int, _c_dbl, _c_dbl, _vp, _c_int, _c_dbl, _c_dbl, _c_int, _c_int,
                                       _c_int, _vp, _vp, _vp, _c_sz, _vp]),
    "impdar_phsh_set_legacy": (_c_int, [_c_int]),
    "impdar_phsh_workspace_bytes": (_c_sz, [_c_int, _c_int]),
    "impdar_phsh_ffd_workspace_bytes": (_c_sz, [_c_int, _c_int]),
    "impdar_phsh_ffd_f64": (_c_int, [_vp, _vp, _c_int, _c_int, _c_dbl, _c_dbl, _c_dbl, _vp, _vp, _c_dbl, _c_dbl,
                                     _vp, _c_sz, _vp]),
    "impdar_phsh_f32": (_c_int, [_vp, _vp, _c_int, _c_int, _c_dbl, _c_dbl, _c_dbl, _vp, _vp, _c_dbl, _c_dbl,
                                 _vp, _c_sz, _vp]),
    "impdar_wiener_f32": (_c_int, [_vp, _vp, _c_int, _c_int, _c_int, _c_int, _c_int, _c_dbl, _vp, _vp]),
    "impdar_wiener_f64": (_c_int, [_vp, _vp, _c_int, _c_int, _c_int, _c_int, _c_int, _c_dbl, _vp, _vp]),
    "impdar_median_f32": (_c_int, [_vp, _vp, _c_int, _c_int, _c_int, _c_int, _vp]),
    "impdar_median_f64": (_c_int, [_vp, _vp, _c_int, _c_int, _c_int, _c_int, _vp]),
    "impdar_interp_node_bytes": (_c_sz, []),
    "impdar_crop_f32": (_c_int, [_vp, _vp, _c_int, _c_int, _c_int, _c_int, _c_int, _c_int, _c_int, _c_int, _vp]),
    "impdar_crop_f64": (_c_int, [_vp, _vp, _c_int, _c_int, _c_int, _c_int, _c_int, _c_int, _c_int, _c_int, _vp]),
    "impdar_crop_bytes": (_c_int, [_vp, _vp, _c_int, _c_int, _c_int, _c_int, _c_int, _c_int, _c_int, _c_int, _c_int, _vp]),
    "impdar_shift_traces_f32": (_c_int, [_vp, _vp, _c_int, _c_int, _c_int, _vp, _vp]),
    "impdar_shift_traces_f32_f64": (_c_int, [_vp, _vp, _c_int, _c_int, _c_int, _vp, _vp]),
    "impdar_shift_traces_f64": (_c_int, [_vp, _vp, _c_int, _c_int, _c_int, _vp, _vp]),
    "impdar_restack_f32": (_c_int, [_vp, _vp, _c_int, _c_int, _c_int, _vp]),
    "impdar_restack_f32_f64": (_c_int, [_vp, _vp, _c_int, _c_int, _c_int, _vp]),
    "impdar_restack_f64": (_c_int, [_vp, _vp, _c_int, _c_int, _c_int, _vp]),
    "impdar_interp_rows_f32": (_c_int, [_vp, _vp, _c_int, _c_int, _c_int, _vp, _c_int, _vp]),
    "impdar_interp_rows_f32_f64": (_c_int, [_vp, _vp, _c_int, _c_int, _c_int, _vp, _c_int, _vp]),
    "impdar_interp_rows_f64": (_c_int, [_vp, _vp, _c_int, _c_int, _c_int, _vp, _c_int, _vp]),
    "impdar_interp_cols_f32": (_c_int, [_vp, _vp, _c_int, _c_int, _c_int, _vp, _c_int, _vp]),
    "impdar_interp_cols_f32_f64": (_c_int, [_vp, _vp, _c_int, _c_int, _c_int, _vp, _c_int, _vp]),
    "impdar_interp_cols_f64": (_c_int, [_vp, _vp, _c_int, _c_int, _c_int, _vp, _c_int, _vp]),
    "impdar_depth_workspace_bytes": (_c_sz, [_c_int, _c_int, _c_int, _c_int]),
    "impdar_depth_convert_f32": (_c_int, [_vp, _vp, _c_int, _c_int, _c_int, _vp, _vp, _c_int, _vp, _vp, _vp, _c_sz,
                                          _vp]),
    "impdar_depth_convert_f32_f64": (_c_int, [_vp, _vp, _c_int, _c_int, _c_int, _vp, _vp, _c_int, _vp, _vp, _vp,
                                              _c_sz, _vp]),
    "impdar_depth_convert_f64": (_c_int, [_vp, _vp, _c_int, _c_int, _c_int, _vp, _vp, _c_int, _vp, _vp, _vp, _c_sz,
                                          _vp]),
}

_lib = None
_lock = threading.Lock()


class BackendError(RuntimeError):
    """The CUDA backend reported a failure (CUDA / cuFFT error)."""


def load():
    """Load the shared library (once).  Raises if it has not been built: there is no fallback."""
    global _lib
    if _lib is not None:
        return _lib
    with _lock:
        if _lib is not None:
            return _lib
        if not os.path.exists(LIB_PATH):
            raise ImportError(
                "impdar_b200: %s is missing - build it with `python -m impdar_b200._build` "
                "(there is no CPU fallback)" % LIB_PATH)
        lib = ctypes.CDLL(LIB_PATH, mode=ctypes.RTLD_GLOBAL)
        for name, (res, args) in PROTOTYPES.items():
            fn = getattr(lib, name)  # AttributeError if the library does not export a declared symbol
            fn.restype = res
            fn.argtypes = args
        _lib = lib
    return _lib


def last_error():
    return load().impdar_b200_last_error().decode("utf-8", "replace")


def check(rc, exc_for_bad_arg=ValueError):
    """Turn a C status into the exception type the reference would raise."""
    if rc == 0:
        return
    msg = last_error()
    if rc == 1:
        raise exc_for_bad_arg(msg)
    raise BackendError("impdar_b200 backend failure (status %d): %s" % (rc, msg))
