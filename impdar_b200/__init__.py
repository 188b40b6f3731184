"""impdar_b200 - B200 (sm_100a) backend for ImpDAR's radargram migration + filtering hot path.

    import impdar_b200
    impdar_b200.install()          # rebinds impdar.lib.migrationlib.* and the RadarData filter methods
    dat.migrate(mtype='kirch')     # unchanged ImpDAR call, now running on the GPU

or, without ImpDAR installed, ``impdar_b200.RadarData`` offers the same hot-path methods.
"""
from . import migrationlib, filtering, processing, process  # noqa: F401  (process.process mirrors impdar.lib.process.process)
from .radardata import RadarData, RadarFlags  # noqa: F401
from .matio import load_mat  # noqa: F401  (StoDeep / ImpDAR .mat files, SURVEY.md 8f rank 4)
from .migrationlib import (migrationKirchhoff, migrationStolt, migrationPhaseShift,  # noqa: F401
                           migrationTimeWavenumber, getVelocityProfile, migrationKirchhoffLayered, rms_velocity,
                           migrationKirchhoffLateral)

__version__ = "0.1.0"

_MIGRATION_NAMES = ('migrationKirchhoff', 'migrationStolt', 'migrationPhaseShift', 'migrationTimeWavenumber')
_FILTER_NAMES = ('vertical_band_pass', 'horizontalfilt', 'adaptivehfilt',
                 # sibling filters on the same kernels (SURVEY.md 8f rank 2)
                 'highpass', 'lowpass', 'horizontal_band_pass', 'winavg_hfilt', 'rangegain', 'agc', 'denoise')
# index / resampling operations either side of the path (SURVEY.md 8f rank 3), bound from impdar_b200.processing
_PROCESSING_NAMES = ('reverse', 'crop', 'hcrop', 'restack', 'nmo', 'constant_sample_depth_spacing',
                     'traveltime_to_depth', 'constant_space', 'elev_correct', 'clean_GPS')
_saved = {}


def install():
    """Bind the backend behind the reference's seam (SURVEY.md 8b): the four migration callables on the
    ``impdar.lib.migrationlib`` module (looked up by RadarData.migrate at call time,
    _RadarDataFiltering.py:610-631) and vertical_band_pass / horizontalfilt / adaptivehfilt on the RadarData
    class (RadarData/__init__.py:119-121).  mtype 'su*' keeps routing to the reference's SeisUnix shim."""
    import impdar.lib.migrationlib as ref_mig
    from impdar.lib.RadarData import RadarData as RefRadarData
    if _saved:
        return
    for name in _MIGRATION_NAMES:
        _saved[('mig', name)] = getattr(ref_mig, name)
        setattr(ref_mig, name, getattr(migrationlib, name))
    for name in _FILTER_NAMES:
        _saved[('rd', name)] = getattr(RefRadarData, name)
        setattr(RefRadarData, name, getattr(filtering, name))
    for name in _PROCESSING_NAMES:
        _saved[('rd', name)] = getattr(RefRadarData, name)
        setattr(RefRadarData, name, getattr(processing, name))


def uninstall():
    """Restore the reference's own callables."""
    if not _saved:
        return
    import impdar.lib.migrationlib as ref_mig
    from impdar.lib.RadarData import RadarData as RefRadarData
    for (kind, name), fn in list(_saved.items()):
        setattr(ref_mig if kind == 'mig' else RefRadarData, name, fn)
    _saved.clear()
