"""StoDeep / ImpDAR .mat files (SURVEY.md 8f rank 4): impdar_b200.load_mat / RadarData.save against the reference's own
loader and writer.  Fixtures tests/golden/mat_*.mat were written by the UNMODIFIED reference
(tests/golden/make_golden_mat.py); the `reference`-marked tests additionally run the reference itself on its own test
input files (an ImpDAR checkout at IMPDAR_REFERENCE_SRC, default /root/reference/src) and skip without it."""
import os

import numpy as np
import pytest
from scipy.io import loadmat

import impdar_b200
from impdar_b200 import matio
from conftest import GOLDEN_DIR

ATTRS = matio.ATTRS_GUARANTEED + matio.ATTRS_OPTIONAL + ['data_dtype']
FLAG_ATTRS = ['batch', 'bpass', 'hfilt', 'rgain', 'agc', 'restack', 'reverse', 'crop', 'nmo', 'interp', 'mig', 'elev']


def _same(x, y):
    if x is None or y is None:
        return x is None and y is None
    return type(x) is type(y) and np.array_equal(np.asarray(x), np.asarray(y))


def _mat_equal(a, b):
    """Two loadmat dicts carry the same variables with the same shapes, dtypes and values (structs field by field)."""
    ka = sorted(k for k in a if not k.startswith('__'))
    kb = sorted(k for k in b if not k.startswith('__'))
    assert ka == kb
    for k in ka:
        x, y = a[k], b[k]
        assert x.dtype == y.dtype and x.shape == y.shape, k
        if x.dtype.names:
            for f in x.dtype.names:
                assert np.array_equal(np.asarray(x[f][0][0]), np.asarray(y[f][0][0])), (k, f)
        else:
            assert np.array_equal(x, y, equal_nan=x.dtype.kind == 'f'), k


def test_load_fixture_written_by_reference():
    d = impdar_b200.load_mat(os.path.join(GOLDEN_DIR, 'mat_ref_saved.mat'))
    assert d.data.shape == (17, 40) and d.data.dtype == np.float64 and d.data_dtype == np.float64
    assert d.snum == 17 and d.tnum == 40 and d.nmo_depth.shape == (17,) and d.travel_time.shape == (17,)
    assert d.flags.mig == 'stolt' and np.array_equal(d.flags.bpass, [1., 2., 10.]) and d.flags.crop[0] == 1
    assert d.flags.crop[1] == 13 and d.flags.nmo[0] == 1     # the source file was already cropped by 10
    assert d.flags.reverse in (False, 0) and d.picks is None
    assert isinstance(d.trig, np.ndarray) and d.trig.shape == (40,)


def test_round_trip_equals_reference_round_trip(tmp_path):
    """load -> save of a reference-written file gives the file the reference's own load -> save gives."""
    d = impdar_b200.load_mat(os.path.join(GOLDEN_DIR, 'mat_ref_saved.mat'))
    out = os.path.join(str(tmp_path), 'again.mat')
    d.save(out)
    want = loadmat(os.path.join(GOLDEN_DIR, 'mat_ref_resaved.mat'))
    got = loadmat(out)
    want.pop('picks', None)          # the reference attaches an empty Picks object on load; picks are not carried here
    want['fn'] = got['fn']           # the path the file was read from
    _mat_equal(got, want)
    again = impdar_b200.load_mat(out)
    for a in ATTRS:
        if a != 'fn':
            assert _same(getattr(d, a), getattr(again, a)), a


def test_dtype_preservation_rules(tmp_path):
    d = impdar_b200.load_mat(os.path.join(GOLDEN_DIR, 'mat_ref_f32.mat'))
    assert d.data.dtype == np.float32 and d.data_dtype == np.float32 and d.elev is None
    out = os.path.join(str(tmp_path), 'x.mat')
    d.data = d.data.astype(np.float64) * 1.5              # processing widened the radargram: the file keeps float32
    d.save(out)
    assert loadmat(out)['data'].dtype == np.float32
    # (the reference picks float16 for int16 data; MAT v5 has no half type, scipy's writer stores it as double)
    for want, expect in ((np.dtype(np.int16), np.float64), (np.dtype(np.int32), np.float32), (np.dtype(np.int64), np.float64)):
        d.data_dtype = want
        d.data = np.arange(20 * 40, dtype=np.float64).reshape(20, 40)
        d.save(out)
        assert loadmat(out)['data'].dtype == want         # no NaNs: back to the integer type the file came with
        d.data[3, 4] = np.nan
        d.save(out)
        assert loadmat(out)['data'].dtype == expect       # NaNs appeared: the smallest float that keeps them
    d.trig_level = None                                   # None in a guaranteed attribute is written as 0
    d.save(out)
    assert loadmat(out)['trig_level'].shape == (1, 1) and loadmat(out)['trig_level'][0, 0] == 0


def test_format_errors(tmp_path):
    from scipy.io import savemat
    bad = os.path.join(str(tmp_path), 'bad.mat')
    savemat(bad, {'data': np.zeros((3, 4))})
    with pytest.raises(KeyError):
        impdar_b200.load_mat(bad)
    savemat(bad, {'chan': 1, 'dt': 1.0})
    with pytest.raises(KeyError):
        impdar_b200.load_mat(bad)
    good = loadmat(os.path.join(GOLDEN_DIR, 'mat_ref_saved.mat'))
    good = {k: v for k, v in good.items() if not k.startswith('__')}
    good['snum'] = 5                                      # inconsistent with the radargram
    good['flags'] = impdar_b200.RadarFlags().to_matlab()
    good.pop('elev')
    savemat(bad, good)
    with pytest.raises(matio.ImpdarError):
        impdar_b200.load_mat(bad)
    good['filtdata'] = good.pop('data')                   # lower-priority StoDeep name is promoted to `data`
    good['snum'] = 17
    savemat(bad, good)
    d = impdar_b200.load_mat(bad)
    assert d.data.shape == (17, 40) and not hasattr(d, 'filtdata')


@pytest.mark.reference
@pytest.mark.parametrize('name', ['small_data.mat', 'small_data_otherstodeepattrs.mat', 'small_just_otherstodeepattrs.mat',
                                  'small_data_picks.mat'])
def test_load_matches_reference_loader(name):
    from oracle._refimport import import_reference, REFERENCE_SRC
    _, RefRadarData, _ = import_reference()
    fn = os.path.join(os.path.dirname(REFERENCE_SRC), 'test', 'input_data', name)
    r, d = RefRadarData(fn), impdar_b200.load_mat(fn)
    for a in ATTRS:
        assert _same(getattr(r, a), getattr(d, a)), a
    for a in matio.STODEEP_ATTRS[1:]:
        assert _same(getattr(r, a, None), getattr(d, a, None)), a
    for a in FLAG_ATTRS:
        assert np.array_equal(np.asarray(getattr(r.flags, a)), np.asarray(getattr(d.flags, a))), a


@pytest.mark.reference
@pytest.mark.parametrize('name', ['nonimpdar_matlab.mat', 'nonimpdar_justmissingdat.mat'])
def test_bad_files_raise_like_reference(name):
    from oracle._refimport import import_reference, REFERENCE_SRC
    _, RefRadarData, _ = import_reference()
    fn = os.path.join(os.path.dirname(REFERENCE_SRC), 'test', 'input_data', name)
    with pytest.raises(KeyError):
        RefRadarData(fn)
    with pytest.raises(KeyError):
        impdar_b200.load_mat(fn)


def test_save_matches_reference_writer(tmp_path):
    """The same object written by both: the reference loaded mat_ref_picks.mat and saved it as
    mat_ref_picks_resaved.mat; load_mat -> save of that file gives identical variables, shapes, dtypes, values (the
    picks struct, which the reference re-boxes on every pass, is compared field by field in
    test_picks_survive_load_filter_save)."""
    d = impdar_b200.load_mat(os.path.join(GOLDEN_DIR, 'mat_ref_picks.mat'), pinned=False)
    b = os.path.join(str(tmp_path), 'mine.mat')
    d.save(b)
    got, want = loadmat(b), loadmat(os.path.join(GOLDEN_DIR, 'mat_ref_picks_resaved.mat'))
    got.pop('picks')
    want.pop('picks')
    want['fn'] = got['fn']           # the path the file was read from
    _mat_equal(got, want)


@pytest.mark.gpu
def test_loaded_radargram_is_page_locked_and_feeds_the_device_chain():
    import torch
    d = impdar_b200.load_mat(os.path.join(GOLDEN_DIR, 'mat_ref_f32.mat'))
    assert torch.from_numpy(d.data).is_pinned()
    d.trig = np.zeros(d.tnum)
    d.hfilt(ftype='hfilt', bounds=(0, d.tnum))
    assert d.data.dtype == np.float32 and d.flags.hfilt[0] == 1


def _struct_equal(x, y, path=''):
    if x.dtype.names:
        assert x.dtype.names == y.dtype.names and x.shape == y.shape, path
        for f in x.dtype.names:
            _struct_equal(x[f][0, 0], y[f][0, 0], path + '.' + f)
    elif x.dtype == object:
        assert y.dtype == object and x.shape == y.shape, path
        for a, b in zip(x.flat, y.flat):
            _struct_equal(a, b, path + '[]')
    else:
        assert x.shape == y.shape and x.dtype == y.dtype and np.array_equal(x, y, equal_nan=x.dtype.kind == 'f'), path


def test_picks_survive_load_filter_save(tmp_path):
    """A picked profile written by the reference: load_mat -> (a step that keeps both axes) -> save writes the picks back
    verbatim; once a step has changed an axis the stale struct is not written and save says so."""
    import warnings
    src = os.path.join(GOLDEN_DIR, 'mat_ref_picks.mat')
    d = impdar_b200.load_mat(src, pinned=False)
    assert d.picks is None and d.picks_struct is not None
    d.flags.bpass = np.array([1., 2., 10.])              # host-side stand-in for an in-place filter step
    out = os.path.join(str(tmp_path), 'picks_again.mat')
    with warnings.catch_warnings():
        warnings.simplefilter('error')
        d.save(out)
    got = loadmat(out)
    assert 'picks' in got
    _struct_equal(got['picks'], loadmat(src)['picks'])           # field by field, nested pickparams included
    # ... and once more: the round trip is the identity (the reference's own load -> save re-boxes the nested struct
    # fields at every pass, mat_ref_picks_resaved.mat; its numeric fields agree with ours)
    impdar_b200.load_mat(out, pinned=False).save(out)
    _struct_equal(loadmat(out)['picks'], loadmat(src)['picks'])
    want = loadmat(os.path.join(GOLDEN_DIR, 'mat_ref_picks_resaved.mat'))['picks']
    for f in ('samp1', 'samp2', 'samp3', 'time', 'power', 'picknums'):
        assert np.array_equal(got['picks'][f][0, 0], want[f][0, 0], equal_nan=True), f
    # an axis changed (hcrop-like): the raw struct no longer describes the radargram
    d2 = impdar_b200.load_mat(src, pinned=False)
    d2.data = np.ascontiguousarray(d2.data[:, :30])
    d2.tnum = 30
    with pytest.warns(RuntimeWarning, match='picks'):
        d2.save(os.path.join(str(tmp_path), 'picks_cropped.mat'))
    assert 'picks' not in loadmat(os.path.join(str(tmp_path), 'picks_cropped.mat'))
