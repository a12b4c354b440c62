"""-m "not gpu": host side of the time-mean section -- window bounds from the calendar (standard, noleap, 360_day) and
from a step count, the error without a time axis, --timeMean parsing and the series window means, the --section
writer's time_bnds / cell_methods, the new exports."""
import argparse
import ctypes
import datetime

import numpy
import pytest

from nemoflux_b200 import timeobj


class _Var(object):
    """what TimeObj reads from a variable of a dataset"""

    def __init__(self, data, **attrs):
        self.data = numpy.asarray(data)
        self.__dict__.update(attrs)

    def __getitem__(self, idx):
        return self.data[idx]

    def __len__(self):
        return len(self.data)


def _axis(values, units='days since 2000-01-01', calendar=None, bounds=None):
    attrs = dict(standard_name='time', units=units)
    if calendar:
        attrs['calendar'] = calendar
    nc = {}
    if bounds is not None:
        attrs['bounds'] = 'time_centered_bounds'
        nc['time_centered_bounds'] = _Var(bounds)
    nc['time_centered'] = _Var(values, **attrs)
    return timeobj.TimeObj(nc)


def _expected(keys):
    return [0] + [i for i in range(1, len(keys)) if keys[i] != keys[i - 1]] + [len(keys)]


def test_windows_of_n_steps():
    t = _axis(numpy.arange(10.))
    assert timeobj.timeWindows(t, 10, 3) == [0, 3, 6, 9, 10]
    assert timeobj.timeWindows(t, 10, '5') == [0, 5, 10]
    assert timeobj.timeWindows(t, 10, 10) == [0, 10]
    assert timeobj.timeWindows(t, 10, 20) == [0, 10]
    assert timeobj.timeWindows(None, 4, 1) == [0, 1, 2, 3, 4]
    for bad in (0, -2, 'week', 2.5, None):
        with pytest.raises(ValueError):
            timeobj.timeWindows(t, 10, bad)


def test_windows_by_month_and_year_standard():
    days = numpy.arange(0., 800., 5.) + 0.5          # every 5 days from 2000-01-01, over a leap year
    t = _axis(days)
    origin = datetime.date(2000, 1, 1)
    dates = [origin + datetime.timedelta(days=float(d)) for d in days]
    assert timeobj.timeWindows(t, days.size, 'month') == _expected([(d.year, d.month) for d in dates])
    assert timeobj.timeWindows(t, days.size, 'year') == _expected([d.year for d in dates])
    assert len(timeobj.timeWindows(t, days.size, 'year')) == 4      # 2000, 2001, 2002
    # 29 February 2000 exists: a daily axis puts 29 days in February
    daily = _axis(numpy.arange(70.) * 86400., units='seconds since 2000-01-01 00:00:00')
    b = timeobj.timeWindows(daily, 70, 'month')
    assert b == [0, 31, 60, 70]


def test_windows_by_month_and_year_noleap_and_360_day():
    for cal in ('noleap', '365_day'):
        t = _axis(numpy.arange(400.), units='days since 1999-01-01', calendar=cal)
        b = timeobj.timeWindows(t, 400, 'month')
        lengths = numpy.diff(b)
        assert list(lengths[:12]) == [31, 28, 31, 30, 31, 30, 31, 31, 30, 31, 30, 31], cal
        assert timeobj.timeWindows(t, 400, 'year') == [0, 365, 400]
    t = _axis(numpy.arange(0., 800., 1.), units='days since 1990-01-01', calendar='360_day')
    b = timeobj.timeWindows(t, 800, 'month')
    assert all(x == 30 for x in numpy.diff(b)[:-1]) and b[-1] == 800
    assert timeobj.timeWindows(t, 800, 'year') == [0, 360, 720, 800]
    # monthly means stamped mid-month (NEMO's time_centered): one window each
    mid = numpy.array([15.5 + 30 * k for k in range(24)])
    assert timeobj.timeWindows(_axis(mid, calendar='360_day'), 24, 'month') == list(range(25))


def test_calendar_windows_need_a_time_axis():
    none = timeobj.TimeObj({})
    for spec in ('month', 'year'):
        with pytest.raises(ValueError, match='time axis'):
            timeobj.timeWindows(none, 6, spec)
        with pytest.raises(ValueError, match='time axis'):      # a time axis of another length
            timeobj.timeWindows(_axis(numpy.arange(4.)), 6, spec)
        with pytest.raises(ValueError, match='time axis'):      # undecodable units
            timeobj.timeWindows(_axis(numpy.arange(6.), units='days'), 6, spec)
    assert timeobj.timeWindows(none, 6, 4) == [0, 4, 6]


def test_time_bounds_variable():
    b = numpy.stack([numpy.arange(3.) * 10, numpy.arange(3.) * 10 + 10], 1)
    t = _axis(numpy.arange(3.) * 10 + 5, bounds=b)
    assert numpy.array_equal(t.getBounds(), b)
    assert _axis(numpy.arange(3.)).getBounds() is None


def test_time_mean_flag_and_series_means():
    from nemoflux_b200 import fluxplot
    assert fluxplot.parseTimeMean('3') == 3 and fluxplot.parseTimeMean('month') == 'month'
    assert fluxplot.parseTimeMean(' Year ') == 'year'
    for bad in ('0', '-1', '2.5', 'week', ''):
        with pytest.raises(argparse.ArgumentTypeError):
            fluxplot.parseTimeMean(bad)
    base = ['-t', 'T.nc', '-u', 'U.nc', '-v', 'V.nc', '-l', '(0,0),(1,1)']
    for bad in (['--timeMean'], ['--timeMean', 'week'], ['--timeMean', '0']):
        with pytest.raises(SystemExit) as e:                # refused before any file is opened
            fluxplot.main(base + bad)
        assert e.value.code == 2
    rng = numpy.random.default_rng(1)
    x = rng.standard_normal((7, 3, 2)) * 10. ** rng.integers(-5, 5, (7, 3, 2))
    x[2, 0, 0] = -0.0
    b = [0, 2, 3, 7]
    m = fluxplot.windowMeans(x, b)
    assert m.shape == (3, 3, 2)
    for w in range(3):
        acc = numpy.zeros((3, 2))
        for t in range(b[w], b[w + 1]):
            acc = acc + x[t]
        assert numpy.array_equal(m[w], acc / (b[w + 1] - b[w]))
    assert not numpy.signbit(m[1, 0, 0])                  # a one-step window of -0 is +0


class _FakeField(object):
    """what fluxplot.writeSection reads from a Field, with a time axis of nt values and optional CF bounds"""

    def __init__(self, nt, nz, nsub, bounds=None):
        from nemoflux_b200 import nemoflux_gpu
        self.nt, self.nz, self.nsub = nt, nz, nsub
        offs = numpy.array([0, nsub // 3, nsub], numpy.int64)
        rng = numpy.random.default_rng(3)
        sub = dict(offsets=offs, cell=rng.integers(0, 40, nsub), seg=numpy.zeros(nsub, numpy.int32),
                   ta=numpy.linspace(0, 1, nsub + 1)[:-1], tb=numpy.linspace(0, 1, nsub + 1)[1:])
        geo = nemoflux_gpu.sectionGeometry(sub, [numpy.array([[0., 0., 0.], [3., 1., 0.]])] * 2, 8)
        self.pli = type('P', (), {'getSectionGeometry': lambda _self: geo})()
        self.timeObj = _axis(numpy.arange(nt) * 86400. + 43200., units='seconds since 1900-01-01', calendar='noleap',
                             bounds=bounds)
        self.rng = rng
        self.asked = []

    def layerInterfaces(self):
        return 10. * numpy.arange(self.nz + 1)

    def fluxSection(self, layers, windows=None):
        self.asked.append((list(layers), windows))
        self.sec = self.rng.standard_normal((self.nt if windows is None else len(windows) - 1, len(layers) - 1,
                                             self.nsub))
        return self.sec


@pytest.mark.parametrize('with_bounds', [False, True])
def test_section_writer_time_bnds(tmp_path, with_bounds):
    from nemoflux_b200 import fluxplot, ncio
    nt = 5
    stamps = numpy.arange(nt) * 86400. + 43200.
    bnds = numpy.stack([stamps - 43200., stamps + 43200.], 1) if with_bounds else None
    fld = _FakeField(nt=nt, nz=4, nsub=7, bounds=bnds)
    path = str(tmp_path / 'mean.nc')
    W = [0, 2, 4, 5]
    assert fluxplot.writeSection(path, fld, [0, 1, 4], 'Sv', W) == 7
    assert fld.asked == [([0, 1, 4], W)]
    with ncio.open_dataset(path) as nc:
        tr_ = nc['transport']
        assert tuple(tr_.shape) == (3, 2, 7)
        assert numpy.array_equal(numpy.asarray(tr_[:]), fld.sec)
        assert getattr(tr_, 'cell_methods', None) == 'time: mean'
        assert getattr(nc['time'], 'bounds', None) == 'time_bnds'
        assert numpy.array_equal(nc['time'][:], [stamps[0:2].mean(), stamps[2:4].mean(), stamps[4]])
        tb = numpy.asarray(nc['time_bnds'][:])
        if with_bounds:
            assert numpy.array_equal(tb, [[0., 2 * 86400.], [2 * 86400., 4 * 86400.], [4 * 86400., 5 * 86400.]])
        else:
            assert numpy.array_equal(tb, [[stamps[0], stamps[1]], [stamps[2], stamps[3]], [stamps[4], stamps[4]]])
    # without windows: the per-step file, no time_bnds, no cell_methods
    path2 = str(tmp_path / 'steps.nc')
    fluxplot.writeSection(path2, fld, [0, 1, 4], 'Sv')
    assert fld.asked[-1] == ([0, 1, 4], None)
    with ncio.open_dataset(path2) as nc:
        assert tuple(nc['transport'].shape) == (nt, 2, 7)
        assert getattr(nc['transport'], 'cell_methods', None) is None
        assert 'time_bnds' not in nc


def test_section_mean_entry_points_are_exported():
    from nemoflux_b200 import _lib
    lib = ctypes.CDLL(_lib.LIB_PATH)
    for name in ('nfx_flux_section_window_sums', 'nfx_flux_section_window_sums_host'):
        assert hasattr(lib, name) and name in _lib.SIGNATURES
    assert len(_lib.SIGNATURES['nfx_flux_section_window_sums']) == 22
    assert len(_lib.SIGNATURES['nfx_flux_section_window_sums_host']) == 22
