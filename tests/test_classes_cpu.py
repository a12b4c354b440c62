"""-m "not gpu": host side of the class transport -- the --classField / --classBounds flags and their conflicts, the
column headings and CSV of a class series (a stand-in Field), --timeMean on class columns, the new exports."""
import ctypes

import numpy
import pytest

BASE = ['-t', 'T.nc', '-u', 'U.nc', '-v', 'V.nc', '-l', '[(0,0),(1,1)],[(2,2),(3,1)]']


class _FakeField(object):
    """what fluxplot.main reads from a Field, with fluxClasses returning seeded numbers"""
    made = []

    def __init__(self, tFile, uFile, vFile, pts, sverdrup=False, meshFile=None):
        self.nt, self.nz = 5, 4
        self.asked = []
        self.timeObj = type('T', (), {'getTimeAsDate': lambda _self, i: f'day{i}'})()
        _FakeField.made.append(self)

    def fluxClasses(self, var, bounds, file=None):
        self.asked.append((var, list(bounds), file))
        self.series = numpy.random.default_rng(7).standard_normal((self.nt, len(bounds) - 1, 2))
        return self.series


@pytest.fixture
def fake(monkeypatch):
    from nemoflux_b200 import fluxplot
    _FakeField.made = []
    monkeypatch.setattr(fluxplot, 'Field', _FakeField)
    return fluxplot


def test_class_flags_are_parsed_and_checked(fake):
    assert fake.parseList('-inf,-1.5, 0,27.8,inf') == [-numpy.inf, -1.5, 0.0, 27.8, numpy.inf]
    for bad in (['--classField', 'thetao'], ['--classBounds', '0,1'], ['--classField', 'thetao', '--classBounds', '3'],
                ['--classField', 'so', '--classBounds', '0,x'],
                ['--classField', 'so', '--classBounds', '0,1', '--layers', '0,2,4'],
                ['--classField', 'so', '--classBounds', '0,1', '--depthLayers', '0,100']):
        with pytest.raises(SystemExit) as e:                # refused before any file is opened
            fake.main(BASE + bad)
        assert e.value.code == 2
    assert _FakeField.made == []
    fake.main(BASE + ['--classField', 'sigma0:rho.nc', '--classBounds=-inf,27.8,inf'])   # '=': a leading minus
    fake.main(BASE + ['--classField', 'thetao', '--classBounds=-2,0,4'])
    assert [f.asked for f in _FakeField.made] == [[('sigma0', [-numpy.inf, 27.8, numpy.inf], 'rho.nc')],
                                                 [('thetao', [-2.0, 0.0, 4.0], None)]]


def test_class_columns_and_csv(fake, tmp_path, capsys):
    labels = fake.classLabels(['S1', 'S2'], [-numpy.inf, 0.0, 27.8, numpy.inf])
    assert labels == ['S1[-inf–0)', 'S1[0–27.8)', 'S1[27.8–inf)', 'S2[-inf–0)', 'S2[0–27.8)', 'S2[27.8–inf)']
    csv = str(tmp_path / 'c.csv')
    series = fake.main(BASE + ['--classField', 'so', '--classBounds', '33,34.8,36', '-o', csv])
    fld = _FakeField.made[-1]
    assert numpy.array_equal(series, fld.series)
    out = capsys.readouterr().out
    with open(csv, encoding='utf-8') as fh:
        rows = [r.rstrip('\n').split(',') for r in fh]
    heads = rows[0]
    assert heads[0] == 'time' and len(heads) == 5
    assert [h[h.index('['):] for h in heads[1:]] == ['[33–34.8)', '[34.8–36)'] * 2
    assert heads[1][:heads[1].index('[')] == heads[2][:heads[2].index('[')] != heads[3][:heads[3].index('[')]
    assert 'time,' + ','.join(heads[1:]) in out
    vals = numpy.array([[float(x) for x in r[1:]] for r in rows[1:]])
    assert numpy.array_equal(vals, fld.series.transpose(0, 2, 1).reshape(5, -1))     # transect-major columns
    assert [r[0] for r in rows[1:]] == [f'day{i}' for i in range(5)]


def test_class_columns_time_mean(fake, tmp_path):
    csv = str(tmp_path / 'm.csv')
    series = fake.main(BASE + ['--classField', 'so', '--classBounds', '33,34.8,36', '--timeMean', '2', '-o', csv])
    fld = _FakeField.made[-1]
    assert numpy.array_equal(series, fake.windowMeans(fld.series, [0, 2, 4, 5]))
    with open(csv, encoding='utf-8') as fh:
        rows = [r.rstrip('\n').split(',') for r in fh]
    assert [r[0] for r in rows[1:]] == ['day0/day1', 'day2/day3', 'day4/day4']


def test_class_entry_points_are_exported():
    from nemoflux_b200 import _lib, nemoflux_gpu
    from nemoflux_b200.field import Field
    lib = ctypes.CDLL(_lib.LIB_PATH)
    for name in ('nfx_flux_classes', 'nfx_flux_classes_host'):
        assert hasattr(lib, name) and name in _lib.SIGNATURES
    assert len(_lib.SIGNATURES['nfx_flux_classes']) == 22
    assert len(_lib.SIGNATURES['nfx_flux_classes_host']) == 22
    assert callable(nemoflux_gpu.PolylineIntegral.fluxClasses) and callable(Field.fluxClasses)
