"""-m "not gpu": host side of the tracer transport -- the --tracer / --tracerRef flags and their conflicts, the column
headings and CSV of a tracer series (a stand-in Field) with and without layers, --timeMean on tracer columns, the new
exports."""
import ctypes

import numpy
import pytest

BASE = ['-t', 'T.nc', '-u', 'U.nc', '-v', 'V.nc', '-l', '[(0,0),(1,1)],[(2,2),(3,1)]']


class _FakeField(object):
    """what fluxplot.main reads from a Field, with fluxTracer returning seeded numbers"""
    made = []

    def __init__(self, tFile, uFile, vFile, pts, sverdrup=False, meshFile=None):
        self.nt, self.nz = 5, 4
        self.asked = []
        self.timeObj = type('T', (), {'getTimeAsDate': lambda _self, i: f'day{i}'})()
        _FakeField.made.append(self)

    def layerInterfaces(self):
        return numpy.array([0.0, 10.0, 50.0, 200.0, 1000.0])

    def levelsForDepths(self, depths):
        return [int(numpy.argmin(numpy.abs(self.layerInterfaces() - d))) for d in depths]

    def fluxTracer(self, var, file=None, ref=0.0, layers=None):
        self.asked.append((var, file, ref, layers))
        shape = (self.nt, 2) if layers is None else (self.nt, len(layers) - 1, 2)
        self.series = numpy.random.default_rng(7).standard_normal(shape)
        return self.series


@pytest.fixture
def fake(monkeypatch):
    from nemoflux_b200 import fluxplot
    _FakeField.made = []
    monkeypatch.setattr(fluxplot, 'Field', _FakeField)
    return fluxplot


def test_tracer_flags_are_parsed_and_checked(fake):
    for bad in (['--tracerRef', '34.8'], ['--tracer', 'so', '--tracerRef', 'x'],
                ['--tracer', 'so', '--classField', 'thetao', '--classBounds', '0,1'],
                ['--tracer', 'so', '--section', 's.nc']):
        with pytest.raises(SystemExit) as e:                # refused before any file is opened
            fake.main(BASE + bad)
        assert e.value.code == 2
    assert _FakeField.made == []
    fake.main(BASE + ['--tracer', 'so:S.nc', '--tracerRef=34.8'])
    fake.main(BASE + ['--tracer', 'thetao', '--layers', '0,2,4'])
    fake.main(BASE + ['--tracer', 'thetao', '--depthLayers', '0,50,1000', '--tracerRef=-1.5'])
    assert [f.asked for f in _FakeField.made] == [[('so', 'S.nc', 34.8, None)], [('thetao', None, 0.0, [0, 2, 4])],
                                                 [('thetao', None, -1.5, [0, 2, 4])]]


def test_tracer_columns_and_csv(fake, tmp_path, capsys):
    assert fake.tracerLabels(['S1', 'S2'], 'thetao') == ['S1[thetao]', 'S2[thetao]']
    assert fake.tracerLabels(['S1', 'S2'], 'so', [0.0, 10.0, 50.0], [0, 1, 2]) == \
        ['S1[so 0-10 m]', 'S1[so 10-50 m]', 'S2[so 0-10 m]', 'S2[so 10-50 m]']
    csv = str(tmp_path / 't.csv')
    series = fake.main(BASE + ['--tracer', 'thetao', '-o', csv])
    fld = _FakeField.made[-1]
    assert numpy.array_equal(series, fld.series)
    out = capsys.readouterr().out
    with open(csv, encoding='utf-8') as fh:
        rows = [r.rstrip('\n').split(',') for r in fh]
    assert len(rows[0]) == 3 and all(h.endswith('[thetao]') for h in rows[0][1:])
    assert 'time,' + ','.join(rows[0][1:]) + '   [thetao x A m^2/s]' in out
    vals = numpy.array([[float(x) for x in r[1:]] for r in rows[1:]])
    assert numpy.array_equal(vals, fld.series)
    series = fake.main(BASE + ['--tracer', 'so', '--layers', '0,1,3', '-s', '-o', csv])
    fld = _FakeField.made[-1]
    out = capsys.readouterr().out
    with open(csv, encoding='utf-8') as fh:
        rows = [r.rstrip('\n').split(',') for r in fh]
    assert [h[h.index('['):] for h in rows[0][1:]] == ['[so 0-10 m]', '[so 10-200 m]'] * 2
    assert '[so x Sv]' in out
    vals = numpy.array([[float(x) for x in r[1:]] for r in rows[1:]])
    assert numpy.array_equal(vals, fld.series.transpose(0, 2, 1).reshape(5, -1))     # transect-major columns


def test_tracer_columns_time_mean(fake, tmp_path):
    csv = str(tmp_path / 'm.csv')
    series = fake.main(BASE + ['--tracer', 'so', '--timeMean', '2', '-o', csv])
    fld = _FakeField.made[-1]
    assert numpy.array_equal(series, fake.windowMeans(fld.series, [0, 2, 4, 5]))
    with open(csv, encoding='utf-8') as fh:
        rows = [r.rstrip('\n').split(',') for r in fh]
    assert [r[0] for r in rows[1:]] == ['day0/day1', 'day2/day3', 'day4/day4']


def test_tracer_entry_points_are_exported():
    from nemoflux_b200 import _lib, nemoflux_gpu
    from nemoflux_b200.field import Field
    lib = ctypes.CDLL(_lib.LIB_PATH)
    for name in ('nfx_flux_tracer', 'nfx_flux_tracer_host'):
        assert hasattr(lib, name) and name in _lib.SIGNATURES
    assert len(_lib.SIGNATURES['nfx_flux_tracer']) == 24
    assert len(_lib.SIGNATURES['nfx_flux_tracer_host']) == 24
    assert callable(nemoflux_gpu.PolylineIntegral.fluxTracer) and callable(Field.fluxTracer)
