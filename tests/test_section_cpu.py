"""-m "not gpu": host side of the transport section -- the crossing geometry against the oracle's sub-segments, the
fluxplot --section flag and file, the new exports."""
import ctypes

import numpy
import pytest

from helpers import tr


def _oracle_sub(oracle, points, paths):
    """getSubsegments()-shaped dict from the oracle's emission list of every transect"""
    g = oracle.Grid(points)
    subs = []
    for path in paths:
        p = oracle.PolylineIntegral(g)
        p.computeWeights(tr(path))
        cells, edges, w = p.emission_list()
        assert numpy.array_equal(cells[::4], p.subsegs['cell']) and numpy.array_equal(edges[:4], [0, 1, 2, 3])
        subs.append(p.subsegs)
    allsub = numpy.concatenate(subs)
    offs = numpy.concatenate([[0], numpy.cumsum([len(s) for s in subs])]).astype(numpy.int64)
    return dict(offsets=offs, cell=allsub['cell'], seg=allsub['seg'], ta=allsub['ta'], tb=allsub['tb'],
                coeff=allsub['coeff'])


def _gc(a, b):
    from nemoflux_b200.nemoflux_gpu import _great_circle_km
    return float(_great_circle_km(numpy.array([a], float), numpy.array([b], float))[0])


def test_section_geometry_against_the_oracle(oracle):
    from nemoflux_b200.nemoflux_gpu import sectionGeometry
    d = oracle.DataGen(nx=72, ny=36)                                  # 5 degree cells
    paths = [[(-33.3, -61.2), (-33.3, 48.9)],                         # meridional, off the grid lines: a great circle
             [(-120.2, -40.1), (-33.3, 12.6), (70.4, -60.3), (100.1, 50.2)],
             [(-30., -40.), (-30., 40.)],                             # along a grid line: cells on both sides
             [(170.2, 10.3), (189.6, 10.3)]]                          # across the x-period seam
    sub = _oracle_sub(oracle, d.points(), paths)
    geo = sectionGeometry(sub, [numpy.asarray(tr(p)) for p in paths], 72)
    offs = sub['offsets']
    assert numpy.array_equal(geo['offsets'], offs)
    assert numpy.array_equal(geo['cell_j'] * 72 + geo['cell_i'], sub['cell'])
    for m, path in enumerate(paths):
        a, b = offs[m], offs[m + 1]
        assert b > a and numpy.all(geo['transect'][a:b] == m)
        dist = geo['distance_km'][a:b]
        assert numpy.all(numpy.diff(dist) >= -1e-9), m             # emission order runs along the transect
        seg = geo['segment'][a:b]
        assert numpy.all(numpy.diff(seg) >= 0)
        for j in range(len(path) - 1):
            k = seg == j
            ln = (geo['length_km'][a:b][k] * sub['coeff'][a:b][k]).sum()
            full = _gc(path[j], path[j + 1])
            # a meridian is a great circle: the crossings add up to its length; elsewhere the segment (a straight
            # line in lon/lat) is longer than the great circle, and its crossings' chords come close to its length
            if path[j][0] == path[j + 1][0]:
                assert abs(ln - full) <= 1e-9 * full, (m, j, ln, full)
            else:
                from nemoflux_b200.nemoflux_gpu import _great_circle_km
                fine = numpy.asarray(path[j]) + numpy.linspace(0., 1., 20001)[:, None] * numpy.subtract(path[j + 1], path[j])
                curve = _great_circle_km(fine[:-1], fine[1:]).sum()
                assert full < ln <= curve + 1e-9 and ln >= (1 - 1e-3) * curve, (m, j, ln, full, curve)
            # end points on the polyline, in its own coordinates (no x-period image shift)
            lo, hi = numpy.minimum(path[j], path[j + 1]), numpy.maximum(path[j], path[j + 1])
            for key, c in (('lon0', 0), ('lon1', 0), ('lat0', 1), ('lat1', 1)):
                x = geo[key][a:b][k]
                assert numpy.all(x >= lo[c] - 1e-9) and numpy.all(x <= hi[c] + 1e-9), (m, key)
        # the first crossing starts at the transect's start (inside the grid), the midpoint distance is measured
        # from there
        assert numpy.allclose([geo['lon0'][a], geo['lat0'][a]], path[0], atol=1e-12)
        mid = (0.5 * (geo['lon0'][a] + geo['lon1'][a]), 0.5 * (geo['lat0'][a] + geo['lat1'][a]))
        assert abs(geo['distance_km'][a] - _gc(path[0], mid)) <= 1e-9 * max(1., geo['distance_km'][a])
    # the grid-line transect: the cells on both sides hold its crossings, with duplicity coefficients (the length
    # check above weighs the crossings with them)
    a, b = offs[2], offs[3]
    assert numpy.any(sub['coeff'][a:b] != 1.) and (b - a) % 2 == 0
    # the seam: longitudes run on continuously past 180
    a, b = offs[3], offs[4]
    assert geo['lon1'][a:b].max() > 180. and numpy.all(numpy.diff(geo['lon0'][a:b]) > 0)
    # later segments start where the earlier ones end
    a, b = offs[1], offs[2]
    first = geo['segment'][a:b] == 1
    start1 = _gc(paths[1][0], paths[1][1])
    assert geo['distance_km'][a:b][first].min() >= start1 - 1e-9


def test_section_geometry_of_no_crossing():
    from nemoflux_b200.nemoflux_gpu import sectionGeometry
    empty = dict(offsets=numpy.zeros(3, numpy.int64), cell=numpy.zeros(0, numpy.int64), seg=numpy.zeros(0, numpy.int32),
                 ta=numpy.zeros(0), tb=numpy.zeros(0))
    geo = sectionGeometry(empty, [numpy.zeros((2, 3)), numpy.zeros((3, 3))], 8)
    assert geo['transect'].size == 0 and geo['distance_km'].size == 0 and geo['offsets'].size == 3


class _FakeField(object):
    """what fluxplot.writeSection reads from a Field"""

    def __init__(self, nt, nz, nsub, with_time=True):
        from nemoflux_b200 import nemoflux_gpu
        self.nt, self.nz, self.nsub = nt, nz, nsub
        rng = numpy.random.default_rng(3)
        self._sec = {}
        self.asked = []
        offs = numpy.array([0, nsub // 3, nsub], numpy.int64)
        sub = dict(offsets=offs, cell=rng.integers(0, 40, nsub), seg=numpy.zeros(nsub, numpy.int32),
                   ta=numpy.linspace(0, 1, nsub + 1)[:-1], tb=numpy.linspace(0, 1, nsub + 1)[1:])
        geo = nemoflux_gpu.sectionGeometry(sub, [numpy.array([[0., 0., 0.], [3., 1., 0.]])] * 2, 8)
        self.pli = type('P', (), {'getSectionGeometry': lambda _self: geo})()
        self.timeObj = type('T', (), {'getSize': lambda _s: nt if with_time else 0,
                                      'getValues': lambda _s: numpy.arange(nt) * 86400. + 43200.,
                                      'units': 'seconds since 1900-01-01', 'calendar': 'noleap'})()
        self.rng = rng

    def layerInterfaces(self):
        return 10. * numpy.arange(self.nz + 1)

    def fluxSection(self, layers):
        self.asked.append(list(layers))
        self.sec = self.rng.standard_normal((self.nt, len(layers) - 1, self.nsub))
        return self.sec


@pytest.mark.parametrize('layers', [None, [0, 2, 5]])
def test_fluxplot_section_file(tmp_path, layers):
    from nemoflux_b200 import fluxplot, ncio
    fld = _FakeField(nt=3, nz=5, nsub=7)
    path = str(tmp_path / 'sec.nc')
    assert fluxplot.writeSection(path, fld, layers, 'Sv') == 7
    lev = list(range(6)) if layers is None else layers
    assert fld.asked == [lev]
    with ncio.open_dataset(path) as nc:
        tr_ = nc['transport']
        assert tuple(tr_.shape) == (3, len(lev) - 1, 7)
        assert numpy.array_equal(numpy.asarray(tr_[:]), fld.sec)
        assert getattr(tr_, 'units', None) == 'Sv' or tr_.attrs.get('units') == 'Sv'
        assert numpy.array_equal(nc['layer_top'][:], 10. * numpy.array(lev[:-1]))
        assert numpy.array_equal(nc['layer_bottom'][:], 10. * numpy.array(lev[1:]))
        assert numpy.array_equal(nc['transect_offsets'][:], [0, 2, 7])
        assert numpy.dtype(nc['transect_offsets'].dtype).newbyteorder('=') == numpy.int32
        assert numpy.dtype(nc['cell_i'].dtype).newbyteorder('=') == numpy.int32
        assert numpy.array_equal(nc['time'][:], numpy.arange(3) * 86400. + 43200.)
        assert nc['distance_km'].shape == (7,) and nc['lon0'].shape == (7,)
    with open(path, 'rb') as f:
        head = f.read(4)
    assert head == b'CDF\x02'                       # classic, 64-bit offsets
    from scipy.io import netcdf_file
    with netcdf_file(path, 'r', mmap=False) as nc:
        assert nc._recs == 3 and nc.dimensions['time'] is None     # time is the record dimension


def test_fluxplot_section_flag():
    from nemoflux_b200 import fluxplot
    base = ['-t', 'T.nc', '-u', 'U.nc', '-v', 'V.nc', '-l', '(0,0),(1,1)']
    with pytest.raises(SystemExit) as e:                    # refused before any file is opened
        fluxplot.main(base + ['--section'])
    assert e.value.code == 2
    with pytest.raises(SystemExit) as e:
        fluxplot.main(base + ['--section', 's.nc', '--layers', '0,10', '--depthLayers', '0,100'])
    assert e.value.code == 2


def test_section_entry_points_are_exported():
    from nemoflux_b200 import _lib
    lib = ctypes.CDLL(_lib.LIB_PATH)
    for name in ('nfx_flux_section', 'nfx_flux_section_host'):
        assert hasattr(lib, name) and name in _lib.SIGNATURES
    assert len(_lib.SIGNATURES['nfx_flux_section']) == 19
    assert len(_lib.SIGNATURES['nfx_flux_section_host']) == 19
