"""-m "not gpu": host side of the layered flux series -- depth snapping, the fluxplot flags, the exports."""
import ctypes

import numpy
import pytest


def _datagen_bounds(tmp_path, nz):
    from nemoflux_b200 import datagen, ncio
    prefix = str(tmp_path) + '/'
    datagen.cli(['--nx=8', '--ny=4', f'--nz={nz}', '--nt=1', f'--prefix={prefix}'])
    with ncio.open_dataset(prefix + 'T.nc') as nc:
        return numpy.asarray(nc['deptht_bounds'][:], numpy.float64)


def test_depth_snapping_on_datagen_levels(tmp_path):
    """datagen writes ztop = (k+1) dz, zbot = (k+2) dz: the first interface is dz, not the surface, so 0 m snaps to
    level 0 and the bottom of the last level is (nz+1) dz"""
    from nemoflux_b200.field import layerInterfaces, levelsForDepths
    b = _datagen_bounds(tmp_path, 10)
    iface = layerInterfaces(b)
    dz = b[0, 1] - b[0, 0]
    assert iface.size == 11 and numpy.allclose(iface, dz * numpy.arange(1, 12))
    assert levelsForDepths(b, [0.0, iface[-1]]) == [0, 10]
    assert levelsForDepths(b, [0.0, 1e9]) == [0, 10]                       # beyond the bottom: the last interface
    assert levelsForDepths(b, [iface[2] + 0.4 * dz, iface[7] - 0.4 * dz, iface[9]]) == [2, 7, 9]
    assert levelsForDepths(b, [iface[3] + 0.5 * dz, iface[5]]) == [3, 5]   # a tie goes to the shallower interface


def test_depth_snapping_errors():
    from nemoflux_b200.field import levelsForDepths
    b = numpy.stack([numpy.arange(0., 50., 10.), numpy.arange(10., 60., 10.)], 1)    # interfaces 0, 10, ..., 50
    with pytest.raises(ValueError, match='same level interface'):
        levelsForDepths(b, [0, 200, 1000, 6000])                                          # 200, 1000, 6000 -> 50 m
    with pytest.raises(ValueError, match='same level interface'):
        levelsForDepths(b, [12, 14])
    with pytest.raises(ValueError, match='ascending'):
        levelsForDepths(b, [40, 10])
    with pytest.raises(ValueError):
        levelsForDepths(b, [5])
    with pytest.raises(ValueError):
        levelsForDepths(b, [0, float('nan')])
    assert levelsForDepths(b, [0, 24, 26, 50]) == [0, 2, 3, 5]


def test_fluxplot_layer_flags():
    import argparse
    from nemoflux_b200 import fluxplot
    assert fluxplot.parseList('0,10, 35,75', int) == [0, 10, 35, 75]
    assert fluxplot.parseList('0,200,1000,6000') == [0.0, 200.0, 1000.0, 6000.0]
    for bad in ('0', '0,1.5x', ''):
        with pytest.raises(argparse.ArgumentTypeError):
            fluxplot.parseList(bad)
    with pytest.raises(argparse.ArgumentTypeError):
        fluxplot.parseList('0,2.5', int)
    base = ['-t', 'T.nc', '-u', 'U.nc', '-v', 'V.nc', '-l', '(0,0),(1,1)']
    with pytest.raises(SystemExit) as e:                    # mutually exclusive: refused before any file is opened
        fluxplot.main(base + ['--layers', '0,10', '--depthLayers', '0,100'])
    assert e.value.code == 2
    with pytest.raises(SystemExit):
        fluxplot.main(base + ['--layers', '0,x'])


def test_layer_argument_forms():
    from nemoflux_b200.nemoflux_gpu import _layer_levels
    assert _layer_levels(None) is None
    for form in ([0, 10, 75], (0, 10, 75), numpy.array([0, 10, 75], numpy.int64), numpy.array([0., 10., 75.]), range(0, 76, 75)):
        a = _layer_levels(form)
        assert a.dtype == numpy.int32 and a.flags.c_contiguous and a[0] == 0 and a[-1] == 75
    for bad in ([3], [], [[0, 1], [1, 2]], [0, 1.5], [0, 2 ** 40]):
        with pytest.raises(ValueError):
            _layer_levels(bad)


def test_layer_entry_points_are_exported():
    from nemoflux_b200 import _lib
    lib = ctypes.CDLL(_lib.LIB_PATH)
    for name in ('nfx_flux_series_layers', 'nfx_flux_series_layers_host'):
        assert hasattr(lib, name) and name in _lib.SIGNATURES
    assert len(_lib.SIGNATURES['nfx_flux_series_layers']) == 21
    assert len(_lib.SIGNATURES['nfx_flux_series_layers_host']) == 20
