"""-m "not gpu": host-side logic of the package (no compute calls) -- C ABI exports, loud failure without a
GPU, file formats, CLI flag parsing, time sharding with a 2-rank gloo group."""
import json
import os
import re
import subprocess
import sys

import numpy
import pytest

from conftest import GOLDEN, ROOT


# ---- the C ABI -----------------------------------------------------------------------------------------
def _declared_symbols():
    text = open(os.path.join(ROOT, 'include', 'nemoflux_gpu.h')).read()
    text = re.sub(r'/\*.*?\*/', '', text, flags=re.S)
    return sorted(set(re.findall(r'\b(nfx_[a-z0-9_]+)\s*\(', text)))


def test_library_exports_every_declared_symbol():
    import ctypes
    from nemoflux_b200 import _lib
    names = _declared_symbols()
    assert len(names) >= 30
    lib = ctypes.CDLL(_lib.LIB_PATH)
    missing = [n for n in names if not hasattr(lib, n)]
    assert not missing, f'declared in include/nemoflux_gpu.h but not exported: {missing}'
    # the python binding covers the same set
    bound = set(_lib.SIGNATURES) | {'nfx_last_error'}
    assert set(names) == bound, set(names) ^ bound
    assert _lib.load().nfx_version() >= 100


def test_no_silent_cpu_fallback():
    """without a CUDA device every entry point must fail loudly (there is no CPU path in the product)"""
    import torch
    if torch.cuda.is_available():
        pytest.skip('a GPU is present')
    from nemoflux_b200 import nemoflux_gpu, _lib
    with pytest.raises(_lib.NemofluxGpuError) as e:
        nemoflux_gpu.Grid()
    assert e.value.code == 3 and 'CUDA' in str(e.value)
    with pytest.raises(_lib.NemofluxGpuError):
        nemoflux_gpu.PolylineIntegral()
    with pytest.raises(TypeError):
        nemoflux_gpu.edgeFluxAssemble(torch.zeros(1, 1, 4, dtype=torch.float64), torch.zeros(1, 1, 4, dtype=torch.float64),
                                      torch.ones(1, dtype=torch.float64), torch.ones(4, dtype=torch.float64),
                                      torch.ones(4, dtype=torch.float64))


def test_product_never_imports_the_oracle():
    for d, _, files in os.walk(os.path.join(ROOT, 'nemoflux_b200')):
        for fn in files:
            if fn.endswith(('.py', '.cu', '.cuh', '.h')):
                src = open(os.path.join(d, fn)).read()
                assert 'import oracle' not in src and 'from oracle' not in src and 'libnfx_oracle' not in src, fn


# ---- file formats ----------------------------------------------------------------------------------------
WOCE_HEADER = ('EXPOCODE 09AR9404_1    S3 (P12)\n                                  CORR\n'
               'STA. DIST(KM)   LAT      LONG     DEPTH\n-----------------------------------------\n')


def test_latlonreader_matches_reference_outputs(tmp_path):
    """golden = what the reference's LatLonReader returned for its 12 transect files; the files are rebuilt in
    the same WOCE layout from the golden points"""
    from nemoflux_b200.latlonreader import LatLonReader
    gold = json.load(open(os.path.join(GOLDEN, 'golden_summary.json')))['latlonreader']
    assert len(gold) == 12 and len(gold['S3_sta_bdep.txt']) == 50 and len(gold['atlantic/S3.txt']) == 10
    assert gold['sa/S3_sa.txt'] == [[16.0, -40.4], [28.0, -34.5], [31.0, -28.5], [36.0, -30.5]]
    for name, pts in gold.items():
        p = tmp_path / name.replace('/', '_')
        with open(p, 'w') as f:
            f.write(WOCE_HEADER)
            for n, (lon, lat) in enumerate(pts):
                f.write(f'  {55 + n}   {93.7 * n:8.1f}   {lat!r}   {lon!r}   802.4\n')
            f.write('\n')
        got = LatLonReader(str(p)).getLonLats()
        assert got.shape == (len(pts), 2) and numpy.array_equal(got, numpy.array(pts))
    # integer-looking coordinates and lines that must be skipped
    p = tmp_path / 'odd.txt'
    p.write_text(WOCE_HEADER + '  0      0.0   63     -10  0\n  x      0.0   1 2\n  0      5   63 -10\n  0  0.0 -46.0  164 0')
    assert LatLonReader(str(p)).getLonLats().tolist() == [[-10.0, 63.0], [164.0, -46.0]]


def test_subsetnemo_cuts_the_index_window(tmp_path):
    """subsetNEMO.py:6-93: x/y dimensions shrunk, bounds and uo/vo cut, everything else and all attributes kept"""
    from nemoflux_b200 import datagen, ncio, subsetnemo
    src, dst = str(tmp_path) + '/', str(tmp_path / 'sub')
    datagen.cli(['-s', '(1+z)*(t+1)*x*y', '--nx=24', '--ny=12', '--nz=3', '--nt=2', '--deltaDeg=20,30', '-p', src])
    w = ncio.Writer(src + 'U2.nc')                  # a U file with a time axis, as real NEMO output has
    with ncio.open_dataset(src + 'U.nc') as nc:
        for name, n in (('t', 2), ('z', 3), ('y', 12), ('x', 24)):
            w.createDimension(name, n)
        w.createVariable('time_counter', 'float64', ('t',), attrs={'standard_name': 'time', 'units': 'days since 2000-01-01'},
                         data=numpy.array([10., 11.]))
        w.createVariable('uo', 'float32', ('t', 'z', 'y', 'x'), fill_value=1.e20, attrs={'units': 'm/s'},
                         data=nc['uo'].raw().astype(numpy.float32))
        w.setAttr('earthRadius', nc.attrs['earthRadius'])
    w.close()
    subsetnemo.main(['-t', src + 'T.nc', '-u', src + 'U2.nc', '-v', src + 'V.nc', '-o', dst,
                     '--jmin=2', '--jmax=9', '--imin=5', '--imax=20'])
    with ncio.open_dataset(src + 'T.nc') as a, ncio.open_dataset(dst + '/T.nc') as b:
        assert b['bounds_lon'].shape == (7, 15, 4) and b['bounds_lon'].dimensions == ('y', 'x', 'nvertex')
        assert numpy.array_equal(b['bounds_lon'][:], a['bounds_lon'][:][2:9, 5:20])
        assert numpy.array_equal(b['bounds_lat'][:], a['bounds_lat'][:][2:9, 5:20])
        assert numpy.array_equal(b['deptht_bounds'][:], a['deptht_bounds'][:]) and 'deptht' not in b
    with ncio.open_dataset(src + 'U2.nc') as a, ncio.open_dataset(dst + '/U.nc') as b:
        assert b['uo'].shape == (2, 3, 7, 15) and b['uo'].dtype.itemsize == 4 and b['uo'].units == 'm/s'
        assert float(b['uo'].attrs['_FillValue']) == float(numpy.float32(1.e20))
        assert numpy.array_equal(b['uo'].raw(), a['uo'].raw()[:, :, 2:9, 5:20])
        assert numpy.array_equal(b['time_counter'][:], [10., 11.]) and b['time_counter'].standard_name == 'time'
        assert 'timestamp' in b.attrs and 'earth radius' in b.attrs['earthRadius']
    with ncio.open_dataset(src + 'V.nc') as a, ncio.open_dataset(dst + '/V.nc') as b:
        assert numpy.array_equal(b['vo'].raw(), a['vo'].raw()[:, :, 2:9, 5:20])
    with pytest.raises(ValueError):
        subsetnemo.subset(tfile=src + 'T.nc', outputdir=dst, jmin=0, jmax=13, imin=0, imax=4, verbose=False)


def test_datagen_cli_writes_nemo_conventions(tmp_path):
    from nemoflux_b200 import datagen, ncio
    prefix = str(tmp_path) + '/'
    datagen.cli(['--streamFunction=x', f'--prefix={prefix}'])
    g = numpy.load(os.path.join(GOLDEN, 'c1_simple.npz'))
    with ncio.open_dataset(prefix + 'T.nc') as nc:
        assert nc['bounds_lon'].dimensions == ('y', 'x', 'nvertex') and nc['bounds_lon'].shape == (18, 36, 4)
        assert numpy.array_equal(nc['bounds_lon'][:], g['bounds_lon']) and numpy.array_equal(nc['bounds_lat'][:], g['bounds_lat'])
        assert nc['deptht_bounds'].dimensions == ('z', 'axis_nbounds')
        assert numpy.array_equal(nc['deptht_bounds'][:], numpy.stack([g['ztop'], g['zbot']], 1))
    with ncio.open_dataset(prefix + 'U.nc') as nc:
        uo = nc['uo']
        assert uo.dimensions == ('t', 'z', 'y', 'x') and uo.standard_name == 'sea_water_x_velocity' and uo.units == 'm/s'
        assert float(uo.attrs['_FillValue']) == 1.e20 and 'earth radius' in nc.attrs['earthRadius']
        assert numpy.array_equal(uo[:], g['u'])            # the reference's own datagen output, bit for bit
    with ncio.open_dataset(prefix + 'V.nc') as nc:
        assert nc['vo'].standard_name == 'sea_water_y_velocity' and numpy.array_equal(nc['vo'][:], g['v'])
    # README.md:89-91 flags
    datagen.cli(['-s', '(1+10*z)*(t+1)*(cos(2*pi*y/360) + sin(2*pi*x/360))', '--nx=24', '--ny=12', '--nz=3', '--nt=2',
                 '--deltaDeg=20,30', '-p', prefix + 'r'])
    g = numpy.load(os.path.join(GOLDEN, 'rot24x12_t0_sv0.npz'))
    with ncio.open_dataset(prefix + 'rU.nc') as nc:
        m = ~g['mask']
        assert nc['uo'].shape == (2, 3, 12, 24) and numpy.array_equal(nc['uo'][:][:, m], g['u'][:, m])
    # missing values come back as NaN (xarray semantics the Field relies on, field.py:157)
    w = ncio.Writer(prefix + 'm.nc')
    w.createDimension('x', 3)
    w.createVariable('a', 'float64', ('x',), fill_value=1.e20, data=numpy.array([1., 1.e20, 3.]))
    w.close()
    with ncio.open_dataset(prefix + 'm.nc') as nc:
        a = nc['a'][:]
        assert a[0] == 1. and numpy.isnan(a[1]) and a[2] == 3. and nc['a'].raw()[1] == 1.e20
    with pytest.raises(ValueError):
        datagen.parseDeltaDeg('1,2,3')
    with pytest.raises(Exception):
        datagen.eval_stream_function('__import__("os").system("true")', 0., 0., 0., 0, 1, 0., 1.)


def test_datagen_mesh_mask(tmp_path):
    """datagen --meshMask [--partialCells f]: NEMO mesh_mask names and shapes; e3 = layer thickness except in the
    thinned deepest level; e2u/e1v = the arc lengths of field.py:170-181 on the saved bounds, in metres"""
    from nemoflux_b200 import datagen, geo, ncio
    prefix = str(tmp_path) + '/'
    datagen.cli(['-s', 'x', '--nx=24', '--ny=12', '--nz=3', '--nt=1', '--zmax=30', '--deltaDeg=20,30', '-p', prefix,
                 '--meshMask', '--partialCells=0.5'])
    with ncio.open_dataset(prefix + 'T.nc') as nc:
        lon, lat, zb = nc['bounds_lon'][:], nc['bounds_lat'][:], nc['deptht_bounds'][:]
    with ncio.open_dataset(prefix + 'mesh_mask.nc') as nc:
        assert nc['e3u_0'].dimensions == ('t', 'z', 'y', 'x') and nc['e3u_0'].shape == (1, 3, 12, 24)
        assert nc['e2u'].dimensions == ('t', 'y', 'x') and nc['e1v'].shape == (1, 12, 24)
        e3u, e3v, e2u, e1v = nc['e3u_0'][:][0], nc['e3v_0'][:][0], nc['e2u'][:][0], nc['e1v'][:][0]
    dz = zb[:, 1] - zb[:, 0]
    assert numpy.array_equal(e3u[:2], numpy.broadcast_to(dz[:2, None, None], (2, 12, 24)))
    assert numpy.array_equal(e3v[:2], e3u[:2])
    for e3 in (e3u, e3v):
        assert (e3[2] <= dz[2]).all() and (e3[2] > 0.5 * dz[2] - 1e-12).all() and len(numpy.unique(e3[2])) > 50
    pts = numpy.zeros((12 * 24, 4, 3))
    pts[:, :, 0], pts[:, :, 1] = lon.reshape(-1, 4), lat.reshape(-1, 4)
    arc = geo.cellArcLengths(pts)
    assert numpy.array_equal(e2u.reshape(-1), arc[:, 1] * 6371000.0) and numpy.array_equal(e1v.reshape(-1), arc[:, 2] * 6371000.0)
    # without the flag no mesh file is written
    datagen.cli(['-s', 'x', '-p', prefix + 'n'])
    assert not os.path.exists(prefix + 'nmesh_mask.nc')


def test_hdf5_reader_on_the_reference_grid_file(tmp_path):
    """nemoflux's real-data files are NetCDF-4 (HDF5); the reference ships one, data/sa/T.nc (README.md:118ff), whose
    arrays and dimension names are committed as tests/golden/sa_T_grid.npz.  Those must be a sane NEMO T grid:
    vertices SW, SE, NE, NW, neighbours sharing their nodes, S3_sa.txt inside.  A NetCDF-4 file with the same
    variables, dimension scales (_Netcdf4Dimid / _Netcdf4Coordinates, dimensions without a variable) and attributes
    is written from them by tests/h5build.py (version-2 object headers, contiguous float32 data); the package's own
    reader (h5lite via ncio) must give back the committed arrays, and the reference's data-preparation tool must cut it"""
    import h5build
    from nemoflux_b200 import ncio
    g = numpy.load(os.path.join(GOLDEN, 'sa_T_grid.npz'))
    lon, lat, zb = g['bounds_lon'], g['bounds_lat'], g['deptht_bounds']
    assert lon.shape == lat.shape == (100, 100, 4) and zb.shape == (75, 2) and lon.dtype == numpy.float32
    assert (lon[..., 1] > lon[..., 0]).all() and (lon[..., 2] == lon[..., 1]).all() and (lon[..., 3] == lon[..., 0]).all()
    assert (lat[..., 3] > lat[..., 0]).all() and (lat[..., 2] > lat[..., 1]).all()
    assert numpy.array_equal(lon[:, 1:, 0], lon[:, :-1, 1]) and numpy.array_equal(lat[1:, :, 0], lat[:-1, :, 3])
    assert (zb[1:, 0] == zb[:-1, 1]).all() and zb[0, 0] == 0.0 and 5000. < zb[-1, 1] < 6500.     # 75 NEMO levels
    for x, y in ((16., -40.4), (28., -34.5), (31., -28.5), (36., -30.5)):                       # data/sa/S3_sa.txt:5-8
        assert lon.min() < x < lon.max() and lat.min() < y < lat.max()
    dims = {str(name): str(d).split('|') for name, d in g['dims']}
    sizes = {}
    for name, dn in sorted(dims.items()):
        sizes.update(zip(dn, g[name].shape))
    dimid = {dn: numpy.int32(i) for i, dn in enumerate(sizes)}
    variables = {dn: dict(data=numpy.zeros(n, numpy.float32),
                          attrs={'CLASS': 'DIMENSION_SCALE', '_Netcdf4Dimid': dimid[dn],
                                 'NAME': f'This is a netCDF dimension but not a netCDF variable.{n:10d}'})
                 for dn, n in sizes.items() if dn not in dims}
    for name, dn in dims.items():
        variables[name] = dict(data=g[name], attrs={'_Netcdf4Coordinates': numpy.array([dimid[d] for d in dn])})
    variables['deptht']['attrs'] = {'CLASS': 'DIMENSION_SCALE', 'NAME': 'deptht', '_Netcdf4Dimid': dimid['deptht'],
                                    'standard_name': 'depth', 'units': 'm', 'bounds': 'deptht_bounds'}
    path = str(tmp_path / 'T.nc')
    h5build.write_new(path, variables)
    with ncio.open_dataset(path) as nc:
        assert set(nc.variables) == {'bounds_lon', 'bounds_lat', 'deptht', 'deptht_bounds'}
        assert nc['bounds_lon'].dimensions == ('y', 'x', 'nvertex') and nc['deptht_bounds'].dimensions == ('deptht', 'axis_nbounds')
        assert nc['deptht'].standard_name == 'depth' and nc['deptht'].units == 'm' and nc['deptht'].bounds == 'deptht_bounds'
        for name in ('bounds_lon', 'bounds_lat', 'deptht_bounds', 'deptht'):
            assert numpy.array_equal(nc[name][:], g[name]), name
        assert numpy.array_equal(nc['bounds_lat'][3, 5:7], g['bounds_lat'][3, 5:7])             # partial reads (memmap)
    # the reference's data-preparation tool on its grid file (subsetNEMO.py:6-93): NetCDF-4 in, classic out
    from nemoflux_b200 import subsetnemo
    out = tmp_path / 'subset'
    subsetnemo.subset(tfile=path, outputdir=str(out), jmin=10, jmax=40, imin=20, imax=90, verbose=False)
    with ncio.open_dataset(str(out / 'T.nc')) as nc:
        assert nc['bounds_lon'].dimensions == ('y', 'x', 'nvertex') and nc['bounds_lon'].shape == (30, 70, 4)
        assert numpy.array_equal(nc['bounds_lon'][:], g['bounds_lon'][10:40, 20:90])
        assert numpy.array_equal(nc['bounds_lat'][:], g['bounds_lat'][10:40, 20:90])
        assert numpy.array_equal(nc['deptht_bounds'][:], g['deptht_bounds']) and nc['deptht'].units == 'm'


def test_hdf5_chunked_deflate_shuffle_decoding():
    """the chunked layout of h5lite on a hand-built version-1 chunk B-tree (two levels, edge chunks hanging over the
    dataset, a missing chunk = fill value, deflate + shuffle + fletcher32 filters, one chunk with deflate skipped)"""
    import struct
    import zlib
    from nemoflux_b200 import h5lite
    rng = numpy.random.default_rng(1)
    shape, cdims = (5, 7), (2, 4)
    dtype = numpy.dtype('<f4')
    data = rng.standard_normal(shape).astype(dtype)
    filters = [(2, [4]), (1, [4]), (3, [])]                    # shuffle, deflate, fletcher32 (order of application)
    buf = bytearray(b'\0' * 64)

    def put(b):
        addr = len(buf)
        buf.extend(b)
        buf.extend(b'\0' * (-len(buf) % 8))
        return addr

    def encode(chunk, skip_deflate):
        raw = chunk.tobytes()
        raw = numpy.frombuffer(raw, numpy.uint8).reshape(-1, 4).T.tobytes()        # shuffle
        if not skip_deflate:
            raw = zlib.compress(raw, 4)
        return raw + b'ABCD'                                                       # fletcher32 checksum (not verified)

    entries = []
    for j0 in range(0, shape[0], cdims[0]):
        for i0 in range(0, shape[1], cdims[1]):
            if (j0, i0) == (2, 4):
                continue                                        # never written
            chunk = numpy.zeros(cdims, dtype)
            sub = data[j0:j0 + cdims[0], i0:i0 + cdims[1]]
            chunk[:sub.shape[0], :sub.shape[1]] = sub
            skip = (j0, i0) == (0, 4)
            raw = encode(chunk, skip)
            entries.append(((j0, i0), len(raw), 2 if skip else 0, put(raw)))

    def node(level, items):                                     # items: (offsets, nbytes, mask, child address)
        b = b'TREE' + bytes([1, level]) + struct.pack('<H', len(items)) + struct.pack('<QQ', h5lite.UNDEF, h5lite.UNDEF)
        for offs, nbytes, mask, child in items:
            b += struct.pack('<II', nbytes, mask) + struct.pack('<QQQ', offs[0], offs[1], 0) + struct.pack('<Q', child)
        b += struct.pack('<II', 0, 0) + struct.pack('<QQQ', shape[0], shape[1], 0)
        return put(b)

    leaf_a, leaf_b = node(0, entries[:3]), node(0, entries[3:])
    root = node(1, [(entries[0][0], 0, 0, leaf_a), (entries[3][0], 0, 0, leaf_b)])
    f = h5lite.File.__new__(h5lite.File)
    f._buf, f._base, f.path = bytes(buf), 0, '<memory>'
    ds = h5lite.Dataset(f, 'v', shape, dtype, ('chunked', root, cdims), filters, {}, numpy.float32(-9.).tobytes())
    got = ds.read()
    want = data.copy()
    want[2:4, 4:7] = -9.
    assert numpy.array_equal(got, want)
    # partial reads decode only the chunks under the block (what a time slice of uo/vo does)
    from nemoflux_b200 import ncio
    lazy = ncio._H5Data('<memory>', f, h5lite.Dataset(f, 'v', shape, dtype, ('chunked', root, cdims), filters, {},
                                                      numpy.float32(-9.).tobytes()))
    reads = []
    orig = f._read
    f._read = lambda addr, n: (reads.append(addr), orig(addr, n))[1]
    assert numpy.array_equal(lazy[1, 1:3], want[1, 1:3])
    assert len([a for a in reads if a in {e[3] for e in entries}]) == 1          # one chunk was enough
    assert numpy.array_equal(lazy[3:5, 2:7], want[3:5, 2:7]) and numpy.array_equal(lazy[-1], want[-1])
    assert numpy.array_equal(lazy[4, -1], want[4, -1]) and numpy.array_equal(lazy[::2, 1], want[::2, 1])
    assert numpy.array_equal(lazy[...], want)
    with pytest.raises(IndexError):
        lazy[5]
    with pytest.raises(h5lite.H5Error):
        h5lite.apply_filters_reverse(b'1234', [(32015, [])], 0, 4)
    for size in (1, 2, 3, 4, 8, 16):                             # the vectorised unshuffle against a plain transpose
        elems = rng.integers(0, 256, (37, size), dtype=numpy.uint8)
        planes = elems.T.tobytes()
        assert h5lite.unshuffle(planes, size, 37) == elems.tobytes(), size


def test_hdf5_old_style_file_roundtrip(tmp_path):
    """a file in the oldest HDF5 flavour (symbol-table group, version-1 object headers, chunked + shuffle + deflate
    data, version-1 attribute messages) written by tests/h5build.py: variables, attributes, partial reads"""
    import h5build
    from nemoflux_b200 import ncio
    rng = numpy.random.default_rng(0)
    uo = rng.standard_normal((3, 4, 9, 11)).astype('<f4')
    uo[:, :, 2:4, 5:8] = numpy.float32(1.e20)
    vo = rng.standard_normal((3, 4, 9, 11)).astype('>f8')
    tc = numpy.arange(3, dtype='<f8') * 86400.
    path = str(tmp_path / 'old.nc')
    h5build.write(path, {
        'uo': dict(data=uo, chunks=(1, 2, 9, 11), deflate=True, shuffle=True,
                   attrs={'_FillValue': numpy.float32(1.e20), 'units': 'm/s', 'standard_name': 'sea_water_x_velocity'}),
        'vo': dict(data=vo, attrs={'units': 'm/s'}),
        'time_counter': dict(data=tc, chunks=(2,), attrs={'standard_name': 'time'}),
        'many': dict(data=numpy.arange(40, dtype='<i4').reshape(20, 2), chunks=(3, 2))})      # two-level chunk tree
    with ncio.open_dataset(path) as nc:
        assert set(nc.variables) == {'uo', 'vo', 'time_counter', 'many'}
        assert nc['uo'].shape == (3, 4, 9, 11) and nc['uo'].units == 'm/s' and nc['uo'].fill_value() == float(numpy.float32(1.e20))
        assert numpy.array_equal(nc['uo'].raw(), uo) and numpy.array_equal(nc['uo'].raw((1, slice(1, 3))), uo[1, 1:3])
        assert numpy.isnan(nc['uo'][0, 0, 2, 5]) and nc['uo'][0, 0, 0, 0] == uo[0, 0, 0, 0]
        assert numpy.array_equal(nc['vo'].raw(), vo.astype('<f8')) and nc['vo'].raw().dtype.isnative
        dst = numpy.zeros((2, 9, 11), numpy.float32)
        nc['uo'].read_into(dst, (2, slice(2, 4)))
        assert numpy.array_equal(dst, uo[2, 2:4])
        assert numpy.array_equal(nc['time_counter'][:], tc) and nc['time_counter'].standard_name == 'time'
        assert numpy.array_equal(nc['many'][:], numpy.arange(40).reshape(20, 2)) and numpy.array_equal(nc['many'][7:15, 1], numpy.arange(15, 31, 2))
    with open(str(tmp_path / 'bad.nc'), 'wb') as f:
        f.write(b'not a netcdf file at all')
    with pytest.raises(RuntimeError):
        ncio.open_dataset(str(tmp_path / 'bad.nc'))


def test_hdf5_new_style_file_roundtrip(tmp_path):
    """the newer HDF5 structures written by tests/h5build.write_new: superblock 2, version-2 object headers with
    times / creation order / a continuation block, link messages, variable-length strings in a global heap, and a
    variable whose many attributes live in dense storage (fractal heap with an indirect root block + version-2
    B-tree) -- what real NEMO uo/vo variables with their ~10 attributes look like"""
    import h5build
    from nemoflux_b200 import ncio
    rng = numpy.random.default_rng(5)
    uo = rng.standard_normal((3, 4, 9, 11)).astype('<f4')
    attrs = {'_FillValue': numpy.float32(1.e20), 'units': 'm/s', 'standard_name': 'sea_water_x_velocity',
             'long_name': 'vlen:ocean current along i-axis', 'online_operation': 'average', 'interval_operation': '1 h',
             'interval_write': '1 month', 'cell_methods': 'time: mean (interval: 1 h)', 'missing_value': numpy.float32(1.e20),
             'coordinates': 'time_centered nav_lat nav_lon', 'valid_range': numpy.array([-10., 10.]),
             'comment': 'x' * 300, 'comment2': 'y' * 200, 'comment3': 'z' * 180}
    path = str(tmp_path / 'new.nc')
    h5build.write_new(path, {
        'uo': dict(data=uo, chunks=(1, 2, 9, 11), deflate=True, shuffle=True, attrs=attrs, dense_attrs=True),
        'vo': dict(data=uo.astype('>f8'), attrs={'units': 'm/s', 'title': 'vlen:northward'}),
        'time_counter': dict(data=numpy.arange(3.), attrs={'standard_name': 'time'})})
    with ncio.open_dataset(path) as nc:
        assert nc.attrs == {'Conventions': 'CF-1.6'} and set(nc.variables) == {'uo', 'vo', 'time_counter'}
        got = nc['uo'].attrs
        assert set(got) == set(attrs)
        for k, v in attrs.items():
            want = v[5:] if isinstance(v, str) and v.startswith('vlen:') else v
            assert numpy.array_equal(got[k], want), k
        assert numpy.array_equal(nc['uo'].raw(), uo) and numpy.array_equal(nc['uo'].raw((2, slice(0, 2))), uo[2, :2])
        assert numpy.array_equal(nc['vo'].raw(), uo.astype('f8')) and nc['vo'].title == 'northward'
        assert nc['time_counter'].standard_name == 'time' and numpy.array_equal(nc['time_counter'][:], [0., 1., 2.])


def test_transect_argument_forms(tmp_path):
    from nemoflux_b200.field import parseLonLatPoints
    from nemoflux_b200.fluxviz import parseTransects
    flat = parseLonLatPoints('(-180,-70),(-160,-10),(-35,40)')                 # README.md:32
    assert len(flat) == 1 and flat[0].shape == (3, 3) and flat[0][1].tolist() == [-160., -10., 0.]
    many = parseLonLatPoints('[(0,0),(1,1)],[(2,2),(3,3),(4,4)]')               # fluxviz.py:378
    assert [m.shape[0] for m in many] == [2, 3]
    one = parseLonLatPoints('[(0,0),(1,1)]')
    assert len(one) == 1 and one[0].shape == (2, 3)
    with pytest.raises(RuntimeError):
        parseTransects('', '')
    a = tmp_path / 'S1.txt'
    b = tmp_path / 'S2.txt'
    a.write_text(WOCE_HEADER + '  0      0.0   -31.4   152.0   0\n  0      0.0   -34.5   172.0   0\n')
    b.write_text(WOCE_HEADER + '  0      0.0   -46.0      164    0\n  0      0.0   -48.0      170    0\n  0 0.0 -40.0 179 0\n')
    pts, names = parseTransects('', str(tmp_path / 'S*.txt'))
    assert [p.shape[0] for p in pts] == [2, 3] and pts[0][0].tolist() == [152.0, -31.4, 0.0]
    pts, names = parseTransects('', repr([str(a)]))
    assert len(pts) == 1 and names == [str(a)]


def test_fluxexact_cli(capsys):
    from nemoflux_b200 import fluxexact
    res = fluxexact.main(['--potentialFunction=x', '-l', '(-180,-70),(-160,-10),(180,40)', '--nz', '2'])
    assert numpy.allclose(res, [360.0])
    res = fluxexact.exactFlux('(1+10*z)*(t+1)*(cos(2*pi*y/360) + sin(2*pi*x/360))',
                              numpy.array([(-100., -80.), (0., 80.)]), nz=10, nt=3)
    assert numpy.allclose(res / res[0], [1, 2, 3])


def test_timeobj():
    from nemoflux_b200.timeobj import TimeObj
    from nemoflux_b200.ncio import Variable
    nc = {'uo': Variable('uo', numpy.zeros((2, 1)), ('t', 'x'), {}),
          'time_counter': Variable('time_counter', numpy.array([0., 86400. * 31]), ('t',),
                                   {'standard_name': 'time', 'units': 'seconds since 1950-01-01 00:00:00'})}
    t = TimeObj(nc)
    assert t.getSize() == 2 and t.getTimeAsString(1) == '1950-2-1'
    t = TimeObj({'uo': nc['uo']})
    assert t.getSize() == 0 and t.getTimeAsString(3) == 'time index 3'     # mock data has no time axis


# ---- time sharding -------------------------------------------------------------------------------------------
def test_shard_time_partitions():
    from nemoflux_b200 import dist
    assert dist.shard_counts(73, 8) == [10, 9, 9, 9, 9, 9, 9, 9]                 # SURVEY.md 8e
    assert dist.shard_counts(365, 2) == [183, 182] and dist.shard_counts(365, 4) == [92, 91, 91, 91]
    for nt in (0, 1, 5, 73, 365):
        for world in (1, 2, 3, 8):
            assert dist.check_partition(nt, world)
    with pytest.raises(ValueError):
        dist.shard_time(10, 2, 2)


def test_shard_batches_balanced():
    from nemoflux_b200 import dist
    for nt, npanels, world in ((73, 26, 8), (7, 2, 3), (5, 1, 8), (365, 3, 4)):
        covered = 0
        sizes = []
        for r in range(world):
            s = dist.shard_batches(nt, npanels, world, r)
            assert s['g0'] == covered
            covered = s['g1']
            sizes.append(s['g1'] - s['g0'])
            if s['nt_touched']:
                assert s['t_first'] * npanels + s['b0'] == s['g0'] and s['t_first'] * npanels + s['b1'] == s['g1']
                assert 0 <= s['b0'] < npanels and s['b1'] <= s['nt_touched'] * npanels
        assert covered == nt * npanels and max(sizes) - min(sizes) <= 1
    assert [dist.shard_batches(73, 26, 8, r)['nt_touched'] for r in range(8)] == [10] * 8      # 9.125 steps each


WORKER = r'''
import os, sys
import numpy, torch
import torch.distributed as dist
sys.path.insert(0, sys.argv[1])
from nemoflux_b200 import dist as nd
rank, world, nt, m = int(sys.argv[2]), int(sys.argv[3]), int(sys.argv[4]), 5
os.environ['MASTER_ADDR'] = '127.0.0.1'
os.environ['MASTER_PORT'] = sys.argv[5]
dist.init_process_group('gloo', rank=rank, world_size=world)
full = torch.arange(nt * m, dtype=torch.float64).reshape(nt, m) * 0.5 + 1.0     # the 1-rank answer
def compute_local(t0, n):      # stands for K2+K3 on this rank's time steps
    return full[t0:t0 + n].clone()
out = nd.sharded_flux_series(compute_local, nt)
assert out.shape == (nt, m) and torch.equal(out, full), (rank, out)
mx = nd.allreduce_max(float(rank + 1))
assert mx == world
# balanced sharding: 3 panels per time step, the partial sums of shared time steps add up
npanels = 3
contrib = torch.arange(nt * npanels * m, dtype=torch.float64).reshape(nt, npanels, m) + 1.0
s = nd.shard_batches(nt, npanels, world, rank)
part = torch.zeros((s['nt_touched'], m), dtype=torch.float64)
for b in range(s['b0'], s['b1']):
    part[b // npanels] += contrib[s['t_first'] + b // npanels, b % npanels]
tot = nd.combine_partial_series(part, nt, npanels)
assert torch.equal(tot, contrib.sum(1)), (rank, tot)
# the same with shares proportional to each rank's measured rate (every rank passes the same weights)
weights = [1.0 + 0.25 * r for r in range(world)]
s = nd.shard_batches(nt, npanels, world, rank, weights)
part = torch.zeros((s['nt_touched'], m), dtype=torch.float64)
for b in range(s['b0'], s['b1']):
    part[b // npanels] += contrib[s['t_first'] + b // npanels, b % npanels]
tot = nd.combine_partial_series(part, nt, npanels, weights=weights)
assert torch.equal(tot, contrib.sum(1)), (rank, tot)
# host-fed time steps apportioned by rate: the blocks tile the series, the gathered result is the 1-rank answer
counts = nd.apportion_by_rate(nt, [23.0, 35.0][:world] if world == 2 else [1.0] * world)
t0, n = nd.blocks_from_counts(counts)[rank]
cm = max(max(counts), 1)
blk = torch.zeros((cm, m), dtype=torch.float64)
blk[:n] = full[t0:t0 + n]
parts = [torch.zeros((cm, m), dtype=torch.float64) for _ in range(world)]
dist.all_gather(parts, blk)
got = torch.cat([parts[r][:counts[r]] for r in range(world)], 0)
assert torch.equal(got, full), (rank, counts)
dist.barrier()
dist.destroy_process_group()
print('ok', rank)
'''


def test_bench_reference_arm_contract():
    """bench.py --impl reference (the CPU arm the driver times next to ours): one JSON line with the contract's keys,
    no GPU needed; under a multi-rank launch only rank 0 prints"""
    cmd = [sys.executable, os.path.join(ROOT, 'bench.py'), '--impl', 'reference', '--workload', 'tiny', '--steps', '2',
           '--warmup', '1', '--cpu-steps', '3']
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=300, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [ln for ln in out.stdout.splitlines() if ln.startswith('{')]
    assert len(lines) == 1
    d = json.loads(lines[0])
    for key in ('impl', 'metric', 'value', 'unit', 'n_gpus', 'steps', 'warmup', 'ms_per_step', 'higher_is_better', 'scaling',
                'vs_baseline', 'dtype', 'data', 'config', 'cpu_baseline', 'e2e'):
        assert key in d, key
    assert d['impl'] == 'reference' and d['value'] > 0 and d['steps'] == 2 and d['vs_baseline'] is None
    assert d['cpu_baseline']['kind'] == 'port' and d['cpu_baseline']['value'] == d['value'] and d['cpu_baseline']['cores'] >= 1
    assert d['e2e'] == {'value': d['value'], 'unit': d['unit'], 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0}
    assert 'workload' in d['config'] and 'model' not in d['config']
    env = dict(os.environ, RANK='1', WORLD_SIZE='2', LOCAL_RANK='1')
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=300, cwd=ROOT, env=env)
    assert out.returncode == 0 and not [ln for ln in out.stdout.splitlines() if ln.startswith('{')]


def test_bench_dump_outputs_reference_arm(oracle, tmp_path):
    """bench.py --dump-outputs DIR writes the flux series of the last timed step as float64 .npy: the same file from
    run to run whatever the number of steps, equal to the oracle's series of the sampled time steps; --steps 0 is
    refused instead of timing nothing"""
    from nemoflux_b200 import synth
    cmd = [sys.executable, os.path.join(ROOT, 'bench.py'), '--impl', 'reference', '--workload', 'tiny', '--warmup', '0',
           '--cpu-steps', '3']
    got = []
    for steps in (1, 2):
        d = tmp_path / f'steps{steps}'
        out = subprocess.run(cmd + ['--steps', str(steps), '--dump-outputs', str(d)], capture_output=True, text=True,
                             timeout=300, cwd=ROOT)
        assert out.returncode == 0, out.stderr[-2000:]
        assert os.listdir(d) == ['flux_series.npy']
        got.append(numpy.load(d / 'flux_series.npy'))
    assert got[0].dtype == numpy.float64 and got[0].shape == (3, 12) and numpy.array_equal(got[0], got[1])
    syn = synth.make('tiny')
    uh = numpy.stack([syn.uv_host(t)[0] for t in range(3)])
    vh = numpy.stack([syn.uv_host(t)[1] for t in range(3)])
    ref = oracle.flux_series(syn.points, syn.transects, uh, vh, syn.thickness)
    assert numpy.abs(got[0] - ref).max() <= 1e-12 * numpy.abs(ref).max()
    out = subprocess.run(cmd + ['--steps', '0'], capture_output=True, text=True, timeout=300, cwd=ROOT)
    assert out.returncode != 0 and '--steps must be at least 1' in out.stderr


def test_f32_bit_shuffle_conversion_in_emulation():
    """nfx_stream_ops.cuh::clean_scaled restated with numpy integer arithmetic: the float's bits moved into the double
    layout without re-biasing are exactly x * 2^-896 for every finite float (normals, denormals, +-0, FLT_MAX), 0 for
    NaN and the missing-value marker, and every infinity is flagged by the running maximum (those threads recompute
    with the plain conversion).  (A second flavour with one ordered compare and one wide multiply gave the same bits
    and the same speed on the device -- profiles/r2_fused_experiments.md -- and was dropped.)"""
    rng = numpy.random.default_rng(12)
    bits = rng.integers(0, 2 ** 32, 200000, dtype=numpy.uint64).astype(numpy.uint32)
    special = numpy.array([0x00000000, 0x80000000, 0x00000001, 0x80000001, 0x007fffff, 0x00800000, 0x7f7fffff, 0xff7fffff,
                           0x7f800000, 0xff800000, 0x7fc00000, 0xffc00000, 0x7f800001, 0x60ad78ec, 0xe0ad78ec], numpy.uint32)
    bits = numpy.concatenate([special, bits])
    x = bits.view(numpy.float32)
    marker = numpy.float32(1.e20)                               # bits 0x60ad78ec

    def pack(b):                                                # hi = (b >> 3 arithmetic) & 0x8fffffff, lo = b << 29
        hi = (b.astype(numpy.int32) >> 3).astype(numpy.uint32) & numpy.uint32(0x8fffffff)
        lo = (b.astype(numpy.uint64) << numpy.uint64(29)).astype(numpy.uint32)
        return ((hi.astype(numpy.uint64) << numpy.uint64(32)) | lo.astype(numpy.uint64)).view(numpy.float64)

    for fill in (marker, numpy.float32('nan')):
        has_fill = not numpy.isnan(fill)
        with numpy.errstate(invalid='ignore'):
            keep = (~(x == fill) | numpy.isnan(x)) & (numpy.abs(x) <= numpy.finfo(numpy.float32).max)   # NEU and |x| <= FLT_MAX
            keep &= ~numpy.isnan(x)
        v1 = pack(numpy.where(keep, bits, numpy.uint32(0)))
        finite = numpy.isfinite(x)
        with numpy.errstate(invalid='ignore'):
            want = numpy.where(has_fill & (x == fill), 0.0, x.astype(numpy.float64) * 2.0 ** -896)[finite]
        assert numpy.array_equal(v1[finite], want) and numpy.array_equal(numpy.signbit(v1[finite]), numpy.signbit(want))
        assert (v1[numpy.isnan(x)] == 0).all()
        inf = numpy.isinf(x)
        assert inf.any() and numpy.isinf(numpy.abs(x[inf]).max())         # what the FMNMX3 running maximum sees


def test_gpu_cpu_binding_is_harmless_without_nvml_affinity():
    """bind_to_gpu_cpus: no GPU / no affinity information -> nothing changes and 0 is returned"""
    from nemoflux_b200 import dist
    before = os.sched_getaffinity(0)
    import torch
    if not torch.cuda.is_available():
        assert dist.gpu_local_cpus(0) == set()
        assert dist.bind_to_gpu_cpus(0) == 0
    else:
        n = dist.bind_to_gpu_cpus(0)
        assert n == 0 or n == len(os.sched_getaffinity(0))
        os.sched_setaffinity(0, before)
    assert os.sched_getaffinity(0) == before


@pytest.mark.parametrize('nt', [7, 8])
def test_allgather_series_two_ranks_gloo(tmp_path, nt):
    """world_size 2 on CPU: uneven (4+3) and even shards assemble to the single-rank series bit for bit"""
    script = tmp_path / 'worker.py'
    script.write_text(WORKER)
    port = str(29500 + (os.getpid() + nt) % 2000)
    procs = [subprocess.Popen([sys.executable, str(script), ROOT, str(r), '2', str(nt), port],
                              stdout=subprocess.PIPE, stderr=subprocess.STDOUT) for r in range(2)]
    outs = [p.communicate(timeout=180)[0].decode() for p in procs]
    for p, o in zip(procs, outs):
        assert p.returncode == 0, o


def test_bench_arms_share_config_and_defaults():
    """bench.py: at N = 1 the workload is BASELINE config 3, at N >= 2 config 4 sharded by time (strong scaling); the
    `config` dict is a function of (workload, N, dtype) only, so the reference arm and the GPU arm print the same one"""
    import importlib.util
    spec = importlib.util.spec_from_file_location('nfx_bench', os.path.join(ROOT, 'bench.py'))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    from nemoflux_b200 import synth

    class A(object):
        workload, nt_local, nt_total = 'auto', 0, 0
    assert bench.pick_workload(A, 1) == ('C3', 365, 'weak')
    for n in (2, 4, 8):
        assert bench.pick_workload(A, n) == ('C4', 365, 'strong')
    c1 = bench.make_config('C4', synth.CONFIGS['C4'], 8, 'f64', 365, 'strong')
    c2 = bench.make_config('C4', dict(synth.CONFIGS['C4']), 8, 'f64', 365, 'strong')
    assert c1 == c2 and c1['workload'].startswith('C4') and 'model' not in c1
    assert c1['sharding'].startswith('time steps [46, 46, 46, 46, 46, 45, 45, 45]')
    assert bench.make_config('C3', synth.CONFIGS['C3'], 1, 'f32', 365, 'weak')['storage_dtype'] == 'f32'


def test_apportion_by_rate():
    """dist.apportion_by_rate: host-fed time steps in proportion to the measured H2D rates (the 8-GPU boxes of the pool
    give GPUs 0-3 23 GB/s and 4-7 35 GB/s, profiles/r1_numa_probe8.md); never worse than equal shards"""
    from nemoflux_b200 import dist as nd
    rates = [23, 23, 23, 23, 35, 35, 35, 35]
    c = nd.apportion_by_rate(32, rates)
    assert sum(c) == 32 and c == [3, 3, 3, 3, 5, 5, 5, 5]
    span = lambda cc: max(x / r for x, r in zip(cc, rates))   # noqa: E731
    for total in (1, 7, 8, 24, 33, 100, 365):
        c = nd.apportion_by_rate(total, rates)
        assert sum(c) == total and min(c) >= 0
        assert span(c) <= span(nd.shard_counts(total, 8)) + 1e-12
    assert nd.apportion_by_rate(9, [1.0, 1.0, 1.0]) == [3, 3, 3]
    assert nd.apportion_by_rate(0, [3.0, 4.0]) == [0, 0]
    assert sum(nd.apportion_by_rate(5, [0.0, 0.0])) == 5
    assert nd.blocks_from_counts([2, 0, 3]) == [(0, 2), (2, 0), (2, 3)]
    with pytest.raises(ValueError):
        nd.apportion_by_rate(3, [])
    with pytest.raises(ValueError):
        nd.apportion_by_rate(3, [1.0, float('nan')])


def test_ncio_decoding_matches_xarray_conventions():
    """ncio.Variable: scale_factor / add_offset and BOTH missing-value attributes are honoured when decoded values are
    asked for (xarray.open_dataset's mask_and_scale, which the reference relies on, field.py:22-35); the raw fast path
    refuses packed data instead of handing out counts as metres per second"""
    from nemoflux_b200 import ncio
    raw = numpy.array([[1, 2, -32767], [4, -999, 6]], numpy.int16)
    v = ncio.Variable('uo', raw, ('y', 'x'), {'scale_factor': numpy.float32(0.01), 'add_offset': numpy.float32(1.5),
                                              '_FillValue': numpy.int16(-32767), 'missing_value': numpy.int16(-999)})
    assert v.packed and v.fill_values() == [-32767.0, -999.0]
    d = v[...]
    assert d.dtype == numpy.float32
    assert numpy.isnan(d[0, 2]) and numpy.isnan(d[1, 1])
    assert numpy.allclose(d[0, :2], [1.51, 1.52]) and numpy.allclose(d[1, ::2], [1.54, 1.56])
    with pytest.raises(NotImplementedError):
        v.raw()
    with pytest.raises(NotImplementedError):
        v.read_into(numpy.zeros((2, 3), numpy.int16))
    with pytest.raises(ValueError):
        v.fill_value()
    f = ncio.Variable('vo', numpy.array([1.0, 1e20, -9e33, 4.0], numpy.float32), ('x',),
                      {'_FillValue': numpy.float32(1e20), 'missing_value': numpy.float32(-9e33)})
    assert not f.packed and numpy.array_equal(numpy.isnan(f[...]), [False, True, True, False])
    g = ncio.Variable('wo', numpy.array([1.0, 1e20], numpy.float32), ('x',),
                      {'_FillValue': numpy.float32(1e20), 'missing_value': numpy.float32(1e20)})
    assert g.fill_value() == float(numpy.float32(1e20)) and numpy.array_equal(g.raw(), [1.0, numpy.float32(1e20)])


def test_ncio_serialises_reads_of_a_thread_unsafe_backend():
    """netCDF4-python releases the GIL around nc_get_vara and libnetcdf / HDF5 are not thread-safe: Variables of that
    backend carry ncio's process-wide lock, every read takes it, and Field reads them with one worker"""
    import threading
    import time
    from nemoflux_b200 import ncio

    class Unsafe(object):           # raises when two reads overlap
        shape, dtype = (8, 4), numpy.dtype('f8')

        def __init__(self):
            self.inside, self.max_inside = 0, 0

        def __getitem__(self, idx):
            self.inside += 1
            self.max_inside = max(self.max_inside, self.inside)
            time.sleep(0.005)
            self.inside -= 1
            return numpy.zeros(self.shape)[idx]

    for lock, expect in ((ncio._NETCDF4_LOCK, 1), (None, None)):
        data = Unsafe()
        v = ncio.Variable('uo', data, ('t', 'x'), {}, lock=lock)
        assert v.thread_safe == (lock is None)
        dst = numpy.zeros((8, 4))
        ths = [threading.Thread(target=v.read_into, args=(dst[i], i)) for i in range(8)]
        ths += [threading.Thread(target=v.raw, args=(i,)) for i in range(4)]
        for t in ths:
            t.start()
        for t in ths:
            t.join()
        if expect is not None:
            assert data.max_inside == expect
        else:
            assert data.max_inside > 1          # the mmap-style backends do read in parallel


def test_timeobj_calendars():
    """CF calendars NEMO commonly runs with: noleap has no 29 February, 360_day has twelve 30-day months"""
    from nemoflux_b200 import ncio, timeobj

    def tobj(values, calendar):
        attrs = {'standard_name': 'time', 'units': 'days since 2000-01-01'}
        if calendar:
            attrs['calendar'] = calendar
        return timeobj.TimeObj({'time_counter': ncio.Variable('time_counter', numpy.array(values, numpy.float64), ('t',), attrs)})

    assert tobj([59.0, 60.0], None).getTimeAsString(1) == '2000-3-1'              # 2000 is a leap year: day 59 = 29 Feb
    assert tobj([59.0, 60.0], None).getTimeAsString(0) == '2000-2-29'
    assert tobj([59.0, 365.0], 'noleap').getTimeAsString(0) == '2000-3-1'
    assert tobj([59.0, 365.0], 'noleap').getTimeAsString(1) == '2001-1-1'
    assert tobj([59.0, 360.0], '360_day').getTimeAsString(0) == '2000-2-30'
    assert tobj([59.0, 360.0], '360_day').getTimeAsString(1) == '2001-1-1'


def test_weighted_batch_sharding_tiles_the_batch_space():
    """dist.shard_batches(weights=): contiguous ranges proportional to each rank's measured rate that tile the
    (time step, panel) space exactly; equal weights reproduce the unweighted cut"""
    from nemoflux_b200 import dist as nd
    nt, npanels, world = 73, 51, 8
    for weights in (None, [1.0] * 8, [1.0, 0.97, 1.0, 0.95, 1.0, 1.0, 0.98, 1.0], [3.0, 1, 1, 1, 1, 1, 1, 1]):
        covered = numpy.zeros(nt * npanels, int)
        sizes = []
        for r in range(world):
            s = nd.shard_batches(nt, npanels, world, r, weights)
            covered[s['g0']:s['g1']] += 1
            sizes.append(s['g1'] - s['g0'])
            assert s['t_first'] * npanels + s['b0'] == s['g0'] and s['t_first'] * npanels + s['b1'] == s['g1']
            assert s['nt_touched'] == (s['g1'] - 1) // npanels - s['g0'] // npanels + 1
        assert (covered == 1).all()
        if weights is not None:
            w = numpy.array(weights) / sum(weights)
            assert numpy.abs(numpy.array(sizes) - w * nt * npanels).max() <= 1.0
    for r in range(world):          # equal weights: the unweighted cut up to the rounding of a boundary
        a, b = nd.shard_batches(nt, npanels, world, r), nd.shard_batches(nt, npanels, world, r, [2.0] * 8)
        assert abs(a['g0'] - b['g0']) <= 3 and abs(a['g1'] - b['g1']) <= 3 and abs((a['g1'] - a['g0']) - (b['g1'] - b['g0'])) <= 1
    with pytest.raises(ValueError):
        nd.shard_batches(nt, npanels, world, 0, [1.0] * 7)
    with pytest.raises(ValueError):
        nd.batch_bounds(10, 2, [1.0, 0.0])


def test_netcdf4_backend_reads_are_serialised_when_it_is_installed(tmp_path):
    """with netCDF4-python importable ncio prefers it (what the reference requires): its variables carry the lock, and
    the parallel readers of Field.fluxSeries (read_into from a thread pool + a prefetch thread) get the right values"""
    pytest.importorskip('netCDF4')
    import threading
    from nemoflux_b200 import ncio
    path = str(tmp_path / 'U.nc')
    data = numpy.arange(6 * 5 * 8 * 9, dtype=numpy.float32).reshape(6, 5, 8, 9)
    w = ncio.Writer(path)
    for name, n in (('t', 6), ('z', 5), ('y', 8), ('x', 9)):
        w.createDimension(name, n)
    w.createVariable('uo', 'float32', ('t', 'z', 'y', 'x'), fill_value=1.e20, data=data)
    w.close()
    with ncio.open_dataset(path) as nc:
        var = nc['uo']
        assert not var.thread_safe and var._lock is ncio._NETCDF4_LOCK
        dst = numpy.zeros_like(data)
        ths = [threading.Thread(target=var.read_into, args=(dst[t, z0:z0 + 1], (t, slice(z0, z0 + 1))))
               for t in range(6) for z0 in range(5)]
        for th in ths:
            th.start()
        for th in ths:
            th.join()
        assert numpy.array_equal(dst, data)


def test_fused_pass_queue_order_cannot_deadlock():
    """csrc/nfx_k23_fused.cu hands out work items from one counter in the order
        ... | K2 tiles of batch b | K3 items of batch b - lag | K2 tiles of batch b + 1 | ...
    A K2 tile of batch b waits for the K3 items of batch b - R (its ring slot), a K3 item of batch b for the K2 tiles of
    batch b.  The pass cannot deadlock, whatever the number of resident CTAs, iff every wait targets items with a SMALLER
    id (items a running CTA already holds) -- which needs R > lag.  This model restates the host-side choice of
    (ring slots R, lag) of flux_series_fused and checks the invariant, then runs the queue with 1..many CTAs."""
    def choose(resident, ntiles, slot_bytes, npanels, ring_max=24 << 20, lag_opt=0):
        slots = (2 * resident + ntiles - 1) // ntiles + 1
        cap = max(3, ring_max // slot_bytes)
        slots = min(max(slots, 3), cap)
        lag = lag_opt if lag_opt > 0 else ((resident + ntiles - 1) // ntiles + 1 if npanels == 1 else 1)
        lag = max(1, min(lag, cap - 2))
        slots = min(max(slots, lag + 2), cap)
        return slots, lag

    def item_ids(nb, ntiles, nk3, lag):
        per = ntiles + nk3
        k2 = lambda b: range(b * per, b * per + ntiles)                               # noqa: E731
        k3 = lambda b: range((b + lag) * per + ntiles, (b + lag) * per + per)         # noqa: E731
        return k2, k3, (nb + lag) * per

    rng = numpy.random.default_rng(17)
    shapes = [(444, 118, 1923 * 1024, 1), (592, 118, 1923 * 1024, 1), (444, 256, 4 << 20, 51), (592, 512, 8 << 20, 26),
              (444, 480, 8 << 20, 3), (3, 1, 64, 1), (1, 7, 1 << 20, 4)]
    shapes += [(int(rng.integers(1, 700)), int(rng.integers(1, 600)), int(rng.integers(1, 9)) << 20, int(rng.integers(1, 60)))
               for _ in range(40)]
    for resident, ntiles, slot_bytes, npanels in shapes:
        for lag_opt in (0, 1, 5, 60):
            R, lag = choose(resident, ntiles, slot_bytes, npanels, lag_opt=lag_opt)
            assert R > lag >= 1 and R * slot_bytes <= max(24 << 20, 3 * slot_bytes)
            nb, nk3 = 40, 3
            k2, k3, nitems = item_ids(nb, ntiles, nk3, lag)
            for b in range(nb):
                assert max(k2(b)) < min(k3(b))                                         # K3 of b waits for K2 of b
                if b >= R:
                    assert max(k3(b - R)) < min(k2(b))                                 # K2 of b waits for K3 of b - R
    # the queue itself, event by event, with few and many CTAs (a CTA holds one item and blocks until its counter is full)
    for ncta in (1, 2, 5, 64):
        for ntiles, nk3, nb, (R, lag) in ((3, 2, 12, (3, 1)), (2, 1, 9, (4, 2)), (5, 3, 7, (9, 7)), (1, 1, 30, (3, 1))):
            per = ntiles + nk3
            nitems = (nb + lag) * per
            k2done, k3done = [0] * nb, [0] * nb
            nxt, running, finished = 0, {}, 0
            for _ in range(100000):
                for c in range(ncta):                                                   # idle CTAs take the next item
                    if c not in running and nxt < nitems:
                        running[c] = nxt
                        nxt += 1
                progressed = False
                for c, it in sorted(running.items(), key=lambda kv: -kv[1]):          # worst case: newest item first
                    bb, r = divmod(it, per)
                    if r < ntiles:
                        b = bb
                        ok = b >= nb or b < R or k3done[b - R] == nk3
                        if ok:
                            if b < nb:
                                k2done[b] += 1
                    else:
                        b = bb - lag
                        ok = not (0 <= b < nb) or k2done[b] == ntiles
                        if ok and 0 <= b < nb:
                            k3done[b] += 1
                    if ok:
                        del running[c]
                        finished += 1
                        progressed = True
                        break
                if finished == nitems:
                    break
                assert progressed, (ncta, ntiles, nk3, nb, R, lag, running)
            assert finished == nitems and k2done == [ntiles] * nb and k3done == [nk3] * nb


def test_hdf5_random_hyperslabs_and_chunk_plans(tmp_path):
    """read_region on random blocks of chunked variables (both file generations, 2-4 axes, edge chunks that hang over
    the dataset, with and without shuffle + deflate) equals numpy slicing, and chunk_plan lists exactly the chunks a
    brute-force walk over the chunk grid finds -- the list the device decoder is fed with"""
    import itertools
    import h5build
    from nemoflux_b200 import h5lite
    rng = numpy.random.default_rng(77)
    cases = [((9, 14), (4, 5)), ((5, 3, 11, 13), (1, 1, 4, 6)), ((7, 6, 10), (2, 6, 3)), ((4, 20), (4, 20)), ((3, 17), (1, 40))]
    for writer in (h5build.write, h5build.write_new):
        variables = {}
        for k, (shape, chunks) in enumerate(cases):
            dt = ('<f4', '>f8', '<f8', '>f4', '<f4')[k]
            variables['v%d' % k] = dict(data=rng.standard_normal(shape).astype(dt), chunks=chunks,
                                        deflate=k % 2 == 0, shuffle=k % 3 != 1)
        path = str(tmp_path / ('slabs_%s.h5' % writer.__name__))
        writer(path, variables)
        f = h5lite.File(path)
        for name, v in variables.items():
            ds, data = f.datasets[name], v['data']
            assert ds.chunk_dims[:data.ndim] == tuple(v['chunks'])
            for trial in range(25):
                starts = [int(rng.integers(0, n)) for n in data.shape]
                stops = [int(rng.integers(a, n + 1)) for a, n in zip(starts, data.shape)]
                if trial == 0:
                    starts, stops = [0] * data.ndim, list(data.shape)
                got = ds.read_region(starts, stops)
                want = data[tuple(slice(a, b) for a, b in zip(starts, stops))]
                assert got.dtype == data.dtype and got.shape == want.shape and numpy.array_equal(got, want)
                origins = set()
                for idx in itertools.product(*[range(0, n, c) for n, c in zip(data.shape, v['chunks'])]):
                    if all(max(o, a) < min(o + c, b) for o, c, a, b in zip(idx, v['chunks'], starts, stops)):
                        origins.add(tuple(idx))
                plan = ds.chunk_plan(starts, stops)
                assert {tuple(p[3][:data.ndim]) for p in plan} == origins and len(plan) == len(origins)
                assert all(p[1] > 0 and p[0] > 0 for p in plan)
        f.close()
