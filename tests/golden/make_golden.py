"""Generate golden vectors from the REAL reference code (run once, in the build container).

The reference (/root/reference/nemoflux/*.py) cannot run end to end here: mint, vtk, xarray, netCDF4,
defopt and matplotlib are not installed.  Its numpy-only pieces can: this script stubs the missing
modules in sys.modules, imports the reference's own ``datagen``, ``geo``, ``field`` and
``latlonreader`` modules from /root/reference and calls

  * DataGen.build / rotatePole / applyStreamFunction / computeUVFromPotential (datagen.py:31-166),
  * geo.lonLat2XYZArray / geo.getArcLengthArray through Field.computeArcLengths (field.py:170-181),
  * Field.readField (field.py:145-163) and Field.computeIntegratedFlux (field.py:183-234),
  * LatLonReader (latlonreader.py:8-20) on every transect file under /root/reference/data,

writing the outputs to tests/golden/*.npz / *.json.  Nothing here is read at test time from
/root/reference; the fixtures are committed.  The mint-dependent pieces (computeWeights,
getIntegral) cannot be generated this way -- that part of the oracle stays "parity unpinned".

Usage:  python tests/golden/make_golden.py
"""
import hashlib
import json
import os
import sys
import types

import numpy

REF = '/root/reference/nemoflux'
OUT = os.environ.get('NFX_GOLDEN_OUT') or os.path.dirname(os.path.abspath(__file__))   # regenerate elsewhere to compare


def _stub_modules():
    for name in ('netCDF4', 'defopt', 'xarray', 'mint', 'vtk', 'matplotlib', 'matplotlib.pyplot',
                 'matplotlib.dates'):
        if name not in sys.modules:
            sys.modules[name] = types.ModuleType(name)
    sys.modules['defopt'].run = lambda *a, **k: None
    sys.path.insert(0, REF)


class _Var(object):
    """stands in for an xarray variable: nc[name][t, :, :, :].fillna(0.0)"""

    def __init__(self, arr):
        self.arr = arr
        self.shape = arr.shape

    def __getitem__(self, idx):
        return _Var(self.arr[idx])

    def fillna(self, value):
        return numpy.where(numpy.isnan(self.arr), value, self.arr)


class _Grid(object):
    def __init__(self, points):
        self.points = points

    def getPoints(self):
        return self.points


def sha(a):
    return hashlib.sha256(numpy.ascontiguousarray(a).tobytes()).hexdigest()


def run_datagen(datagen, streamFunction, nx=36, ny=18, nz=1, nt=1, deltaDeg=(0., 0.),
                xmin=-180., xmax=180., ymin=-90., ymax=90., zmin=0., zmax=1.):
    g = datagen.DataGen('')
    g.setSizes(nx, ny, nz, nt)
    g.setBoundingBox(xmin=xmin, xmax=xmax, ymin=ymin, ymax=ymax, zmin=zmin, zmax=zmax)
    g.build()
    if deltaDeg[0] != 0 or deltaDeg[1] != 0:
        g.rotatePole(deltaDeg=deltaDeg)
    g.applyStreamFunction(streamFunction)
    g.computeUVFromPotential()
    return g


def run_field(field_mod, g, timeIndex=0, sverdrup=False, landmask=None):
    """Field.computeArcLengths + readField + computeIntegratedFlux on DataGen output."""
    F = field_mod.Field
    f = F.__new__(F)
    f.sverdrup = sverdrup
    f.nt, f.nz, f.ny, f.nx = g.nt, g.nz, g.ny, g.nx
    ncell = g.ny * g.nx
    pts = numpy.zeros((g.ny, g.nx, 4, 3), numpy.float64)   # horizgrid.py:17-22
    pts[..., 0] = g.bounds_lon
    pts[..., 1] = g.bounds_lat
    f.gr = _Grid(pts.reshape((ncell, 4, 3)))
    f.arcLengths = numpy.zeros((ncell, 4), numpy.float64)
    f.computeArcLengths()
    bounds_depth = numpy.stack([g.ztop, g.zbot], axis=1)    # datagen.py:176-178
    f.thickness = bounds_depth[:, 1] - bounds_depth[:, 0]   # field.py:51
    u, v = g.u.copy(), g.v.copy()
    if landmask is not None:
        u[:, landmask] = numpy.nan
        v[:, landmask] = numpy.nan
    f.ncU = {'uo': _Var(u)}
    f.ncV = {'vo': _Var(v)}
    f.timeIndex = timeIndex
    f.edgeFluxesUArray = numpy.zeros((ncell,), numpy.float64)
    f.edgeFluxesVArray = numpy.zeros((ncell,), numpy.float64)
    f.integratedVelocity = numpy.zeros((ncell, 4), numpy.float64)
    f.maxAbsFlux = 0.
    U, V = f.getUV()
    f.computeIntegratedFlux(U, V)
    return dict(arcLengths=f.arcLengths, thickness=numpy.asarray(f.thickness), U=numpy.asarray(U),
                V=numpy.asarray(V), iV=f.integratedVelocity, absEU=f.edgeFluxesUArray,
                absEV=f.edgeFluxesVArray, maxAbsFlux=numpy.float64(f.maxAbsFlux), u=u, v=v)


def main():
    _stub_modules()
    import datagen
    import field as field_mod
    import latlonreader

    summary = {}

    # C1 (README.md:26): --streamFunction="x", defaults
    g = run_datagen(datagen, 'x')
    r = run_field(field_mod, g)
    numpy.savez_compressed(os.path.join(OUT, 'c1_simple.npz'), bounds_lon=g.bounds_lon,
                           bounds_lat=g.bounds_lat, ztop=g.ztop, zbot=g.zbot, **r)
    summary['c1_simple'] = dict(maxAbsFlux=float(r['maxAbsFlux']))

    # singular (README.md:50)
    g = run_datagen(datagen, 'arctan2(y, x+180)/(2*pi)')
    r = run_field(field_mod, g)
    numpy.savez_compressed(os.path.join(OUT, 'singular.npz'), bounds_lon=g.bounds_lon,
                           bounds_lat=g.bounds_lat, ztop=g.ztop, zbot=g.zbot, **r)
    summary['singular'] = dict(maxAbsFlux=float(r['maxAbsFlux']))

    # small pole-displaced case with depth/time dependence, a land mask (NaN) and Sverdrup units
    sf = '(1+10*z)*(t+1)*(cos(2*pi*y/360) + sin(2*pi*x/360))'
    g = run_datagen(datagen, sf, nx=24, ny=12, nz=3, nt=2, deltaDeg=(20., 30.))
    mask = numpy.zeros((3, 12, 24), bool)
    mask[:, 3:6, 4:9] = True
    mask[2, :, 15:] = True
    for ti in (0, 1):
        for sv in (False, True):
            r = run_field(field_mod, g, timeIndex=ti, sverdrup=sv, landmask=mask)
            numpy.savez_compressed(os.path.join(OUT, f'rot24x12_t{ti}_sv{int(sv)}.npz'),
                                   bounds_lon=g.bounds_lon, bounds_lat=g.bounds_lat, ztop=g.ztop,
                                   zbot=g.zbot, mask=mask, **r)

    # C2 (README.md:89-91): too large to commit in full -> digests + the vertically integrated fields
    g = run_datagen(datagen, sf, nx=360, ny=180, nz=10, nt=20, deltaDeg=(20., 30.))
    dig = dict(bounds_lon=sha(g.bounds_lon), bounds_lat=sha(g.bounds_lat), u=sha(g.u), v=sha(g.v))
    keep = {}
    for ti in (0, 19):
        r = run_field(field_mod, g, timeIndex=ti)
        dig[f'iV_t{ti}'] = sha(r['iV'])
        dig[f'arcLengths'] = sha(r['arcLengths'])
        keep[f'U_t{ti}'] = r['U']
        keep[f'V_t{ti}'] = r['V']
        keep[f'iV_t{ti}_rows'] = r['iV'][::997]        # sparse sample of rows
        dig[f'maxAbsFlux_t{ti}'] = float(r['maxAbsFlux'])
    numpy.savez_compressed(os.path.join(OUT, 'c2_sample.npz'), ztop=g.ztop, zbot=g.zbot,
                           bounds_lon_rows=g.bounds_lon[::17, ::13], bounds_lat_rows=g.bounds_lat[::17, ::13],
                           **keep)
    summary['c2_digests'] = dig

    # a plain 360x180 rectilinear grid, closed-loop case of README.md:65-66 (digests only)
    g = run_datagen(datagen, 'cos(2*pi*y/360) + sin(2*pi*x/360)', nx=360, ny=180)
    r = run_field(field_mod, g)
    summary['closed2_digests'] = dict(u=sha(g.u), v=sha(g.v), iV=sha(r['iV']),
                                      maxAbsFlux=float(r['maxAbsFlux']))

    # LatLonReader on every transect file (latlonreader.py:8-20)
    ll = {}
    root = '/root/reference/data'
    for d, _, files in sorted(os.walk(root)):
        for fn in sorted(files):
            if fn.endswith('.txt'):
                p = os.path.join(d, fn)
                ll[os.path.relpath(p, root)] = latlonreader.LatLonReader(p).getLonLats().tolist()
    summary['latlonreader'] = ll

    with open(os.path.join(OUT, 'golden_summary.json'), 'w') as f:
        json.dump(summary, f, indent=1, sort_keys=True)
    print('wrote', sorted(os.listdir(OUT)))


if __name__ == '__main__':
    main()
