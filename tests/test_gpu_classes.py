"""Class transport (fluxClasses): every transect's flux binned by a T-grid field -- against numpy built from the
per-level section and the class field at the crossings' cells on every storage type, metric, plane layout and special
value; the invariants against the layered and plain series; the infinity rule; bit-identical results across calls,
chunkings, byte orders and entry points; the errors; the Field / fluxplot --classField path."""
import numpy
import pytest

from helpers import README_C2, SF_C2, random_transects, tr

pytestmark = pytest.mark.gpu

NZ = 75
NFX_E_INVALID = 1          # include/nemoflux_gpu.h
PER_LEVEL = list(range(NZ + 1))
INF = numpy.inf


def _handle(gpu, points, ny, nx, transects):
    g = gpu.Grid()
    g.setPoints(points)
    g.setCGridShape(ny, nx)
    p = gpu.PolylineIntegral()
    p.build(g)
    p.computeWeights(transects)
    return g, p


def _np(x):
    return x if isinstance(x, numpy.ndarray) else x.cpu().numpy()


def _same(a, b, what=''):
    a, b = _np(a), _np(b)
    assert a.shape == b.shape, (what, a.shape, b.shape)
    assert numpy.array_equal(a.view(numpy.int64), b.view(numpy.int64)), (what, numpy.nanmax(numpy.abs(a - b)))


@pytest.fixture(scope='module')
def small(oracle):
    """76 800 cells, 75 levels, NaN land, denormals and the fill value -7 in u/v; transects that start in row 0 (south
    edges that are never written), in column 0 (x-periodic west edges), and one along a grid row (crossings shared by
    the two cells beside it)"""
    nx, ny, nt = 320, 240, 3
    g = oracle.DataGen(nx=nx, ny=ny, nz=NZ, nt=nt, deltaDeg=(20., 30.))
    P, arc = g.points(), oracle.arc_lengths(g.points())

    def center(c):
        lon = P[c, :, 0] - 360. * numpy.round((P[c, :, 0] - P[c, 0, 0]) / 360.)
        return float(lon.mean()), float(P[c, :, 1].mean())
    transects = random_transects(numpy.random.default_rng(3), 6, max_pts=4) + [tr(README_C2)]
    for a, b in (((0, nx // 3), (4, nx // 3 + 5)), ((ny // 2, 0), (ny // 2 + 3, 4))):
        pa, pb = center(a[0] * nx + a[1]), center(b[0] * nx + b[1])
        transects.append(tr([pa, (pb[0] - 360. * round((pb[0] - pa[0]) / 360.), pb[1])]))
    row = [P[(ny // 3) * nx + i, 0] for i in range(nx // 2, nx // 2 + 12)]    # south-west corners along one grid row
    transects.append(tr([(float(q[0]), float(q[1])) for q in row]))
    u, v = g.uv(SF_C2)
    u[:, :, 10:14, 20:40] = numpy.nan
    rng = numpy.random.default_rng(11)
    cf = rng.uniform(-2.0, 30.0, (nt, NZ, ny, nx))
    cf[:, :, 100:110, 50:90] = numpy.nan
    cf[:, 40:, 60:70, :] = 1e20                                    # the class field's marker
    cf[:, ::7] = numpy.round(cf[:, ::7])                           # values exactly on a bound
    return dict(nx=nx, ny=ny, nt=nt, P=P, arc=arc, transects=transects, u=u, v=v, cf=cf,
                th=numpy.linspace(1.0, 40.0, NZ))


BOUNDS = [-INF, 0.0, 4.0, 10.0, 17.0, 25.0]          # the top class ends at 25: values >= 25 count nowhere


def _fields(s, dtype):
    u, v = s['u'].astype(dtype), s['v'].astype(dtype)
    tiny = numpy.finfo(dtype).tiny
    u[:, ::2, 30:33, 5:60] = tiny / 8
    v[:, 1::3, 40:42, 10:70] = -tiny / 16
    v[:, :, 50:52, 100:120] = -7.0
    return u, v


def _reference(p, sec, cf, cfill, bounds):
    """classes of the definition in numpy: sec (nt, nz, nsub) the per-level section, cf (1 or nt, nz, ncell) in the
    storage type -> (classes, sum of |f| over the terms of every entry)"""
    sub = p.getSubsegments()
    x = cf[:, :, sub['cell']]
    bad = numpy.isnan(x) | (x == x.dtype.type(cfill))
    j = numpy.searchsorted(numpy.asarray(bounds), x.astype(numpy.float64), side='right') - 1
    j = numpy.where(bad | (j >= len(bounds) - 1), -1, j)
    j = numpy.broadcast_to(j, sec.shape)
    nt, K, M = sec.shape[0], len(bounds) - 1, len(sub['offsets']) - 1
    out, bar = numpy.zeros((nt, K, M)), numpy.zeros((nt, K, M))
    for m in range(M):
        a, b = sub['offsets'][m], sub['offsets'][m + 1]
        for c in range(K):
            f = numpy.where(j[..., a:b] == c, sec[..., a:b], 0.0)
            out[:, c, m] = f.sum((1, 2))
            bar[:, c, m] = numpy.abs(f).sum((1, 2))
    return out, bar


def _close(got, ref, bar, what=''):
    got = _np(got)
    assert got.shape == ref.shape, (what, got.shape, ref.shape)
    assert (numpy.abs(got - ref) <= 1e-12 * bar + 1e-300).all(), (what, numpy.abs(got - ref).max())


@pytest.mark.parametrize('dtype', [numpy.float64, numpy.float32])
@pytest.mark.parametrize('sverdrup', [False, True])
@pytest.mark.parametrize('padded', [False, True])
def test_classes_against_numpy(gpu, small, dtype, sverdrup, padded):
    """thickness and e3 (1 and nt steps), class field of 1 and nt steps: numpy's binning of the per-level section within
    1e-12 * sum |f|; row-0 south, x-periodic west edges and a transect along a grid line are read"""
    import torch
    s = small
    nx, ny, nt = s['nx'], s['ny'], s['nt']
    ncell = nx * ny
    u, v = _fields(s, dtype)
    _, p = _handle(gpu, s['P'], ny, nx, s['transects'])
    geo = p.getSectionGeometry()
    assert (geo['cell_j'] == 0).any() and (geo['cell_i'] == 0).any() and (p.getSubsegments()['coeff'] < 1).any()
    tdt = torch.float64 if dtype == numpy.float64 else torch.float32
    pad = 4 if dtype == numpy.float64 else 8
    ld = (ncell + 1 + pad - 1) // pad * pad if padded else ncell

    def dev(x):
        x = numpy.ascontiguousarray(x).reshape(x.shape[0], NZ, ncell)
        if not padded:
            return torch.from_numpy(x).to('cuda')
        t = torch.full((x.shape[0], NZ, ld), 3.0, dtype=tdt, device='cuda')[:, :, :ncell]
        t.copy_(torch.from_numpy(x))
        return t
    ud, vd = dev(u), dev(v)
    a1, a2, th = (torch.from_numpy(x).to('cuda') for x in (s['arc'][:, 1].copy(), s['arc'][:, 2].copy(), s['th']))
    kw = dict(sverdrup=sverdrup, fill=-7.0)
    cf = s['cf'].astype(dtype).reshape(nt, NZ, ncell)
    rng = numpy.random.default_rng(9)
    e3h = rng.uniform(0.5, 30., (nt, NZ, ny, nx)).astype(dtype)
    metrics = [('thickness', th, {})] + [(f'e3 {n}', None, dict(e3u=dev(e3h[:n]), e3v=dev(e3h[:n, ..., ::-1])))
                                         for n in (1, nt)]
    for name, thk, e3 in metrics:
        sec = _np(p.fluxSection(ud, vd, thk, a1, a2, layers=PER_LEVEL, **e3, **kw))
        for c_nt in (1, nt):
            for bounds, cfill in ((BOUNDS, 1e20), ([1.0, 2.0, 3.0, 5.0, 8.0, 13.0, 21.0, INF], float('nan'))):
                got = p.fluxClasses(ud, vd, thk, a1, a2, dev(cf[:c_nt]), bounds, cfill=cfill, **e3, **kw)
                assert got.dtype == torch.float64 and tuple(got.shape) == (nt, len(bounds) - 1, len(s['transects']))
                ref, bar = _reference(p, sec, cf[:c_nt], cfill, bounds)
                assert (bar > 0).sum() > len(s['transects'])
                _close(got, ref, bar, (name, c_nt, bounds))


def _per_level_bar(p, args, ny, nx, **kw):
    """(nt, nz, nsub) sum over the 4 edges of |w_e E_e| of every crossing and level: the scale of a series entry"""
    import torch
    u = args[0]
    nt, ncell = u.shape[0], nx * ny
    E = torch.empty((nt, NZ, 2 * ncell), dtype=torch.float64, device='cuda')
    p.fluxSeries(*args, eflux=E, layers=PER_LEVEL, **kw)
    E = E.cpu().numpy()
    sub = p.getSubsegments()
    cell = sub['cell']
    j, i = cell // nx, cell % nx
    idx = numpy.stack([numpy.where(j >= 1, ncell + cell - nx, -1), cell, ncell + cell,
                       numpy.where(i >= 1, cell - 1, cell + nx - 1)], 1)
    Eg = numpy.where(idx >= 0, E[..., numpy.maximum(idx, 0)], 0.0)
    return numpy.abs(sub['w'] * Eg).sum(-1)


def _transect_sum(p, x):
    offs = p.getSubsegments()['offsets']
    return numpy.stack([x[..., a:b].sum(-1) for a, b in zip(offs[:-1], offs[1:])], -1)


@pytest.mark.parametrize('dtype', [numpy.float64, numpy.float32])
def test_classes_invariants(gpu, small, dtype):
    """a field k + 0.5 with bounds on layer boundaries gives the layered series; one class (-inf, inf) on a finite field
    gives the plain series; classes covering the field's range add up to it (all within 1e-12)"""
    import torch
    s = small
    nx, ny, nt = s['nx'], s['ny'], s['nt']
    ncell = nx * ny
    u, v = _fields(s, dtype)
    _, p = _handle(gpu, s['P'], ny, nx, s['transects'])
    args = [torch.from_numpy(numpy.ascontiguousarray(x)).to('cuda')
            for x in (u, v, s['th'], s['arc'][:, 1].copy(), s['arc'][:, 2].copy())]
    bar_k = _per_level_bar(p, args, ny, nx, fill=-7.0)                      # (nt, nz, nsub)
    levels = numpy.broadcast_to((numpy.arange(NZ) + 0.5)[None, :, None], (1, NZ, ncell)).astype(dtype).copy()
    for L in ([0, NZ], [0, 1, 7, 23, 75], [10, 40], PER_LEVEL):
        got = _np(p.fluxClasses(*args, torch.from_numpy(levels).to('cuda'), numpy.array(L, numpy.float64), fill=-7.0))
        ser = _np(p.fluxSeries(*args, layers=L, fill=-7.0))
        bar = numpy.stack([_transect_sum(p, bar_k[:, L[i]:L[i + 1]].sum(1)) for i in range(len(L) - 1)], 1)
        assert (bar > 0).any()
        assert (numpy.abs(got - ser) <= 1e-12 * bar + 1e-300).all(), L
    plain = _np(p.fluxSeries(*args, fill=-7.0))
    bar = _transect_sum(p, bar_k.sum(1))
    finite = s['cf'][:1].astype(dtype).reshape(1, NZ, ncell)
    finite = numpy.where(numpy.isfinite(finite) & (finite < 1e19), finite, 3.0).astype(dtype)
    one = _np(p.fluxClasses(*args, torch.from_numpy(finite).to('cuda'), [-INF, INF], fill=-7.0))
    assert (numpy.abs(one[:, 0] - plain) <= 1e-12 * bar + 1e-300).all()
    cover = _np(p.fluxClasses(*args, torch.from_numpy(finite).to('cuda'), [-2.0, 0.0, 3.0, 3.5, 9.0, 20.0, 30.5],
                              fill=-7.0))
    assert (numpy.abs(cover.sum(1) - plain) <= 1e-12 * bar + 1e-300).all()


@pytest.mark.parametrize('dtype', [numpy.float64, numpy.float32])
def test_infinity_reaches_only_its_class(gpu, small, dtype):
    """+-inf on level 30 of 4 columns, a class field k + 0.5: the class holding level 30 is not finite in exactly the
    transects with a crossing that reads one of those columns; every other entry equals the classes of the data with 0
    there, bit for bit"""
    import torch
    s = small
    nx, ny, nt = s['nx'], s['ny'], s['nt']
    ncell = nx * ny
    u, v = _fields(s, dtype)
    _, p = _handle(gpu, s['P'], ny, nx, s['transects'])
    a1, a2, th = (torch.from_numpy(x).to('cuda') for x in (s['arc'][:, 1].copy(), s['arc'][:, 2].copy(), s['th']))
    sub = p.getSubsegments()
    cell = sub['cell']
    idx = numpy.stack([numpy.where(cell >= nx, ncell + cell - nx, -1), cell, ncell + cell,
                       numpy.where(cell % nx >= 1, cell - 1, cell + nx - 1)], 1)
    c0 = int(idx[len(idx) // 2, 1]) // 4 * 4
    reads = (((idx % ncell) >= c0) & ((idx % ncell) < c0 + 4) & (idx >= 0)).any(1)
    hit = numpy.array([reads[a:b].any() for a, b in zip(sub['offsets'][:-1], sub['offsets'][1:])])
    assert hit.any() and not hit.all()
    levels = numpy.broadcast_to((numpy.arange(NZ) + 0.5)[None, :, None], (1, NZ, ncell))
    levels = torch.from_numpy(levels.astype(dtype))
    bounds = [0.0, 10.0, 20.0, 30.0, 40.0, 75.0]
    dev = lambda x: torch.from_numpy(x).to('cuda')          # noqa: E731
    for val in (numpy.inf, -numpy.inf):
        ui, vi, u0, v0 = u.copy(), v.copy(), u.copy(), v.copy()
        for a, x in ((ui, val), (vi, val), (u0, 0), (v0, 0)):
            a.reshape(nt, NZ, -1)[:, 30, c0:c0 + 4] = x
        got = _np(p.fluxClasses(dev(ui), dev(vi), th, a1, a2, levels.cuda(), bounds, fill=-7.0))
        ref = _np(p.fluxClasses(dev(u0), dev(v0), th, a1, a2, levels.cuda(), bounds, fill=-7.0))
        assert not numpy.isfinite(got[:, 3][:, hit]).any()
        _same(got[:, 3][:, ~hit], ref[:, 3][:, ~hit], val)
        for c in (0, 1, 2, 4):
            _same(got[:, c], ref[:, c], (val, c))


@pytest.mark.parametrize('dtype', [numpy.float64, numpy.float32])
def test_classes_are_deterministic(gpu, small, dtype):
    """repeated device calls, the host entry point with every chunking, native and big-endian buffers, class field and
    e3 of 1 and nt steps on the host: the bits of the device call"""
    import torch
    s = small
    nx, ny, nt = s['nx'], s['ny'], s['nt']
    ncell = nx * ny
    u, v = _fields(s, dtype)
    _, p = _handle(gpu, s['P'], ny, nx, s['transects'])
    a1, a2 = s['arc'][:, 1].copy(), s['arc'][:, 2].copy()
    dargs = [torch.from_numpy(numpy.ascontiguousarray(x)).to('cuda') for x in (u, v, s['th'], a1, a2)]
    cf = s['cf'].astype(dtype)
    rng = numpy.random.default_rng(5)
    e3u = rng.uniform(0.5, 30., (nt, NZ, ny * nx)).astype(dtype)
    e3v = rng.uniform(0.5, 30., (nt, NZ, ny * nx)).astype(dtype)
    for c_nt in (1, nt):
        dc = torch.from_numpy(cf[:c_nt].reshape(c_nt, NZ, ncell)).to('cuda')
        ref = _np(p.fluxClasses(*dargs, dc, BOUNDS, cfill=1e20, fill=-7.0))
        for _ in range(3):
            _same(p.fluxClasses(*dargs, dc, BOUNDS, cfill=1e20, fill=-7.0), ref, 'repeat')
        for be in (False, True):
            to = (lambda x: x.astype(x.dtype.newbyteorder('>'))) if be else (lambda x: x)    # noqa: E731
            for cs in (1, 2, 0):
                out = p.fluxClasses(to(u), to(v), s['th'], a1, a2, to(cf[:c_nt]), BOUNDS, cfill=1e20, fill=-7.0,
                                    chunk_steps=cs)
                assert isinstance(out, numpy.ndarray)
                _same(out, ref, (c_nt, be, cs))
        for e3_nt in (1, nt):
            de3 = dict(e3u=torch.from_numpy(e3u[:e3_nt]).to('cuda'), e3v=torch.from_numpy(e3v[:e3_nt]).to('cuda'))
            ref = _np(p.fluxClasses(dargs[0], dargs[1], None, *dargs[3:], dc, BOUNDS, cfill=1e20, fill=-7.0, **de3))
            for be in (False, True):
                to = (lambda x: x.astype(x.dtype.newbyteorder('>'))) if be else (lambda x: x)    # noqa: E731
                for cs in (1, 0):
                    _same(p.fluxClasses(to(u), to(v), None, a1, a2, to(cf[:c_nt]), BOUNDS, cfill=1e20, fill=-7.0,
                                        chunk_steps=cs, e3u=to(e3u[:e3_nt]), e3v=to(e3v[:e3_nt])),
                          ref, ('host e3', c_nt, e3_nt, be, cs))


def test_classes_errors_and_edge_cases(gpu, small):
    import ctypes
    import torch
    from nemoflux_b200 import _lib
    s = small
    nx, ny, nt = s['nx'], s['ny'], s['nt']
    ncell = nx * ny
    _, p = _handle(gpu, s['P'], ny, nx, s['transects'])
    u, v = _fields(s, numpy.float64)
    args = [torch.from_numpy(x).to('cuda') for x in (u, v, s['th'], s['arc'][:, 1].copy(), s['arc'][:, 2].copy())]
    hargs = (u, v, s['th'], s['arc'][:, 1].copy(), s['arc'][:, 2].copy())
    cf = s['cf'][:1].reshape(1, NZ, ncell)
    dc = torch.from_numpy(cf).to('cuda')
    n0 = _lib.launch_count()
    for bad in ([0.0, numpy.nan, 1.0], [0.0, 1.0, 1.0], [2.0, 1.0], [INF, INF], list(range(98))):
        with pytest.raises(_lib.NemofluxGpuError) as e:
            p.fluxClasses(*args, dc, bad)
        assert e.value.code == NFX_E_INVALID and 'class' in str(e.value)
        with pytest.raises(_lib.NemofluxGpuError):
            p.fluxClasses(*hargs, cf, bad, chunk_steps=1)
    assert _lib.launch_count() == n0
    assert p.fluxClasses(*args, dc, list(range(97))).shape == (nt, 96, len(s['transects']))     # the largest K
    with pytest.raises(ValueError):
        p.fluxClasses(*args, dc, [1.0])
    with pytest.raises(TypeError):
        p.fluxClasses(*args, dc.float(), BOUNDS)                              # dtype of the class field
    with pytest.raises(ValueError):
        p.fluxClasses(*args, dc[:, :-1], BOUNDS)                              # levels
    with pytest.raises(ValueError):
        p.fluxClasses(*args, torch.cat([dc, dc]), BOUNDS)                     # 2 steps, nt = 3
    # one level on padded planes (ld > ncell): a class field or e3 of nt steps must step time by nz * ld as uo/vo do
    def padded():
        return torch.ones((nt, 1, ncell + 8), dtype=torch.float64, device='cuda')[:, :, :ncell]
    flat = torch.ones((nt, 1, ncell), dtype=torch.float64, device='cuda')
    one = [padded(), padded(), args[2][:1], args[3], args[4]]
    assert tuple(p.fluxClasses(*one, padded(), BOUNDS).shape) == (nt, 5, len(s['transects']))
    with pytest.raises(ValueError):
        p.fluxClasses(*one, flat, BOUNDS)
    with pytest.raises(ValueError):
        p.fluxClasses(one[0], one[1], None, *one[3:], padded(), BOUNDS, e3u=flat, e3v=flat)
    with pytest.raises(ValueError):
        p.fluxClasses(*hargs, cf.astype(numpy.float32), BOUNDS)              # host: dtype
    with pytest.raises(ValueError):
        p.fluxClasses(*hargs, cf.astype('>f8'), BOUNDS)                      # host: byte order
    # NULL pointers and a handle without a C-grid shape: refused, nothing launched
    lib = _lib.load()
    b = numpy.array(BOUNDS)
    ptr = [ctypes.c_void_p(a.data_ptr()) for a in args]
    out = torch.zeros((nt, 5, len(s['transects'])), dtype=torch.float64, device='cuda')
    n0 = _lib.launch_count()
    for cfp, outp in ((None, out.data_ptr()), (dc.data_ptr(), None)):
        assert lib.nfx_flux_classes(ctypes.byref(p._h), ptr[0], ptr[1], None, None, _lib.NFX_F64, 0, ptr[2], ptr[3],
                                    ptr[4], nt, NZ, ncell, cfp, 1, float('nan'), 5, b.ctypes.data_as(ctypes.c_void_p),
                                    0, float('nan'), outp, None) == NFX_E_INVALID
    assert lib.nfx_flux_classes(ctypes.byref(p._h), ptr[0], ptr[1], None, None, _lib.NFX_F64, 0, ptr[2], ptr[3],
                                ptr[4], nt, NZ, ncell, dc.data_ptr(), 1, float('nan'), 5, None, 0, float('nan'),
                                out.data_ptr(), None) == NFX_E_INVALID
    assert _lib.launch_count() == n0
    g2 = gpu.Grid()
    g2.setPoints(s['P'])
    p2 = gpu.PolylineIntegral()
    p2.build(g2)
    p2.computeWeights(s['transects'])
    n0 = _lib.launch_count()
    with pytest.raises(_lib.NemofluxGpuError) as e:
        p2.fluxClasses(*args, dc, BOUNDS)
    assert e.value.code == NFX_E_INVALID and 'cgrid' in str(e.value)
    with pytest.raises(_lib.NemofluxGpuError):
        p2.fluxClasses(*hargs, cf, BOUNDS)
    assert _lib.launch_count() == n0
    # no step, no transect, and a transect that crosses no cell (outside the grid)
    assert tuple(p.fluxClasses(*(a[:0] for a in args[:2]), *args[2:], dc, BOUNDS).shape) == (0, 5, len(s['transects']))
    assert p.fluxClasses(u[:0], v[:0], *hargs[2:], cf, BOUNDS).shape == (0, 5, len(s['transects']))
    assert _lib.launch_count() == n0
    _, p0 = _handle(gpu, s['P'], ny, nx, [])
    assert tuple(p0.fluxClasses(*args, dc, BOUNDS).shape) == (nt, 5, 0)
    assert p0.fluxClasses(*hargs, cf, BOUNDS).shape == (nt, 5, 0)
    lines = [s['transects'][0], tr([(0., 100.), (10., 120.)]), s['transects'][1]]
    _, pe = _handle(gpu, s['P'], ny, nx, lines)
    offs = pe.getSubsegments()['offsets']
    assert offs[2] == offs[1] and offs[1] > 0 and offs[3] > offs[2]
    got = _np(pe.fluxClasses(*args, dc, BOUNDS, cfill=1e20))
    assert (got[:, :, 1] == 0).all()
    _, p1 = _handle(gpu, s['P'], ny, nx, [lines[0], lines[2]])
    _same(got[:, :, [0, 2]], p1.fluxClasses(*args, dc, BOUNDS, cfill=1e20))
    _same(pe.fluxClasses(*hargs, cf, BOUNDS, cfill=1e20), got)


def _files(tmp_path, nt, nz):
    """datagen's T/U/V files, the T file rewritten with a thetao (t, z, y, x) float32 variable (_FillValue 1e20 on a
    patch of land), and a separate file with a time-invariant float64 so (z, y, x)"""
    from nemoflux_b200 import datagen, ncio
    prefix = str(tmp_path) + '/'
    datagen.cli([f'--streamFunction={SF_C2}', '--nx=72', '--ny=36', f'--nz={nz}', f'--nt={nt}', '--deltaDeg=20,30',
                 f'--prefix={prefix}'])
    with ncio.open_dataset(prefix + 'T.nc') as nc:
        grid = {k: numpy.asarray(nc[k][:]) for k in ('deptht_bounds', 'bounds_lat', 'bounds_lon')}
    rng = numpy.random.default_rng(21)
    thetao = rng.uniform(-2.0, 20.0, (nt, nz, 36, 72)).astype(numpy.float32)
    thetao[:, 3:, 10:14, 30:40] = 1e20
    so = rng.uniform(33.0, 36.0, (nz, 36, 72))
    T2 = prefix + 'T2.nc'
    w = ncio.Writer(T2)
    for name, n in (('t', nt), ('z', nz), ('y', 36), ('x', 72), ('nvertex', 4), ('axis_nbounds', 2)):
        w.createDimension(name, n)
    w.createVariable('deptht_bounds', 'f8', ('z', 'axis_nbounds'), data=grid['deptht_bounds'])
    w.createVariable('bounds_lat', 'f8', ('y', 'x', 'nvertex'), data=grid['bounds_lat'])
    w.createVariable('bounds_lon', 'f8', ('y', 'x', 'nvertex'), data=grid['bounds_lon'])
    w.createVariable('thetao', 'f4', ('t', 'z', 'y', 'x'), fill_value=1e20, data=thetao)
    w.close()
    S = prefix + 'S.nc'
    w = ncio.Writer(S)
    for name, n in (('z', nz), ('y', 36), ('x', 72)):
        w.createDimension(name, n)
    w.createVariable('so', 'f8', ('z', 'y', 'x'), data=so)
    w.close()
    return T2, prefix + 'U.nc', prefix + 'V.nc', S, thetao, so


def test_field_and_fluxplot_classes(gpu, oracle, tmp_path, capsys):
    """Field.fluxClasses on classic files (big-endian; the class field from the T file, f32 next to f64 uo/vo, and
    time-invariant from another file) and on deflated NetCDF-4 uo/vo (device decode): PolylineIntegral.fluxClasses of
    the same data, bit for bit; fluxplot --classField prints and writes one column per (transect, class), and
    --timeMean averages them"""
    import h5build
    from nemoflux_b200 import fluxplot
    from nemoflux_b200.field import Field
    nt, nz = 4, 8
    T, U, V, S, thetao, so = _files(tmp_path, nt, nz)
    lines = [tr([(-100, -70), (100, -70), (0, 70)]), tr([(-150, -20), (-20, 35), (60, -40)])]
    tb, sb = [-2.0, 0.0, 5.0, 10.0, 20.0], [33.0, 34.0, 34.8, 36.0]

    def direct(f, c, bounds, cfill):
        u, v, fill = f._uv_slabs(0, f.nt)
        c = c.astype(u.dtype).reshape(-1, nz, 36, 72)
        return f.pli.fluxClasses(u, v, f.thickness, f.arcLengths[:, 1].copy(), f.arcLengths[:, 2].copy(), c, bounds,
                                 cfill=cfill, sverdrup=f.sverdrup, fill=fill)
    f = Field(T, U, V, lines, sverdrup=True, verbose=False)
    ref_t = direct(f, thetao, tb, float(numpy.float32(1e20)))
    assert numpy.abs(ref_t).max() > 0
    for cs in (1, 0):
        _same(f.fluxClasses('thetao', tb, chunk_steps=cs), ref_t, ('thetao', cs))
    ref_s = direct(f, so, sb, float('nan'))
    _same(f.fluxClasses('so', sb, file=S, chunk_steps=3), ref_s, 'so')
    d = oracle.DataGen(nx=72, ny=36, nz=nz, nt=nt, deltaDeg=(20., 30.))
    u, v = d.uv(SF_C2)
    U4, V4 = str(tmp_path / 'U4.nc'), str(tmp_path / 'V4.nc')
    for fname, vname, a in ((U4, 'uo', u), (V4, 'vo', v)):
        h5build.write(fname, {vname: dict(data=a, chunks=(1, 2, 36, 72), deflate=True, shuffle=True),
                              'time_counter': dict(data=numpy.arange(float(nt)), chunks=(1,))})
    f4 = Field(T, U4, V4, lines, verbose=False)
    got = f4.fluxClasses('thetao', tb, chunk_steps=2)
    assert f4.last_ingest['path'] == 'device decode'
    _same(got, direct(f4, thetao, tb, float(numpy.float32(1e20))), 'device decode')
    _same(f4.fluxClasses('thetao', tb, chunk_steps=2, device_decode=False), got, 'host zlib')
    # fluxplot --classField
    pts = '[(-100,-70),(100,-70),(0,70)],[(-150,-20),(-20,35),(60,-40)]'
    csv = str(tmp_path / 'classes.csv')
    series = fluxplot.main(['-t', T, '-u', U, '-v', V, '-l', pts, '-s', '--classField', 'thetao',
                            '--classBounds=-2,0,5,10,20', '-o', csv])
    out = capsys.readouterr().out
    _same(series, ref_t, 'fluxplot')
    heads = [f'{lab}[{a:g}–{b:g})' for lab in ('transect0', 'transect1') for a, b in zip(tb[:-1], tb[1:])]
    with open(csv, encoding='utf-8') as fh:
        rows = [r.rstrip('\n').split(',') for r in fh]
    assert len(rows[0]) == 9 and len(rows) == nt + 1
    assert all(h.endswith(w[w.index('['):]) for h, w in zip(rows[0][1:], heads))
    assert rows[0][1][rows[0][1].index('['):] in out
    vals = numpy.array([[float(x) for x in r[1:]] for r in rows[1:]])
    _same(vals, ref_t.transpose(0, 2, 1).reshape(nt, -1), 'csv')
    series = fluxplot.main(['-t', T, '-u', U, '-v', V, '-l', pts, '-s', '--classField', f'so:{S}', '--classBounds',
                            '33,34,34.8,36', '--timeMean', '2'])
    capsys.readouterr()
    _same(series, fluxplot.windowMeans(ref_s, [0, 2, 4]), 'timeMean')
