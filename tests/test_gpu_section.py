"""The transport section (fluxSection): per cell crossing, layer and time step, the weighted sum of the 4 layered edge
fluxes fluxSeries(layers=, eflux=) writes -- bit for bit against numpy on every storage type, layering, metric, plane
layout and entry point; its sums against the layered series and the oracle; the analytic per-crossing answer; the
infinity rule; the errors; the Field / fluxplot --section path."""
import numpy
import pytest

from helpers import README_C2, SF_C2, random_transects, tr

pytestmark = pytest.mark.gpu

NZ = 75
NFX_E_INVALID = 1          # include/nemoflux_gpu.h
ONE, RAGGED, PER_LEVEL, PARTIAL = [0, NZ], [0, 1, 7, 23, 75], list(range(NZ + 1)), [10, 40]
LAYERINGS = {'one': ONE, 'ragged': RAGGED, 'per-level': PER_LEVEL, 'partial': PARTIAL}


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
    assert numpy.array_equal(a, b, equal_nan=True), (what, numpy.nanmax(numpy.abs(a - b)))


def _center(P, c):
    """a point inside cell c: the mean of its vertices, longitudes unwrapped around vertex 0"""
    lon = P[c, :, 0] - 360. * numpy.round((P[c, :, 0] - P[c, 0, 0]) / 360.)
    return float(lon.mean()), float(P[c, :, 1].mean())


@pytest.fixture(scope='module')
def small(oracle):
    """the data of test_gpu_layers.py: 76 800 cells, 75 levels, NaN land, denormals and the fill value -7; plus two
    transects that start in row 0 (south edges that are never written) and in column 0 (x-periodic west edges)"""
    nx, ny, nt = 320, 240, 2
    g = oracle.DataGen(nx=nx, ny=ny, nz=NZ, nt=nt, deltaDeg=(20., 30.))
    P, arc = g.points(), oracle.arc_lengths(g.points())
    transects = random_transects(numpy.random.default_rng(3), 6, max_pts=4) + [tr(README_C2)]
    for a, b in (((0, nx // 3), (4, nx // 3 + 5)), ((ny // 2, 0), (ny // 2 + 3, 4))):
        pa = _center(P, a[0] * nx + a[1])
        pb = _center(P, b[0] * nx + b[1])
        pb = (pb[0] - 360. * round((pb[0] - pa[0]) / 360.), pb[1])
        transects.append(tr([pa, pb]))
    u, v = g.uv(SF_C2)
    u[:, :, 10:14, 20:40] = numpy.nan
    return dict(nx=nx, ny=ny, nt=nt, g=g, P=P, arc=arc, transects=transects, u=u, v=v,
                th=numpy.linspace(1.0, 40.0, NZ))


def _fields(s, dtype):
    u, v = s['u'].astype(dtype), s['v'].astype(dtype)
    tiny = numpy.finfo(dtype).tiny
    u[:, ::2, 30:33, 5:60] = tiny / 8
    v[:, 1::3, 40:42, 10:70] = -tiny / 16
    v[:, :, 50:52, 100:120] = -7.0
    return u, v


def _flux_index(cell, ny, nx):
    """(nsub, 4) list-order compact index of the edges S, E, N, W of every crossing's cell (-1: south edge of row 0)"""
    ncell = ny * nx
    j, i = cell // nx, cell % nx
    return numpy.stack([numpy.where(j >= 1, ncell + cell - nx, -1), cell, ncell + cell,
                        numpy.where(i >= 1, cell - 1, cell + nx - 1)], 1)


def _gather(p, ny, nx, E):
    """(w, E at the 4 edges of every crossing): E (..., 2*ncell) -> (..., nsub, 4)"""
    sub = p.getSubsegments()
    idx = _flux_index(sub['cell'], ny, nx)
    Eg = numpy.where(idx >= 0, E[..., numpy.maximum(idx, 0)], 0.0)
    return sub['w'], Eg


def _reference(p, ny, nx, E):
    """the section of the definition, in numpy (float64 multiplies and adds, no FMA)"""
    w, Eg = _gather(p, ny, nx, E)
    with numpy.errstate(all='ignore'):
        return ((w[:, 0] * Eg[..., 0] + w[:, 1] * Eg[..., 1]) + w[:, 2] * Eg[..., 2]) + w[:, 3] * Eg[..., 3]


def _eflux(p, u, v, th, a1, a2, L, **kw):
    import torch
    nt, ncell = u.shape[0], a1.numel()
    buf = torch.full((nt, len(L) - 1, 2 * ncell), 5.0, dtype=torch.float64, device=u.device)
    p.fluxSeries(u, v, th, a1, a2, eflux=buf, layers=L, **kw)
    return buf.cpu().numpy()


@pytest.mark.parametrize('dtype', [numpy.float64, numpy.float32])
@pytest.mark.parametrize('sverdrup', [False, True])
@pytest.mark.parametrize('padded', [False, True])
def test_section_bit_contract(gpu, small, dtype, sverdrup, padded):
    """every layering, thickness and e3 (1 and nt steps): the numpy evaluation of the definition from the layered
    edge fluxes, bit for bit; row-0 south and x-periodic west edges are read"""
    import torch
    s = small
    nx, ny, nt = s['nx'], s['ny'], s['nt']
    ncell = nx * ny
    u, v = _fields(s, dtype)
    _, p = _handle(gpu, s['P'], ny, nx, s['transects'])
    geo = p.getSectionGeometry()
    assert (geo['cell_j'] == 0).any() and (geo['cell_i'] == 0).any()
    d = 'cuda'
    tdt = torch.float64 if dtype == numpy.float64 else torch.float32
    pad = 4 if dtype == numpy.float64 else 8
    ld = (ncell + 1 + pad - 1) // pad * pad if padded else ncell

    def dev(x):
        x = numpy.ascontiguousarray(x).reshape(x.shape[0], NZ, ncell)
        if not padded:
            return torch.from_numpy(x).to(d)
        t = torch.full((x.shape[0], NZ, ld), 3.0, dtype=tdt, device=d)[:, :, :ncell]
        t.copy_(torch.from_numpy(x))
        return t
    ud, vd = dev(u), dev(v)
    a1, a2, th = (torch.from_numpy(x).to(d) for x in (s['arc'][:, 1].copy(), s['arc'][:, 2].copy(), s['th']))
    kw = dict(sverdrup=sverdrup, fill=-7.0)
    nsub = p.getNumberOfSubsegments()
    for name, L in LAYERINGS.items():
        sec = p.fluxSection(ud, vd, th, a1, a2, layers=L, **kw)
        assert sec.shape == (nt, len(L) - 1, nsub) and sec.dtype == torch.float64
        _same(sec, _reference(p, ny, nx, _eflux(p, ud, vd, th, a1, a2, L, **kw)), ('thickness', name))
    _same(p.fluxSection(ud, vd, th, a1, a2, **kw), p.fluxSection(ud, vd, th, a1, a2, layers=PER_LEVEL, **kw))
    rng = numpy.random.default_rng(9)
    for e3_nt in (1, nt):
        e3h = rng.uniform(0.5, 30., (e3_nt, NZ, ny, nx)).astype(dtype)
        e3 = dict(e3u=dev(e3h), e3v=dev(e3h[..., ::-1]))
        for name, L in (('one', ONE), ('ragged', RAGGED), ('partial', PARTIAL)):
            sec = p.fluxSection(ud, vd, None, a1, a2, layers=L, **e3, **kw)
            _same(sec, _reference(p, ny, nx, _eflux(p, ud, vd, None, a1, a2, L, **e3, **kw)), ('e3', e3_nt, name))


def _l1(p, ny, nx, E):
    """sum over a transect's crossings of sum_e |w_e E_e|: (..., M)"""
    w, Eg = _gather(p, ny, nx, E)
    per = numpy.abs(w * Eg).sum(-1)
    offs = p.getSubsegments()['offsets']
    return numpy.stack([per[..., a:b].sum(-1) for a, b in zip(offs[:-1], offs[1:])], -1)


def _by_transect(p, sec):
    offs = p.getSubsegments()['offsets']
    return numpy.stack([sec[..., a:b].sum(-1) for a, b in zip(offs[:-1], offs[1:])], -1)


@pytest.mark.parametrize('dtype', [numpy.float64, numpy.float32])
def test_section_sums_to_the_layered_series(gpu, small, dtype):
    import torch
    s = small
    u, v = _fields(s, dtype)
    _, p = _handle(gpu, s['P'], s['ny'], s['nx'], s['transects'])
    d = 'cuda'
    args = [torch.from_numpy(numpy.ascontiguousarray(x)).to(d)
            for x in (u, v, s['th'], s['arc'][:, 1].copy(), s['arc'][:, 2].copy())]
    for L in (ONE, RAGGED, PER_LEVEL):
        sec = _np(p.fluxSection(*args, layers=L, fill=-7.0))
        tot = _by_transect(p, sec)
        bar = _l1(p, s['ny'], s['nx'], _eflux(p, *args, L, fill=-7.0))
        assert (bar > 0).any()
        for order in ('list', 'map'):
            ser = _np(p.fluxSeries(*args, layers=L, fill=-7.0, order=order))
            assert (numpy.abs(tot - ser) <= 1e-12 * bar + 1e-300).all(), (L, order)


def test_section_sums_to_the_oracle(gpu, oracle):
    import torch
    nz = 12
    g = oracle.DataGen(nx=72, ny=36, nz=nz, nt=3, deltaDeg=(20., 30.))
    P, arc = g.points(), oracle.arc_lengths(g.points())
    u, v = g.uv(SF_C2)
    rng = numpy.random.default_rng(99)
    land = rng.random((nz, g.ny, g.nx)) < 0.15
    u[:, land] = numpy.nan
    v[:, land] = numpy.nan
    transects = random_transects(rng, 10) + [tr(README_C2)]
    th = g.thickness()
    _, p = _handle(gpu, P, g.ny, g.nx, transects)
    d = 'cuda'
    args = [torch.from_numpy(numpy.ascontiguousarray(x)).to(d) for x in (u, v, th, arc[:, 1].copy(), arc[:, 2].copy())]
    for L in ([0, 3, 4, 12], [2, 9]):
        sec = _np(p.fluxSection(*args, layers=L))
        tot = _by_transect(p, sec)
        bar = _l1(p, g.ny, g.nx, _eflux(p, *args, L))
        for i in range(len(L) - 1):
            thm = th.copy()
            thm[:L[i]] = 0.
            thm[L[i + 1]:] = 0.
            ref = oracle.flux_series(P, transects, u, v, thm)
            assert (numpy.abs(tot[:, i] - ref) <= 2e-12 * bar[:, i] + 1e-300).all(), (L, i)


def test_section_analytic_per_crossing(gpu):
    """unrotated regular grid, nodal stream function psi_k = a1_k g1 + a2_k g2: every crossing of cell (j, i) carries
    coeff * dz_k * (psi_h(end) - psi_h(start)) on level k, psi_h bilinear in the cell; a closed loop adds up to 0"""
    import torch
    from nemoflux_b200 import synth
    syn = synth.make('tiny', deltaDeg=(0., 0.), land=False)
    d = torch.device('cuda', 0)
    _, p = _handle(gpu, syn.points, syn.ny, syn.nx, syn.transects)
    u, v = syn.fill_device(0, 2, d)
    th, a1, a2 = (torch.from_numpy(x).to(d) for x in (syn.thickness, syn.arc1, syn.arc2))
    sec = _np(p.fluxSection(u, v, th, a1, a2))
    sub = p.getSubsegments()
    j, i = sub['cell'] // syn.nx, sub['cell'] % syn.nx

    def bilinear(g, xi):
        s_, t_ = xi[:, 0], xi[:, 1]
        return ((1 - s_) * (1 - t_) * g[j, i] + s_ * (1 - t_) * g[j, i + 1] + s_ * t_ * g[j + 1, i + 1] +
                (1 - s_) * t_ * g[j + 1, i])
    d1 = bilinear(syn.g1, sub['xib']) - bilinear(syn.g1, sub['xia'])
    d2 = bilinear(syn.g2, sub['xib']) - bilinear(syn.g2, sub['xia'])
    inner = (j >= 1) & (i >= 1)        # row 0 has no south flux, and g2 is not periodic across column 0
    assert inner.sum() > 100
    scale = 0.
    for t in range(2):
        c1, c2 = syn.coeffs(t)
        ex = sub['coeff'][None] * syn.thickness[:, None] * (c1[:, None] * d1[None] + c2[:, None] * d2[None])
        scale = max(scale, numpy.abs(ex).max())
        assert numpy.abs(sec[t][:, inner] - ex[:, inner]).max() <= 1e-11 * scale, t
    offs = sub['offsets']
    loops = [m for m, k in enumerate(syn.kinds) if k == 'loop']
    assert loops
    for m in loops:
        assert numpy.abs(sec[:, :, offs[m]:offs[m + 1]].sum(-1)).max() <= 1e-11 * scale, m


@pytest.mark.parametrize('dtype', [numpy.float64, numpy.float32])
def test_infinity_reaches_only_its_crossings(gpu, small, dtype):
    """+-inf on level 30 of 4 columns: in the layer holding level 30, exactly the crossings that read one of those
    columns are not finite; every other value equals the section of the data with 0 there, bit for bit"""
    import torch
    s = small
    nx, ny, nt = s['nx'], s['ny'], s['nt']
    ncell = nx * ny
    u, v = _fields(s, dtype)
    _, p = _handle(gpu, s['P'], ny, nx, s['transects'])
    d = 'cuda'
    a1, a2, th = (torch.from_numpy(x).to(d) for x in (s['arc'][:, 1].copy(), s['arc'][:, 2].copy(), s['th']))
    idx = _flux_index(p.getSubsegments()['cell'], ny, nx)
    c0 = int(idx[len(idx) // 2, 1]) // 4 * 4
    col = slice(c0, c0 + 4)
    reads = (((idx % ncell) >= c0) & ((idx % ncell) < c0 + 4) & (idx >= 0)).any(1)
    assert reads.any() and not reads.all()
    dev = lambda x: torch.from_numpy(x).to(d)          # noqa: E731
    for val in (numpy.inf, -numpy.inf):
        ui, vi, u0, v0 = u.copy(), v.copy(), u.copy(), v.copy()
        for a, x in ((ui, val), (vi, val), (u0, 0), (v0, 0)):
            a.reshape(nt, NZ, -1)[:, 30, col] = x
        sec = _np(p.fluxSection(dev(ui), dev(vi), th, a1, a2, layers=RAGGED, fill=-7.0))
        ref = _np(p.fluxSection(dev(u0), dev(v0), th, a1, a2, layers=RAGGED, fill=-7.0))
        for i in range(len(RAGGED) - 1):
            if RAGGED[i] <= 30 < RAGGED[i + 1]:
                assert not numpy.isfinite(sec[:, i][:, reads]).any()
                _same(sec[:, i][:, ~reads], ref[:, i][:, ~reads], (val, i))
            else:
                _same(sec[:, i], ref[:, i], (val, i))


@pytest.mark.parametrize('dtype', [numpy.float64, numpy.float32])
@pytest.mark.parametrize('big_endian', [False, True])
def test_section_host_entry_point(gpu, small, dtype, big_endian):
    """host buffers (native / big-endian, chunks of 1 step and automatic, e3 on the device, on the host invariant and on
    the host per step): the device path, bit for bit"""
    import torch
    s = small
    nx, ny, nt = s['nx'], s['ny'], s['nt']
    u, v = _fields(s, dtype)
    _, p = _handle(gpu, s['P'], ny, nx, s['transects'])
    d = 'cuda'
    a1, a2 = s['arc'][:, 1].copy(), s['arc'][:, 2].copy()
    dargs = [torch.from_numpy(numpy.ascontiguousarray(x)).to(d) for x in (u, v, s['th'], a1, a2)]
    hu, hv = (u.astype(u.dtype.newbyteorder('>')), v.astype(v.dtype.newbyteorder('>'))) if big_endian else (u, v)
    for L in (ONE, RAGGED, PER_LEVEL):
        ref = _np(p.fluxSection(*dargs, layers=L, fill=-7.0))
        for cs in (1, 0):
            out = p.fluxSection(hu, hv, s['th'], a1, a2, layers=L, fill=-7.0, chunk_steps=cs)
            assert isinstance(out, numpy.ndarray)
            _same(out, ref, (L, cs))
    rng = numpy.random.default_rng(5)
    for e3_nt in (1, nt):
        e3u = rng.uniform(0.5, 30., (e3_nt, NZ, ny * nx)).astype(dtype)
        e3v = rng.uniform(0.5, 30., (e3_nt, NZ, ny * nx)).astype(dtype)
        de3 = dict(e3u=torch.from_numpy(e3u).to(d), e3v=torch.from_numpy(e3v).to(d))
        ref = _np(p.fluxSection(*dargs[:2], None, *dargs[3:], layers=RAGGED, fill=-7.0, **de3))
        he3 = (e3u.astype(hu.dtype), e3v.astype(hu.dtype))
        for cs in (1, 0):
            _same(p.fluxSection(hu, hv, None, a1, a2, layers=RAGGED, fill=-7.0, chunk_steps=cs, e3u=he3[0], e3v=he3[1]),
                  ref, ('host e3', e3_nt, cs))
            if e3_nt == 1:
                _same(p.fluxSection(hu, hv, None, a1, a2, layers=RAGGED, fill=-7.0, chunk_steps=cs, **de3), ref,
                      ('device e3', cs))


def test_section_errors_and_edge_cases(gpu, small):
    import ctypes
    import torch
    from nemoflux_b200 import _lib
    s = small
    nx, ny, nt = s['nx'], s['ny'], s['nt']
    _, p = _handle(gpu, s['P'], ny, nx, s['transects'])
    d = 'cuda'
    u, v = _fields(s, numpy.float64)
    args = [torch.from_numpy(x).to(d) for x in (u, v, s['th'], s['arc'][:, 1].copy(), s['arc'][:, 2].copy())]
    nsub = p.getNumberOfSubsegments()
    n0 = _lib.launch_count()
    for bad in ([5, 5], [0, 10, 7], [-1, 10], [0, NZ + 1], [40, 10]):
        out = torch.full((nt, len(bad) - 1, nsub), 42.0, dtype=torch.float64, device=d)
        with pytest.raises(_lib.NemofluxGpuError) as e:
            p.fluxSection(*args, layers=bad, out=out)
        assert e.value.code == NFX_E_INVALID and 'layers' in str(e.value)
        assert (out == 42.0).all()
        with pytest.raises(_lib.NemofluxGpuError):
            p.fluxSection(u, v, s['th'], s['arc'][:, 1].copy(), s['arc'][:, 2].copy(), chunk_steps=1, layers=bad)
    assert _lib.launch_count() == n0
    for bad in ([3], [[0, 1]], [0, 2.5]):
        with pytest.raises(ValueError):
            p.fluxSection(*args, layers=bad)
    out = torch.full((nt, 4, nsub), 42.0, dtype=torch.float64, device=d)
    with pytest.raises(ValueError):
        p.fluxSection(*args, layers=[0, 10, 75], out=out)                   # wrong size
    with pytest.raises(TypeError):
        p.fluxSection(*args, layers=RAGGED, out=out.float())                # wrong dtype
    with pytest.raises(ValueError):
        p.fluxSection(args[0], args[1][:, :, :-1], *args[2:], layers=RAGGED)   # u / v shapes differ
    with pytest.raises(TypeError):
        p.fluxSection(args[0].float(), args[1].float(), *args[2:], layers=RAGGED, e3u=args[0], e3v=args[1])
    with pytest.raises(ValueError):
        p.fluxSection(*args[:3], args[3][:-1], args[4], layers=RAGGED)    # arc1 size
    assert (out == 42.0).all()
    # NULL section pointer and a handle without a C-grid shape: refused, nothing launched
    lib = _lib.load()
    lev = numpy.array(RAGGED, numpy.int32)
    ptr = [ctypes.c_void_p(a.data_ptr()) for a in args]
    assert lib.nfx_flux_section(ctypes.byref(p._h), ptr[0], ptr[1], None, None, _lib.NFX_F64, 0, ptr[2], ptr[3], ptr[4],
                                nt, NZ, nx * ny, len(RAGGED) - 1, lev.ctypes.data_as(ctypes.c_void_p), 0, float('nan'),
                                None, None) == NFX_E_INVALID
    g2 = gpu.Grid()
    g2.setPoints(s['P'])
    p2 = gpu.PolylineIntegral()
    p2.build(g2)
    p2.computeWeights(s['transects'])
    n0 = _lib.launch_count()
    with pytest.raises(_lib.NemofluxGpuError) as e:
        p2.fluxSection(*args, layers=RAGGED)
    assert e.value.code == NFX_E_INVALID and 'cgrid' in str(e.value)
    assert _lib.launch_count() == n0
    # two calls, identical bits
    a = _np(p.fluxSection(*args, layers=PER_LEVEL))
    _same(p.fluxSection(*args, layers=PER_LEVEL), a)
    # no transect, and a transect that crosses no cell (outside the grid)
    _, p0 = _handle(gpu, s['P'], ny, nx, [])
    sec0 = p0.fluxSection(*args, layers=RAGGED)
    assert tuple(sec0.shape) == (nt, len(RAGGED) - 1, 0)
    assert p0.fluxSection(u, v, s['th'], s['arc'][:, 1].copy(), s['arc'][:, 2].copy(), layers=RAGGED).shape == \
        (nt, len(RAGGED) - 1, 0)
    lines = [s['transects'][0], tr([(0., 100.), (10., 120.)]), s['transects'][1]]
    _, pe = _handle(gpu, s['P'], ny, nx, lines)
    offs = pe.getSubsegments()['offsets']
    assert offs[2] == offs[1] and offs[1] > 0 and offs[3] > offs[2]
    sec = _np(pe.fluxSection(*args, layers=RAGGED))
    _, p1 = _handle(gpu, s['P'], ny, nx, [lines[0], lines[2]])
    _same(sec, p1.fluxSection(*args, layers=RAGGED))
    assert (pe.seriesStatus() == 0)


def _files(tmp_path, *args):
    from nemoflux_b200 import datagen
    prefix = str(tmp_path) + '/'
    datagen.cli(list(args) + [f'--prefix={prefix}'])
    return prefix + 'T.nc', prefix + 'U.nc', prefix + 'V.nc'


def test_field_and_fluxplot_section(gpu, oracle, tmp_path, capsys):
    """Field.fluxSection on classic (big-endian), NetCDF-4 contiguous, deflated (device-decoded) and meshFile= inputs:
    PolylineIntegral.fluxSection of the same data, bit for bit; fluxplot --section writes it and reads back equal"""
    import h5build
    from nemoflux_b200 import fluxplot, ncio
    from nemoflux_b200.field import Field
    nz = 8
    T, U, V = _files(tmp_path, f'--streamFunction={SF_C2}', '--nx=72', '--ny=36', f'--nz={nz}', '--nt=4',
                     '--deltaDeg=20,30', '--meshMask', '--partialCells=0.5')
    mesh = str(tmp_path / 'mesh_mask.nc')
    lines = [tr([(-100, -70), (100, -70), (0, 70)]), tr([(-150, -20), (-20, 35), (60, -40)])]

    def direct(f, L):
        u, v, fill = f._uv_slabs(0, f.nt)
        return f.pli.fluxSection(u, v, f.thickness, f.arcLengths[:, 1].copy(), f.arcLengths[:, 2].copy(),
                                 sverdrup=f.sverdrup, fill=fill, layers=L, e3u=f._d_e3u, e3v=f._d_e3v)
    f = Field(T, U, V, lines, verbose=False)
    for L in (None, [0, 2, 5, 8]):
        sec = f.fluxSection(layers=L, chunk_steps=1)
        assert sec.shape == (4, nz if L is None else 3, f.pli.getNumberOfSubsegments())
        _same(sec, direct(f, L), ('classic', L))
        _same(f.fluxSection(layers=L), sec)
    fm = Field(T, U, V, lines, sverdrup=True, verbose=False, meshFile=mesh)
    assert fm._d_e3u is not None
    _same(fm.fluxSection(layers=[0, 3, 8], chunk_steps=2), direct(fm, [0, 3, 8]), 'meshFile')
    # the same data as NetCDF-4 files: contiguous (host read) and chunked + deflated (device decode)
    d = oracle.DataGen(nx=72, ny=36, nz=nz, nt=4, deltaDeg=(20., 30.))
    u, v = d.uv(SF_C2)
    for kind, chunks in (('contiguous', None), ('deflated', (1, 2, 36, 72))):
        U4, V4 = str(tmp_path / f'U4{kind}.nc'), str(tmp_path / f'V4{kind}.nc')
        for fname, vname, a in ((U4, 'uo', u), (V4, 'vo', v)):
            h5build.write(fname, {vname: dict(data=a, chunks=chunks, deflate=chunks is not None,
                                              shuffle=chunks is not None),
                                  'time_counter': dict(data=numpy.arange(4.), chunks=(1,) if chunks else None)})
        f4 = Field(T, U4, V4, lines, verbose=False)
        sec = f4.fluxSection(layers=[0, 2, 5, 8], chunk_steps=2)
        if kind == 'deflated':
            assert f4.last_ingest['path'] == 'device decode'
            _same(f4.fluxSection(layers=[0, 2, 5, 8], chunk_steps=2, device_decode=False), sec, 'host zlib')
        _same(sec, direct(f4, [0, 2, 5, 8]), kind)
    # fluxplot --section
    pts = '[(-100,-70),(100,-70),(0,70)],[(-150,-20),(-20,35),(60,-40)]'
    path = str(tmp_path / 'section.nc')
    series = fluxplot.main(['-t', T, '-u', U, '-v', V, '-l', pts, '-s', '--layers', '0,2,5,8', '--section', path])
    out = capsys.readouterr().out
    assert 'crossings written' in out and series.shape == (4, 3, 2)
    fs = Field(T, U, V, lines, sverdrup=True, verbose=False)
    ref = fs.fluxSection(layers=[0, 2, 5, 8])
    geo = fs.pli.getSectionGeometry()
    with ncio.open_dataset(path) as nc:
        assert tuple(nc['transport'].shape) == ref.shape and ref.shape[2] == fs.pli.getNumberOfSubsegments()
        _same(numpy.asarray(nc['transport'][:], numpy.float64), ref, 'file')
        assert numpy.array_equal(nc['transect_offsets'][:], geo['offsets'])
        assert numpy.array_equal(nc['distance_km'][:], geo['distance_km'])
        assert numpy.array_equal(nc['cell_i'][:], geo['cell_i'])
        iface = fs.layerInterfaces()
        assert numpy.array_equal(nc['layer_top'][:], iface[[0, 2, 5]])
        assert numpy.array_equal(nc['layer_bottom'][:], iface[[2, 5, 8]])
    assert numpy.abs(_by_transect(fs.pli, ref) - series).max() <= 1e-12 * numpy.abs(series).max() * 100
