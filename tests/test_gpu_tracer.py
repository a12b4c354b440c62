"""Tracer transport (fluxTracer): the flux of every crossing with each level term weighted by a tracer at the C-grid
face of its edge -- bit for bit against the section for a tracer of 1 (and of 2^p), against numpy restating the
definition, and the series against numpy's tile-tree fold of the section, on every storage type, metric, plane layout
and special value; the missing-value rules; layers and ref; bit-identical results across calls, chunkings, byte orders
and entry points; the errors; the Field / fluxplot --tracer path."""
import numpy
import pytest

from helpers import tr
from test_gpu_classes import NZ, _fields, _files, _handle, _np, _same, small  # noqa: F401 (small: a fixture)

pytestmark = pytest.mark.gpu

NFX_E_INVALID = 1          # include/nemoflux_gpu.h
PER_LEVEL = list(range(NZ + 1))
LAYERS = [0, 1, 7, 23, 60, 75]


def _faces(p, nx, ny):
    """per crossing and edge (S, E, N, W): the flux index (-1: none), the face's T cells a, b and whether b exists"""
    ncell = nx * ny
    c = p.getSubsegments()['cell'].astype(numpy.int64)
    j, i = c // nx, c % nx
    east = numpy.where(i + 1 < nx, c + 1, c + 1 - nx)
    west = numpy.where(i >= 1, c - 1, c + nx - 1)
    north = numpy.where(j + 1 < ny, c + nx, c)
    south = numpy.where(j >= 1, c - nx, c)
    idx = numpy.stack([numpy.where(j >= 1, ncell + c - nx, -1), c, ncell + c, west], 1)
    a = numpy.stack([south, c, c, west], 1)
    b = numpy.stack([c, east, north, c], 1)
    has_b = numpy.stack([j >= 0, j >= 0, j + 1 < ny, j >= 0], 1)
    return idx, a, b, has_b


def _reference(p, nx, ny, u, v, tau, arc1, arc2, layers, th=None, e3u=None, e3v=None, ref=0.0, tfill=numpy.nan,
               fill=numpy.nan, sverdrup=False):
    """the section of the definition in numpy, sequential over k, every operation elementwise in float64: u, v
    (nt, nz, ncell), tau / e3u / e3v (1 or nt, nz, ncell) in the storage type -> (section (nt, N, nsub), sum of |terms|)"""
    ncell = nx * ny
    idx, a, b, has_b = _faces(p, nx, ny)
    w = p.getSubsegments()['w']
    live = idx >= 0
    isv = idx >= ncell
    col = numpy.where(live, numpy.where(isv, idx - ncell, idx), 0)
    arc = numpy.where(live, numpy.where(isv, -arc2[col], arc1[col]), 0.0)
    dt = u.dtype.type

    def clean(x):
        return numpy.where(numpy.isnan(x) | (x == dt(fill)), 0.0, x.astype(numpy.float64))
    miss = lambda x: numpy.isnan(x) | (x == dt(tfill))                       # noqa: E731
    nt, nsub = u.shape[0], len(w)
    out = numpy.zeros((nt, len(layers) - 1, nsub))
    bar = numpy.zeros_like(out)
    for li in range(len(layers) - 1):
        A = numpy.zeros((nt, nsub, 4))
        B = numpy.zeros((nt, nsub, 4))
        for k in range(layers[li], layers[li + 1]):
            x = clean(numpy.where(isv, v[:, k][:, col], u[:, k][:, col]))
            if th is not None:
                d = th[k]
            else:
                d = clean(numpy.where(isv, e3v[:, k][:, col], e3u[:, k][:, col]))
            ta, tb = tau[:, k][:, a], tau[:, k][:, b]
            pa, pb = ~miss(ta), ~miss(tb) & has_b
            fa, fb = ta.astype(numpy.float64), tb.astype(numpy.float64)
            with numpy.errstate(invalid='ignore', over='ignore'):
                q = numpy.where(pa & pb, 0.5 * (fa + fb) - ref,
                                numpy.where(pa, fa - ref, numpy.where(pb, fb - ref, 0.0)))
                term = (d * x) * q
            A = A + term
            B = B + numpy.abs(term)
        with numpy.errstate(invalid='ignore', over='ignore'):
            f = A * arc
            g = B * numpy.abs(arc)
            if sverdrup:
                f = f * (6371000.0 / 1.e6)
                g = g * (6371000.0 / 1.e6)
            f = numpy.where(live, f, 0.0)
            g = numpy.where(live, g, 0.0)
            r = w[:, 0] * f[..., 0]
            for e in range(1, 4):
                r = r + w[:, e] * f[..., e]
        out[:, li] = r
        bar[:, li] = (numpy.abs(w) * g).sum(-1)
    return out, bar


def _tile_fold(p, sec):
    """the series of a section (nt, N, nsub): per transect tiles of 32 crossings in emission order, each folded by the
    shuffle tree (lane l + lane l + o, o = 16 .. 1, absent lanes +0), then the tiles in ascending order from +0"""
    offs = p.getSubsegments()['offsets']
    nt, n = sec.shape[:2]
    out = numpy.zeros((nt, n, len(offs) - 1))
    for m in range(len(offs) - 1):
        acc = numpy.zeros((nt, n))
        for t0 in range(offs[m], offs[m + 1], 32):
            lanes = numpy.zeros((nt, n, 32))
            t1 = min(t0 + 32, offs[m + 1])
            lanes[..., :t1 - t0] = sec[..., t0:t1]
            for o in (16, 8, 4, 2, 1):
                lanes[..., :o] = lanes[..., :o] + lanes[..., o:2 * o]
            acc = acc + lanes[..., 0]
        out[..., m] = acc
    return out


def _tracer(s, dtype, tfill):
    """a tracer of nt steps with NaN land, the marker on a patch (one reaching the top row) and rows of equal values"""
    nx, ny, nt = s['nx'], s['ny'], s['nt']
    rng = numpy.random.default_rng(17)
    t = rng.uniform(-2.0, 30.0, (nt, NZ, ny, nx))
    t[:, :, 100:110, 50:90] = numpy.nan
    t[:, :, 10:12, 20:30] = numpy.nan                                 # land beside u's NaN patch
    t[:, 40:, 60:70, :] = tfill
    t[:, :, ny - 2:, 100:160] = tfill                                 # the top row: N faces with no north cell
    t[:, ::5, 30:35, :] = 4.0
    return t.astype(dtype).reshape(nt, NZ, nx * ny)


@pytest.mark.parametrize('dtype', [numpy.float64, numpy.float32])
@pytest.mark.parametrize('sverdrup', [False, True])
@pytest.mark.parametrize('padded', [False, True])
def test_tracer_contracts(gpu, small, dtype, sverdrup, padded):
    """thickness and e3 (1 and nt steps), tracer of 1 and nt steps, padded planes: tau == 1 gives fluxSection bit for
    bit and tau == 2^p its 2^p multiple; numpy's restatement of the definition is met bit for bit, and the series is
    numpy's tile-tree fold of the section bit for bit"""
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
    a1h, a2h = s['arc'][:, 1].copy(), s['arc'][:, 2].copy()
    a1, a2, th = (torch.from_numpy(x).to('cuda') for x in (a1h, a2h, s['th']))
    kw = dict(sverdrup=sverdrup, fill=-7.0)
    tau = _tracer(s, dtype, 1e20)
    e3h = numpy.random.default_rng(9).uniform(0.5, 30., (nt, NZ, ny, nx)).astype(dtype).reshape(nt, NZ, ncell)
    e3vh = e3h.reshape(nt, NZ, ny, nx)[..., ::-1].reshape(nt, NZ, ncell)
    metrics = [('thickness', th, {}, dict(th=s['th']))] + \
        [(f'e3 {n}', None, dict(e3u=dev(e3h[:n]), e3v=dev(e3vh[:n])), dict(e3u=e3h[:n], e3v=e3vh[:n])) for n in (1, nt)]
    uh, vh = u.reshape(nt, NZ, ncell), v.reshape(nt, NZ, ncell)
    ud0, vd0 = dev(s['u'].astype(dtype)), dev(s['v'].astype(dtype))     # without the denormals
    for name, thk, e3, e3r in metrics:
        for L in (PER_LEVEL, LAYERS):
            sec = p.fluxSection(ud, vd, thk, a1, a2, layers=L, **e3, **kw)
            sec0 = p.fluxSection(ud0, vd0, thk, a1, a2, layers=L, **e3, **kw)
            for tr_nt in (1, nt):
                one = dev(numpy.ones((tr_nt, NZ, ncell), dtype))
                _same(p.fluxTracer(ud, vd, thk, a1, a2, one, layers=L, section=True, **e3, **kw), sec, (name, 'tau 1'))
                # 2^p: exact wherever no intermediate value is subnormal
                four = dev(numpy.full((tr_nt, NZ, ncell), 4.0, dtype))
                _same(p.fluxTracer(ud0, vd0, thk, a1, a2, four, layers=L, section=True, **e3, **kw), 4.0 * sec0,
                      (name, 'tau 4'))
        for tr_nt in (1, nt):
            got = p.fluxTracer(ud, vd, thk, a1, a2, dev(tau[:tr_nt]), tfill=1e20, layers=LAYERS, section=True, **e3,
                               **kw)
            assert got.dtype == torch.float64 and tuple(got.shape) == (nt, len(LAYERS) - 1, len(geo['cell_j']))
            ref, bar = _reference(p, nx, ny, uh, vh, tau[:tr_nt], a1h, a2h, LAYERS, tfill=1e20, fill=-7.0,
                                  sverdrup=sverdrup, **e3r)
            assert numpy.isfinite(ref).all() and (bar > 0).sum() > 100
            _same(got, ref, (name, tr_nt, 'numpy'))
            ser = p.fluxTracer(ud, vd, thk, a1, a2, dev(tau[:tr_nt]), tfill=1e20, layers=LAYERS, **e3, **kw)
            _same(ser, _tile_fold(p, _np(got)), (name, tr_nt, 'fold'))
    whole = p.fluxTracer(ud, vd, th, a1, a2, dev(tau), tfill=1e20, **kw)
    assert tuple(whole.shape) == (nt, len(s['transects']))
    _same(whole, p.fluxTracer(ud, vd, th, a1, a2, dev(tau), tfill=1e20, layers=[0, NZ], **kw)[:, 0], 'layers=None')


@pytest.mark.parametrize('dtype', [numpy.float64, numpy.float32])
def test_missing_values_and_faces(gpu, small, dtype):
    """a tracer missing (NaN or the marker) on one side of a face takes the other side, on both sides counts 0, and the
    N face of the top row takes its own cell: numpy's restatement on a tracer with every such case, bit for bit; a
    tracer missing everywhere gives 0"""
    import torch
    s = small
    nx, ny, nt = s['nx'], s['ny'], s['nt']
    ncell = nx * ny
    u, v = _fields(s, dtype)
    P = s['P']

    def center(c):
        lon = P[c, :, 0] - 360. * numpy.round((P[c, :, 0] - P[c, 0, 0]) / 360.)
        return float(lon.mean()), float(P[c, :, 1].mean())
    pa, pb = center((ny - 1) * nx + 100), center((ny - 2) * nx + 106)   # through cells of the top row
    lines = s['transects'] + [tr([pa, (pb[0] - 360. * round((pb[0] - pa[0]) / 360.), pb[1])])]
    _, p = _handle(gpu, P, ny, nx, lines)
    cells = p.getSubsegments()['cell']
    a1h, a2h = s['arc'][:, 1].copy(), s['arc'][:, 2].copy()
    dev = lambda x: torch.from_numpy(numpy.ascontiguousarray(x)).to('cuda')   # noqa: E731
    uh, vh = u.reshape(nt, NZ, ncell), v.reshape(nt, NZ, ncell)
    args = [dev(uh), dev(vh), dev(s['th']), dev(a1h), dev(a2h)]
    rng = numpy.random.default_rng(23)
    tau = rng.uniform(-2.0, 30.0, (nt, NZ, ncell)).astype(dtype)
    # every other crossing cell missing (NaN or the marker) on alternate levels; some neighbours as well
    tau[:, ::2, cells[::2]] = numpy.nan
    tau[:, 1::2, cells[1::3]] = -999.0
    tau[:, :, (cells[::5] + 1) % ncell] = -999.0
    tau[:, 3::4, (cells[::7] + nx) % ncell] = numpy.nan
    for tfill in (-999.0, float('nan')):
        got = p.fluxTracer(*args, dev(tau), tfill=tfill, ref=1.5, layers=LAYERS, section=True, fill=-7.0)
        ref, _ = _reference(p, nx, ny, uh, vh, tau, a1h, a2h, LAYERS, th=s['th'], ref=1.5, tfill=tfill, fill=-7.0)
        _same(got, ref, tfill)
    assert (cells >= ncell - nx).any()                                      # the top row is crossed
    nan = numpy.full((1, NZ, ncell), numpy.nan, dtype)
    assert (_np(p.fluxTracer(*args, dev(nan), layers=LAYERS, section=True, fill=-7.0)) == 0).all()


@pytest.mark.parametrize('dtype', [numpy.float64, numpy.float32])
def test_layers_and_ref(gpu, small, dtype):
    """the layers of a column add up to the whole column, and ref: the series with ref equals the series with ref = 0
    minus ref times the volume series (both within 1e-12 * sum |terms|)"""
    import torch
    s = small
    nx, ny, nt = s['nx'], s['ny'], s['nt']
    ncell = nx * ny
    u, v = _fields(s, dtype)
    _, p = _handle(gpu, s['P'], ny, nx, s['transects'])
    a1h, a2h = s['arc'][:, 1].copy(), s['arc'][:, 2].copy()
    uh, vh = u.reshape(nt, NZ, ncell), v.reshape(nt, NZ, ncell)
    dev = lambda x: torch.from_numpy(numpy.ascontiguousarray(x)).to('cuda')   # noqa: E731
    args = [dev(uh), dev(vh), dev(s['th']), dev(a1h), dev(a2h)]
    tau = numpy.random.default_rng(29).uniform(-2.0, 30.0, (nt, NZ, ncell)).astype(dtype)
    _, bar_k = _reference(p, nx, ny, uh, vh, tau, a1h, a2h, PER_LEVEL, th=s['th'], fill=-7.0)
    offs = p.getSubsegments()['offsets']
    tsum = lambda x: numpy.stack([x[..., a:b].sum(-1) for a, b in zip(offs[:-1], offs[1:])], -1)   # noqa: E731
    whole = _np(p.fluxTracer(*args, dev(tau), fill=-7.0))
    bar = tsum(bar_k.sum(1))
    assert (bar > 0).all()
    layered = _np(p.fluxTracer(*args, dev(tau), layers=LAYERS, fill=-7.0))
    assert (numpy.abs(layered.sum(1) - whole) <= 1e-12 * bar).all()
    per_level = _np(p.fluxTracer(*args, dev(tau), layers=PER_LEVEL, fill=-7.0))
    assert (numpy.abs(per_level.sum(1) - whole) <= 1e-12 * bar).all()
    vol = _np(p.fluxSeries(*args, fill=-7.0))
    _, bar_v = _reference(p, nx, ny, uh, vh, numpy.ones_like(tau), a1h, a2h, [0, NZ], th=s['th'], fill=-7.0)
    for r in (34.8, -3.0):
        got = _np(p.fluxTracer(*args, dev(tau), ref=r, fill=-7.0))
        assert (numpy.abs(got - (whole - r * vol)) <= 1e-12 * (bar + abs(r) * tsum(bar_v[:, 0]))).all(), r


@pytest.mark.parametrize('dtype', [numpy.float64, numpy.float32])
def test_tracer_is_deterministic(gpu, small, dtype):
    """repeated device calls, the host entry point with every chunking, native and big-endian buffers, tracer and e3 of
    1 and nt steps, series and section: the bits of the device call"""
    import torch
    s = small
    nx, ny, nt = s['nx'], s['ny'], s['nt']
    ncell = nx * ny
    u, v = _fields(s, dtype)
    _, p = _handle(gpu, s['P'], ny, nx, s['transects'])
    a1, a2 = s['arc'][:, 1].copy(), s['arc'][:, 2].copy()
    dargs = [torch.from_numpy(numpy.ascontiguousarray(x)).to('cuda') for x in (u, v, s['th'], a1, a2)]
    tau = _tracer(s, dtype, 1e20).reshape(nt, NZ, ny, nx)
    rng = numpy.random.default_rng(5)
    e3u = rng.uniform(0.5, 30., (nt, NZ, ny * nx)).astype(dtype)
    e3v = rng.uniform(0.5, 30., (nt, NZ, ny * nx)).astype(dtype)
    kw = dict(tfill=1e20, ref=2.5, fill=-7.0)
    be_ = lambda x: x.astype(x.dtype.newbyteorder('>'))                  # noqa: E731
    for tr_nt in (1, nt):
        dt = torch.from_numpy(tau[:tr_nt].reshape(tr_nt, NZ, ncell)).to('cuda')
        for layers, section in ((None, False), (LAYERS, False), (None, True)):
            ref = _np(p.fluxTracer(*dargs, dt, layers=layers, section=section, **kw))
            for _ in range(2):
                _same(p.fluxTracer(*dargs, dt, layers=layers, section=section, **kw), ref, 'repeat')
            for be in (False, True):
                to = be_ if be else (lambda x: x)
                for cs in (1, 2, 0):
                    out = p.fluxTracer(to(u), to(v), s['th'], a1, a2, to(tau[:tr_nt]), layers=layers, section=section,
                                       chunk_steps=cs, **kw)
                    assert isinstance(out, numpy.ndarray)
                    _same(out, ref, (tr_nt, layers, section, be, cs))
        for e3_nt in (1, nt):
            de3 = dict(e3u=torch.from_numpy(e3u[:e3_nt]).to('cuda'), e3v=torch.from_numpy(e3v[:e3_nt]).to('cuda'))
            ref = _np(p.fluxTracer(dargs[0], dargs[1], None, *dargs[3:], dt, layers=LAYERS, **kw, **de3))
            for be in (False, True):
                to = be_ if be else (lambda x: x)
                for cs in (1, 0):
                    _same(p.fluxTracer(to(u), to(v), None, a1, a2, to(tau[:tr_nt]), layers=LAYERS, chunk_steps=cs,
                                       e3u=to(e3u[:e3_nt]), e3v=to(e3v[:e3_nt]), **kw),
                          ref, ('host e3', tr_nt, e3_nt, be, cs))


def test_tracer_errors_and_edge_cases(gpu, small):
    import ctypes
    import torch
    from nemoflux_b200 import _lib
    s = small
    nx, ny, nt = s['nx'], s['ny'], s['nt']
    ncell = nx * ny
    _, p = _handle(gpu, s['P'], ny, nx, s['transects'])
    u, v = _fields(s, numpy.float64)
    M = len(s['transects'])
    args = [torch.from_numpy(x).to('cuda') for x in (u, v, s['th'], s['arc'][:, 1].copy(), s['arc'][:, 2].copy())]
    hargs = (u, v, s['th'], s['arc'][:, 1].copy(), s['arc'][:, 2].copy())
    tau = numpy.ones((1, NZ, ncell))
    dtau = torch.from_numpy(tau).to('cuda')
    n0 = _lib.launch_count()
    for bad in ([0, 0, 5], [5, 2], [0, NZ + 1], [-1, 3]):
        with pytest.raises(_lib.NemofluxGpuError) as e:
            p.fluxTracer(*args, dtau, layers=bad)
        assert e.value.code == NFX_E_INVALID and 'layers' in str(e.value)
        with pytest.raises(_lib.NemofluxGpuError):
            p.fluxTracer(*hargs, tau, layers=bad, chunk_steps=1)
    assert _lib.launch_count() == n0
    with pytest.raises(TypeError):
        p.fluxTracer(*args, dtau.float())                                     # dtype of the tracer
    with pytest.raises(ValueError):
        p.fluxTracer(*args, dtau[:, :-1])                                     # levels
    with pytest.raises(ValueError):
        p.fluxTracer(*args, torch.cat([dtau, dtau]))                          # 2 steps, nt = 3
    with pytest.raises(ValueError):
        p.fluxTracer(*hargs, tau.astype(numpy.float32))                       # host: dtype
    with pytest.raises(ValueError):
        p.fluxTracer(*hargs, tau.astype('>f8'))                               # host: byte order
    # one level on padded planes (ld > ncell): a tracer of nt steps must step time by nz * ld as uo/vo do

    def padded():
        return torch.ones((nt, 1, ncell + 8), dtype=torch.float64, device='cuda')[:, :, :ncell]
    flat = torch.ones((nt, 1, ncell), dtype=torch.float64, device='cuda')
    one = [padded(), padded(), args[2][:1], args[3], args[4]]
    assert tuple(p.fluxTracer(*one, padded()).shape) == (nt, M)
    with pytest.raises(ValueError):
        p.fluxTracer(*one, flat)
    # NULL pointers, tr_nt outside {1, nt}, no output: refused, nothing launched
    lib = _lib.load()
    lev = numpy.array([0, NZ], numpy.int32)
    lp = lev.ctypes.data_as(ctypes.c_void_p)
    ptr = [ctypes.c_void_p(a.data_ptr()) for a in args]
    out = torch.zeros((nt, 1, M), dtype=torch.float64, device='cuda')
    n0 = _lib.launch_count()
    for tp, tr_nt, sp, secp in ((None, 1, out.data_ptr(), None), (dtau.data_ptr(), 2, out.data_ptr(), None),
                                (dtau.data_ptr(), 1, None, None), (dtau.data_ptr(), 1, out.data_ptr(), 'nolev')):
        levp = None if secp == 'nolev' else lp
        assert lib.nfx_flux_tracer(ctypes.byref(p._h), ptr[0], ptr[1], None, None, _lib.NFX_F64, 0, ptr[2], ptr[3],
                                   ptr[4], nt, NZ, ncell, tp, tr_nt, float('nan'), 0.0, 1, levp, 0, float('nan'), sp,
                                   None, None) == NFX_E_INVALID
    assert lib.nfx_flux_tracer_host(ctypes.byref(p._h), u.ctypes.data, v.ctypes.data, None, None, _lib.NFX_F64, 0, 0,
                                    hargs[2].ctypes.data, hargs[3].ctypes.data, hargs[4].ctypes.data, nt, NZ,
                                    tau.ctypes.data, 1, float('nan'), 0.0, 1, lp, 0, float('nan'), 0, None,
                                    None) == NFX_E_INVALID
    assert _lib.launch_count() == n0
    g2 = gpu.Grid()
    g2.setPoints(s['P'])
    p2 = gpu.PolylineIntegral()
    p2.build(g2)
    p2.computeWeights(s['transects'])
    n0 = _lib.launch_count()
    with pytest.raises(_lib.NemofluxGpuError) as e:
        p2.fluxTracer(*args, dtau)
    assert e.value.code == NFX_E_INVALID and 'cgrid' in str(e.value)
    with pytest.raises(_lib.NemofluxGpuError):
        p2.fluxTracer(*hargs, tau)
    assert _lib.launch_count() == n0
    # no step, no transect, and a transect that crosses no cell (outside the grid)
    assert tuple(p.fluxTracer(*(a[:0] for a in args[:2]), *args[2:], dtau).shape) == (0, M)
    assert p.fluxTracer(u[:0], v[:0], *hargs[2:], tau, section=True).shape == (0, NZ, p.getNumberOfSubsegments())
    assert _lib.launch_count() == n0
    _, p0 = _handle(gpu, s['P'], ny, nx, [])
    assert tuple(p0.fluxTracer(*args, dtau, layers=LAYERS).shape) == (nt, len(LAYERS) - 1, 0)
    assert p0.fluxTracer(*hargs, tau, section=True).shape == (nt, NZ, 0)
    lines = [s['transects'][0], tr([(0., 100.), (10., 120.)]), s['transects'][1]]
    _, pe = _handle(gpu, s['P'], ny, nx, lines)
    offs = pe.getSubsegments()['offsets']
    assert offs[2] == offs[1] and offs[1] > 0 and offs[3] > offs[2]
    got = _np(pe.fluxTracer(*args, dtau * 3.0))
    assert (got[:, 1] == 0).all()
    _, p1 = _handle(gpu, s['P'], ny, nx, [lines[0], lines[2]])
    _same(got[:, [0, 2]], p1.fluxTracer(*args, dtau * 3.0))
    _same(pe.fluxTracer(*hargs, tau * 3.0), got)


# blocks of cells [j0, j1) x [i0, i1) (i modulo nx) whose node-to-node loops cross only the cells on their boundary:
# one inside the grid, one against column 0 (its west faces are the x-periodic eU[c + nx - 1]), one across the x-wrap
# and a larger one
LOOP_BLOCKS = [(60, 63, 100, 104), (50, 53, 0, 3), (40, 43, 318, 322), (30, 36, 300, 310)]


def _node_loop(P, nx, j0, j1, i0, i1):
    """the closed loop through the cell corners around the block, counterclockwise in index space, one vertex per node
    (node (j, i): the south-west corner of cell j * nx + i mod nx), longitudes continuous along the loop"""
    node = [(j0, i) for i in range(i0, i1 + 1)] + [(j, i1) for j in range(j0 + 1, j1 + 1)] + \
        [(j1, i) for i in range(i1 - 1, i0 - 1, -1)] + [(j, i0) for j in range(j1 - 1, j0 - 1, -1)]
    pts = numpy.array([P[j * nx + i % nx, 0, :2] for j, i in node])
    pts[:, 0] = pts[0, 0] + (pts[:, 0] - pts[0, 0] + 180.) % 360. - 180.
    return tr(pts)


def _face_fluxes(nx, ny, u, v, tau, th, arc1, arc2, layers, tfill, fill, ref=0.0):
    """per layer the centred tracer flux through every east face eU[c] (c -> east(c)) and north face eV[c] (c ->
    north(c), none in the top row), positive eastward / northward: sum_k (dz_k u_k) q_k times the face's arc, q the face
    rule on the two T cells beside the face -> (FE, FN, |FE|, |FN|), each (nt, nlayers, ncell)"""
    ncell = nx * ny
    c = numpy.arange(ncell)
    east = numpy.where(c % nx + 1 < nx, c + 1, c + 1 - nx)
    north = numpy.where(c + nx < ncell, c + nx, c)
    dt = u.dtype.type

    def clean(x):
        return numpy.where(numpy.isnan(x) | (x == dt(fill)), 0.0, x.astype(numpy.float64))

    def face(ta, tb, has_b):
        pa = ~(numpy.isnan(ta) | (ta == dt(tfill)))
        pb = ~(numpy.isnan(tb) | (tb == dt(tfill))) & has_b
        fa, fb = ta.astype(numpy.float64), tb.astype(numpy.float64)
        with numpy.errstate(invalid='ignore', over='ignore'):
            return numpy.where(pa & pb, 0.5 * (fa + fb) - ref,
                               numpy.where(pa, fa - ref, numpy.where(pb, fb - ref, 0.0)))
    nt, nl = u.shape[0], len(layers) - 1
    out = [numpy.zeros((nt, nl, ncell)) for _ in range(4)]
    for li in range(nl):
        for k in range(layers[li], layers[li + 1]):
            t = tau[:, k] if tau.shape[0] == nt else numpy.broadcast_to(tau[:, k], (nt, ncell))
            fe = th[k] * clean(u[:, k]) * face(t, t[:, east], numpy.ones(ncell, bool)) * arc1
            fn = th[k] * clean(v[:, k]) * face(t, t[:, north], c + nx < ncell) * arc2
            for o, x in zip(out, (fe, fn, numpy.abs(fe), numpy.abs(fn))):
                o[:, li] += x
    return out


def _divergence(nx, block, FE, FN, AE, AN):
    """the net outward flux of the block's cells: east minus west plus north minus south, and its sum of |terms|"""
    j0, j1, i0, i1 = block
    cells = numpy.array([j * nx + i % nx for j in range(j0, j1) for i in range(i0, i1)])
    west = cells - cells % nx + (cells % nx - 1) % nx
    south = cells - nx
    div = (FE[..., cells] - FE[..., west] + FN[..., cells] - FN[..., south]).sum(-1)
    bar = (AE[..., cells] + AE[..., west] + AN[..., cells] + AN[..., south]).sum(-1)
    return div, bar


@pytest.mark.parametrize('dtype', [numpy.float64, numpy.float32])
def test_closed_loops_return_the_enclosed_divergence(gpu, small, dtype):
    """a closed node-to-node loop around a block of cells returns the net centred tracer flux out of those cells --
    numpy's east-minus-west plus north-minus-south of the face fluxes of the enclosed cells, built from the grid alone
    (no K1 weights) -- within 1e-12 * sum |terms|, for the [0, nz] series and per layer, with ref 0 and ref 2.5.  The
    loops run along grid lines, so K1 shares every crossing between the two cells beside it (duplicity coefficients
    below 1); the face value is the same from both.  The volume series of the same loops is the divergence with q = 1."""
    import torch
    s = small
    nx, ny, nt = s['nx'], s['ny'], s['nt']
    ncell = nx * ny
    u, v = _fields(s, dtype)
    loops = [_node_loop(s['P'], nx, *b) for b in LOOP_BLOCKS]
    _, p = _handle(gpu, s['P'], ny, nx, loops)
    sub = p.getSubsegments()
    for m, (j0, j1, i0, i1) in enumerate(LOOP_BLOCKS):
        a, b = sub['offsets'][m], sub['offsets'][m + 1]
        J, I = sub['cell'][a:b] // nx, sub['cell'][a:b] % nx
        # the loop crosses only the cells on either side of the block's boundary, and shares crossings between them
        assert b > a and ((J >= j0 - 1) & (J <= j1) & ((I - (i0 - 1)) % nx <= i1 - i0 + 1)).all(), m
        assert (sub['coeff'][a:b] < 1).any(), m
    a1h, a2h = s['arc'][:, 1].copy(), s['arc'][:, 2].copy()
    uh, vh = u.reshape(nt, NZ, ncell), v.reshape(nt, NZ, ncell)
    dev = lambda x: torch.from_numpy(numpy.ascontiguousarray(x)).to('cuda')   # noqa: E731
    args = [dev(uh), dev(vh), dev(s['th']), dev(a1h), dev(a2h)]
    tau = _tracer(s, dtype, 1e20)
    for L in ([0, NZ], LAYERS):
        for ref in (0.0, 2.5):
            FE, FN, AE, AN = _face_fluxes(nx, ny, uh, vh, tau, s['th'], a1h, a2h, L, 1e20, -7.0, ref)
            got = _np(p.fluxTracer(*args, dev(tau), tfill=1e20, ref=ref, layers=L, fill=-7.0))
            for m, block in enumerate(LOOP_BLOCKS):
                want, bar = _divergence(nx, block, FE, FN, AE, AN)
                assert (bar > 0).all()
                assert (numpy.abs(got[:, :, m] - want) <= 1e-12 * bar).all(), (L, ref, block, got[:, :, m], want)
    FE, FN, AE, AN = _face_fluxes(nx, ny, uh, vh, numpy.ones((1, NZ, ncell), dtype), s['th'], a1h, a2h, [0, NZ],
                                  1e20, -7.0)
    vol = _np(p.fluxSeries(*args, fill=-7.0))
    for m, block in enumerate(LOOP_BLOCKS):
        want, bar = _divergence(nx, block, FE, FN, AE, AN)
        assert (numpy.abs(vol[:, m] - want[:, 0]) <= 1e-12 * bar[:, 0]).all(), block


def test_field_and_fluxplot_tracer(gpu, oracle, tmp_path, capsys):
    """Field.fluxTracer on classic files (big-endian; the tracer from the T file, f32 next to f64 uo/vo, and
    time-invariant f64 from another file) and on deflated NetCDF-4 uo/vo (device decode): PolylineIntegral.fluxTracer of
    the same data, bit for bit; fluxplot --tracer prints and writes one column per transect (per (transect, layer) with
    --layers), and --timeMean averages them"""
    import h5build
    from helpers import SF_C2
    from nemoflux_b200 import fluxplot
    from nemoflux_b200.field import Field
    nt, nz = 4, 8
    T, U, V, S, thetao, so = _files(tmp_path, nt, nz)
    lines = [tr([(-100, -70), (100, -70), (0, 70)]), tr([(-150, -20), (-20, 35), (60, -40)])]

    def direct(f, c, tfill, **kw):
        u, v, fill = f._uv_slabs(0, f.nt)
        c = c.astype(u.dtype).reshape(-1, nz, 36, 72)
        return f.pli.fluxTracer(u, v, f.thickness, f.arcLengths[:, 1].copy(), f.arcLengths[:, 2].copy(), c,
                                tfill=tfill, sverdrup=f.sverdrup, fill=fill, **kw)
    f = Field(T, U, V, lines, sverdrup=True, verbose=False)
    t_fill = float(numpy.float32(1e20))
    ref_t = direct(f, thetao, t_fill)
    assert numpy.abs(ref_t).max() > 0
    for cs in (1, 0):
        _same(f.fluxTracer('thetao', chunk_steps=cs), ref_t, ('thetao', cs))
    _same(f.fluxTracer('thetao', layers=[0, 3, nz], section=True, chunk_steps=3),
          direct(f, thetao, t_fill, layers=[0, 3, nz], section=True), 'section')
    ref_s = direct(f, so, float('nan'), ref=34.8, layers=[0, 2, nz])
    _same(f.fluxTracer('so', file=S, ref=34.8, layers=[0, 2, nz], chunk_steps=3), ref_s, 'so')
    d = oracle.DataGen(nx=72, ny=36, nz=nz, nt=nt, deltaDeg=(20., 30.))
    u, v = d.uv(SF_C2)
    U4, V4 = str(tmp_path / 'U4.nc'), str(tmp_path / 'V4.nc')
    for fname, vname, a in ((U4, 'uo', u), (V4, 'vo', v)):
        h5build.write(fname, {vname: dict(data=a, chunks=(1, 2, 36, 72), deflate=True, shuffle=True),
                              'time_counter': dict(data=numpy.arange(float(nt)), chunks=(1,))})
    f4 = Field(T, U4, V4, lines, verbose=False)
    got = f4.fluxTracer('thetao', chunk_steps=2)
    assert f4.last_ingest['path'] == 'device decode'
    _same(got, direct(f4, thetao, t_fill), 'device decode')
    _same(f4.fluxTracer('thetao', chunk_steps=2, device_decode=False), got, 'host zlib')
    _same(f4.fluxTracer('so', file=S, chunk_steps=2), direct(f4, so, float('nan')), 'device decode, steady')
    # fluxplot --tracer
    pts = '[(-100,-70),(100,-70),(0,70)],[(-150,-20),(-20,35),(60,-40)]'
    csv = str(tmp_path / 'tracer.csv')
    series = fluxplot.main(['-t', T, '-u', U, '-v', V, '-l', pts, '-s', '--tracer', 'thetao', '-o', csv])
    out = capsys.readouterr().out
    _same(series, ref_t, 'fluxplot')
    with open(csv, encoding='utf-8') as fh:
        rows = [r.rstrip('\n').split(',') for r in fh]
    assert rows[0] == ['time', 'line0[thetao]', 'line1[thetao]'] and len(rows) == nt + 1
    assert 'line0[thetao]' in out
    _same(numpy.array([[float(x) for x in r[1:]] for r in rows[1:]]), ref_t, 'csv')
    series = fluxplot.main(['-t', T, '-u', U, '-v', V, '-l', pts, '-s', '--tracer', f'so:{S}', '--tracerRef=34.8',
                            '--layers', f'0,2,{nz}', '--timeMean', '2', '-o', csv])
    capsys.readouterr()
    _same(series, fluxplot.windowMeans(ref_s, [0, 2, 4]), 'layers, time mean')
    with open(csv, encoding='utf-8') as fh:
        heads = fh.readline().rstrip('\n').split(',')
    assert len(heads) == 5 and all(h.split('[')[1].startswith('so ') for h in heads[1:])
