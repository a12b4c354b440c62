"""The time-mean transport section (fluxSection(windows=)): per window of time steps, layer and cell crossing, the
per-step section summed in ascending step order from +0 and divided by the window's length -- bit for bit against a
numpy loop over fluxSection's per-step output on every storage type, layering, metric, plane layout, window list and
entry point; steps outside the windows are not read; chunking and split calls do not change the bits; the sums against
the layered series and the analytic answer; the errors; the Field / fluxplot --timeMean path."""
import numpy
import pytest

from helpers import README_C2, SF_C2, random_transects, tr

pytestmark = pytest.mark.gpu

NZ = 75
NT = 7
NFX_E_INVALID = 1          # include/nemoflux_gpu.h
ONE, RAGGED, PER_LEVEL, PARTIAL = [0, NZ], [0, 1, 7, 23, 75], list(range(NZ + 1)), [10, 40]
LAYERINGS = {'one': ONE, 'ragged': RAGGED, 'per-level': PER_LEVEL, 'partial': PARTIAL}
# the whole record, ragged, one step each, and lists that leave steps out at either end
WINDOWS = {'all': [0, NT], 'ragged': [0, 1, 4, NT], 'steps': list(range(NT + 1)), 'inner': [2, 5],
           'late': [1, 2, 6]}


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
    num = ~numpy.isnan(a)                      # -0 and +0 apart (NaN payloads and signs are not part of the contract)
    assert numpy.array_equal(numpy.signbit(a[num]), numpy.signbit(b[num])), what


def _mean_ref(sec, bounds):
    """the definition in numpy: a sequential sum over the steps of every window from +0, then one division"""
    sec = _np(sec)
    out = numpy.empty((len(bounds) - 1,) + sec.shape[1:])
    with numpy.errstate(all='ignore'):
        for w in range(len(bounds) - 1):
            acc = numpy.zeros(sec.shape[1:])
            for t in range(bounds[w], bounds[w + 1]):
                acc = acc + sec[t]
            out[w] = acc / float(bounds[w + 1] - bounds[w])
    return out


def _center(P, c):
    lon = P[c, :, 0] - 360. * numpy.round((P[c, :, 0] - P[c, 0, 0]) / 360.)
    return float(lon.mean()), float(P[c, :, 1].mean())


@pytest.fixture(scope='module')
def data(oracle):
    """NT steps of 19 200 cells and 75 levels: NaN land, denormals, the fill value -7 and -0 columns; transects that
    start in row 0 (south edges never written) and column 0 (x-periodic west edges)"""
    nx, ny = 160, 120
    g = oracle.DataGen(nx=nx, ny=ny, nz=NZ, nt=NT, deltaDeg=(20., 30.))
    P, arc = g.points(), oracle.arc_lengths(g.points())
    transects = random_transects(numpy.random.default_rng(3), 5, max_pts=4) + [tr(README_C2)]
    for a, b in (((0, nx // 3), (4, nx // 3 + 5)), ((ny // 2, 0), (ny // 2 + 3, 4))):
        pa = _center(P, a[0] * nx + a[1])
        pb = _center(P, b[0] * nx + b[1])
        pb = (pb[0] - 360. * round((pb[0] - pa[0]) / 360.), pb[1])
        transects.append(tr([pa, pb]))
    u, v = g.uv(SF_C2)
    u[:, :, 10:14, 20:40] = numpy.nan
    return dict(nx=nx, ny=ny, g=g, P=P, arc=arc, transects=transects, u=u, v=v, th=numpy.linspace(1.0, 40.0, NZ))


def _fields(s, dtype):
    u, v = s['u'].astype(dtype), s['v'].astype(dtype)
    tiny = numpy.finfo(dtype).tiny
    u[:, ::2, 30:33, 5:60] = tiny / 8
    v[:, 1::3, 40:42, 10:70] = -tiny / 16
    v[:, :, 50:52, 100:120] = -7.0
    u[:, :, 60:70, 60:80] = -0.0
    v[:, :, 60:70, 60:80] = -0.0
    return u, v


def _args(s, u, v, d='cuda'):
    import torch
    return [torch.from_numpy(numpy.ascontiguousarray(x)).to(d)
            for x in (u, v, s['th'], s['arc'][:, 1].copy(), s['arc'][:, 2].copy())]


@pytest.mark.parametrize('dtype', [numpy.float64, numpy.float32])
@pytest.mark.parametrize('sverdrup', [False, True])
@pytest.mark.parametrize('padded', [False, True])
def test_mean_bit_contract(gpu, data, dtype, sverdrup, padded):
    """every layering and window list, thickness and e3 (1 and nt steps): the numpy loop over the per-step section,
    bit for bit"""
    import torch
    s = data
    nx, ny = s['nx'], s['ny']
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
        for wname, W in WINDOWS.items():
            m = p.fluxSection(ud, vd, th, a1, a2, layers=L, windows=W, **kw)
            assert m.shape == (len(W) - 1, len(L) - 1, nsub) and m.dtype == torch.float64 and m.is_cuda
            _same(m, _mean_ref(sec, W), ('thickness', name, wname))
    _same(p.fluxSection(ud, vd, th, a1, a2, windows=[0, 3, NT], **kw),
          p.fluxSection(ud, vd, th, a1, a2, layers=PER_LEVEL, windows=[0, 3, NT], **kw))
    rng = numpy.random.default_rng(9)
    for e3_nt in (1, NT):
        e3h = rng.uniform(0.5, 30., (e3_nt, NZ, ny, nx)).astype(dtype)
        e3 = dict(e3u=dev(e3h), e3v=dev(e3h[..., ::-1]))
        for name, L in (('one', ONE), ('ragged', RAGGED), ('partial', PARTIAL)):
            sec = p.fluxSection(ud, vd, None, a1, a2, layers=L, **e3, **kw)
            for wname in ('ragged', 'inner'):
                W = WINDOWS[wname]
                _same(p.fluxSection(ud, vd, None, a1, a2, layers=L, windows=W, **e3, **kw), _mean_ref(sec, W),
                      ('e3', e3_nt, name, wname))


def test_steps_outside_the_windows_are_not_read(gpu, data):
    """+inf in every value of the steps before b0 and from bK on: the means stay finite and identical"""
    s = data
    u, v = _fields(s, numpy.float64)
    u, v = numpy.nan_to_num(u, nan=0.0), numpy.nan_to_num(v, nan=0.0)
    _, p = _handle(gpu, s['P'], s['ny'], s['nx'], s['transects'])
    W = [2, 4, 5]
    ui, vi = u.copy(), v.copy()
    for a in (ui, vi):
        a[:W[0]] = numpy.inf
        a[W[-1]:] = numpy.inf
    ref = _np(p.fluxSection(*_args(s, u, v), layers=RAGGED, windows=W))
    assert numpy.isfinite(ref).all()
    _same(p.fluxSection(*_args(s, ui, vi), layers=RAGGED, windows=W), ref, 'device')
    a = _args(s, ui, vi, 'cpu')
    for cs in (1, 2, 0):
        _same(p.fluxSection(ui, vi, s['th'], a[3].numpy(), a[4].numpy(), layers=RAGGED, windows=W, chunk_steps=cs),
              ref, ('host', cs))


@pytest.mark.parametrize('dtype', [numpy.float64, numpy.float32])
def test_infinity_inside_a_window(gpu, data, dtype):
    """+-inf on level 30 of 4 columns at step 3: the means are those of the numpy loop, bit for bit"""
    s = data
    u, v = _fields(s, dtype)
    _, p = _handle(gpu, s['P'], s['ny'], s['nx'], s['transects'])
    c0 = int(p.getSubsegments()['cell'][3]) // 4 * 4
    for val in (numpy.inf, -numpy.inf):
        ui, vi = u.copy(), v.copy()
        for a in (ui, vi):
            a.reshape(NT, NZ, -1)[3, 30, c0:c0 + 4] = val
        args = _args(s, ui, vi)
        sec = p.fluxSection(*args, layers=RAGGED, fill=-7.0)
        assert not numpy.isfinite(_np(sec)).all()
        for W in (WINDOWS['ragged'], WINDOWS['all'], WINDOWS['steps']):
            _same(p.fluxSection(*args, layers=RAGGED, fill=-7.0, windows=W), _mean_ref(sec, W), (val, W))


@pytest.mark.parametrize('dtype', [numpy.float64, numpy.float32])
@pytest.mark.parametrize('big_endian', [False, True])
def test_chunks_and_split_calls(gpu, data, dtype, big_endian):
    """host buffers with chunk_steps 1, 2, 3, nt and automatic (windows straddling the chunks), native and big-endian,
    e3 on the host (1 and nt steps) and on the device: the device path bit for bit; two device calls with
    continue_first equal one call"""
    import torch
    s = data
    nx, ny = s['nx'], s['ny']
    u, v = _fields(s, dtype)
    _, p = _handle(gpu, s['P'], ny, nx, s['transects'])
    d = 'cuda'
    a1, a2 = s['arc'][:, 1].copy(), s['arc'][:, 2].copy()
    dargs = _args(s, u, v)
    hu, hv = (u.astype(u.dtype.newbyteorder('>')), v.astype(v.dtype.newbyteorder('>'))) if big_endian else (u, v)
    for L in (ONE, RAGGED, PER_LEVEL):
        for W in (WINDOWS['ragged'], WINDOWS['late'], [0, 5, NT]):
            ref = _np(p.fluxSection(*dargs, layers=L, fill=-7.0, windows=W))
            for cs in (1, 2, 3, NT, 0):
                out = p.fluxSection(hu, hv, s['th'], a1, a2, layers=L, fill=-7.0, chunk_steps=cs, windows=W)
                assert isinstance(out, numpy.ndarray)
                _same(out, ref, (L, W, cs))
    rng = numpy.random.default_rng(5)
    W = [0, 3, 5, NT]
    for e3_nt in (1, NT):
        e3u = rng.uniform(0.5, 30., (e3_nt, NZ, ny * nx)).astype(dtype)
        e3v = rng.uniform(0.5, 30., (e3_nt, NZ, ny * nx)).astype(dtype)
        de3 = dict(e3u=torch.from_numpy(e3u).to(d), e3v=torch.from_numpy(e3v).to(d))
        for Wx in (W, [1, 4]):
            ref = _np(p.fluxSection(*dargs[:2], None, *dargs[3:], layers=RAGGED, fill=-7.0, windows=Wx, **de3))
            he3 = (e3u.astype(hu.dtype), e3v.astype(hu.dtype))
            for cs in (2, 0):
                _same(p.fluxSection(hu, hv, None, a1, a2, layers=RAGGED, fill=-7.0, chunk_steps=cs, windows=Wx,
                                    e3u=he3[0], e3v=he3[1]), ref, ('host e3', e3_nt, cs, Wx))
                if e3_nt == 1:
                    _same(p.fluxSection(hu, hv, None, a1, a2, layers=RAGGED, fill=-7.0, chunk_steps=cs, windows=Wx,
                                        **de3), ref, ('device e3', cs, Wx))
    # window [3, 5) split over two device calls (steps [0, 4) and [4, 7)), and over two host calls
    one = p.sectionWindowSums(*dargs, W, layers=RAGGED, fill=-7.0)
    part = torch.full((3, len(RAGGED) - 1, p.getNumberOfSubsegments()), 99.0, dtype=torch.float64, device=d)
    p.sectionWindowSums(dargs[0][:4], dargs[1][:4], *dargs[2:], [0, 3, 4], layers=RAGGED, fill=-7.0, sums=part[:2])
    p.sectionWindowSums(dargs[0][4:], dargs[1][4:], *dargs[2:], [0, 1, 3], layers=RAGGED, fill=-7.0, sums=part[1:],
                        continue_first=True)
    _same(part, one, 'device split')
    hpart = numpy.full(tuple(part.shape), 99.0)
    p.sectionWindowSums(hu[:4], hv[:4], s['th'], a1, a2, [0, 3, 4], layers=RAGGED, fill=-7.0, sums=hpart[:2])
    p.sectionWindowSums(hu[4:], hv[4:], s['th'], a1, a2, [0, 1, 3], layers=RAGGED, fill=-7.0, sums=hpart[1:],
                        continue_first=True, chunk_steps=1)
    _same(hpart, one, 'host split')


def _by_transect(p, x):
    offs = p.getSubsegments()['offsets']
    return numpy.stack([x[..., a:b].sum(-1) for a, b in zip(offs[:-1], offs[1:])], -1)


def test_means_sum_to_the_windowed_layered_series(gpu, data):
    """a transect's crossings add up to the window mean of its layered series within 1e-12 * the window mean of
    sum |w f| (the edge fluxes of fluxSeries(eflux=))"""
    import torch
    s = data
    nx, ny = s['nx'], s['ny']
    u, v = _fields(s, numpy.float64)
    _, p = _handle(gpu, s['P'], ny, nx, s['transects'])
    args = _args(s, u, v)
    ncell = nx * ny
    sub = p.getSubsegments()
    j, i = sub['cell'] // nx, sub['cell'] % nx
    idx = numpy.stack([numpy.where(j >= 1, ncell + sub['cell'] - nx, -1), sub['cell'], ncell + sub['cell'],
                       numpy.where(i >= 1, sub['cell'] - 1, sub['cell'] + nx - 1)], 1)
    for L in (ONE, RAGGED):
        ef = torch.zeros((NT, len(L) - 1, 2 * ncell), dtype=torch.float64, device='cuda')
        ser = _np(p.fluxSeries(*args, layers=L, fill=-7.0, order='list', eflux=ef))
        ef = ef.cpu().numpy()
        Eg = numpy.where(idx >= 0, ef[..., numpy.maximum(idx, 0)], 0.0)
        bar = _by_transect(p, numpy.abs(sub['w'] * Eg).sum(-1))
        for W in (WINDOWS['ragged'], WINDOWS['all'], WINDOWS['inner']):
            m = _by_transect(p, _np(p.fluxSection(*args, layers=L, fill=-7.0, windows=W)))
            assert (bar > 0).any()
            ok = numpy.abs(m - _mean_ref(ser, W)) <= 1e-12 * _mean_ref(bar, W) + 1e-300
            assert ok.all(), (L, W)


def test_mean_analytic_per_crossing(gpu):
    """synthetic stream function with coefficients proportional to (t + 1): every crossing's mean is the per-step
    analytic answer of step 0 times the window mean of (t + 1)"""
    import torch
    from nemoflux_b200 import synth
    syn = synth.make('tiny', deltaDeg=(0., 0.), land=False)
    d = torch.device('cuda', 0)
    _, p = _handle(gpu, syn.points, syn.ny, syn.nx, syn.transects)
    nt = 5
    u, v = syn.fill_device(0, nt, d)
    th, a1, a2 = (torch.from_numpy(x).to(d) for x in (syn.thickness, syn.arc1, syn.arc2))
    W = [0, 2, 5]
    m = _np(p.fluxSection(u, v, th, a1, a2, windows=W))
    sub = p.getSubsegments()
    j, i = sub['cell'] // syn.nx, sub['cell'] % syn.nx

    def bilinear(g, xi):
        s_, t_ = xi[:, 0], xi[:, 1]
        return ((1 - s_) * (1 - t_) * g[j, i] + s_ * (1 - t_) * g[j, i + 1] + s_ * t_ * g[j + 1, i + 1] +
                (1 - s_) * t_ * g[j + 1, i])
    d1 = bilinear(syn.g1, sub['xib']) - bilinear(syn.g1, sub['xia'])
    d2 = bilinear(syn.g2, sub['xib']) - bilinear(syn.g2, sub['xia'])
    inner = (j >= 1) & (i >= 1)
    assert inner.sum() > 100
    c1, c2 = syn.coeffs(0)
    ex0 = sub['coeff'][None] * syn.thickness[:, None] * (c1[:, None] * d1[None] + c2[:, None] * d2[None])
    scale = numpy.abs(ex0).max() * nt
    for w in range(len(W) - 1):
        f = numpy.mean(numpy.arange(W[w], W[w + 1]) + 1.0)
        assert numpy.abs(m[w][:, inner] - f * ex0[:, inner]).max() <= 1e-11 * scale, w


def test_mean_errors_and_edge_cases(gpu, data):
    import torch
    from nemoflux_b200 import _lib
    s = data
    nx, ny = s['nx'], s['ny']
    _, p = _handle(gpu, s['P'], ny, nx, s['transects'])
    d = 'cuda'
    u, v = _fields(s, numpy.float64)
    args = _args(s, u, v)
    hargs = (u, v, s['th'], s['arc'][:, 1].copy(), s['arc'][:, 2].copy())
    nsub = p.getNumberOfSubsegments()
    n0 = _lib.launch_count()
    for bad in ([3, 3], [0, 4, 2], [-1, 3], [0, NT + 1], [5, 1]):
        out = torch.full((len(bad) - 1, len(RAGGED) - 1, nsub), 42.0, dtype=torch.float64, device=d)
        with pytest.raises(_lib.NemofluxGpuError) as e:
            p.fluxSection(*args, layers=RAGGED, windows=bad, out=out)
        assert e.value.code == NFX_E_INVALID and 'windows' in str(e.value)
        assert (out == 42.0).all()
        with pytest.raises(_lib.NemofluxGpuError) as e:
            p.fluxSection(*hargs, layers=RAGGED, windows=bad, chunk_steps=1)
        assert e.value.code == NFX_E_INVALID and 'windows' in str(e.value)
    # a bad layering with good windows, and nt == 0 (no window can hold a step)
    with pytest.raises(_lib.NemofluxGpuError) as e:
        p.fluxSection(*args, layers=[0, 5, 5], windows=[0, 2])
    assert e.value.code == NFX_E_INVALID and 'layers' in str(e.value)
    with pytest.raises(_lib.NemofluxGpuError) as e:
        p.fluxSection(args[0][:0], args[1][:0], *args[2:], layers=RAGGED, windows=[0, 1])
    assert e.value.code == NFX_E_INVALID
    with pytest.raises(_lib.NemofluxGpuError) as e:
        p.fluxSection(u[:0], v[:0], *hargs[2:], layers=RAGGED, windows=[0, 1])
    assert e.value.code == NFX_E_INVALID
    assert _lib.launch_count() == n0
    for bad in ([3], [[0, 1]], [0, 2.5]):
        with pytest.raises(ValueError):
            p.fluxSection(*args, windows=bad)
    out = torch.full((2, len(RAGGED) - 1, nsub), 42.0, dtype=torch.float64, device=d)
    with pytest.raises(ValueError):
        p.fluxSection(*args, layers=RAGGED, windows=[0, 2, 4, 6], out=out)      # wrong shape
    with pytest.raises(ValueError):
        p.fluxSection(*args, layers=RAGGED, windows=[0, 2, 4], out=out.view(2, nsub, -1))
    with pytest.raises(TypeError):
        p.fluxSection(*args, layers=RAGGED, windows=[0, 2, 4], out=out.float())
    with pytest.raises(ValueError):
        p.sectionWindowSums(*hargs, [0, 2, 4], layers=RAGGED, sums=numpy.zeros((2, 3, nsub)))
    assert (out == 42.0).all() and _lib.launch_count() == n0
    # out= is filled with the means and returned
    m = p.fluxSection(*args, layers=RAGGED, windows=[0, 2, 4], out=out)
    assert m.data_ptr() == out.data_ptr()
    _same(out, _mean_ref(p.fluxSection(*args, layers=RAGGED), [0, 2, 4]))
    # no crossing: an empty result, nothing launched
    _, p0 = _handle(gpu, s['P'], ny, nx, [])
    n0 = _lib.launch_count()
    assert tuple(p0.fluxSection(*args, layers=RAGGED, windows=[0, 3]).shape) == (1, len(RAGGED) - 1, 0)
    assert p0.fluxSection(*hargs, layers=RAGGED, windows=[0, 3]).shape == (1, len(RAGGED) - 1, 0)
    assert _lib.launch_count() == n0
    with pytest.raises(_lib.NemofluxGpuError):
        p0.fluxSection(*args, layers=RAGGED, windows=[0, NT + 3])
    # two calls, identical bits
    _same(p.fluxSection(*args, windows=[0, 2, NT]), p.fluxSection(*args, windows=[0, 2, NT]))
    assert p.seriesStatus() == 0


def _files(tmp_path, *args):
    from nemoflux_b200 import datagen
    prefix = str(tmp_path) + '/'
    datagen.cli(list(args) + [f'--prefix={prefix}'])
    return prefix + 'T.nc', prefix + 'U.nc', prefix + 'V.nc'


def test_field_and_fluxplot_time_mean(gpu, oracle, tmp_path, capsys):
    """Field.fluxSection(windows=) on classic (big-endian) and deflated NetCDF-4 (device-decoded) files, with read blocks
    that split windows: PolylineIntegral.fluxSection(windows=) of the whole record, bit for bit; fluxplot --timeMean 2
    --section writes the window means with time_bnds and cell_methods"""
    import h5build
    from nemoflux_b200 import fluxplot, ncio
    from nemoflux_b200.field import Field
    nz, nt = 8, 5
    T, U, V = _files(tmp_path, f'--streamFunction={SF_C2}', '--nx=72', '--ny=36', f'--nz={nz}', f'--nt={nt}',
                     '--deltaDeg=20,30')
    lines = [tr([(-100, -70), (100, -70), (0, 70)]), tr([(-150, -20), (-20, 35), (60, -40)])]

    def direct(f, L, W):
        u, v, fill = f._uv_slabs(0, f.nt)
        return f.pli.fluxSection(u, v, f.thickness, f.arcLengths[:, 1].copy(), f.arcLengths[:, 2].copy(),
                                 sverdrup=f.sverdrup, fill=fill, layers=L, windows=W)
    f = Field(T, U, V, lines, verbose=False)
    for L in (None, [0, 2, 5, 8]):
        for W in ([0, 3, 5], [1, 2, 4], [0, 5]):
            ref = direct(f, L, W)
            for cs in (1, 2, 0):
                _same(f.fluxSection(layers=L, windows=W, chunk_steps=cs), ref, ('classic', L, W, cs))
    with pytest.raises(ValueError):
        f.fluxSection(windows=[0, nt + 1])
    d = oracle.DataGen(nx=72, ny=36, nz=nz, nt=nt, deltaDeg=(20., 30.))
    u, v = d.uv(SF_C2)
    U4, V4 = str(tmp_path / 'U4.nc'), str(tmp_path / 'V4.nc')
    for fname, vname, a in ((U4, 'uo', u), (V4, 'vo', v)):
        h5build.write(fname, {vname: dict(data=a, chunks=(1, 2, 36, 72), deflate=True, shuffle=True),
                              'time_counter': dict(data=numpy.arange(float(nt)), chunks=(1,))})
    f4 = Field(T, U4, V4, lines, verbose=False)
    for W in ([0, 3, 5], [1, 2, 4]):
        ref = direct(f4, [0, 2, 5, 8], W)
        for cs in (2, 0):
            m = f4.fluxSection(layers=[0, 2, 5, 8], windows=W, chunk_steps=cs)
            assert f4.last_ingest['path'] == 'device decode'
            _same(m, ref, ('deflated', W, cs))
    # fluxplot --timeMean 2 --section
    pts = '[(-100,-70),(100,-70),(0,70)],[(-150,-20),(-20,35),(60,-40)]'
    path = str(tmp_path / 'mean.nc')
    series = fluxplot.main(['-t', T, '-u', U, '-v', V, '-l', pts, '-s', '--layers', '0,2,5,8', '--section', path,
                            '--timeMean', '2'])
    out = capsys.readouterr().out
    assert 'crossings written' in out and series.shape == (3, 3, 2)
    fs = Field(T, U, V, lines, sverdrup=True, verbose=False)
    W = [0, 2, 4, 5]
    _same(series, fluxplot.windowMeans(fs.fluxSeries(layers=[0, 2, 5, 8]), W))
    ref = fs.fluxSection(layers=[0, 2, 5, 8], windows=W)
    with ncio.open_dataset(path) as nc:
        _same(numpy.asarray(nc['transport'][:], numpy.float64), ref, 'file')
        assert getattr(nc['transport'], 'cell_methods', None) == 'time: mean' or \
            nc['transport'].attrs.get('cell_methods') == 'time: mean'
        assert tuple(nc['time_bnds'].shape) == (3, 2)
        assert nc['time'].shape == (3,)
    assert numpy.abs(_by_transect(fs.pli, ref) - series).max() <= 1e-12 * numpy.abs(series).max() * 100
