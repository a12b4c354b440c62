"""The layered flux series (fluxSeries(layers=)): layer i of the series is the plain series with the thickness (or
e3u/e3v) zeroed outside the levels [l_i, l_{i+1}), bit for bit on finite data, on every path -- fused or two launches,
sparse or dense, one or several panels, device or host buffers -- and the same numbers as the oracle and the analytic
answer.  The only intended difference from masking: an infinity outside the layer does not reach it."""
import numpy
import pytest

from helpers import README_C2, SF_C2, random_transects, tr

pytestmark = pytest.mark.gpu

NZ = 75
ONE, RAGGED, PER_LEVEL, PARTIAL = [0, NZ], [0, 1, 7, 23, 75], list(range(NZ + 1)), [10, 40]
LAYERINGS = {'one': ONE, 'ragged': RAGGED, 'per-level': PER_LEVEL, 'partial': PARTIAL}


@pytest.fixture(autouse=True)
def _reset_options():
    from nemoflux_b200 import _lib
    yield
    for opt, val in ((_lib.NFX_OPT_SPARSE_COLUMNS, 1), (_lib.NFX_OPT_RING_SLOT_MB, 0), (_lib.NFX_OPT_FAST_SERIES, 1),
                     (_lib.NFX_OPT_FUSED_ORDER, 3), (_lib.NFX_OPT_FUSED_K3_LAG, 0), (_lib.NFX_OPT_RING_MAX_MB, 0)):
        _lib.set_option(opt, val)


def _handle(gpu, points, ny, nx, transects):
    g = gpu.Grid()
    g.setPoints(points)
    g.setCGridShape(ny, nx)
    p = gpu.PolylineIntegral()
    p.build(g)
    p.computeWeights(transects)
    return g, p


def _mask(layers, i, nz=NZ):
    m = numpy.zeros(nz)
    m[layers[i]:layers[i + 1]] = 1.0
    return m


def _np(x):
    return x if isinstance(x, numpy.ndarray) else x.cpu().numpy()


def _same(a, b, what=''):
    a, b = _np(a), _np(b)
    assert a.shape == b.shape, (what, a.shape, b.shape)
    assert numpy.array_equal(a, b, equal_nan=True), (what, numpy.nanmax(numpy.abs(a - b)))


@pytest.fixture(scope='module')
def small(oracle):
    """76 800 cells (two panels with a 1 MB ring slot), 75 levels, NaN land, denormals and the fill value -7"""
    nx, ny, nt = 320, 240, 2
    g = oracle.DataGen(nx=nx, ny=ny, nz=NZ, nt=nt, deltaDeg=(20., 30.))
    P, arc = g.points(), oracle.arc_lengths(g.points())
    transects = random_transects(numpy.random.default_rng(3), 6, max_pts=4) + [tr(README_C2)]
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


def _run(p, u, v, th, a1, a2, layers=None, two_launch=False, e3=None, **kw):
    """one series call on the device path; two_launch: with an eflux buffer (returned too)"""
    import torch
    nt, ncell = u.shape[0], a1.numel()
    eflux = None
    if two_launch:
        shape = (nt, 2 * ncell) if layers is None else (nt, len(layers) - 1, 2 * ncell)
        eflux = torch.full(shape, 5.0, dtype=torch.float64, device=u.device)
    e3kw = {} if e3 is None else dict(e3u=e3[0], e3v=e3[1])
    s = p.fluxSeries(u, v, th, a1, a2, eflux=eflux, layers=layers, **e3kw, **kw)
    assert p.seriesStatus() == 0
    return _np(s), eflux


@pytest.mark.parametrize('dtype', [numpy.float64, numpy.float32])
@pytest.mark.parametrize('order', ['map', 'list'])
@pytest.mark.parametrize('sparse', [0, 2])
@pytest.mark.parametrize('two_launch', [False, True])
@pytest.mark.parametrize('slot_mb', [0, 1])
def test_layers_equal_masked_thickness(gpu, small, dtype, order, sparse, two_launch, slot_mb):
    """every layering, every layer: the masked-thickness series of the same path bit for bit; [0, nz] is the plain
    series; the layered edge fluxes are edgeFluxAssemble's with the masked thickness"""
    import torch
    from nemoflux_b200 import _lib
    _lib.set_option(_lib.NFX_OPT_SPARSE_COLUMNS, sparse)
    _lib.set_option(_lib.NFX_OPT_RING_SLOT_MB, slot_mb)
    s = small
    u, v = _fields(s, dtype)
    _, p = _handle(gpu, s['P'], s['ny'], s['nx'], s['transects'])
    d = 'cuda'
    ud, vd = torch.from_numpy(u).to(d), torch.from_numpy(v).to(d)
    a1, a2, th = (torch.from_numpy(x).to(d) for x in (s['arc'][:, 1].copy(), s['arc'][:, 2].copy(), s['th']))
    kw = dict(order=order, fill=-7.0, two_launch=two_launch)
    plain, _ = _run(p, ud, vd, th, a1, a2, **kw)
    path = _lib.get_option(_lib.NFX_OPT_LAST_SERIES_PATH)
    assert path == (0 if two_launch else 1) and numpy.isfinite(plain).all()
    for name, L in LAYERINGS.items():
        lay, ef = _run(p, ud, vd, th, a1, a2, layers=L, **kw)
        assert _lib.get_option(_lib.NFX_OPT_LAST_SERIES_PATH) == path
        assert lay.shape == (s['nt'], len(L) - 1, len(s['transects']))
        if name == 'one':
            _same(lay[:, 0], plain, name)
        for i in range(len(L) - 1):
            thm = th * torch.from_numpy(_mask(L, i)).to(d)
            ref, _ = _run(p, ud, vd, thm, a1, a2, **kw)
            _same(lay[:, i], ref, (name, i))
            if two_launch and i in (0, len(L) - 2):
                _same(ef[:, i], gpu.edgeFluxAssemble(ud, vd, thm, a1, a2, fill=-7.0), (name, 'eflux', i))


@pytest.mark.parametrize('dtype', [numpy.float64, numpy.float32])
def test_layers_padded_planes_and_scale_factors(gpu, small, dtype):
    """padded level planes (the widest loads), e3u/e3v time-invariant and time-varying: the mask goes onto e3"""
    import torch
    s = small
    nx, ny, nt = s['nx'], s['ny'], s['nt']
    ncell = nx * ny
    u, v = _fields(s, dtype)
    _, p = _handle(gpu, s['P'], ny, nx, s['transects'])
    d = 'cuda'
    tdt = torch.float64 if dtype == numpy.float64 else torch.float32
    pad = 4 if dtype == numpy.float64 else 8
    ld = (ncell + 1 + pad - 1) // pad * pad

    def dev(x):
        t = torch.full((x.shape[0], NZ, ld), 3.0, dtype=tdt, device=d)[:, :, :ncell]
        t.copy_(torch.from_numpy(numpy.ascontiguousarray(x).reshape(x.shape[0], NZ, ncell)))
        return t
    ud, vd = dev(u), dev(v)
    a1, a2, th = (torch.from_numpy(x).to(d) for x in (s['arc'][:, 1].copy(), s['arc'][:, 2].copy(), s['th']))
    rng = numpy.random.default_rng(9)
    for two_launch in (False, True):
        lay, _ = _run(p, ud, vd, th, a1, a2, layers=RAGGED, two_launch=two_launch)
        for i in range(len(RAGGED) - 1):
            _same(lay[:, i], _run(p, ud, vd, th * torch.from_numpy(_mask(RAGGED, i)).to(d), a1, a2,
                                  two_launch=two_launch)[0], ('thickness', two_launch, i))
        for e3_nt in (1, nt):
            e3h = rng.uniform(0.5, 30., (e3_nt, NZ, ny, nx)).astype(dtype)
            e3 = (dev(e3h), dev(e3h[..., ::-1]))
            for L in (ONE, RAGGED, PARTIAL):
                lay, ef = _run(p, ud, vd, None, a1, a2, layers=L, two_launch=two_launch, e3=e3)
                if L is ONE:
                    _same(lay[:, 0], _run(p, ud, vd, None, a1, a2, two_launch=two_launch, e3=e3)[0])
                for i in range(len(L) - 1):
                    m = torch.from_numpy(_mask(L, i).astype(dtype)).to(d)[None, :, None]
                    e3m = (dev((e3[0] * m).cpu().numpy()), dev((e3[1] * m).cpu().numpy()))
                    ref, _ = _run(p, ud, vd, None, a1, a2, two_launch=two_launch, e3=e3m)
                    _same(lay[:, i], ref, ('e3', two_launch, e3_nt, L, i))
                    if two_launch:
                        _same(ef[:, i], gpu.edgeFluxAssemble(ud, vd, None, a1, a2, e3u=e3m[0], e3v=e3m[1]))


@pytest.mark.parametrize('dtype', [numpy.float64, numpy.float32])
@pytest.mark.parametrize('big_endian', [False, True])
def test_layers_host_buffers(gpu, small, dtype, big_endian):
    """host buffers streamed in chunks (native and big-endian bytes, thickness and host e3): the masked host series"""
    s = small
    u, v = _fields(s, dtype)
    if big_endian:
        u, v = u.astype(u.dtype.newbyteorder('>')), v.astype(v.dtype.newbyteorder('>'))
    _, p = _handle(gpu, s['P'], s['ny'], s['nx'], s['transects'])
    a1, a2 = s['arc'][:, 1].copy(), s['arc'][:, 2].copy()
    for L in (ONE, RAGGED, PER_LEVEL):
        lay = p.fluxSeries(u, v, s['th'], a1, a2, fill=-7.0, chunk_steps=1, layers=L)
        assert isinstance(lay, numpy.ndarray) and lay.shape == (s['nt'], len(L) - 1, len(s['transects']))
        if L is ONE:
            _same(lay[:, 0], p.fluxSeries(u, v, s['th'], a1, a2, fill=-7.0, chunk_steps=1))
        for i in range(0, len(L) - 1, 7 if L is PER_LEVEL else 1):
            _same(lay[:, i], p.fluxSeries(u, v, s['th'] * _mask(L, i), a1, a2, fill=-7.0, chunk_steps=1), (L, i))
    e3 = numpy.random.default_rng(5).uniform(0.5, 30., (1, NZ, s['ny'] * s['nx'])).astype(u.dtype)
    lay = p.fluxSeries(u, v, None, a1, a2, chunk_steps=1, layers=RAGGED, e3u=e3, e3v=e3)
    for i in range(len(RAGGED) - 1):
        e3m = (e3 * _mask(RAGGED, i)[None, :, None]).astype(u.dtype)
        _same(lay[:, i], p.fluxSeries(u, v, None, a1, a2, chunk_steps=1, e3u=e3m, e3v=e3m), i)


@pytest.mark.parametrize('dtype', [numpy.float64, numpy.float32])
def test_layers_on_the_c2_and_c3_grids(gpu, oracle, dtype):
    """C2 (README) and C3 (ORCA1-shaped, 75 levels): one layer is the plain series, ragged layers the masked ones"""
    import torch
    from nemoflux_b200 import synth
    d = torch.device('cuda', 0)
    tdt = torch.float64 if dtype == numpy.float64 else torch.float32
    g = oracle.DataGen(nx=360, ny=180, nz=NZ, nt=2)
    u2, v2 = g.uv(SF_C2)
    arc = oracle.arc_lengths(g.points())
    c2 = (g.points(), g.ny, g.nx, [tr(README_C2)], torch.from_numpy(u2.astype(dtype)).to(d),
          torch.from_numpy(v2.astype(dtype)).to(d), g.thickness(), arc[:, 1].copy(), arc[:, 2].copy())
    syn = synth.make('C3')
    u3, v3 = syn.fill_device(0, 2, d, dtype=tdt, pad=8)
    c3 = (syn.points, syn.ny, syn.nx, syn.transects, u3, v3, syn.thickness, syn.arc1, syn.arc2)
    for P, ny, nx, transects, ud, vd, th, a1, a2 in (c2, c3):
        _, p = _handle(gpu, P, ny, nx, transects)
        th, a1, a2 = (torch.from_numpy(numpy.ascontiguousarray(x)).to(d) for x in (th, a1, a2))
        for two_launch in (False, True):
            plain, _ = _run(p, ud, vd, th, a1, a2, two_launch=two_launch)
            _same(_run(p, ud, vd, th, a1, a2, layers=ONE, two_launch=two_launch)[0][:, 0], plain)
            lay, _ = _run(p, ud, vd, th, a1, a2, layers=RAGGED, two_launch=two_launch)
            for i in range(len(RAGGED) - 1):
                ref, _ = _run(p, ud, vd, th * torch.from_numpy(_mask(RAGGED, i)).to(d), a1, a2, two_launch=two_launch)
                _same(lay[:, i], ref, i)


def _l1_scale(oracle, P, transects, u, v, th, arc):
    """sum |w*f| per (t, transect), the bar of DESIGN 2"""
    og = oracle.Grid(P)
    maps = []
    for xyz in transects:
        op = oracle.PolylineIntegral(og)
        op.computeWeights(xyz)
        maps.append(op.merged_map())
    out = numpy.zeros((u.shape[0], len(transects)))
    for t in range(u.shape[0]):
        iV, _, _ = oracle.edgeflux_step_c(u[t], v[t], th, arc[:, 1].copy(), arc[:, 2].copy(), False)
        f = iV.reshape(-1)
        for m, (keys, ws) in enumerate(maps):
            out[t, m] = numpy.abs(ws * f[keys]).sum()
    return out


def test_layers_match_the_oracle(gpu, oracle):
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
    for L in ([0, 3, 4, 12], list(range(nz + 1)), [2, 9]):
        lay = _np(p.fluxSeries(*args, layers=L))
        for i in range(len(L) - 1):
            thm = th * _mask(L, i, nz)
            ref = oracle.flux_series(P, transects, u, v, thm)
            scale = _l1_scale(oracle, P, transects, u, v, thm, arc)
            assert (numpy.abs(lay[:, i] - ref) <= 1e-12 * scale + 1e-300).all(), (L, i)


def test_per_level_layers_analytic(gpu):
    """node-to-node transects on a z-dependent stream function: layer k carries dz_k (psi_k(B) - psi_k(A)), and the
    layers add up to the plain series"""
    import torch
    from nemoflux_b200 import synth
    syn = synth.make('small')
    d = torch.device('cuda', 0)
    _, p = _handle(gpu, syn.points, syn.ny, syn.nx, syn.transects)
    u, v = syn.fill_device(0, 2, d)
    th, a1, a2 = (torch.from_numpy(x).to(d) for x in (syn.thickness, syn.arc1, syn.arc2))
    plain = _np(p.fluxSeries(u, v, th, a1, a2))
    lay = _np(p.fluxSeries(u, v, th, a1, a2, layers=range(syn.nz + 1)))
    scale = numpy.abs(plain).max()
    assert scale > 1.0
    assert numpy.abs(lay.sum(axis=1) - plain).max() <= 1e-12 * scale
    nexact = 0
    for m in range(syn.ntransects):
        if syn.node_ends[m] is None:
            continue
        (ja, ia), (jb, ib) = syn.node_ends[m]
        for t in range(2):
            a1k, a2k = syn.coeffs(t)
            ex = syn.thickness * (a1k * (syn.g1[jb, ib] - syn.g1[ja, ia]) + a2k * (syn.g2[jb, ib] - syn.g2[ja, ia]))
            assert numpy.abs(lay[t, :, m] - ex).max() <= 1e-11 * scale, (m, t)
        nexact += 1
    assert nexact >= syn.ntransects // 2


@pytest.mark.parametrize('dtype', [numpy.float64, numpy.float32])
@pytest.mark.parametrize('two_launch', [False, True])
def test_infinity_outside_the_layer(gpu, small, dtype, two_launch):
    """+-inf on a level outside a layer, in a column the transects read: that layer stays finite and equals the masked
    series of the data with the infinity replaced by 0; the layer holding it is not finite"""
    import torch
    s = small
    u, v = _fields(s, dtype)
    _, p = _handle(gpu, s['P'], s['ny'], s['nx'], s['transects'])
    d = 'cuda'
    a1, a2, th = (torch.from_numpy(x).to(d) for x in (s['arc'][:, 1].copy(), s['arc'][:, 2].copy(), s['th']))
    offs, grp = p.getColumnGroups('float64' if dtype == numpy.float64 else 'float32', 'map', 4)
    g0 = int(grp[offs[0] + (offs[1] - offs[0]) // 2]) * 4
    col = slice(g0, g0 + 4)                              # a group of 4 columns in which some transect reads eU or eV
    for val in (numpy.inf, -numpy.inf):
        ui, vi = u.copy(), v.copy()
        ui.reshape(s['nt'], NZ, -1)[:, 30, col] = val
        vi.reshape(s['nt'], NZ, -1)[:, 30, col] = val
        u0, v0 = u.copy(), v.copy()
        u0.reshape(s['nt'], NZ, -1)[:, 30, col] = 0
        v0.reshape(s['nt'], NZ, -1)[:, 30, col] = 0
        dev = lambda x: torch.from_numpy(x).to(d)          # noqa: E731
        lay, _ = _run(p, dev(ui), dev(vi), th, a1, a2, layers=RAGGED, two_launch=two_launch, fill=-7.0)
        for i in range(len(RAGGED) - 1):
            if RAGGED[i] <= 30 < RAGGED[i + 1]:
                assert not numpy.isfinite(lay[:, i]).all()
                continue
            assert numpy.isfinite(lay[:, i]).all()
            ref, _ = _run(p, dev(u0), dev(v0), th * torch.from_numpy(_mask(RAGGED, i)).to(d), a1, a2,
                          two_launch=two_launch, fill=-7.0)
            _same(lay[:, i], ref, (val, i))


def test_determinism_and_options_leave_the_bits(gpu, small):
    """run to run, and whatever the visiting order, the K3 lag, the ring size and the slot size of a one-panel grid"""
    import torch
    from nemoflux_b200 import _lib
    s = small
    u, v = _fields(s, numpy.float64)
    _, p = _handle(gpu, s['P'], s['ny'], s['nx'], s['transects'])
    d = 'cuda'
    args = [torch.from_numpy(x).to(d) for x in (u, v, s['th'], s['arc'][:, 1].copy(), s['arc'][:, 2].copy())]
    for L in (RAGGED, PER_LEVEL):
        base = _np(p.fluxSeries(*args, layers=L))
        for _ in range(3):
            _same(p.fluxSeries(*args, layers=L), base)
        for opt, vals in ((_lib.NFX_OPT_FUSED_ORDER, (0, 1, 2, 3)), (_lib.NFX_OPT_FUSED_K3_LAG, (1, 2, 7, 0)),
                          (_lib.NFX_OPT_RING_MAX_MB, (1, 4, 0)), (_lib.NFX_OPT_RING_SLOT_MB, (2, 8, 0))):
            for val in vals:
                _lib.set_option(opt, val)
                _same(p.fluxSeries(*args, layers=L), base, (opt, val))
                assert _lib.get_option(_lib.NFX_OPT_LAST_SERIES_PATH) == 1
        _lib.set_option(_lib.NFX_OPT_RING_SLOT_MB, 1)          # two panels: another summation order, deterministic
        two = _np(p.fluxSeries(*args, layers=L))
        for lag in (1, 3, 0):
            _lib.set_option(_lib.NFX_OPT_FUSED_K3_LAG, lag)
            _same(p.fluxSeries(*args, layers=L), two, ('two panels', lag))
        assert numpy.abs(two - base).max() <= 1e-12 * numpy.abs(base).max()
        _lib.set_option(_lib.NFX_OPT_RING_SLOT_MB, 0)


def test_invalid_layerings_raise_and_leave_the_output(gpu, small):
    import torch
    from nemoflux_b200 import _lib
    s = small
    _, p = _handle(gpu, s['P'], s['ny'], s['nx'], s['transects'])
    d = 'cuda'
    u, v = _fields(s, numpy.float64)
    args = [torch.from_numpy(x).to(d) for x in (u, v, s['th'], s['arc'][:, 1].copy(), s['arc'][:, 2].copy())]
    M = len(s['transects'])
    n0 = _lib.launch_count()
    for bad in ([5, 5], [0, 10, 7], [-1, 10], [0, NZ + 1], [40, 10]):
        out = torch.full((s['nt'], len(bad) - 1, M), 42.0, dtype=torch.float64, device=d)
        with pytest.raises(_lib.NemofluxGpuError) as e:
            p.fluxSeries(*args, layers=bad, out=out)
        assert e.value.code == 1 and 'layers' in str(e.value)
        assert (out == 42.0).all()
        with pytest.raises(_lib.NemofluxGpuError):
            p.fluxSeries(u, v, s['th'], s['arc'][:, 1].copy(), s['arc'][:, 2].copy(), chunk_steps=1, layers=bad)
    assert _lib.launch_count() == n0
    for bad in ([3], [[0, 1]], [0, 2.5]):
        with pytest.raises(ValueError):
            p.fluxSeries(*args, layers=bad)
    with pytest.raises(ValueError):
        p.fluxSeries(*args, layers=RAGGED, batch_range=(0, 1))
    out = torch.full((s['nt'], 4, M), 42.0, dtype=torch.float64, device=d)
    for shape in ((s['nt'], 2 * s['nx'] * s['ny']), (s['nt'], 3, 2 * s['nx'] * s['ny'])):
        with pytest.raises(ValueError):
            p.fluxSeries(*args, layers=RAGGED, out=out, eflux=torch.zeros(shape, dtype=torch.float64, device=d))
    assert (out == 42.0).all()
    # a layering whose (pseudo-step, panel) batches overflow an int is refused before anything runs
    lib = _lib.load()
    import ctypes
    lev = numpy.array([0, 1, 2], numpy.int32)
    nt_huge = 2 ** 30 + 1
    assert lib.nfx_flux_series_layers(ctypes.byref(p._h), ctypes.c_void_p(args[0].data_ptr()),
                                      ctypes.c_void_p(args[1].data_ptr()), None, None, _lib.NFX_F64, 0,
                                      ctypes.c_void_p(args[2].data_ptr()), ctypes.c_void_p(args[3].data_ptr()),
                                      ctypes.c_void_p(args[4].data_ptr()), nt_huge, NZ, s['nx'] * s['ny'], 2,
                                      lev.ctypes.data_as(ctypes.c_void_p), 0, float('nan'), _lib.NFX_ORDER_MAP, None,
                                      ctypes.c_void_p(out.data_ptr()), None) == 1
    assert 'overflows' in lib.nfx_last_error().decode()
    assert _lib.launch_count() == n0


def _files(tmp_path, *args):
    from nemoflux_b200 import datagen
    prefix = str(tmp_path) + '/'
    datagen.cli(list(args) + [f'--prefix={prefix}'])
    return prefix + 'T.nc', prefix + 'U.nc', prefix + 'V.nc'


def test_field_and_fluxplot_layers(gpu, oracle, tmp_path, capsys):
    """fluxplot --depthLayers / --layers on datagen files: snapped headers, per-layer columns that add up to the plain
    column, on the host-streamed path (classic files) and the device-decoded path (deflated NetCDF-4)"""
    import h5build
    from nemoflux_b200 import fluxplot
    from nemoflux_b200.field import Field
    nz = 8
    T, U, V = _files(tmp_path, f'--streamFunction={SF_C2}', '--nx=72', '--ny=36', f'--nz={nz}', '--nt=4',
                     '--deltaDeg=20,30')
    pts = '[(-100,-70),(100,-70),(0,70)],[(-150,-20),(-20,35),(60,-40)]'
    plain = fluxplot.main(['-t', T, '-u', U, '-v', V, '-l', pts])
    capsys.readouterr()
    csv = str(tmp_path / 'layers.csv')
    lay = fluxplot.main(['-t', T, '-u', U, '-v', V, '-l', pts, '--depthLayers', '0,0.3,2', '-o', csv])
    out = capsys.readouterr().out
    f = Field(T, U, V, [tr([(-100, -70), (100, -70), (0, 70)])], verbose=False)
    iface = f.layerInterfaces()
    L = f.levelsForDepths([0, 0.3, 2])
    assert L[0] == 0 and L[-1] == nz and lay.shape == (4, 2, 2)
    want = [f'line{m}[{iface[a]:g}-{iface[b]:g} m]' for m in range(2) for a, b in zip(L[:-1], L[1:])]
    assert 'time,' + ','.join(want) in out
    rows = open(csv).read().strip().split('\n')
    assert rows[0] == 'time,' + ','.join(want) and len(rows) == 5
    assert numpy.allclose([float(x) for x in rows[2].split(',')[1:]], lay[1].T.reshape(-1), rtol=0, atol=0)
    scale = numpy.abs(plain).max()
    assert numpy.abs(lay.sum(axis=1) - plain).max() <= 1e-12 * scale
    lay2 = fluxplot.main(['-t', T, '-u', U, '-v', V, '-l', pts, '--layers', '0,2,5,8'])
    out = capsys.readouterr().out
    assert f'line1[{iface[5]:g}-{iface[8]:g} m]' in out and lay2.shape == (4, 3, 2)
    assert numpy.abs(lay2.sum(axis=1) - plain).max() <= 1e-12 * scale
    # the device-decoded path: the same data as deflated NetCDF-4 files
    d = oracle.DataGen(nx=72, ny=36, nz=nz, nt=4, deltaDeg=(20., 30.))
    u, v = d.uv(SF_C2)
    U4, V4 = str(tmp_path / 'U4.nc'), str(tmp_path / 'V4.nc')
    for fname, vname, a in ((U4, 'uo', u), (V4, 'vo', v)):
        h5build.write(fname, {vname: dict(data=a, chunks=(1, 2, 36, 72), deflate=True, shuffle=True),
                              'time_counter': dict(data=numpy.arange(4.), chunks=(1,))})
    lines = [tr([(-100, -70), (100, -70), (0, 70)]), tr([(-150, -20), (-20, 35), (60, -40)])]
    f4 = Field(T, U4, V4, lines, verbose=False)
    s4 = f4.fluxSeries(chunk_steps=2, layers=[0, 2, 5, 8])
    assert f4.last_ingest['path'] == 'device decode'
    assert numpy.abs(s4 - lay2).max() <= 1e-12 * scale
    assert numpy.abs(s4.sum(axis=1) - plain).max() <= 1e-12 * scale
    assert numpy.array_equal(f4.fluxSeries(chunk_steps=2, layers=[0, 2, 5, 8], device_decode=False), s4)
