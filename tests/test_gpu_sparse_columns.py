"""The sparse fused pass (NFX_OPT_SPARSE_COLUMNS): its K2 tiles load only the column groups whose edge fluxes the
transects read.  The group list must be exactly the columns the oracle's map touches, and the series must be the dense
pass's series bit for bit, whatever the data, layout, path or transect set."""
import numpy
import pytest

from helpers import README_C2, SF_C2, random_transects, tr

pytestmark = pytest.mark.gpu

DENSE, AUTO, SPARSE = 0, 1, 2


@pytest.fixture(autouse=True)
def _reset_options():
    from nemoflux_b200 import _lib
    yield
    for opt in (_lib.NFX_OPT_SPARSE_COLUMNS, _lib.NFX_OPT_RING_SLOT_MB, _lib.NFX_OPT_FAST_SERIES):
        _lib.set_option(opt, 1 if opt != _lib.NFX_OPT_RING_SLOT_MB else 0)


def _handle(gpu, points, ny, nx, transects):
    g = gpu.Grid()
    g.setPoints(points)
    g.setCGridShape(ny, nx)
    p = gpu.PolylineIntegral()
    p.build(g)
    p.computeWeights(transects)
    return g, p


def _groups_ref(oracle, points, nx, transects, panel, vec):
    """numpy restatement: the u and v columns of every key of the oracle's merged maps -> per panel, sorted groups"""
    og = oracle.Grid(points)
    keys = [numpy.zeros(0, numpy.int64)]
    for xyz in transects:
        op = oracle.PolylineIntegral(og)
        op.computeWeights(xyz)
        keys.append(op.merged_map()[0])
    keys = numpy.concatenate(keys)
    cell, e = keys >> 2, keys & 3
    j, i = cell // nx, cell % nx
    ucols = numpy.concatenate([cell[e == 1], numpy.where(i >= 1, cell - 1, cell + nx - 1)[e == 3]])
    vcols = numpy.concatenate([cell[e == 2], (cell - nx)[(e == 0) & (j >= 1)]])   # south edge of row 0: always 0
    cols = numpy.unique(numpy.concatenate([ucols, vcols]))
    q = cols // panel
    g = (cols - q * panel) // vec
    return q, g


def _check_groups(gpu, oracle, syn_points, ny, nx, transects, dtype, vec):
    _, p = _handle(gpu, syn_points, ny, nx, transects)
    npanels, panel = p.getNumberOfPanels(dtype)
    offs, grp = p.getColumnGroups(dtype, 'map', vec)
    offs_l, grp_l = p.getColumnGroups(dtype, 'list', vec)
    assert numpy.array_equal(offs, offs_l) and numpy.array_equal(grp, grp_l)
    q, g = _groups_ref(oracle, syn_points, nx, transects, panel, vec)
    assert offs.size == npanels + 1 and offs[0] == 0 and offs[-1] == grp.size
    for k in range(npanels):
        want = numpy.unique(g[q == k])
        assert numpy.array_equal(grp[offs[k]:offs[k + 1]], want), (k, vec)
    return npanels


@pytest.mark.parametrize('dtype,vec', [('float64', 1), ('float64', 2), ('float64', 4), ('float32', 4), ('float32', 8)])
@pytest.mark.parametrize('slot_mb', [0, 1])
def test_group_list_matches_oracle_map(gpu, oracle, dtype, vec, slot_mb):
    """C3 grid and transects; a 1 MB ring slot cuts the grid into two panels"""
    from nemoflux_b200 import _lib, synth
    _lib.set_option(_lib.NFX_OPT_RING_SLOT_MB, slot_mb)
    syn = synth.make('C3')
    npanels = _check_groups(gpu, oracle, syn.points, syn.ny, syn.nx, syn.transects, dtype, vec)
    assert npanels == (1 if slot_mb == 0 else 2)


def _fields(dtype, specials, rng, nt, nz, ny, nx, g):
    u, v = g.uv(SF_C2)
    u, v = u[:nt, :nz].astype(dtype), v[:nt, :nz].astype(dtype)
    u[:, :, 10:14, 20:40] = numpy.nan
    if specials:
        tiny = numpy.finfo(dtype).tiny
        u[:, ::2, 30:33, 5:60] = tiny / 8                 # denormals
        v[:, 1::3, 40:42, 10:70] = -tiny / 16
        v[:, :, 50:52, 100:120] = -7.0                     # the fill value
    return u, v


def _series(p, mode, *args, **kw):
    from nemoflux_b200 import _lib
    _lib.set_option(_lib.NFX_OPT_SPARSE_COLUMNS, mode)
    s = p.fluxSeries(*args, **kw)
    s = s if isinstance(s, numpy.ndarray) else s.cpu().numpy()
    assert p.seriesStatus() == 0
    return s, _lib.get_option(_lib.NFX_OPT_LAST_SERIES_SPARSE)


def _same(a, b):
    assert numpy.array_equal(a, b, equal_nan=True)


@pytest.fixture(scope='module')
def small(oracle):
    nx, ny, nz, nt = 320, 240, 7, 4          # 76 800 cells: a 1 MB ring slot cuts them into two panels
    g = oracle.DataGen(nx=nx, ny=ny, nz=nz, nt=nt, deltaDeg=(20., 30.))
    P, arc = g.points(), oracle.arc_lengths(g.points())
    transects = random_transects(numpy.random.default_rng(3), 6, max_pts=4) + [tr(README_C2)]
    return dict(nx=nx, ny=ny, nz=nz, nt=nt, g=g, P=P, arc=arc, transects=transects,
                th=numpy.linspace(1.0, 40.0, nz))


@pytest.mark.parametrize('dtype', [numpy.float64, numpy.float32])
@pytest.mark.parametrize('order', ['list', 'map'])
@pytest.mark.parametrize('sverdrup', [False, True])
@pytest.mark.parametrize('slot_mb', [0, 1])
def test_sparse_equals_dense(gpu, small, dtype, order, sverdrup, slot_mb):
    """f64/f32 storage, both orders, sverdrup, a fill value, NaN / denormals; one and two panels; an infinity in a column
    no transect reads leaves the series unchanged, one in a touched column reaches it the same way in both passes"""
    import torch
    from nemoflux_b200 import _lib
    _lib.set_option(_lib.NFX_OPT_RING_SLOT_MB, slot_mb)
    s = small
    nx, ny = s['nx'], s['ny']
    u, v = _fields(dtype, True, None, s['nt'], s['nz'], ny, nx, s['g'])
    _, p = _handle(gpu, s['P'], ny, nx, s['transects'])
    vec = 4
    offs, grp = p.getColumnGroups('float64' if dtype == numpy.float64 else 'float32', order, vec)
    touched = numpy.zeros(ny * nx, bool)
    panel = p.getNumberOfPanels('float64' if dtype == numpy.float64 else 'float32')[1]
    for q in range(offs.size - 1):
        for gg in grp[offs[q]:offs[q + 1]]:
            touched[q * panel + gg * vec: q * panel + gg * vec + vec] = True
    assert touched.any() and not touched.all()
    d = 'cuda'
    a1, a2, th = (torch.from_numpy(x).to(d) for x in (s['arc'][:, 1].copy(), s['arc'][:, 2].copy(), s['th']))
    kw = dict(order=order, sverdrup=sverdrup, fill=-7.0)

    def run(uu, vv):
        ud, vd = torch.from_numpy(uu).to(d), torch.from_numpy(vv).to(d)
        dense, sp0 = _series(p, DENSE, ud, vd, th, a1, a2, **kw)
        sparse, sp2 = _series(p, SPARSE, ud, vd, th, a1, a2, **kw)
        assert (sp0, sp2) == (0, 1) and _lib.get_option(_lib.NFX_OPT_LAST_SERIES_PATH) == 1
        _same(dense, sparse)
        return sparse

    base = run(u, v)
    assert numpy.isfinite(base).all()
    untouched = numpy.nonzero(~touched)[0]
    uu = u.copy()
    uu.reshape(s['nt'], s['nz'], -1)[1, 2, untouched[len(untouched) // 2]] = numpy.inf
    vv = v.copy()
    vv.reshape(s['nt'], s['nz'], -1)[2, 0, untouched[len(untouched) // 3]] = -numpy.inf
    _same(run(uu, vv), base)
    hit = numpy.nonzero(touched)[0]
    uu.reshape(s['nt'], s['nz'], -1)[0, 1, hit[len(hit) // 2]] = numpy.inf
    run(uu, v)


@pytest.mark.parametrize('dtype', [numpy.float64, numpy.float32])
@pytest.mark.parametrize('layout', ['padded', 'misaligned'])
def test_sparse_equals_dense_layouts_ranges_e3(gpu, small, dtype, layout):
    """padded planes (widest vectors) and a view one element off alignment (vec 1), batch-range partial sums on two
    panels, and the fused e3 path"""
    import torch
    from nemoflux_b200 import _lib
    s = small
    nx, ny, nz, nt = s['nx'], s['ny'], s['nz'], s['nt']
    ncell = nx * ny
    u, v = _fields(dtype, True, None, nt, nz, ny, nx, s['g'])
    _, p = _handle(gpu, s['P'], ny, nx, s['transects'])
    d = 'cuda'
    tdt = torch.float64 if dtype == numpy.float64 else torch.float32
    pad = 4 if dtype == numpy.float64 else 8
    ld = (ncell + 1 + pad - 1) // pad * pad

    def dev(x):
        if layout == 'padded':
            t = torch.full((x.shape[0], nz, ld), 3.0, dtype=tdt, device=d)[:, :, :ncell]
        else:
            t = torch.full((x.shape[0] * nz * ncell + 1,), 3.0, dtype=tdt, device=d)[1:].view(x.shape[0], nz, ncell)
        t.copy_(torch.from_numpy(x.reshape(x.shape[0], nz, ncell)))
        return t
    ud, vd = dev(u), dev(v)
    a1, a2, th = (torch.from_numpy(x).to(d) for x in (s['arc'][:, 1].copy(), s['arc'][:, 2].copy(), s['th']))
    _lib.set_option(_lib.NFX_OPT_FAST_SERIES, 2)
    _same(*[_series(p, m, ud, vd, th, a1, a2)[0] for m in (DENSE, SPARSE)])
    e3 = dev(numpy.random.default_rng(9).uniform(0.5, 30., (1, nz, ny, nx)).astype(dtype))
    _same(*[_series(p, m, ud, vd, None, a1, a2, e3u=e3, e3v=e3)[0] for m in (DENSE, SPARSE)])
    _lib.set_option(_lib.NFX_OPT_RING_SLOT_MB, 1)
    npanels = p.getNumberOfPanels('float64' if dtype == numpy.float64 else 'float32')[0]
    assert npanels == 2
    for b0, b1 in ((0, 3), (3, nt * npanels - 2)):
        _same(*[_series(p, m, ud, vd, th, a1, a2, batch_range=(b0, b1))[0] for m in (DENSE, SPARSE)])
        _same(*[_series(p, m, ud, vd, None, a1, a2, e3u=e3, e3v=e3, batch_range=(b0, b1))[0] for m in (DENSE, SPARSE)])


@pytest.mark.parametrize('dtype', [numpy.float64, numpy.float32])
def test_sparse_equals_dense_host_buffers(gpu, small, dtype):
    from nemoflux_b200 import _lib
    s = small
    u, v = _fields(dtype, True, None, s['nt'], s['nz'], s['ny'], s['nx'], s['g'])
    _, p = _handle(gpu, s['P'], s['ny'], s['nx'], s['transects'])
    args = (u, v, s['th'], s['arc'][:, 1].copy(), s['arc'][:, 2].copy())
    dense, sp0 = _series(p, DENSE, *args, chunk_steps=3)
    sparse, sp2 = _series(p, SPARSE, *args, chunk_steps=3)
    assert _lib.get_option(_lib.NFX_OPT_LAST_SERIES_PATH) == 1 and (sp0, sp2) == (0, 1)
    _same(dense, sparse)


def test_transect_sets_empty_one_cell_whole_grid(gpu, oracle):
    """no sub-segment, one cell, and zonal transects through every row: there automatic mode keeps the dense pass"""
    import torch
    nx, ny, nz, nt = 64, 32, 5, 3
    g = oracle.DataGen(nx=nx, ny=ny, nz=nz, nt=nt)
    P, arc = g.points(), oracle.arc_lengths(g.points())
    u, v = g.uv(SF_C2)
    d = 'cuda'
    args = [torch.from_numpy(numpy.ascontiguousarray(x)).to(d)
            for x in (u, v, numpy.linspace(1., 2., nz), arc[:, 1].copy(), arc[:, 2].copy())]
    dlat = 180.0 / ny
    rows = [tr([(lon, -90 + (j + 0.5) * dlat) for lon in (-179.9, -90.0, 0.0, 90.0, 179.9)]) for j in range(ny)]
    cases = {'empty': [tr([(10.0, 10.0)])], 'one cell': [tr([(1.0, 1.0), (2.0, 2.0)])], 'whole grid': rows}
    for name, transects in cases.items():
        _, p = _handle(gpu, P, ny, nx, transects)
        dense, _ = _series(p, DENSE, *args)
        sparse, sp = _series(p, SPARSE, *args)
        assert sp == 1
        _same(dense, sparse)
        auto, sp_auto = _series(p, AUTO, *args)
        _same(auto, dense)
        share = p.getColumnGroups('float64', 'map', 4)[1].size * 4 / (nx * ny)
        assert sp_auto == (0 if name == 'whole grid' else 1), (name, share)
        if name == 'empty':
            assert share == 0 and (dense == 0).all()
        if name == 'whole grid':
            assert share > 0.95


def test_recompute_weights_on_the_same_handle(gpu, small):
    """computeWeights with another transect set rebuilds the group list: same series as a fresh handle"""
    import torch
    s = small
    u, v = _fields(numpy.float64, False, None, s['nt'], s['nz'], s['ny'], s['nx'], s['g'])
    d = 'cuda'
    args = [torch.from_numpy(numpy.ascontiguousarray(x)).to(d)
            for x in (u, v, s['th'], s['arc'][:, 1].copy(), s['arc'][:, 2].copy())]
    other = random_transects(numpy.random.default_rng(11), 5, max_pts=5)
    _, p = _handle(gpu, s['P'], s['ny'], s['nx'], s['transects'])
    _series(p, SPARSE, *args)
    p.computeWeights(other)
    again, sp = _series(p, SPARSE, *args)
    _, fresh = _handle(gpu, s['P'], s['ny'], s['nx'], other)
    ref, _ = _series(fresh, SPARSE, *args)
    dense, _ = _series(fresh, DENSE, *args)
    assert sp == 1
    _same(again, ref)
    _same(again, dense)


def test_c3_automatic_mode_takes_the_sparse_pass(gpu):
    """the flagship workload: its groups cover well under the threshold, so the default takes the sparse pass"""
    import torch
    from nemoflux_b200 import _lib, synth
    syn = synth.make('C3')
    _, p = _handle(gpu, syn.points, syn.ny, syn.nx, syn.transects)
    dev = torch.device('cuda', 0)
    u, v = syn.fill_device(0, 3, dev)
    args = [u, v] + [torch.from_numpy(x).to(dev) for x in (syn.thickness, syn.arc1, syn.arc2)]
    auto, sp = _series(p, AUTO, *args)
    dense, _ = _series(p, DENSE, *args)
    assert sp == 1 and _lib.get_option(_lib.NFX_OPT_SPARSE_COLUMNS) == DENSE
    _same(auto, dense)
