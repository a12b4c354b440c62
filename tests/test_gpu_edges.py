"""The section, window, class, tracer and series kernels at their loop and launch edges, against a float64 numpy
restatement of the per-crossing, per-level operations built from host inputs and the oracle's sub-segments only:
every level count from 1 to 7, 11 and 16 (the unroll tails of every kernel), both storage types, thickness and e3 of
1 or nt steps, dense and padded planes, layerings whose boundaries fall inside an unroll batch, transects of 31, 32,
33 and 65 crossings (the 32-crossing tiles); the second and later launch slices of every kernel (nt = 65 537, window
rows > 65 535, pseudo-steps > 65 535, several partial-sum batches of one class call, 96 classes on 3000 levels); the
two-launch series over more than 65 535 steps; every selectable K2 and fused instance against the oracle."""
import numpy
import pytest

from helpers import tr

pytestmark = pytest.mark.gpu

SCALE = 6371000.0 / 1.e6                    # sverdrup, as K2
FILL = -7.0                                 # the u/v marker of these tests (exact in float32)
TFILL = 1e20                                # the tracer / class-field marker (compared in the storage type)
NX, NY = 72, 24                             # 5-degree cells, 60S..60N
LEVELS = [1, 2, 3, 4, 5, 6, 7, 11, 16]


def _centre(j, i):
    return (-180. + 5. * i + 2.5, -60. + 5. * j + 2.5)


# crossings 31, 32, none, 33, 65 (along rows through the cell centres), one from row 0, one from column 0, one across
# the x-period seam: the 32-crossing tiles end inside, at and just past a tile
TRANSECTS = [tr([_centre(10, 3), _centre(10, 33)]), tr([_centre(12, 40), _centre(12, 71)]),
             tr([(0., 100.), (10., 120.)]), tr([_centre(14, 1), _centre(14, 33)]),
             tr([_centre(20, 2), _centre(20, 66)]), tr([_centre(0, 10), _centre(6, 14)]),
             tr([_centre(17, 0), _centre(22, 3)]), tr([_centre(15, 68), (_centre(17, 4)[0] + 360., _centre(17, 4)[1])])]
COUNTS = [31, 32, 0, 33, 65]


# ---- the reference ---------------------------------------------------------------------------------------------
def oracle_crossings(oracle, points, transects):
    """the oracle's sub-segments of every transect in emission order: cell (nsub), w (nsub, 4), offsets (M + 1)"""
    g = oracle.Grid(points)
    subs = []
    for xyz in transects:
        p = oracle.PolylineIntegral(g)
        p.computeWeights(xyz)
        subs.append(p.subsegs)
    s = numpy.concatenate(subs) if subs else numpy.zeros(0, oracle.SUBSEG_DTYPE)
    offs = numpy.concatenate([[0], numpy.cumsum([len(x) for x in subs])]).astype(numpy.int64)
    return dict(cell=s['cell'].astype(numpy.int64), w=numpy.ascontiguousarray(s['w']), offsets=offs)


def _clean(x, fill):
    """NaN and the marker (compared in the storage type) as 0, the rest converted exactly to float64"""
    return numpy.where(numpy.isnan(x) | (x == x.dtype.type(fill)), 0.0, x.astype(numpy.float64))


class Reference(object):
    """float64 restatement of the kernels' operation sequence per crossing s (cell c) and level k, from host inputs:
    edges in the order S, E, N, W read the columns v[south(c)], u[c], v[c], u[west(c)] (x-periodic west, the south
    edge of row 0 dead: its flux is 0); per layer and edge the column sum from +0 over ascending k of dz * u (e3 * u,
    times the face tracer q with a tracer), times arc1 (-arc2 for v), times 6.371 with sverdrup, then
    ((w0 f0 + w1 f1) + w2 f2) + w3 f3.  Every operation is one IEEE float64 operation, as on the device."""

    def __init__(self, sub, nx, ny, arc1, arc2):
        cell = sub['cell']
        self.w, self.offsets, self.nx, self.ncell = sub['w'], sub['offsets'], nx, nx * ny
        j, i = cell // nx, cell % nx
        west = numpy.where(i >= 1, cell - 1, cell + nx - 1)
        east = numpy.where(i + 1 < nx, cell + 1, cell + 1 - nx)
        north = numpy.where(j + 1 < ny, cell + nx, cell)
        south = numpy.where(j >= 1, cell - nx, cell)
        self.cell = cell
        self.col = numpy.stack([numpy.where(j >= 1, cell - nx, 0), cell, cell, west], 1)
        self.isv = numpy.array([True, False, True, False])
        self.live = numpy.stack([j >= 1] + [numpy.ones_like(j, bool)] * 3, 1)
        self.arc = numpy.where(self.live, numpy.where(self.isv, -arc2[self.col], arc1[self.col]), 0.0)
        self.face = (numpy.stack([south, cell, cell, west], 1), numpy.stack([cell, east, north, cell], 1),
                     numpy.stack([numpy.ones_like(j, bool), numpy.ones_like(j, bool), j + 1 < ny,
                                  numpy.ones_like(j, bool)], 1))

    def _term(self, u, v, k, th, e3u, e3v, fill):
        """(nt, nsub, 4): dz (or e3) times u at level k of every edge"""
        x = _clean(numpy.where(self.isv, v[:, k][:, self.col], u[:, k][:, self.col]), fill)
        d = th[k] if th is not None else _clean(numpy.where(self.isv, e3v[:, k][:, self.col],
                                                            e3u[:, k][:, self.col]), fill)
        return d * x

    def _q(self, tau, k, tfill, ref):
        """(1 or nt, nsub, 4): the face value of the tracer at level k of every edge"""
        a, b, has_b = self.face
        ta, tb = tau[:, k][:, a], tau[:, k][:, b]
        dt = tau.dtype.type
        pa = ~(numpy.isnan(ta) | (ta == dt(tfill)))
        pb = ~(numpy.isnan(tb) | (tb == dt(tfill))) & has_b
        fa, fb = ta.astype(numpy.float64), tb.astype(numpy.float64)
        return numpy.where(pa & pb, 0.5 * (fa + fb) - ref,
                           numpy.where(pa, fa - ref, numpy.where(pb, fb - ref, 0.0)))

    def section(self, u, v, levels, th=None, e3u=None, e3v=None, fill=numpy.nan, sverdrup=False, tau=None,
                tfill=numpy.nan, ref=0.0):
        """(section (nt, N, nsub), sum of |w f| over the edges (nt, N, nsub)); u, v (nt, nz, ncell) and e3u, e3v,
        tau (1 or nt, nz, ncell) in the storage type"""
        nt, nsub, n = u.shape[0], len(self.cell), len(levels) - 1
        out, bar = numpy.zeros((nt, n, nsub)), numpy.zeros((nt, n, nsub))
        with numpy.errstate(invalid='ignore', over='ignore'):
            for li in range(n):
                acc = numpy.zeros((nt, nsub, 4))
                for k in range(levels[li], levels[li + 1]):
                    t = self._term(u, v, k, th, e3u, e3v, fill)
                    acc = acc + (t if tau is None else t * self._q(tau, k, tfill, ref))
                f = acc * self.arc
                if sverdrup:
                    f = f * SCALE
                f = numpy.where(self.live, f, 0.0)
                r = self.w[:, 0] * f[..., 0]
                for e in range(1, 4):
                    r = r + self.w[:, e] * f[..., e]
                out[:, li], bar[:, li] = r, (numpy.abs(self.w) * numpy.abs(f)).sum(-1)
        return out, bar

    def per_transect(self, x):
        """(..., nsub) -> (..., M): the sum over every transect's crossings (numpy's order: for the bars)"""
        o = self.offsets
        return numpy.stack([x[..., a:b].sum(-1) for a, b in zip(o[:-1], o[1:])], -1)

    def tile_fold(self, x):
        """(..., nsub) -> (..., M): per transect the 32-crossing tiles in emission order, each folded by the shuffle
        tree (lane l + lane l + o, o = 16 .. 1, absent lanes +0), the tiles added in ascending order from +0"""
        o = self.offsets
        out = numpy.zeros(x.shape[:-1] + (len(o) - 1,))
        for m in range(len(o) - 1):
            acc = numpy.zeros(x.shape[:-1])
            for t0 in range(o[m], o[m + 1], 32):
                t1 = min(t0 + 32, o[m + 1])
                lanes = numpy.zeros(x.shape[:-1] + (32,))
                lanes[..., :t1 - t0] = x[..., t0:t1]
                for h in (16, 8, 4, 2, 1):
                    lanes[..., :h] = lanes[..., :h] + lanes[..., h:2 * h]
                acc = acc + lanes[..., 0]
            out[..., m] = acc
        return out

    def classes(self, u, v, cf, bounds, cfill=numpy.nan, **kw):
        """(classes (nt, K, M) in the kernels' order, sum of |terms| (nt, K, M)): per crossing the one-level section
        of every level added to the class of cf at its cell in ascending k from +0, then the tile fold"""
        nt, nz = u.shape[:2]
        K = len(bounds) - 1
        x = cf[:, :, self.cell]
        bad = numpy.isnan(x) | (x == x.dtype.type(cfill))
        j = numpy.searchsorted(numpy.asarray(bounds, numpy.float64), x.astype(numpy.float64), side='right') - 1
        j = numpy.where(bad | (j >= K), -1, j)
        j = numpy.broadcast_to(j, (nt,) + j.shape[1:])
        per_level, bar_k = self.section(u, v, list(range(nz + 1)), **kw)
        out, bar = numpy.zeros((nt, K, len(self.offsets) - 1)), numpy.zeros((nt, K, len(self.offsets) - 1))
        for c in numpy.unique(j[j >= 0]):
            acc = numpy.zeros((nt, len(self.cell)))
            for k in range(nz):
                acc = numpy.where(j[:, k] == c, acc + per_level[:, k], acc)
            out[:, c] = self.tile_fold(acc)
            bar[:, c] = self.per_transect(numpy.where(j == c, bar_k, 0.0).sum(1))
        return out, bar

    def cell_fluxes(self, u, v, levels, th=None, e3u=None, e3v=None, fill=numpy.nan, sverdrup=False, arc1=None,
                    arc2=None):
        """K2's edge fluxes (nt, N, 2 * ncell) of every cell: [eU | eV] per layer"""
        nt, n = u.shape[0], len(levels) - 1
        out = numpy.zeros((nt, n, 2 * self.ncell))
        with numpy.errstate(invalid='ignore', over='ignore'):
            for li in range(n):
                su, sv = numpy.zeros((nt, self.ncell)), numpy.zeros((nt, self.ncell))
                for k in range(levels[li], levels[li + 1]):
                    du = th[k] if th is not None else _clean(e3u[:, k], fill)
                    dv = th[k] if th is not None else _clean(e3v[:, k], fill)
                    su = su + du * _clean(u[:, k], fill)
                    sv = sv + dv * _clean(v[:, k], fill)
                fu, fv = su * arc1, (-sv) * arc2
                if sverdrup:
                    fu, fv = fu * SCALE, fv * SCALE
                out[:, li, :self.ncell], out[:, li, self.ncell:] = fu, fv
        return out


def window_sums(sec, bounds, start=None):
    """sums over the windows [b_w, b_(w+1)) of a section (nt, N, nsub), steps added in ascending order from +0 (window
    0 from `start` instead: a continued sum)"""
    out = numpy.zeros((len(bounds) - 1,) + sec.shape[1:])
    for w in range(len(bounds) - 1):
        acc = numpy.zeros(sec.shape[1:]) if w or start is None else start.copy()
        for t in range(bounds[w], bounds[w + 1]):
            acc = acc + sec[t]
        out[w] = acc
    return out


# ---- comparisons -----------------------------------------------------------------------------------------------
def _np(x):
    return x if isinstance(x, numpy.ndarray) else x.cpu().numpy()


def _same(got, want, what=''):
    """bit for bit; NaN matches NaN whatever its payload"""
    got, want = _np(got), numpy.asarray(want, numpy.float64)
    assert got.shape == want.shape, (what, got.shape, want.shape)
    gn, wn = numpy.isnan(got), numpy.isnan(want)
    ok = (gn == wn) & ((got.view(numpy.int64) == want.view(numpy.int64)) | gn)
    if not ok.all():
        i = numpy.argwhere(~ok)[0]
        raise AssertionError(f'{what}: {(~ok).sum()} of {ok.size} values differ, first at {tuple(i)}: '
                             f'{got[tuple(i)]!r} vs {want[tuple(i)]!r}')


def _close(got, want, bar, what=''):
    got = _np(got)
    assert got.shape == want.shape, (what, got.shape, want.shape)
    err = numpy.abs(got - want)
    assert (err <= 1e-12 * bar + 1e-300).all(), (what, err.max(), numpy.argwhere(err > 1e-12 * bar + 1e-300)[0])


# ---- fixtures --------------------------------------------------------------------------------------------------
OPTIONS = ('NFX_OPT_K2_VARIANT', 'NFX_OPT_K2_UNROLL', 'NFX_OPT_K2_BLOCK', 'NFX_OPT_K2_ALU_MASK',
           'NFX_OPT_FUSED_F32_SHAPE', 'NFX_OPT_FUSED_F64_CTAS', 'NFX_OPT_FAST_SERIES')


@pytest.fixture(autouse=True)
def _restore_options():
    """every option a test here sets is put back afterwards, also when the test fails"""
    from nemoflux_b200 import _lib
    saved = [(getattr(_lib, n), _lib.get_option(getattr(_lib, n))) for n in OPTIONS]
    yield
    for opt, val in saved:
        _lib.set_option(opt, val)


def _option(name, value):
    from nemoflux_b200 import _lib
    _lib.set_option(getattr(_lib, name), value)


def _handle(gpu, points, ny, nx, transects):
    g = gpu.Grid()
    g.setPoints(points)
    g.setCGridShape(ny, nx)
    p = gpu.PolylineIntegral()
    p.build(g)
    p.computeWeights(transects)
    return g, p


def _checked_handle(gpu, oracle, points, ny, nx, transects):
    """the GPU handle and the oracle's crossings; K1 must have emitted the oracle's cells and weights"""
    _, p = _handle(gpu, points, ny, nx, transects)
    sub = oracle_crossings(oracle, points, transects)
    gs = p.getSubsegments()
    assert numpy.array_equal(gs['offsets'], sub['offsets']) and numpy.array_equal(gs['cell'], sub['cell'])
    assert numpy.array_equal(gs['w'].view(numpy.int64), sub['w'].view(numpy.int64))
    return p, sub


@pytest.fixture(scope='module')
def grid(oracle):
    d = oracle.DataGen(nx=NX, ny=NY, ymin=-60., ymax=60.)
    P = d.points()
    arc = oracle.arc_lengths(P)
    sub = oracle_crossings(oracle, P, TRANSECTS)
    n = numpy.diff(sub['offsets'])
    assert list(n[:5]) == COUNTS and n[5:].min() > 0
    cells = sub['cell'][sub['offsets'][5]:sub['offsets'][6]]
    assert (cells < NX).any() and (sub['cell'][sub['offsets'][6]:sub['offsets'][7]] % NX == 0).any()
    return dict(P=P, arc1=arc[:, 1].copy(), arc2=arc[:, 2].copy())


def _data(rng, dtype, shape, fill=FILL):
    """random values with NaN, the marker, denormals and exact zeros of both signs"""
    x = rng.uniform(-2.0, 2.0, shape)
    flat = x.reshape(-1)
    idx = rng.permutation(flat.size)
    q = max(1, flat.size // 40)
    flat[idx[:q]] = numpy.nan
    flat[idx[q:2 * q]] = fill
    flat[idx[3 * q:4 * q]] = 0.0
    flat[idx[4 * q:5 * q]] = -0.0
    x = x.astype(dtype)
    x.reshape(-1)[idx[2 * q:3 * q]] = numpy.finfo(dtype).tiny / dtype(8) * numpy.sign(flat[idx[2 * q:3 * q]] + 0.5)
    return x


def _tracer(rng, dtype, shape):
    t = rng.uniform(-2.0, 30.0, shape)
    flat = t.reshape(-1)
    idx = rng.permutation(flat.size)
    q = max(1, flat.size // 20)
    flat[idx[:q]] = numpy.nan
    flat[idx[q:2 * q]] = TFILL
    flat[idx[2 * q:3 * q]] = numpy.round(flat[idx[2 * q:3 * q]])        # on the class bounds
    return t.astype(dtype)


def _layerings(nz):
    """the whole column, one layer per level, and layerings starting above level 0 / ending above nz with
    boundaries inside an unroll batch"""
    out = [[0, nz], list(range(nz + 1))]
    if nz >= 2:
        out.append([1, nz])
        out.append([0, nz - 1])
    if nz >= 3:
        out.append([1, 2, nz])
    if nz >= 6:
        out.append([1, 2, 5, nz])
    if nz >= 11:
        out.append([3, 4, 9, 10, nz])
    uniq = []
    for L in out:
        if L not in uniq:
            uniq.append(L)
    return uniq


class Device(object):
    """host arrays (nt, nz, ncell) as CUDA tensors, densely or on padded planes (ld > ncell, ld a multiple of 8)"""

    def __init__(self, ncell, padded):
        self.ncell, self.padded = ncell, padded
        self.ld = (ncell + 8) // 8 * 8 + 8 if padded else ncell

    def __call__(self, x):
        import torch
        x = numpy.ascontiguousarray(x)
        if not self.padded:
            return torch.from_numpy(x).to('cuda')
        t = torch.full(x.shape[:2] + (self.ld,), 3.0, dtype=torch.from_numpy(x[:0]).dtype, device='cuda')
        t = t[:, :, :self.ncell]
        t.copy_(torch.from_numpy(x))
        return t


# ---- 2. the level-count sweep ----------------------------------------------------------------------------------
@pytest.mark.parametrize('nz', LEVELS)
@pytest.mark.parametrize('dtype', [numpy.float64, numpy.float32])
def test_level_sweep(gpu, oracle, grid, dtype, nz):
    """every nz of LEVELS x storage type x {thickness, e3 of 1 step, e3 of nt steps} x {dense, padded planes}: the
    section, the window sums, the tracer section and series and the K2 edge fluxes of every layering bit for bit, the
    classes bit for bit, the layered and whole-column series through the fused pass and two launches within
    1e-12 * sum |terms|"""
    import torch
    nt, ncell = 5, NX * NY
    p, sub = _checked_handle(gpu, oracle, grid['P'], NY, NX, TRANSECTS)
    R = Reference(sub, NX, NY, grid['arc1'], grid['arc2'])
    rng = numpy.random.default_rng(1000 * nz + (dtype == numpy.float32))
    u, v = _data(rng, dtype, (nt, nz, ncell)), _data(rng, dtype, (nt, nz, ncell))
    th = rng.uniform(0.5, 30.0, nz)
    e3u = numpy.abs(_data(rng, dtype, (nt, nz, ncell))) * dtype(10.0)
    e3v = numpy.abs(_data(rng, dtype, (nt, nz, ncell))) * dtype(10.0)
    tau = _tracer(rng, dtype, (nt, nz, ncell))
    bounds = [-numpy.inf, 0.0, 4.0, 10.0, 17.0, 25.0]
    wins = [0, 1, 4, 5]
    a1, a2 = torch.from_numpy(grid['arc1']).to('cuda'), torch.from_numpy(grid['arc2']).to('cuda')
    for padded in (False, True):
        dev = Device(ncell, padded)
        ud, vd = dev(u), dev(v)
        metrics = [('thickness', dict(thickness=torch.from_numpy(th).to('cuda')), dict(th=th))]
        for n in (1, nt):
            metrics.append((f'e3 {n}', dict(thickness=None, e3u=dev(e3u[:n]), e3v=dev(e3v[:n])),
                            dict(e3u=e3u[:n], e3v=e3v[:n])))
        for name, dk, rk in metrics:
            sverdrup = name != 'thickness'
            kw = dict(fill=FILL, sverdrup=sverdrup)
            rkw = dict(rk, fill=FILL, sverdrup=sverdrup)
            what = (name, 'padded' if padded else 'dense')
            tr_nt = 1 if name == 'e3 1' else nt
            taud = dev(tau[:tr_nt])
            dargs = (ud, vd, dk['thickness'], a1, a2)
            e3 = dict(e3u=dk.get('e3u'), e3v=dk.get('e3v'))
            for L in _layerings(nz):
                sec, bar = R.section(u, v, L, **rkw)
                _same(p.fluxSection(*dargs, layers=L, **e3, **kw), sec, what + ('section', L))
                _same(p.sectionWindowSums(*dargs, wins, layers=L, **e3, **kw), window_sums(sec, wins),
                      what + ('windows', L))
                tsec, tbar = R.section(u, v, L, tau=tau[:tr_nt], tfill=TFILL, ref=1.5, **rkw)
                _same(p.fluxTracer(*dargs, taud, tfill=TFILL, ref=1.5, layers=L, section=True, **e3, **kw), tsec,
                      what + ('tracer section', L))
                _same(p.fluxTracer(*dargs, taud, tfill=TFILL, ref=1.5, layers=L, **e3, **kw), R.tile_fold(tsec),
                      what + ('tracer series', L))
                want, wbar = R.per_transect(sec), R.per_transect(bar)
                for fast in (2, 0):
                    _option('NFX_OPT_FAST_SERIES', fast)
                    _close(p.fluxSeries(*dargs, layers=L, **e3, **kw), want, wbar, what + ('series', fast, L))
                ef = torch.zeros((nt, len(L) - 1, 2 * ncell), dtype=torch.float64, device='cuda')
                _close(p.fluxSeries(*dargs, layers=L, eflux=ef, **e3, **kw), want, wbar, what + ('series eflux', L))
                _same(ef, R.cell_fluxes(u, v, L, arc1=grid['arc1'], arc2=grid['arc2'], **rkw), what + ('eflux', L))
            # the whole column without a layering: the plain K2 and fused instances
            sec, bar = R.section(u, v, [0, nz], **rkw)
            want, wbar = R.per_transect(sec[:, 0]), R.per_transect(bar[:, 0])
            for fast in (2, 0):
                _option('NFX_OPT_FAST_SERIES', fast)
                _close(p.fluxSeries(*dargs, **e3, **kw), want, wbar, what + ('whole series', fast))
            ef = torch.zeros((nt, 2 * ncell), dtype=torch.float64, device='cuda')
            _close(p.fluxSeries(*dargs, eflux=ef, **e3, **kw), want, wbar, what + ('whole series eflux',))
            _same(ef, R.cell_fluxes(u, v, [0, nz], arc1=grid['arc1'], arc2=grid['arc2'], **rkw)[:, 0],
                  what + ('whole eflux',))
            # classes: one-level sections binned by a class field of nt steps (1 step with e3 of 1 step)
            cls, cbar = R.classes(u, v, tau[:tr_nt], bounds, cfill=TFILL, **rkw)
            assert (cbar > 0).sum() > 20
            _same(p.fluxClasses(*dargs, taud, bounds, cfill=TFILL, **e3, **kw), cls, what + ('classes',))


# ---- 3. launch-slice edges -------------------------------------------------------------------------------------
@pytest.fixture(scope='module')
def tiny(oracle):
    """9 x 11 cells (99: no 128-bit rows in float32), a transect from row 1 to the top row and one along a grid line
    (crossings shared by the cells on both sides)"""
    d = oracle.DataGen(nx=9, ny=11, ymin=-55., ymax=55., dy=10.)
    P = d.points()
    arc = oracle.arc_lengths(P)
    lines = [tr([(-100., -38.), (-40., -30.)]), tr([(-170., -42.), (150., 37.)])]
    return dict(P=P, arc1=arc[:, 1].copy(), arc2=arc[:, 2].copy(), lines=lines, nx=9, ny=11)


def _tiny_inputs(tiny, dtype, nt, nz, seed):
    rng = numpy.random.default_rng(seed)
    ncell = tiny['nx'] * tiny['ny']
    u, v = _data(rng, dtype, (nt, nz, ncell)), _data(rng, dtype, (nt, nz, ncell))
    return u, v, rng.uniform(0.5, 30.0, nz), _tracer(rng, dtype, (nt, nz, ncell))


def test_second_launch_slices(gpu, oracle, tiny):
    """nt = 65 537 (two slices of gridDim.y): the section, the tracer section and series and the classes bit for bit;
    window sums over 65 537 one-step windows x 2 layers (131 074 rows), continuing a stored sum and through host-buffer
    chunks, bit for bit; the layered two-launch series over 40 000 steps x 2 layers (80 000 pseudo-steps): edge fluxes
    bit for bit, series within 1e-12 * sum |terms|"""
    import torch
    nt, nz, dtype = 65537, 2, numpy.float32
    p, sub = _checked_handle(gpu, oracle, tiny['P'], tiny['ny'], tiny['nx'], tiny['lines'])
    R = Reference(sub, tiny['nx'], tiny['ny'], tiny['arc1'], tiny['arc2'])
    u, v, th, tau = _tiny_inputs(tiny, dtype, nt, nz, 5)
    dev = lambda x: torch.from_numpy(numpy.ascontiguousarray(x)).to('cuda')   # noqa: E731
    dargs = (dev(u), dev(v), dev(th), dev(tiny['arc1']), dev(tiny['arc2']))
    kw = dict(fill=FILL, sverdrup=True)
    L = [0, 1, 2]
    sec, _ = R.section(u, v, L, th=th, **kw)
    _same(p.fluxSection(*dargs, layers=L, **kw), sec, 'section')
    taud = dev(tau)
    tsec, _ = R.section(u, v, L, th=th, tau=tau, tfill=TFILL, ref=2.5, **kw)
    _same(p.fluxTracer(*dargs, taud, tfill=TFILL, ref=2.5, layers=L, section=True, **kw), tsec, 'tracer section')
    _same(p.fluxTracer(*dargs, taud, tfill=TFILL, ref=2.5, layers=L, **kw), R.tile_fold(tsec), 'tracer series')
    bounds = [0.0, 4.0, 10.0, 30.0]
    cls, _ = R.classes(u, v, tau, bounds, cfill=TFILL, th=th, **kw)
    _same(p.fluxClasses(*dargs, taud, bounds, cfill=TFILL, **kw), cls, 'classes')
    del tsec, cls
    # windows: one row per (window, layer) on gridDim.y
    wins = list(range(0, nt + 1))
    start = numpy.random.default_rng(2).uniform(-1, 1, (1, 2, len(sub['cell'])))
    want = window_sums(sec, wins, start[0])
    sums = torch.zeros((nt, 2, len(sub['cell'])), dtype=torch.float64, device='cuda')
    sums[0] = dev(start[0])
    _same(p.sectionWindowSums(*dargs, wins, layers=L, sums=sums, continue_first=True, **kw), want, 'windows')
    hs = numpy.zeros((nt, 2, len(sub['cell'])))
    hs[0] = start[0]
    uh, vh = (x.reshape(nt, nz, tiny['ny'], tiny['nx']) for x in (u, v))
    got = p.sectionWindowSums(uh, vh, th, tiny['arc1'], tiny['arc2'], wins, layers=L, sums=hs, continue_first=True,
                              chunk_steps=20000, **kw)
    _same(got, want, 'windows, host chunks')
    wide = [0, 3, 30001, 30002, nt]                   # windows across the host chunks
    _same(p.sectionWindowSums(uh, vh, th, tiny['arc1'], tiny['arc2'], wide, layers=L, chunk_steps=20000, **kw),
          window_sums(sec, wide), 'long windows, host chunks')
    del want, hs, got
    # the layered two-launch series: 80 000 pseudo-steps, 40 000 time steps
    n = 40000
    _option('NFX_OPT_FAST_SERIES', 0)
    ef = torch.zeros((n, 2, 2 * tiny['nx'] * tiny['ny']), dtype=torch.float64, device='cuda')
    ser = p.fluxSeries(*(x[:n] for x in dargs[:2]), *dargs[2:], layers=L, eflux=ef, **kw)
    _same(ef, R.cell_fluxes(u[:n], v[:n], L, th=th, arc1=tiny['arc1'], arc2=tiny['arc2'], **kw), 'layered eflux')
    _, bar = R.section(u[:n], v[:n], L, th=th, **kw)
    _close(ser, R.per_transect(sec[:n]), R.per_transect(bar), 'layered series')
    _close(p.fluxSeries(*(x[:n] for x in dargs[:2]), *dargs[2:], layers=L, **kw), R.per_transect(sec[:n]),
           R.per_transect(bar), 'layered series, internal eflux')


def test_class_partial_batches(gpu, oracle, grid):
    """96 classes on 24 transects of 65 crossings (72 tiles) over 1300 steps: the 64 MB of partial sums hold 1213
    steps, so one call runs 2 batches of k_flux_classes + k_reduce_class_tiles; the classes bit for bit"""
    import torch
    from nemoflux_b200 import _lib
    nt, nz, ncell, dtype = 1300, 1, NX * NY, numpy.float32
    lines = [tr([_centre(j, 2), _centre(j, 66)]) for j in range(NY)]
    p, sub = _checked_handle(gpu, oracle, grid['P'], NY, NX, lines)
    R = Reference(sub, NX, NY, grid['arc1'], grid['arc2'])
    rng = numpy.random.default_rng(8)
    u, v = _data(rng, dtype, (nt, nz, ncell)), _data(rng, dtype, (nt, nz, ncell))
    th = rng.uniform(0.5, 30.0, nz)
    cf = rng.uniform(0.0, 4.0, (nt, nz, ncell)).astype(dtype)
    cf[:, :, ::11] = numpy.nan
    cf[:, :, ::13] = 95.5                                   # the last class
    bounds = numpy.arange(97.0)
    ntiles = int(sum((b - a + 31) // 32 for a, b in zip(sub['offsets'][:-1], sub['offsets'][1:])))
    steps = max(1, min(nt, (64 << 20) // 8 // (ntiles * 96)))
    nbatch = -(-nt // steps)
    assert ntiles == 72 and nbatch == 2, (ntiles, steps)
    dev = lambda x: torch.from_numpy(numpy.ascontiguousarray(x)).to('cuda')   # noqa: E731
    dargs = (dev(u), dev(v), dev(th), dev(grid['arc1']), dev(grid['arc2']))
    want, _ = R.classes(u, v, cf, bounds, th=th, fill=FILL)
    assert (want[steps:, 95] != 0).any() and (want[steps:, :4] != 0).all()
    n0 = _lib.launch_count()
    got = p.fluxClasses(*dargs, dev(cf), bounds, fill=FILL)
    assert _lib.launch_count() - n0 == 2 * nbatch
    _same(got, want, 'classes')


def test_96_classes_on_3000_levels(gpu, oracle, tiny):
    """K = 96 (the most) with nz = 3000: 221 KB of dynamic shared memory in k_flux_classes; bit for bit"""
    import torch
    nt, nz = 2, 3000
    p, sub = _checked_handle(gpu, oracle, tiny['P'], tiny['ny'], tiny['nx'], tiny['lines'])
    R = Reference(sub, tiny['nx'], tiny['ny'], tiny['arc1'], tiny['arc2'])
    u, v, th, _ = _tiny_inputs(tiny, numpy.float64, nt, nz, 6)
    cf = numpy.random.default_rng(7).uniform(-1.0, 97.0, (1, nz, tiny['nx'] * tiny['ny']))
    bounds = numpy.arange(97.0)
    dev = lambda x: torch.from_numpy(numpy.ascontiguousarray(x)).to('cuda')   # noqa: E731
    want, _ = R.classes(u, v, cf, bounds, th=th, fill=FILL)
    assert (want != 0).sum(1).min() > 10
    got = p.fluxClasses(dev(u), dev(v), dev(th), dev(tiny['arc1']), dev(tiny['arc2']), dev(cf), bounds, fill=FILL)
    _same(got, want, 'classes')


# ---- 4. the two-launch series over more than 65 535 steps ------------------------------------------------------
@pytest.mark.parametrize('dtype', [numpy.float32, numpy.float64])
def test_two_launch_series_over_65535_steps(gpu, oracle, tiny, dtype):
    """70 000 steps on 99 cells: the host-array series (float32: the two-launch path by default, 99 cells give no
    128-bit rows; float64 with NFX_OPT_FAST_SERIES = 0) and the device series with two launches, whole column and
    layered, within 1e-12 * sum |terms| of the reference and of the fused pass"""
    import torch
    from nemoflux_b200 import _lib
    nt, nz = 70000, 2
    p, sub = _checked_handle(gpu, oracle, tiny['P'], tiny['ny'], tiny['nx'], tiny['lines'])
    R = Reference(sub, tiny['nx'], tiny['ny'], tiny['arc1'], tiny['arc2'])
    u, v, th, _ = _tiny_inputs(tiny, dtype, nt, nz, 9)
    a1, a2 = tiny['arc1'], tiny['arc2']
    dev = lambda x: torch.from_numpy(numpy.ascontiguousarray(x)).to('cuda')   # noqa: E731
    dargs = (dev(u), dev(v), dev(th), dev(a1), dev(a2))
    for L in (None, [0, 1, 2]):
        sec, bar = R.section(u, v, [0, nz] if L is None else L, th=th, fill=FILL)
        want, wbar = R.per_transect(sec), R.per_transect(bar)
        if L is None:
            want, wbar = want[:, 0], wbar[:, 0]
        _option('NFX_OPT_FAST_SERIES', 2)
        fused = _np(p.fluxSeries(*dargs, layers=L, fill=FILL))
        assert _lib.get_option(_lib.NFX_OPT_LAST_SERIES_PATH) == 1
        _close(fused, want, wbar, ('fused', L))
        _option('NFX_OPT_FAST_SERIES', 1 if dtype == numpy.float32 else 0)
        host = p.fluxSeries(u.reshape(nt, nz, tiny['ny'], tiny['nx']), v.reshape(nt, nz, tiny['ny'], tiny['nx']), th,
                            a1, a2, layers=L, fill=FILL)
        assert _lib.get_option(_lib.NFX_OPT_LAST_SERIES_PATH) == 0
        _close(host, want, wbar, ('host', L))
        _close(host, fused, wbar, ('host vs fused', L))
        _option('NFX_OPT_FAST_SERIES', 0)
        got = p.fluxSeries(*dargs, layers=L, fill=FILL)
        assert _lib.get_option(_lib.NFX_OPT_LAST_SERIES_PATH) == 0
        _same(got, host, ('device two launches = host', L))


# ---- 5. every selectable K2 and fused instance -----------------------------------------------------------------
K2_PAIRS = [(5, 256), (3, 256), (15, 256), (5, 128), (5, 512)]      # dispatch_ldg


def _k2_configs(dtype):
    """(name, {option: value}) of every K2 instance the options select for this storage type"""
    out = [('ldg', dict(NFX_OPT_K2_VARIANT=1)), ('ldg128', dict(NFX_OPT_K2_VARIANT=3))]
    out += [(f'unroll {a} block {b}', dict(NFX_OPT_K2_UNROLL=a, NFX_OPT_K2_BLOCK=b)) for a, b in K2_PAIRS]
    out += [(f'unroll {a} block {b} ldg', dict(NFX_OPT_K2_VARIANT=1, NFX_OPT_K2_UNROLL=a, NFX_OPT_K2_BLOCK=b))
            for a, b in K2_PAIRS]
    if dtype == numpy.float32:
        out += [(f'alu {m:#x}', dict(NFX_OPT_K2_ALU_MASK=m)) for m in (0, 0x01, 0x09, 0x15, 0x1f)]
    else:
        out += [(f'tma {c}', dict(NFX_OPT_K2_VARIANT=2, NFX_OPT_K2_UNROLL=c)) for c in range(9)]
    return out


@pytest.mark.parametrize('nz', [7, 17])
@pytest.mark.parametrize('dtype', [numpy.float64, numpy.float32])
def test_every_k2_and_fused_instance(gpu, oracle, grid, dtype, nz):
    """with NaN, denormals, the fill marker and +-inf in u/v: every K2 instance's edge fluxes equal
    oracle.edgeflux_step_c bit for bit and its two-launch series the default one; every fused shape's series equals
    the default fused series bit for bit"""
    import torch
    from nemoflux_b200 import _lib
    nt, ncell = 3, NX * NY
    p, _ = _checked_handle(gpu, oracle, grid['P'], NY, NX, TRANSECTS)
    rng = numpy.random.default_rng(77 + nz)
    u, v = _data(rng, dtype, (nt, nz, ncell)), _data(rng, dtype, (nt, nz, ncell))
    u[:, 2, 100:104] = numpy.inf                            # a few columns: the ALU path's re-do loop
    v[:, nz - 1, 900:902] = -numpy.inf
    th = rng.uniform(0.5, 30.0, nz)
    a1, a2 = grid['arc1'], grid['arc2']
    want = numpy.stack([numpy.concatenate(oracle.edgeflux_step_c(u[t].reshape(nz, NY, NX), v[t].reshape(nz, NY, NX),
                                                                 th, a1, a2, True, FILL, want_iV=False)[1:])
                        for t in range(nt)])
    assert numpy.isinf(want).any() and numpy.isfinite(want).mean() > 0.99
    dev = lambda x: torch.from_numpy(numpy.ascontiguousarray(x)).to('cuda')   # noqa: E731
    dargs = (dev(u), dev(v), dev(th), dev(a1), dev(a2))
    kw = dict(fill=FILL, sverdrup=True)
    defaults = {n: _lib.get_option(getattr(_lib, n)) for n in OPTIONS}
    _option('NFX_OPT_FAST_SERIES', 0)
    base = _np(p.fluxSeries(*dargs, **kw))
    assert numpy.isfinite(base).any()
    for name, opts in [('default', {})] + _k2_configs(dtype):
        for k, val in opts.items():
            _option(k, val)
        ef = torch.zeros((nt, 2 * ncell), dtype=torch.float64, device='cuda')
        ser = p.fluxSeries(*dargs, eflux=ef, **kw)
        _same(ef, want, (name, 'eflux'))
        _same(ser, base, (name, 'series'))
        _same(p.fluxSeries(*dargs, **kw), base, (name, 'series, internal eflux'))
        for k in opts:
            _option(k, defaults[k])
    _option('NFX_OPT_FAST_SERIES', 2)
    fused = _np(p.fluxSeries(*dargs, **kw))
    for k, vals in (('NFX_OPT_FUSED_F32_SHAPE', (43, 45, 83, 85)), ('NFX_OPT_FUSED_F64_CTAS', (2, 3, 4))):
        for val in vals:
            _option(k, val)
            _same(p.fluxSeries(*dargs, **kw), fused, (k, val))
            for layered in ([0, nz], [1, 3, nz]):
                _option(k, defaults[k])
                ref = _np(p.fluxSeries(*dargs, layers=layered, **kw))
                _option(k, val)
                _same(p.fluxSeries(*dargs, layers=layered, **kw), ref, (k, val, layered))
        _option(k, defaults[k])
