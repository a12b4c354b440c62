"""-m gpu: the CUDA path (through the C ABI) against the CPU oracle on the same inputs.

Bars: intersected-edge lists bit-exact (cell, segment, image ids equal; ta, tb, coefficient, parametric
coordinates and weights equal bit for bit); K2 bit-exact against the sequential C restatement and
<= 1e-12 against the reference's numpy formulation; flux series <= 1e-12 relative to sum |w*f|.
"""
import os

import numpy
import pytest

from helpers import (README_C1, README_C2, README_LOOP, README_SINGULAR, SF_C2, assert_bitwise, random_transects, tr)

pytestmark = pytest.mark.gpu

FLUX_RTOL = 1.e-12      # north star: fluxes agree to fp64 relative error <= 1e-12


def _build(gpu, points, ny=None, nx=None, periodX=360.):
    g = gpu.Grid()
    g.setPoints(points)
    if ny:
        g.setCGridShape(ny, nx)
    p = gpu.PolylineIntegral()
    p.build(g, periodX=periodX)
    return g, p


def _check_lists(oracle, gpu_pli, ogrid, transects, periodX=360., counterclock=False):
    s = gpu_pli.getSubsegments()
    mp = gpu_pli.getMap()
    assert len(s['offsets']) == len(transects) + 1
    total = 0
    for m, xyz in enumerate(transects):
        op = oracle.PolylineIntegral(ogrid, periodX)
        op.computeWeights(xyz, counterclock=counterclock)
        o = op.subsegs
        a, b = s['offsets'][m], s['offsets'][m + 1]
        assert b - a == len(o), f'transect {m}: {b - a} sub-segments on the GPU, {len(o)} in the oracle'
        assert numpy.array_equal(s['cell'][a:b], o['cell']), f'transect {m}: cell ids differ'
        assert numpy.array_equal(s['seg'][a:b], o['seg'])
        assert numpy.array_equal(s['img'][a:b], o['img'])
        for k in ('ta', 'tb', 'coeff', 'xia', 'xib', 'w'):
            assert_bitwise(s[k][a:b], o[k], f'transect {m} {k}')
        keys, ws = op.merged_map()
        ma, mb = mp['offsets'][m], mp['offsets'][m + 1]
        assert numpy.array_equal(mp['keys'][ma:mb], keys), f'transect {m}: map keys differ'
        assert_bitwise(mp['w'][ma:mb], ws, f'transect {m} map weights')
        # getWeights view
        cells, edges, w = gpu_pli.getWeights(m)
        oc, oe, ow = op.emission_list()
        assert numpy.array_equal(cells, oc) and numpy.array_equal(edges, oe)
        assert_bitwise(w, ow, 'emission weights')
        total += len(o)
    return total


# ---------------------------------------------------------------------------------------------------
# K1
# ---------------------------------------------------------------------------------------------------
def test_k1_c1_list_bit_exact(gpu, oracle):
    g = oracle.DataGen()
    P = g.points()
    _, p = _build(gpu, P, g.ny, g.nx)
    xyz = tr(README_C1)
    p.computeWeights(xyz)
    n = _check_lists(oracle, p, oracle.Grid(P), [xyz])
    assert n == 59
    s = p.getSubsegments()
    assert list(numpy.bincount(s['seg'])) == [6, 15, 14, 12, 12]
    assert list(s['cell'][:6]) == [72, 108, 144, 181, 217, 253]       # SURVEY appendix A


@pytest.mark.parametrize('delta', [(0., 0.), (20., 30.)])
def test_k1_random_transects_bit_exact(gpu, oracle, delta):
    g = oracle.DataGen(nx=90, ny=45, deltaDeg=delta)
    P = g.points()
    rng = numpy.random.default_rng(1234)
    nodes = numpy.stack([g.xx, g.yy], -1) if delta == (0., 0.) else None
    transects = random_transects(rng, 24, nodes=nodes)
    transects += [tr(README_C1), tr(README_SINGULAR), tr(README_LOOP), tr(README_C2)]
    # along grid lines (duplicate sub-segments, coefficient 0/1), across the date line, degenerate pieces
    transects += [tr([(-180, -40), (180, -40)]), tr([(-60, -80), (-60, 80)]), tr([(170, 10), (190, 20)]),
                  tr([(-190, -10), (-170, 5)]), tr([(10, 10), (10, 10)]), tr([(10, 10)]), tr([(0, 0), (4, 4), (4, 4), (8, 0)])]
    _, p = _build(gpu, P, g.ny, g.nx)
    p.computeWeights(transects)
    n = _check_lists(oracle, p, oracle.Grid(P), transects)
    assert n > 1000


def test_k1_real_nemo_grid_bit_exact(gpu, oracle):
    """the reference's real NEMO T grid (data/sa/T.nc, a 100 x 100 ORCA025 window, committed as
    tests/golden/sa_T_grid.npz) with the reference's transect data/sa/S3_sa.txt, transects along its grid lines and
    random ones: lists bit for bit against the oracle; a nodal stream function integrates to psi(B) - psi(A)"""
    import os
    import torch
    from conftest import GOLDEN
    g = numpy.load(os.path.join(GOLDEN, 'sa_T_grid.npz'))
    lon, lat = g['bounds_lon'].astype(numpy.float64), g['bounds_lat'].astype(numpy.float64)
    P = numpy.zeros((100, 100, 4, 3))
    P[..., 0], P[..., 1] = lon, lat
    P = P.reshape(-1, 4, 3)
    rng = numpy.random.default_rng(31)
    transects = [tr([(16., -40.4), (28., -34.5), (31., -28.5), (36., -30.5)])]                 # data/sa/S3_sa.txt:5-8
    transects += random_transects(rng, 12, lon_range=(13., 37.), lat_range=(-41., -21.5))
    transects += [tr([(lon[10, 3, 0], lat[10, 3, 0]), (lon[10, 90, 0], lat[10, 90, 0])]),        # along a grid line
                  tr([(lon[5, 40, 0], lat[5, 40, 0]), (lon[95, 40, 0], lat[95, 40, 0])]),
                  tr([(5., -30.), (45., -30.)])]                                                # enters and leaves the window
    nodes = []
    for _ in range(6):
        ja, ia, jb, ib = (int(v) for v in rng.integers(5, 95, 4))
        a, b = (lon[ja, ia, 0], lat[ja, ia, 0]), (lon[jb, ib, 0], lat[jb, ib, 0])
        transects.append(tr([a, (float(rng.uniform(15., 35.)), float(rng.uniform(-39., -23.))), b]))
        nodes.append((a, b))
    _, p = _build(gpu, P, 100, 100)
    p.computeWeights(transects)
    n = _check_lists(oracle, p, oracle.Grid(P), transects)
    assert n > 1500

    def psi(x, y):
        return numpy.sin(numpy.radians(3 * x)) * (y + 45.) + 0.01 * x * y
    se, ne, nw = psi(lon[..., 1], lat[..., 1]), psi(lon[..., 2], lat[..., 2]), psi(lon[..., 3], lat[..., 3])
    # compact edge fluxes [eU | eV] (field.py:195-196: east edge, north edge) of the nodal stream function
    ef = torch.from_numpy(numpy.concatenate([(ne - se).reshape(-1), (ne - nw).reshape(-1)])[None]).cuda()
    series = p.integrate(ef).cpu().numpy()[0]
    for k, (a, b) in enumerate(nodes):
        exact = psi(*b) - psi(*a)
        assert abs(series[len(transects) - 6 + k] - exact) <= 1e-10 * max(1.0, abs(exact))


def test_k1_record_list_and_fallback_agree(gpu, oracle):
    """the count pass records its hits so that the fill pass is a scatter; when the record list (sized from the
    previous call on the handle) is too small the fill pass traverses again -- same lists either way"""
    g = oracle.DataGen(nx=720, ny=360)
    P = g.points()
    long_tr = [tr([(-179.3, -80.2), (178.9, 79.7)]), tr([(-100, 60), (120, -70), (150, 10)])]
    _, p1 = _build(gpu, P, g.ny, g.nx)
    p1.computeWeights(long_tr)                                  # first call: list sized from the geometry
    a = p1.getSubsegments()
    _, p2 = _build(gpu, P, g.ny, g.nx)
    p2.computeWeights([tr([(10.2, 10.1), (10.9, 10.4)])])       # a handful of sub-segments -> a tiny hint
    p2.computeWeights(long_tr)                                  # list overflows -> second traversal
    b = p2.getSubsegments()
    assert len(a['cell']) > 1500
    for key in ('offsets', 'cell', 'seg', 'ta', 'tb', 'coeff', 'w'):
        assert numpy.array_equal(a[key], b[key]), key
    p2.computeWeights(long_tr)                                  # now the hint fits: record path again
    c = p2.getSubsegments()
    for key in ('cell', 'ta', 'w'):
        assert numpy.array_equal(a[key], c[key]), key
    _check_lists(oracle, p1, oracle.Grid(P), long_tr)


def test_k1_counterclock_and_no_period(gpu, oracle):
    g = oracle.DataGen(nx=36, ny=18)
    P = g.points()
    xyz = tr(README_C1)
    _, p = _build(gpu, P, periodX=0.)
    p.computeWeights(xyz, counterclock=True)
    _check_lists(oracle, p, oracle.Grid(P), [xyz], periodX=0., counterclock=True)


def test_k1_filter_is_superset(gpu, oracle):
    """the oracle's brute force (no candidate filter) agrees with the GPU's bounding-box traversal"""
    g = oracle.DataGen(nx=48, ny=24, deltaDeg=(20., 30.))
    P = g.points()
    rng = numpy.random.default_rng(7)
    transects = random_transects(rng, 6)
    _, p = _build(gpu, P)
    p.computeWeights(transects)
    s = p.getSubsegments()
    og = oracle.Grid(P)
    for m, xyz in enumerate(transects):
        ob = oracle.PolylineIntegral(og, 360., filter_mode=0)
        ob.computeWeights(xyz)
        a, b = s['offsets'][m], s['offsets'][m + 1]
        assert numpy.array_equal(s['cell'][a:b], ob.subsegs['cell'])
        assert_bitwise(s['w'][a:b], ob.subsegs['w'], 'weights vs brute force')


def test_k1_empty_and_errors(gpu, oracle):
    g = oracle.DataGen()
    grid, p = _build(gpu, g.points())
    p.computeWeights([])
    assert p.getNumberOfTransects() == 0
    assert p.getSubsegments()['cell'].size == 0
    # a transect entirely outside the grid gives no sub-segments and integral 0
    p.computeWeights(tr([(0, 100), (10, 120)]))
    assert p.getSubsegments()['cell'].size == 0
    assert p.getIntegral(numpy.ones((grid.getNumberOfCells(), 4))) == 0.0
    with pytest.raises(ValueError):
        p.computeWeights(numpy.zeros((3, 2)))
    with pytest.raises(ValueError):
        p.getIntegral(numpy.ones(5))
    q = gpu.PolylineIntegral()
    with pytest.raises(RuntimeError):
        q.computeWeights(tr(README_C1))          # setGrid/buildLocator missing
    with pytest.raises(RuntimeError):
        q.buildLocator()


# ---------------------------------------------------------------------------------------------------
# K2
# ---------------------------------------------------------------------------------------------------
def _rand_uv(rng, nt, nz, ny, nx, dtype, nan_frac=0.2):
    u = rng.standard_normal((nt, nz, ny, nx)).astype(dtype)
    v = rng.standard_normal((nt, nz, ny, nx)).astype(dtype)
    u[rng.random(u.shape) < nan_frac] = numpy.nan
    v[rng.random(v.shape) < nan_frac] = numpy.nan
    return u, v


@pytest.mark.parametrize('shape', [(3, 7, 9, 11), (2, 75, 12, 20), (2, 5, 10, 13), (4, 10, 16, 32), (1, 1, 3, 5)])
@pytest.mark.parametrize('dtype', [numpy.float64, numpy.float32])
@pytest.mark.parametrize('sverdrup', [False, True])
def test_k2_bit_exact_vs_sequential_oracle(gpu, oracle, shape, dtype, sverdrup):
    import torch
    nt, nz, ny, nx = shape
    rng = numpy.random.default_rng(nt * 1000 + nz * 10 + nx)
    u, v = _rand_uv(rng, nt, nz, ny, nx, dtype)
    th = rng.uniform(0.5, 20., nz)
    arc1 = rng.uniform(1e-3, 2e-2, ny * nx)
    arc2 = rng.uniform(1e-3, 2e-2, ny * nx)
    d = 'cuda'
    ef = gpu.edgeFluxAssemble(torch.from_numpy(u).to(d), torch.from_numpy(v).to(d), torch.from_numpy(th).to(d),
                              torch.from_numpy(arc1).to(d), torch.from_numpy(arc2).to(d), sverdrup=sverdrup)
    iv = gpu.edgeFluxToCellByCell(ef, ny, nx).cpu().numpy()
    efh = ef.cpu().numpy()
    for t in range(nt):
        iV, eU, eV = oracle.edgeflux_step_c(u[t], v[t], th, arc1, arc2, sverdrup)
        assert_bitwise(efh[t, :ny * nx], eU, f'eU t={t}')
        assert_bitwise(efh[t, ny * nx:], eV, f'eV t={t}')
        assert_bitwise(iv[t], iV, f'iV t={t}')
        # the reference's numpy formulation (tensordot) differs only by summation order
        U = oracle.read_field(u[t].astype(numpy.float64), th)
        V = oracle.read_field(v[t].astype(numpy.float64), th)
        arc = numpy.zeros((ny * nx, 4))
        arc[:, 1], arc[:, 2] = arc1, arc2
        iVn, _, _ = oracle.integrated_flux(U, V, arc, sverdrup)
        scale = numpy.abs(iVn).max() + 1e-300
        assert numpy.abs(iv[t] - iVn).max() <= 1e-13 * scale * nz
    assert gpu.edgeFluxAbsMax(ef) == numpy.abs(efh).max()


@pytest.mark.parametrize('thick_max', [20., 2.0e31])
@pytest.mark.parametrize('shape', [(2, 75, 16, 32), (2, 12, 9, 11)])
def test_k2_f32_special_values(gpu, oracle, shape, thick_max):
    """float32 storage takes the bit-shuffle conversion (clean_scaled): denormals, signed zeros, FLT_MAX, the
    smallest normals and infinities must give the bits of the plain (double)x path; thickness >= 2^100 too"""
    import torch
    nt, nz, ny, nx = shape
    rng = numpy.random.default_rng(99)
    u, v = _rand_uv(rng, nt, nz, ny, nx, numpy.float32)
    for a in (u, v):
        r = rng.random(a.shape)
        a[r < 0.02] = 0.0
        a[(r >= 0.02) & (r < 0.04)] = -0.0
        a[(r >= 0.04) & (r < 0.07)] = numpy.float32(1.0e-41)
        a[(r >= 0.07) & (r < 0.09)] = numpy.float32(-1.4e-45)
        a[(r >= 0.09) & (r < 0.11)] = numpy.finfo(numpy.float32).max
        a[(r >= 0.11) & (r < 0.13)] = -numpy.finfo(numpy.float32).tiny
        a[(r >= 0.13) & (r < 0.1305)] = numpy.inf
        a[(r >= 0.1305) & (r < 0.131)] = -numpy.inf
    th = rng.uniform(0.5, thick_max, nz)
    arc1 = rng.uniform(1e-3, 2e-2, ny * nx)
    arc2 = rng.uniform(1e-3, 2e-2, ny * nx)
    d = 'cuda'
    from nemoflux_b200 import _lib
    dev_args = [torch.from_numpy(x).to(d) for x in (u, v, th, arc1, arc2)]
    efh = gpu.edgeFluxAssemble(*dev_args).cpu().numpy()                    # 128-bit loads (the float32 default)
    try:
        _lib.set_option(_lib.NFX_OPT_K2_VARIANT, _lib.NFX_K2_LDG)         # widest loads: float x 8
        assert_bitwise_nan = gpu.edgeFluxAssemble(*dev_args).cpu().numpy()
    finally:
        _lib.set_option(_lib.NFX_OPT_K2_VARIANT, _lib.NFX_K2_AUTO)
    assert numpy.array_equal(assert_bitwise_nan, efh, equal_nan=True)
    if thick_max < 1.e30:
        # the same special values through the e3u/e3v path (both factors float32, bit shuffle + exact rescale):
        # e3 == dz[k] must reproduce the 1-D thickness result bit for bit
        th32 = th.astype(numpy.float32)
        e3 = torch.from_numpy(numpy.ascontiguousarray(numpy.broadcast_to(th32[None, :, None], (1, nz, ny * nx)))).to(d)
        ref_1d = gpu.edgeFluxAssemble(dev_args[0], dev_args[1], torch.from_numpy(th32.astype(numpy.float64)).to(d),
                                      dev_args[3], dev_args[4]).cpu().numpy()
        got_e3 = gpu.edgeFluxAssemble(dev_args[0].reshape(nt, nz, -1), dev_args[1].reshape(nt, nz, -1), None,
                                      dev_args[3], dev_args[4], e3u=e3, e3v=e3).cpu().numpy()
        assert numpy.array_equal(got_e3, ref_1d, equal_nan=True)
    ninf = 0
    for t in range(nt):
        with numpy.errstate(all='ignore'):
            _, eU, eV = oracle.edgeflux_step_c(u[t], v[t], th, arc1, arc2, False, want_iV=False)
        ref = numpy.concatenate([eU, eV])
        nan = numpy.isnan(ref)
        assert numpy.array_equal(nan, numpy.isnan(efh[t]))      # inf - inf: NaN on both sides (payload is not compared)
        assert_bitwise(numpy.where(nan, 0., efh[t]), numpy.where(nan, 0., ref), f't={t}')
        ninf += int(numpy.isinf(ref).sum() + nan.sum())
    assert ninf > 0


def test_k2_fill_value(gpu, oracle):
    import torch
    rng = numpy.random.default_rng(5)
    u, v = _rand_uv(rng, 2, 6, 8, 10, numpy.float64, nan_frac=0.)
    u[rng.random(u.shape) < 0.3] = 1.e20       # raw _FillValue of datagen.py:191
    v[rng.random(v.shape) < 0.3] = 1.e20
    th = rng.uniform(1., 2., 6)
    a1 = rng.uniform(.01, .02, 80)
    a2 = rng.uniform(.01, .02, 80)
    d = 'cuda'
    ef = gpu.edgeFluxAssemble(torch.from_numpy(u).to(d), torch.from_numpy(v).to(d), torch.from_numpy(th).to(d),
                              torch.from_numpy(a1).to(d), torch.from_numpy(a2).to(d), fill=1.e20).cpu().numpy()
    for t in range(2):
        _, eU, eV = oracle.edgeflux_step_c(u[t], v[t], th, a1, a2, False, fill=1.e20)
        assert_bitwise(ef[t, :80], eU)
        assert_bitwise(ef[t, 80:], eV)
    assert numpy.abs(ef).max() < 1e3


def test_k2_golden_reference_outputs(gpu):
    """inputs/outputs produced by the reference's own Field.readField/computeIntegratedFlux code"""
    import torch
    from conftest import GOLDEN
    d = 'cuda'
    for ti in (0, 1):
        for sv in (0, 1):
            g = numpy.load(os.path.join(GOLDEN, f'rot24x12_t{ti}_sv{sv}.npz'))
            u, v = g['u'], g['v']                      # (nt, nz, ny, nx) with NaN land
            nt, nz, ny, nx = u.shape
            th = g['thickness']
            arc = g['arcLengths']
            ef = gpu.edgeFluxAssemble(torch.from_numpy(u).to(d), torch.from_numpy(v).to(d),
                                      torch.from_numpy(th).to(d), torch.from_numpy(arc[:, 1].copy()).to(d),
                                      torch.from_numpy(arc[:, 2].copy()).to(d), sverdrup=bool(sv))
            iv = gpu.edgeFluxToCellByCell(ef, ny, nx).cpu().numpy()[ti]
            ref = g['iV']
            assert numpy.abs(iv - ref).max() <= 1e-13 * numpy.abs(ref).max()
            efh = ef.cpu().numpy()[ti]
            assert numpy.allclose(numpy.abs(efh[:ny * nx]), g['absEU'], rtol=1e-13, atol=0)
            assert abs(gpu.edgeFluxAbsMax(ef[ti:ti + 1]) - float(g['maxAbsFlux'])) <= 1e-13 * float(g['maxAbsFlux'])


# ---------------------------------------------------------------------------------------------------
# K3 and the whole path
# ---------------------------------------------------------------------------------------------------
def _series_gpu(gpu, P, ny, nx, transects, u, v, th, arc, sverdrup=False, order='map', host=False):
    import torch
    _, p = _build(gpu, P, ny, nx)
    p.computeWeights(transects)
    if host:
        return p, p.fluxSeries(u, v, th, arc[:, 1].copy(), arc[:, 2].copy(), sverdrup=sverdrup, order=order,
                               chunk_steps=3)
    d = 'cuda'
    out = p.fluxSeries(torch.from_numpy(u).to(d), torch.from_numpy(v).to(d), torch.from_numpy(th).to(d),
                       torch.from_numpy(arc[:, 1].copy()).to(d), torch.from_numpy(arc[:, 2].copy()).to(d),
                       sverdrup=sverdrup, order=order)
    return p, out.cpu().numpy()


def _l1_scale(oracle, P, transects, u, v, th, arc, sverdrup):
    """sum |w*f| per (t, transect): the scale against which flux errors are measured"""
    og = oracle.Grid(P)
    nt = u.shape[0]
    out = numpy.zeros((nt, len(transects)))
    plis = []
    for xyz in transects:
        op = oracle.PolylineIntegral(og)
        op.computeWeights(xyz)
        plis.append(op.merged_map())
    for t in range(nt):
        iV, _, _ = oracle.edgeflux_step_c(u[t], v[t], th, arc[:, 1].copy(), arc[:, 2].copy(), sverdrup)
        f = iV.reshape(-1)
        for m, (keys, ws) in enumerate(plis):
            out[t, m] = numpy.abs(ws * f[keys]).sum()
    return out


def test_known_answers_readme(gpu, oracle):
    # README.md:26-39: 360
    g = oracle.DataGen()
    P, arc = g.points(), oracle.arc_lengths(g.points())
    u, v = g.uv('x')
    _, s = _series_gpu(gpu, P, g.ny, g.nx, [tr(README_C1)], u, v, g.thickness(), arc)
    assert abs(s[0, 0] - 360.) <= 1e-12 * 360.
    # README.md:50-56: 0.5, node to node around a singular stream function
    u, v = g.uv('arctan2(y, x+180)/(2*pi)')
    _, s = _series_gpu(gpu, P, g.ny, g.nx, [tr(README_SINGULAR)], u, v, g.thickness(), arc)
    assert abs(s[0, 0] - 0.5) <= 2e-15
    # README.md:65-68: closed loop, zero to machine accuracy
    g = oracle.DataGen(nx=360, ny=180)
    P, arc = g.points(), oracle.arc_lengths(g.points())
    u, v = g.uv('cos(2*pi*y/360) + sin(2*pi*x/360)')
    _, s = _series_gpu(gpu, P, g.ny, g.nx, [tr(README_LOOP)], u, v, g.thickness(), arc)
    assert abs(s[0, 0]) <= 1e-13


@pytest.mark.parametrize('order', ['map', 'list'])
@pytest.mark.parametrize('sverdrup', [False, True])
def test_flux_series_vs_oracle(gpu, oracle, order, sverdrup):
    g = oracle.DataGen(nx=72, ny=36, nz=5, nt=4, deltaDeg=(20., 30.))
    P, arc = g.points(), oracle.arc_lengths(g.points())
    u, v = g.uv(SF_C2)
    rng = numpy.random.default_rng(99)
    land = rng.random((g.nz, g.ny, g.nx)) < 0.15
    u[:, land] = numpy.nan
    v[:, land] = numpy.nan
    transects = random_transects(rng, 12) + [tr(README_C2), tr(README_LOOP)]
    th = g.thickness()
    ref = oracle.flux_series(P, transects, u, v, th, sverdrup=sverdrup, order=order)
    refc = oracle.flux_series(P, transects, u, v, th, sverdrup=sverdrup, order=order, use_c=True)
    scale = _l1_scale(oracle, P, transects, u, v, th, arc, sverdrup)
    p, s = _series_gpu(gpu, P, g.ny, g.nx, transects, u, v, th, arc, sverdrup=sverdrup, order=order)
    assert s.shape == ref.shape == (4, 14)
    assert (numpy.abs(s - ref) <= FLUX_RTOL * scale + 1e-300).all()
    assert (numpy.abs(s - refc) <= FLUX_RTOL * scale + 1e-300).all()
    # the host-buffer entry point (double-buffered staging) gives the same numbers as the device one
    _, sh = _series_gpu(gpu, P, g.ny, g.nx, transects, u, v, th, arc, sverdrup=sverdrup, order=order, host=True)
    assert numpy.array_equal(sh, s)
    # mint-style getIntegral on the (ncell,4) array of one time step
    iV, _, _ = oracle.edgeflux_step_c(u[1], v[1], th, arc[:, 1].copy(), arc[:, 2].copy(), sverdrup)
    one = p.getIntegral(iV, order=order)
    assert (numpy.abs(one - ref[1]) <= FLUX_RTOL * scale[1] + 1e-300).all()


def test_c2_series_linear_in_time(gpu, oracle):
    """BASELINE config 2 (README.md:89-91): flux(t) = flux(0)*(t+1)"""
    g = oracle.DataGen(nx=360, ny=180, nz=10, nt=20, deltaDeg=(20., 30.))
    P, arc = g.points(), oracle.arc_lengths(g.points())
    u, v = g.uv(SF_C2)
    p, s = _series_gpu(gpu, P, g.ny, g.nx, [tr(README_C2)], u, v, g.thickness(), arc)
    assert p.getSubsegments()['cell'].size == 361
    ref = oracle.flux_series(P, [tr(README_C2)], u, v, g.thickness())
    assert numpy.abs(s - ref).max() <= 1e-12 * numpy.abs(ref).max()
    assert numpy.allclose(s[:, 0] / s[0, 0], numpy.arange(1, 21), rtol=1e-12)
    assert abs(s[0, 0] - 1.7386322852896516) <= 1e-11


@pytest.mark.parametrize('cfg', [0, 2, 3, 6, 7])
def test_k2_tma_variant_bit_exact(gpu, oracle, cfg):
    """the TMA (cp.async.bulk) staged variant gives the same bits as the direct-load kernel and the oracle,
    including ragged tiles (ncell not a multiple of the tile) and a level count that is no multiple of KL"""
    import torch
    from nemoflux_b200 import _lib
    rng = numpy.random.default_rng(17 + cfg)
    d = 'cuda'
    try:
        for (nt, nz, ny, nx) in [(3, 75, 26, 42), (2, 7, 9, 14), (5, 16, 40, 64), (1, 1, 2, 3)]:
            u, v = _rand_uv(rng, nt, nz, ny, nx, numpy.float64)
            th = rng.uniform(0.5, 20., nz)
            a1 = rng.uniform(1e-3, 2e-2, ny * nx)
            a2 = rng.uniform(1e-3, 2e-2, ny * nx)
            args = [torch.from_numpy(x).to(d) for x in (u, v, th, a1, a2)]
            _lib.set_option(_lib.NFX_OPT_K2_VARIANT, _lib.NFX_K2_TMA)
            _lib.set_option(_lib.NFX_OPT_K2_UNROLL, cfg)
            ef = gpu.edgeFluxAssemble(*args, sverdrup=True).cpu().numpy()
            _lib.set_option(_lib.NFX_OPT_K2_VARIANT, _lib.NFX_K2_LDG)
            _lib.set_option(_lib.NFX_OPT_K2_UNROLL, 0)
            ef2 = gpu.edgeFluxAssemble(*args, sverdrup=True).cpu().numpy()
            assert_bitwise(ef, ef2, 'TMA vs LDG')
            for t in range(nt):
                _, eU, eV = oracle.edgeflux_step_c(u[t], v[t], th, a1, a2, True)
                assert_bitwise(ef[t, :ny * nx], eU, 'eU')
                assert_bitwise(ef[t, ny * nx:], eV, 'eV')
    finally:
        _lib.set_option(_lib.NFX_OPT_K2_VARIANT, _lib.NFX_K2_AUTO)
        _lib.set_option(_lib.NFX_OPT_K2_UNROLL, 0)


@pytest.mark.parametrize('slot_mb,shape', [(16, (72, 36, 5, 9)), (1, (300, 250, 3, 5)), (1, (64, 40, 4, 70))])
def test_fast_series_path_matches_classic(gpu, oracle, slot_mb, shape):
    """nfx_flux_series with eflux == NULL (edge fluxes kept in an L2-resident ring, time batches or cell panels on
    two streams) against the classic K2 -> HBM -> K3 path and the oracle; a 1 MB ring slot forces several panels"""
    import torch
    from nemoflux_b200 import _lib
    nx, ny, nz, nt = shape
    g = oracle.DataGen(nx=nx, ny=ny, nz=nz, nt=nt, deltaDeg=(20., 30.))
    P, arc = g.points(), oracle.arc_lengths(g.points())
    u, v = g.uv(SF_C2)
    rng = numpy.random.default_rng(5)
    land = rng.random((nz, ny, nx)) < 0.1
    u[:, land] = numpy.nan
    v[:, land] = numpy.nan
    transects = random_transects(rng, 9) + [tr(README_C2), tr(README_LOOP), tr([(-180, -40), (180, -40)])]
    th = g.thickness()
    d = 'cuda'
    _, p = _build(gpu, P, ny, nx)
    p.computeWeights(transects)
    args = [torch.from_numpy(x).to(d) for x in (u, v, th, arc[:, 1].copy(), arc[:, 2].copy())]
    try:
        _lib.set_option(_lib.NFX_OPT_RING_SLOT_MB, slot_mb)
        _lib.set_option(_lib.NFX_OPT_FAST_SERIES, 2)           # always the fused pass, also with several panels
        for order in ('map', 'list'):
            fast = p.fluxSeries(*args, order=order).cpu().numpy()
            fast2 = p.fluxSeries(*args, order=order).cpu().numpy()
            assert numpy.array_equal(fast, fast2)                      # deterministic run to run
            ef = torch.empty((nt, 2 * ny * nx), dtype=torch.float64, device=d)
            classic = p.fluxSeries(*args, order=order, eflux=ef).cpu().numpy()
            scale = _l1_scale(oracle, P, transects, u, v, th, arc, False)
            assert (numpy.abs(fast - classic) <= 1e-13 * scale + 1e-300).all()
            ref = oracle.flux_series(P, transects, u, v, th, order=order, use_c=True)
            assert (numpy.abs(fast - ref) <= FLUX_RTOL * scale + 1e-300).all()
            # the eflux the classic path returns is the K2 output
            _, eU, eV = oracle.edgeflux_step_c(u[nt - 1], v[nt - 1], th, arc[:, 1].copy(), arc[:, 2].copy(), False)
            assert_bitwise(ef[nt - 1].cpu().numpy(), numpy.concatenate([eU, eV]), 'eflux')
            host = p.fluxSeries(u, v, th, arc[:, 1].copy(), arc[:, 2].copy(), order=order, chunk_steps=4)
            assert numpy.array_equal(host, fast)
            # big-endian host buffers (a NetCDF classic file as stored): swapped on the device, same bits
            host_be = p.fluxSeries(u.astype('>f8'), v.astype('>f8'), th, arc[:, 1].copy(), arc[:, 2].copy(),
                                   order=order, chunk_steps=4)
            assert numpy.array_equal(host_be, host)
            h32 = p.fluxSeries(u.astype('<f4'), v.astype('<f4'), th, arc[:, 1].copy(), arc[:, 2].copy(),
                               order=order, chunk_steps=3)
            h32_be = p.fluxSeries(u.astype('>f4'), v.astype('>f4'), th, arc[:, 1].copy(), arc[:, 2].copy(),
                                  order=order, chunk_steps=3)
            assert numpy.array_equal(h32_be, h32)
    finally:
        _lib.set_option(_lib.NFX_OPT_RING_SLOT_MB, 0)      # back to automatic
        _lib.set_option(_lib.NFX_OPT_FAST_SERIES, 1)


@pytest.mark.parametrize('dtype', [numpy.float64, numpy.float32])
def test_padded_level_planes(gpu, oracle, dtype):
    """u/v stored with padded level planes (ld > ncell, 32-byte aligned rows): same bits as the dense layout,
    through K2 alone, the two-launch series and the fused series (several panels forced by a 1 MB ring slot)"""
    import torch
    from nemoflux_b200 import _lib
    nx, ny, nz, nt = 301, 251, 4, 5                 # ncell = 75551, odd
    g = oracle.DataGen(nx=nx, ny=ny, nz=nz, nt=nt, deltaDeg=(20., 30.))
    P, arc = g.points(), oracle.arc_lengths(g.points())
    u, v = g.uv(SF_C2)
    u, v = u.astype(dtype), v.astype(dtype)
    u[:, :, 100:120, 50:90] = numpy.nan
    if dtype == numpy.float32:                  # denormals and signed zeros through the bit-shuffle conversion
        u[:, ::2, 10:14, 5:25] = numpy.float32(1.0e-41)
        v[:, ::3, 30:34, 5:25] = numpy.float32(-0.0)
        v[:, 1::3, 30:34, 5:25] = -numpy.finfo(numpy.float32).tiny
    ncell = nx * ny
    pad = 4 if dtype == numpy.float64 else 8
    ld = (ncell + pad - 1) // pad * pad
    d = 'cuda'
    tdt = torch.float64 if dtype == numpy.float64 else torch.float32
    up = torch.full((nt, nz, ld), 7.0, dtype=tdt, device=d)[:, :, :ncell]
    vp = torch.full((nt, nz, ld), 7.0, dtype=tdt, device=d)[:, :, :ncell]
    up.copy_(torch.from_numpy(u.reshape(nt, nz, ncell)))
    vp.copy_(torch.from_numpy(v.reshape(nt, nz, ncell)))
    th, a1, a2 = (torch.from_numpy(x).to(d) for x in (g.thickness(), arc[:, 1].copy(), arc[:, 2].copy()))
    dense = [torch.from_numpy(x).to(d) for x in (u, v)]
    ef_dense = gpu.edgeFluxAssemble(dense[0], dense[1], th, a1, a2).cpu().numpy()
    ef_pad = gpu.edgeFluxAssemble(up, vp, th, a1, a2).cpu().numpy()
    assert_bitwise(ef_pad, ef_dense, 'padded vs dense K2')
    transects = random_transects(numpy.random.default_rng(3), 6) + [tr(README_C2)]
    _, p = _build(gpu, P, ny, nx)
    p.computeWeights(transects)
    try:
        _lib.set_option(_lib.NFX_OPT_RING_SLOT_MB, 1)
        for mode in (0, 2):
            _lib.set_option(_lib.NFX_OPT_FAST_SERIES, mode)
            s_dense = p.fluxSeries(dense[0], dense[1], th, a1, a2).cpu().numpy()
            s_pad = p.fluxSeries(up, vp, th, a1, a2).cpu().numpy()
            assert numpy.array_equal(s_pad, s_dense)
            if mode == 2:                           # the visiting order of the batches cannot change a bit
                for order in (0, 1, 2):
                    _lib.set_option(_lib.NFX_OPT_FUSED_ORDER, order)
                    assert numpy.array_equal(p.fluxSeries(up, vp, th, a1, a2).cpu().numpy(), s_pad)
                _lib.set_option(_lib.NFX_OPT_FUSED_ORDER, 3)
        ref = oracle.flux_series(P, transects, u.astype(numpy.float64), v.astype(numpy.float64), g.thickness(), use_c=True)
        scale = _l1_scale(oracle, P, transects, u.astype(numpy.float64), v.astype(numpy.float64), g.thickness(), arc, False)
        assert (numpy.abs(s_pad - ref) <= FLUX_RTOL * scale + 1e-300).all()
    finally:
        _lib.set_option(_lib.NFX_OPT_RING_SLOT_MB, 0)      # back to automatic
        _lib.set_option(_lib.NFX_OPT_FAST_SERIES, 1)
        _lib.set_option(_lib.NFX_OPT_FUSED_ORDER, 3)
    with pytest.raises(ValueError):
        gpu.edgeFluxAssemble(up.transpose(0, 1), vp.transpose(0, 1), th, a1, a2)


def test_batch_range_partials_add_up(gpu, oracle):
    """balanced multi-GPU sharding, emulated on one GPU: every 'rank' runs its (time step, panel) batch range on
    the time steps it touches; the partial series add up to the full one"""
    import torch
    from nemoflux_b200 import _lib, dist
    nx, ny, nz, nt = 300, 250, 3, 7
    g = oracle.DataGen(nx=nx, ny=ny, nz=nz, nt=nt, deltaDeg=(20., 30.))
    P, arc = g.points(), oracle.arc_lengths(g.points())
    u, v = g.uv(SF_C2)
    transects = random_transects(numpy.random.default_rng(11), 7) + [tr(README_C2), tr(README_LOOP)]
    d = 'cuda'
    _, p = _build(gpu, P, ny, nx)
    p.computeWeights(transects)
    th, a1, a2 = (torch.from_numpy(x).to(d) for x in (g.thickness(), arc[:, 1].copy(), arc[:, 2].copy()))
    ud, vd = torch.from_numpy(u).to(d), torch.from_numpy(v).to(d)
    try:
        _lib.set_option(_lib.NFX_OPT_RING_SLOT_MB, 1)
        _lib.set_option(_lib.NFX_OPT_FAST_SERIES, 2)
        npanels, pc = p.getNumberOfPanels()
        assert npanels == 2 and pc % 1024 == 0
        full = p.fluxSeries(ud, vd, th, a1, a2).cpu().numpy()
        scale = _l1_scale(oracle, P, transects, u, v, g.thickness(), arc, False)
        for world in (1, 2, 3, 5):
            total = numpy.zeros_like(full)
            for r in range(world):
                s = dist.shard_batches(nt, npanels, world, r)
                t0, n = s['t_first'], s['nt_touched']
                if n == 0:
                    continue
                part = p.fluxSeries(ud[t0:t0 + n], vd[t0:t0 + n], th, a1, a2, batch_range=(s['b0'], s['b1']))
                total[t0:t0 + n] += part.cpu().numpy()
            assert (numpy.abs(total - full) <= 1e-13 * scale + 1e-300).all(), world
        # an empty range gives zeros, a bad one is refused
        z = p.fluxSeries(ud[:2], vd[:2], th, a1, a2, batch_range=(1, 1)).cpu().numpy()
        assert (z == 0).all()
        with pytest.raises(RuntimeError):
            p.fluxSeries(ud[:2], vd[:2], th, a1, a2, batch_range=(0, 2 * npanels + 1))
    finally:
        _lib.set_option(_lib.NFX_OPT_RING_SLOT_MB, 0)      # back to automatic
        _lib.set_option(_lib.NFX_OPT_FAST_SERIES, 1)


@pytest.mark.parametrize('dtype', [numpy.float64, numpy.float32])
@pytest.mark.parametrize('e3_nt', [1, 3])
def test_k2_per_column_scale_factors(gpu, oracle, dtype, e3_nt):
    """SURVEY 8f rank 4: e3u/e3v (per column and level, optionally per time step) instead of the 1-D thickness:
    bit-exact against the oracle's definition, and identical to the thickness path when e3[t,k,c] = dz[k]"""
    import torch
    nt, nz, ny, nx = 3, 11, 14, 22
    rng = numpy.random.default_rng(21)
    u, v = _rand_uv(rng, nt, nz, ny, nx, dtype)
    e3u = rng.uniform(0.5, 30., (e3_nt, nz, ny, nx)).astype(dtype)
    e3v = rng.uniform(0.5, 30., (e3_nt, nz, ny, nx)).astype(dtype)
    e3u[:, :, 3, 4] = numpy.nan                       # a missing scale factor counts as 0
    a1 = rng.uniform(1e-3, 2e-2, ny * nx)
    a2 = rng.uniform(1e-3, 2e-2, ny * nx)
    d = 'cuda'
    args = [torch.from_numpy(x).to(d) for x in (u, v)]
    a1d, a2d = torch.from_numpy(a1).to(d), torch.from_numpy(a2).to(d)
    ef = gpu.edgeFluxAssemble(args[0], args[1], None, a1d, a2d, sverdrup=True, e3u=torch.from_numpy(e3u).to(d),
                              e3v=torch.from_numpy(e3v).to(d)).cpu().numpy()
    for t in range(nt):
        te = 0 if e3_nt == 1 else t
        eU, eV = oracle.edgeflux_step_c_e3(u[t].astype(numpy.float64), v[t].astype(numpy.float64),
                                           e3u[te].astype(numpy.float64), e3v[te].astype(numpy.float64), a1, a2, True)
        assert_bitwise(ef[t, :ny * nx], eU, 'eU (e3)')
        assert_bitwise(ef[t, ny * nx:], eV, 'eV (e3)')
    # e3 = dz everywhere reproduces the reference's 1-D thickness path bit for bit
    th = rng.uniform(0.5, 20., nz).astype(dtype).astype(numpy.float64)
    e3c = numpy.broadcast_to(th.astype(dtype)[None, :, None, None], (1, nz, ny, nx)).copy()
    ef_e3 = gpu.edgeFluxAssemble(args[0], args[1], None, a1d, a2d, e3u=torch.from_numpy(e3c).to(d),
                                 e3v=torch.from_numpy(e3c).to(d)).cpu().numpy()
    ef_th = gpu.edgeFluxAssemble(args[0], args[1], torch.from_numpy(th).to(d), a1d, a2d).cpu().numpy()
    assert_bitwise(ef_e3, ef_th, 'e3 = dz')
    # through the series call
    g = oracle.DataGen(nx=nx, ny=ny)
    _, p = _build(gpu, g.points(), ny, nx)
    p.computeWeights([tr([(-150, -50), (-20, 35), (60, -40)])])
    e3d = torch.from_numpy(e3c).to(d)
    ef2 = torch.empty((nt, 2 * ny * nx), dtype=torch.float64, device=d)
    ef3 = torch.empty_like(ef2)
    s_e3 = p.fluxSeries(args[0], args[1], None, a1d, a2d, e3u=e3d, e3v=e3d, eflux=ef3)      # two launches
    s_th = p.fluxSeries(args[0], args[1], torch.from_numpy(th).to(d), a1d, a2d, eflux=ef2)
    assert torch.equal(s_e3, s_th) and torch.equal(ef3, ef2)
    f_e3 = p.fluxSeries(args[0], args[1], None, a1d, a2d, e3u=e3d, e3v=e3d)                 # fused pass
    assert _lib_last_path() == 1
    f_th = p.fluxSeries(args[0], args[1], torch.from_numpy(th).to(d), a1d, a2d)
    assert torch.equal(f_e3, f_th)
    with pytest.raises(ValueError):
        gpu.edgeFluxAssemble(args[0], args[1], None, a1d, a2d, e3u=torch.from_numpy(e3c).to(d))


def _lib_last_path():
    from nemoflux_b200 import _lib
    return _lib.get_option(_lib.NFX_OPT_LAST_SERIES_PATH)


@pytest.mark.parametrize('dtype', [numpy.float64, numpy.float32])
@pytest.mark.parametrize('e3_nt', [1, 5])
@pytest.mark.parametrize('padded', [False, True])
def test_fused_series_with_scale_factors(gpu, oracle, dtype, e3_nt, padded):
    """e3u/e3v through the fused persistent pass (several tiles, several panels forced by a 1 MB ring slot, dense
    and padded planes): identical run to run, equal to the two-launch e3 path to rounding, and to the oracle's
    series built from the oracle's e3 edge fluxes; special float32 values take the same route as in K2"""
    import torch
    from nemoflux_b200 import _lib
    nx, ny, nz, nt = 301, 251, 7, 5                 # ncell = 75551, odd; nz = 7 exercises the level tail (5 + 2, 3 + 3 + 1)
    g = oracle.DataGen(nx=nx, ny=ny, nz=nz, nt=nt, deltaDeg=(20., 30.))
    P, arc = g.points(), oracle.arc_lengths(g.points())
    ncell = nx * ny
    rng = numpy.random.default_rng(77)
    u, v = g.uv(SF_C2)
    u, v = u.astype(dtype), v.astype(dtype)
    u[:, :, 100:120, 50:90] = numpy.nan
    e3u = rng.uniform(0.5, 30., (e3_nt, nz, ny, nx)).astype(dtype)
    e3v = rng.uniform(0.5, 30., (e3_nt, nz, ny, nx)).astype(dtype)
    e3v[:, 2:, 40:44, 60:70] = numpy.nan            # missing scale factor below a synthetic bathymetry: counts as 0
    if dtype == numpy.float32:
        u[:, ::2, 10:14, 5:25] = numpy.float32(1.0e-41)
        v[:, 1::3, 30:34, 5:25] = -numpy.finfo(numpy.float32).tiny
        v[1, 3, 200, 100] = numpy.inf                # an infinity: the thread recomputes its columns with clean()
        e3u[0, 1, 20, 30] = numpy.float32(2.0e-42)
    d = 'cuda'
    tdt = torch.float64 if dtype == numpy.float64 else torch.float32
    pad = (4 if dtype == numpy.float64 else 8) if padded else 1
    ld = (ncell + pad - 1) // pad * pad

    def dev(x):
        t = torch.full((x.shape[0], nz, ld), 7.0, dtype=tdt, device=d)[:, :, :ncell]
        t.copy_(torch.from_numpy(x.reshape(x.shape[0], nz, ncell)))
        return t
    ud, vd, eu, ev = dev(u), dev(v), dev(e3u), dev(e3v)
    a1, a2 = (torch.from_numpy(x).to(d) for x in (arc[:, 1].copy(), arc[:, 2].copy()))
    transects = random_transects(numpy.random.default_rng(5), 6) + [tr(README_C2), tr(README_LOOP)]
    _, p = _build(gpu, P, ny, nx)
    p.computeWeights(transects)
    try:
        ef = torch.empty((nt, 2 * ncell), dtype=torch.float64, device=d)
        classic = p.fluxSeries(ud, vd, None, a1, a2, e3u=eu, e3v=ev, eflux=ef).cpu().numpy()
        assert _lib_last_path() == 0
        # the oracle: its e3 edge fluxes (bit for bit), scattered as field.py:209-223 does, summed over its own map
        og = oracle.Grid(P)
        maps = []
        for xyz in transects:
            op = oracle.PolylineIntegral(og)
            op.computeWeights(xyz)
            maps.append(op.merged_map())
        ref = numpy.zeros((nt, len(transects)))
        scale = numpy.zeros((nt, len(transects)))
        efh = ef.cpu().numpy()
        for t in range(nt):
            te = 0 if e3_nt == 1 else t
            with numpy.errstate(all='ignore'):
                eU, eV = oracle.edgeflux_step_c_e3(u[t].astype(numpy.float64), v[t].astype(numpy.float64),
                                                   e3u[te].astype(numpy.float64), e3v[te].astype(numpy.float64),
                                                   arc[:, 1].copy(), arc[:, 2].copy(), False)
            assert_bitwise(efh[t, :ncell], eU, 'eU (e3)')
            assert_bitwise(efh[t, ncell:], eV, 'eV (e3)')
            iV = numpy.zeros((ny, nx, 4))
            eU2, eV2 = eU.reshape(ny, nx), eV.reshape(ny, nx)
            iV[:, :, 1], iV[:, :, 2] = eU2, eV2
            iV[1:, :, 0] = eV2[:-1, :]
            iV[:, 1:, 3] = eU2[:, :-1]
            iV[:, 0, 3] = eU2[:, -1]
            f = iV.reshape(-1)
            with numpy.errstate(all='ignore'):
                for m, (keys, ws) in enumerate(maps):
                    ref[t, m] = (ws * f[keys]).sum()
                    scale[t, m] = numpy.abs(ws * f[keys]).sum()
        fin = numpy.isfinite(ref)
        assert numpy.array_equal(numpy.isfinite(classic), fin)
        assert fin.sum() >= fin.size - nt * 2           # at most the transects through the one infinite column
        assert (numpy.abs(classic[fin] - ref[fin]) <= FLUX_RTOL * scale[fin] + 1e-300).all()
        for slot_mb in (8, 1):
            _lib.set_option(_lib.NFX_OPT_RING_SLOT_MB, slot_mb)
            _lib.set_option(_lib.NFX_OPT_FAST_SERIES, 2)
            fused = p.fluxSeries(ud, vd, None, a1, a2, e3u=eu, e3v=ev).cpu().numpy()
            assert _lib_last_path() == 1
            assert p.getNumberOfPanels()[0] == (1 if slot_mb == 8 else 2)
            again = p.fluxSeries(ud, vd, None, a1, a2, e3u=eu, e3v=ev).cpu().numpy()
            assert numpy.array_equal(fused, again, equal_nan=True)                       # deterministic
            assert numpy.array_equal(numpy.isfinite(fused), fin)
            assert (numpy.abs(fused[fin] - classic[fin]) <= 1e-13 * scale[fin] + 1e-300).all()
            assert (numpy.abs(fused[fin] - ref[fin]) <= FLUX_RTOL * scale[fin] + 1e-300).all()
            if slot_mb == 1:      # balanced sharding with scale factors: the partial series of 3 'ranks' add up
                from nemoflux_b200 import dist
                total = numpy.zeros_like(fused)
                eu_t = lambda t0, n: eu if e3_nt == 1 else eu[t0:t0 + n]      # noqa: E731
                ev_t = lambda t0, n: ev if e3_nt == 1 else ev[t0:t0 + n]      # noqa: E731
                for r in range(3):
                    sh = dist.shard_batches(nt, 2, 3, r)
                    t0, n = sh['t_first'], sh['nt_touched']
                    part = p.fluxSeries(ud[t0:t0 + n], vd[t0:t0 + n], None, a1, a2, e3u=eu_t(t0, n), e3v=ev_t(t0, n),
                                        batch_range=(sh['b0'], sh['b1']))
                    total[t0:t0 + n] += part.cpu().numpy()
                assert numpy.array_equal(numpy.isfinite(total), fin)
                assert (numpy.abs(total[fin] - fused[fin]) <= 1e-13 * scale[fin] + 1e-300).all()
            # the host-buffer entry point (nfx_flux_series_host_e3): scale factors as host arrays (streamed in the
            # chunks when time-varying, uploaded once otherwise), as device tensors, and big-endian as in a file
            hu, hv = u.reshape(nt, nz, ny, nx), v.reshape(nt, nz, ny, nx)
            host = p.fluxSeries(hu, hv, None, arc[:, 1].copy(), arc[:, 2].copy(), e3u=e3u, e3v=e3v, chunk_steps=2)
            assert _lib_last_path() == 1
            assert numpy.array_equal(host, fused, equal_nan=True)
            dense = [torch.from_numpy(x).to(d) for x in (e3u, e3v)]
            host_d = p.fluxSeries(hu, hv, None, arc[:, 1].copy(), arc[:, 2].copy(), e3u=dense[0], e3v=dense[1], chunk_steps=3)
            assert numpy.array_equal(host_d, fused, equal_nan=True)
            be = '>f8' if dtype == numpy.float64 else '>f4'
            host_be = p.fluxSeries(hu.astype(be), hv.astype(be), None, arc[:, 1].copy(), arc[:, 2].copy(),
                                   e3u=e3u.astype(be), e3v=e3v.astype(be), chunk_steps=2)
            assert numpy.array_equal(host_be, fused, equal_nan=True)
        _lib.set_option(_lib.NFX_OPT_FAST_SERIES, 0)            # two launches per chunk
        host2 = p.fluxSeries(hu, hv, None, arc[:, 1].copy(), arc[:, 2].copy(), e3u=e3u, e3v=e3v, chunk_steps=2)
        assert _lib_last_path() == 0
        assert numpy.array_equal(host2, classic, equal_nan=True)
        with pytest.raises(ValueError):
            p.fluxSeries(hu, hv, None, arc[:, 1].copy(), arc[:, 2].copy(), e3u=e3u.astype(numpy.float16), e3v=e3v)
        with pytest.raises(ValueError):
            p.fluxSeries(hu, hv, None, arc[:, 1].copy(), arc[:, 2].copy(), e3u=e3u)
    finally:
        _lib.set_option(_lib.NFX_OPT_RING_SLOT_MB, 0)      # back to automatic
        _lib.set_option(_lib.NFX_OPT_FAST_SERIES, 1)


def test_device_arc_lengths(gpu, oracle):
    """the optional device metric factors: accurate to a few ulp against an extended-precision evaluation, and
    within the reference formula's own rounding noise (~1e-16/arc) of geo.getArcLengthArray"""
    for nx, ny, delta in ((36, 18, (0., 0.)), (720, 360, (20., 30.))):
        g = oracle.DataGen(nx=nx, ny=ny, deltaDeg=delta, ymin=-80., ymax=80., dy=160. / ny)
        P = g.points()
        grid = gpu.Grid()
        grid.setPoints(P)
        arc = grid.arcLengths().cpu().numpy()
        ld = numpy.longdouble
        d2r = ld(numpy.pi) / 180
        ref = numpy.zeros((P.shape[0], 4), ld)
        for e in range(4):
            p, q = P[:, e].astype(ld), P[:, (e + 1) % 4].astype(ld)
            hav = numpy.sin((q[:, 1] - p[:, 1]) * d2r / 2) ** 2 + \
                numpy.cos(p[:, 1] * d2r) * numpy.cos(q[:, 1] * d2r) * numpy.sin((q[:, 0] - p[:, 0]) * d2r / 2) ** 2
            ref[:, e] = 2 * numpy.arcsin(numpy.sqrt(hav))
        rel = numpy.abs(arc - ref.astype(numpy.float64)) / ref.astype(numpy.float64)
        assert rel.max() < 2e-14, rel.max()            # pi/180 in double limits this, not the kernel
        host = oracle.arc_lengths(P)                   # the reference formula
        noise = 4 * numpy.finfo(float).eps / numpy.maximum(host, 1e-300)
        assert (numpy.abs(arc - host) <= noise * 4 + 1e-15).all()


def test_series_edge_cases(gpu, oracle):
    """degenerate inputs through both series paths: no transects, transects outside the grid, nt = 0 and 1,
    nz = 1, an odd number of cells (scalar loads), a transect that only touches row 0 (always-zero south edges)"""
    import torch
    from nemoflux_b200 import _lib
    d = 'cuda'
    g = oracle.DataGen(nx=37, ny=19, nz=1, nt=2, dy=180. / 19)            # 703 cells: odd
    P, arc = g.points(), oracle.arc_lengths(g.points())
    u, v = g.uv('x + 2*y')
    th = g.thickness()
    args = [torch.from_numpy(x).to(d) for x in (u, v, th, arc[:, 1].copy(), arc[:, 2].copy())]
    _, p = _build(gpu, P, 19, 37)
    try:
        for mode in (0, 2):
            _lib.set_option(_lib.NFX_OPT_FAST_SERIES, mode)
            p.computeWeights([])
            assert tuple(p.fluxSeries(*args).shape) == (2, 0)
            outside = [tr([(0, 100), (10, 120)]), tr([(5, 5)]), tr([(1, 1), (1, 1)])]
            p.computeWeights(outside)
            assert (p.fluxSeries(*args).cpu().numpy() == 0).all()
            row0 = [tr([(-170, -89.5), (170, -89.5)]), tr([(-100, -60), (100, 40)])]
            p.computeWeights(row0)
            s = p.fluxSeries(*args).cpu().numpy()
            ref = oracle.flux_series(P, row0, u, v, th, use_c=True)
            assert numpy.abs(s - ref).max() <= 1e-12 * numpy.abs(ref).max()
            empty = p.fluxSeries(args[0][:0], args[1][:0], *args[2:])
            assert tuple(empty.shape) == (0, 2)
            one = p.fluxSeries(args[0][1:], args[1][1:], *args[2:]).cpu().numpy()
            assert numpy.array_equal(one[0], s[1])
            # host buffers, big-endian, 703 values per chunk: the device byte swap has a tail of < 16 bytes
            for dt in ('f8', 'f4'):
                h_le = p.fluxSeries(u.astype('<' + dt), v.astype('<' + dt), th, arc[:, 1].copy(), arc[:, 2].copy(),
                                    chunk_steps=1)
                h_be = p.fluxSeries(u.astype('>' + dt), v.astype('>' + dt), th, arc[:, 1].copy(), arc[:, 2].copy(),
                                    chunk_steps=1)
                assert numpy.array_equal(h_le, h_be)
                if dt == 'f8':
                    assert numpy.array_equal(h_le, s)
    finally:
        _lib.set_option(_lib.NFX_OPT_FAST_SERIES, 1)
    with pytest.raises(ValueError):
        p.fluxSeries(args[0][:, :, :10], args[1][:, :, :10], *args[2:])         # wrong grid size
    with pytest.raises(TypeError):
        p.fluxSeries(args[0], args[1].cpu(), *args[2:])


@pytest.mark.gpu
def test_guard_bands_catch_an_overrun(gpu):
    """NFX_DEBUG_GUARDS=1 (the stand-in for compute-sanitizer memcheck on pools that refuse it): a byte written right
    before or right behind a library-owned device buffer is reported by nfx_debug_check_guards; a clean run passes"""
    import subprocess
    import sys
    from conftest import ROOT
    code = r'''
import sys
sys.path.insert(0, %r)
import torch
from nemoflux_b200 import _lib, nemoflux_gpu, synth
syn = synth.make('tiny')
g = nemoflux_gpu.Grid(); g.setPoints(syn.points); g.setCGridShape(syn.ny, syn.nx)
p = nemoflux_gpu.PolylineIntegral(); p.build(g); p.computeWeights(syn.transects)
dev = torch.device('cuda', 0)
u, v = syn.fill_device(0, syn.nt, dev)
s = p.fluxSeries(u, v, *(torch.from_numpy(x).to(dev) for x in (syn.thickness, syn.arc1, syn.arc2)))
assert torch.isfinite(s).all()
n = _lib.check_guards()
assert n >= 10, n
for where in (0, 1):
    _lib.call('nfx_debug_poke_guard', where)
    try:
        _lib.check_guards()
    except _lib.NemofluxGpuError as e:
        assert 'guard bytes overwritten' in str(e) and ('BEFORE the start' if where == 0 else 'PAST the end') in str(e), e
    else:
        raise SystemExit('a damaged guard band went unnoticed')
    break       # the band stays damaged: one direction per process
print('ok', n)
''' % ROOT
    for where_first in (0, 1):
        c = code if where_first == 0 else code.replace('for where in (0, 1):', 'for where in (1, 0):')
        out = subprocess.run([sys.executable, '-c', c], capture_output=True, text=True, timeout=300,
                             env=dict(os.environ, NFX_DEBUG_GUARDS='1'))
        assert out.returncode == 0 and out.stdout.startswith('ok'), out.stderr[-2000:] + out.stdout[-500:]


@pytest.mark.gpu
@pytest.mark.parametrize('dtype', [numpy.float64, numpy.float32])
def test_many_levels_up_to_the_shared_memory_limit(gpu, oracle, dtype):
    """the layer thickness (and its 2^896 multiple for float32 storage) lives in dynamic shared memory: 3000 levels
    (47 KB) is the documented limit -- both passes work there (same bits as the sequential oracle), one level more is
    refused with a clear message instead of a launch failure"""
    import torch
    from nemoflux_b200 import _lib
    nx, ny, nt = 24, 12, 2
    rng = numpy.random.default_rng(8)
    for nz in (3000, 1000):
        g = oracle.DataGen(nx=nx, ny=ny, nz=1, nt=1)
        P, arc = g.points(), oracle.arc_lengths(g.points())
        u = rng.normal(size=(nt, nz, ny, nx)).astype(dtype)
        v = rng.normal(size=(nt, nz, ny, nx)).astype(dtype)
        u[:, :, 3:5, 2:9] = numpy.nan
        th = rng.uniform(0.5, 2.0, nz)
        _, p = _build(gpu, P, ny, nx)
        transects = [tr(README_C1), tr([(-100, -40), (80, 30)])]
        p.computeWeights(transects)
        a1, a2 = arc[:, 1].copy(), arc[:, 2].copy()
        args = [torch.from_numpy(x).cuda() for x in (u, v, th, a1, a2)]
        fused = p.fluxSeries(*args).cpu().numpy()
        assert _lib.get_option(_lib.NFX_OPT_LAST_SERIES_PATH) == 1 and p.seriesStatus() == 0
        ef = torch.empty((nt, 2 * ny * nx), dtype=torch.float64, device='cuda')
        classic = p.fluxSeries(*args, eflux=ef).cpu().numpy()
        for t in range(nt):
            _, eU, eV = oracle.edgeflux_step_c(u[t], v[t], th, a1, a2, False)
            assert_bitwise(ef[t].cpu().numpy(), numpy.concatenate([eU, eV]), f'eflux nz={nz}')
        scale = numpy.abs(classic).max()
        assert numpy.abs(fused - classic).max() <= 1e-12 * scale
    nz = 3001
    u = torch.zeros((1, nz, ny, nx), dtype=torch.float64, device='cuda')
    with pytest.raises(_lib.NemofluxGpuError, match='3000 levels'):
        p.fluxSeries(u, u, torch.ones(nz, dtype=torch.float64, device='cuda'), args[3], args[4])
    with pytest.raises(_lib.NemofluxGpuError, match='3000 levels'):
        gpu.edgeFluxAssemble(u, u, torch.ones(nz, dtype=torch.float64, device='cuda'), args[3], args[4])


def test_bench_dump_outputs_is_the_timed_series(gpu, oracle, tmp_path):
    """bench.py --dump-outputs DIR on the GPU arm: the series the last timed step returned, all time steps, equal to the
    oracle's series to the flux bar; a second run with the same arguments writes the same bits"""
    import subprocess
    import sys
    from conftest import ROOT
    from nemoflux_b200 import synth
    got = []
    for run in range(2):
        d = tmp_path / f'run{run}'
        cmd = [sys.executable, os.path.join(ROOT, 'bench.py'), '--workload', 'tiny', '--steps', '2', '--warmup', '1',
               '--no-e2e', '--no-cpu', '--dump-outputs', str(d)]
        out = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=ROOT)
        assert out.returncode == 0, out.stderr[-2000:]
        assert os.listdir(d) == ['flux_series.npy']
        got.append(numpy.load(d / 'flux_series.npy'))
    syn = synth.make('tiny')
    assert got[0].dtype == numpy.float64 and got[0].shape == (syn.nt, syn.ntransects)
    assert numpy.array_equal(got[0], got[1])
    uh = numpy.stack([syn.uv_host(t)[0] for t in range(syn.nt)])
    vh = numpy.stack([syn.uv_host(t)[1] for t in range(syn.nt)])
    ref = oracle.flux_series(syn.points, syn.transects, uh, vh, syn.thickness)
    assert numpy.abs(got[0] - ref).max() <= FLUX_RTOL * numpy.abs(ref).max()
