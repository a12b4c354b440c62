"""-m "not gpu": the oracle against the golden vectors (outputs of the reference's own code), the known
answers the reference records, and its own invariants.  No GPU needed."""
import json
import os

import numpy
import pytest

from conftest import GOLDEN
from helpers import README_C1, README_C2, README_LOOP, README_SINGULAR, SF_C2, random_transects, tr


def _golden(name):
    return numpy.load(os.path.join(GOLDEN, name))


# ---- K2 pinned on the reference's own outputs ------------------------------------------------------------
@pytest.mark.parametrize('name,ti,sv', [('c1_simple.npz', 0, False), ('singular.npz', 0, False),
                                        ('rot24x12_t0_sv0.npz', 0, False), ('rot24x12_t0_sv1.npz', 0, True),
                                        ('rot24x12_t1_sv0.npz', 1, False), ('rot24x12_t1_sv1.npz', 1, True)])
def test_field_restatement_matches_reference_outputs(oracle, name, ti, sv):
    g = _golden(name)
    u, v = g['u'], g['v']
    th = g['zbot'] - g['ztop']
    assert numpy.array_equal(th, g['thickness'])
    ny, nx = u.shape[2:]
    pts = numpy.zeros((ny, nx, 4, 3))
    pts[..., 0], pts[..., 1] = g['bounds_lon'], g['bounds_lat']
    arc = oracle.arc_lengths(pts.reshape(-1, 4, 3))
    assert numpy.allclose(arc, g['arcLengths'], rtol=1e-13, atol=1e-16)
    U = oracle.read_field(u[ti], th)
    V = oracle.read_field(v[ti], th)
    assert numpy.allclose(U, g['U'], rtol=1e-14, atol=1e-300)
    assert numpy.allclose(V, g['V'], rtol=1e-14, atol=1e-300)
    iV, eU, eV = oracle.integrated_flux(U, V, g['arcLengths'], sv)
    scale = numpy.abs(g['iV']).max()
    assert numpy.abs(iV - g['iV']).max() <= 1e-14 * scale
    assert numpy.allclose(numpy.abs(eU), g['absEU'], rtol=1e-14, atol=0)
    assert numpy.allclose(numpy.abs(eV), g['absEV'], rtol=1e-14, atol=0)
    assert abs(max(numpy.abs(eU).max(), numpy.abs(eV).max()) - float(g['maxAbsFlux'])) <= 1e-14 * scale
    # the sequential C restatement (the bit-exact reference of the CUDA kernel) agrees to rounding
    iVc, _, _ = oracle.edgeflux_step_c(u[ti], v[ti], th, g['arcLengths'][:, 1].copy(), g['arcLengths'][:, 2].copy(), sv)
    assert numpy.abs(iVc - g['iV']).max() <= 1e-13 * scale


def test_datagen_restatement_matches_reference_outputs(oracle):
    g = _golden('c1_simple.npz')
    d = oracle.DataGen()
    u, v = d.uv('x')
    assert numpy.array_equal(d.bounds_lon, g['bounds_lon']) and numpy.array_equal(d.bounds_lat, g['bounds_lat'])
    assert numpy.allclose(u, g['u'], rtol=1e-13, atol=1e-13) and numpy.allclose(v, g['v'], rtol=1e-13, atol=1e-13)
    assert numpy.array_equal(d.ztop, g['ztop']) and numpy.array_equal(d.zbot, g['zbot'])
    g = _golden('singular.npz')
    u, v = d.uv('arctan2(y, x+180)/(2*pi)')
    assert numpy.allclose(u, g['u'], rtol=1e-13, atol=1e-14) and numpy.allclose(v, g['v'], rtol=1e-13, atol=1e-14)
    # pole displaced grid: vectorised rotation vs the reference's per-vertex loop (ulp differences only; the
    # longitude of a vertex sitting on the pole is arbitrary in both)
    g = _golden('rot24x12_t0_sv0.npz')
    d = oracle.DataGen(nx=24, ny=12, nz=3, nt=2, deltaDeg=(20., 30.))
    assert numpy.abs(d.bounds_lat - g['bounds_lat']).max() < 1e-12
    notpole = numpy.abs(numpy.abs(g['bounds_lat']) - 90.) > 1e-6
    dl = numpy.abs(d.bounds_lon - g['bounds_lon'])[notpole]
    assert numpy.minimum(dl, numpy.abs(dl - 360.)).max() < 1e-11
    u, v = d.uv(SF_C2)
    m = ~g['mask']
    assert numpy.allclose(u[:, m], g['u'][:, m], rtol=1e-13, atol=1e-13)
    # C2 samples (360x180, nz=10, nt=20)
    g = _golden('c2_sample.npz')
    d = oracle.DataGen(nx=360, ny=180, nz=10, nt=20, deltaDeg=(20., 30.))
    assert numpy.abs(d.bounds_lat[::17, ::13] - g['bounds_lat_rows']).max() < 1e-12
    u, v = d.uv(SF_C2)
    for ti in (0, 19):
        U = oracle.read_field(u[ti], d.thickness())
        assert numpy.allclose(U, g[f'U_t{ti}'], rtol=1e-12, atol=1e-13)
    with open(os.path.join(GOLDEN, 'golden_summary.json')) as f:
        summ = json.load(f)
    arc = oracle.arc_lengths(d.points())
    iV, eU, eV = oracle.integrated_flux(oracle.read_field(u[19], d.thickness()), oracle.read_field(v[19], d.thickness()), arc)
    assert abs(max(numpy.abs(eU).max(), numpy.abs(eV).max()) - summ['c2_digests']['maxAbsFlux_t19']) < 1e-10


# ---- the mint restatement: known answers the reference records --------------------------------------------
def test_known_answer_360(oracle):
    """README.md:26-39, pictures/simple.png"""
    d = oracle.DataGen()
    u, v = d.uv('x')
    s = oracle.flux_series(d.points(), [tr(README_C1)], u, v, d.thickness())
    assert abs(s[0, 0] - 360.) < 1e-12 * 360
    assert abs(numpy.abs(oracle.integrated_flux(oracle.read_field(u[0], d.thickness()), oracle.read_field(v[0], d.thickness()),
                                                oracle.arc_lengths(d.points()))[0]).max() - 10.0) < 1e-12   # colour bar max
    p = oracle.PolylineIntegral(oracle.Grid(d.points()))
    p.computeWeights(tr(README_C1))
    assert len(p.subsegs) == 59                                     # SURVEY.md appendix A
    assert list(numpy.bincount(p.subsegs['seg'])) == [6, 15, 14, 12, 12]
    assert list(p.subsegs['cell'][:6]) == [72, 108, 144, 181, 217, 253]
    assert numpy.allclose(p.subsegs['w'][0], [1 / 6, 1 / 6, 1 / 6, 5 / 6], atol=1e-14)
    assert numpy.allclose(p.subsegs['w'].sum(0), [18., 5.245454545454547, 18., 5.754545454545455], atol=1e-12)
    assert numpy.allclose(p.segment_totals(5), 1.0, atol=1e-14)


def test_known_answer_singular_half(oracle):
    """README.md:50-58: node-to-node path around a singular stream function gives exactly psi(B)-psi(A) = 0.5"""
    d = oracle.DataGen()
    u, v = d.uv('arctan2(y, x+180)/(2*pi)')
    for order in ('map', 'list'):
        s = oracle.flux_series(d.points(), [tr(README_SINGULAR)], u, v, d.thickness(), order=order)
        assert abs(s[0, 0] - 0.5) <= 2e-16 * 4


def test_known_answer_closed_loops(oracle):
    """README.md:65-68 (4.2e-15 in pictures/closed2.png) and README.md:77-79 (2.34e-11 with the displaced pole)"""
    sf = 'cos(2*pi*y/360) + sin(2*pi*x/360)'
    d = oracle.DataGen(nx=360, ny=180)
    u, v = d.uv(sf)
    s = oracle.flux_series(d.points(), [tr(README_LOOP)], u, v, d.thickness())
    assert abs(s[0, 0]) < 1e-13
    d = oracle.DataGen(nx=360, ny=180, deltaDeg=(20., 30.))
    u, v = d.uv(sf)
    s = oracle.flux_series(d.points(), [tr(README_LOOP)], u, v, d.thickness())
    assert abs(s[0, 0]) < 1e-10          # arccos arc lengths vs datagen's un-rotated ds: expected level ~2e-11


def test_c2_series(oracle):
    """BASELINE config 2: 361 sub-segments, flux(t) = 1.7386322852...*(t+1)"""
    d = oracle.DataGen(nx=360, ny=180, nz=10, nt=20, deltaDeg=(20., 30.))
    u, v = d.uv(SF_C2)
    s = oracle.flux_series(d.points(), [tr(README_C2)], u, v, d.thickness())[:, 0]
    assert abs(s[0] - 1.7386322852896516) < 1e-11
    assert numpy.allclose(s / s[0], numpy.arange(1, 21), rtol=1e-12)
    p = oracle.PolylineIntegral(oracle.Grid(d.points()))
    p.computeWeights(tr(README_C2))
    assert len(p.subsegs) == 361
    assert numpy.allclose(p.segment_totals(2), 1.0, atol=1e-13)


def test_node_to_node_exact_and_linear(oracle):
    """fluxexact.py:36-46: F = sum_k dz_k (psi_k(B) - psi_k(A)); linear in u,v and in the thickness"""
    d = oracle.DataGen(nx=36, ny=18, nz=4, nt=3)
    u, v = d.uv(SF_C2)
    path = [(-120, -40), (-33.3, 12.5), (70, -60), (100, 50)]          # ends on nodes, interior points are not
    s = oracle.flux_series(d.points(), [tr(path)], u, v, d.thickness())[:, 0]
    for t in range(3):
        ex = 0.0
        for k in range(4):
            ex += (d.potential_nodes(SF_C2, t, k)[14, 28] - d.potential_nodes(SF_C2, t, k)[5, 6]) * d.thickness()[k]
        assert abs(s[t] - ex) <= 1e-12 * abs(ex)
    s2 = oracle.flux_series(d.points(), [tr(path)], 3 * u, 3 * v, d.thickness())[:, 0]
    s3 = oracle.flux_series(d.points(), [tr(path)], u, v, 2 * d.thickness())[:, 0]
    assert numpy.allclose(s2, 3 * s, rtol=1e-13) and numpy.allclose(s3, 2 * s, rtol=1e-13)


@pytest.mark.parametrize('delta', [(0., 0.), (20., 30.)])
def test_c_oracle_vs_independent_numpy_brute_force(oracle, delta):
    from oracle import brute_numpy
    d = oracle.DataGen(nx=40, ny=20, deltaDeg=delta)
    P = d.points()
    rng = numpy.random.default_rng(3)
    nodes = numpy.stack([d.xx, d.yy], -1) if delta == (0., 0.) else None
    transects = random_transects(rng, 8, nodes=nodes) + [tr(README_C1), tr(README_LOOP), tr([(-180, -40), (180, -40)])]
    g = oracle.Grid(P)
    checked = 0
    for xyz in transects:
        p = oracle.PolylineIntegral(g, filter_mode=1)
        p.computeWeights(xyz)
        pb = oracle.PolylineIntegral(g, filter_mode=0)
        pb.computeWeights(xyz)
        assert numpy.array_equal(p.subsegs, pb.subsegs)              # the bbox filter is a pure superset filter
        b = brute_numpy.compute_weights(P, xyz)
        assert numpy.array_equal(b['cell'], p.subsegs['cell'])
        assert numpy.array_equal(b['seg'], p.subsegs['seg']) and numpy.array_equal(b['img'], p.subsegs['img'])
        assert numpy.allclose(b['ta'], p.subsegs['ta'], atol=1e-13) and numpy.allclose(b['coeff'], p.subsegs['coeff'], atol=1e-12)
        # cells next to the displaced pole are folded quads in the lon-lat plane: the bilinear map has two
        # inverses there and the two solvers may pick different ones -- compare away from the poles
        ok = numpy.abs(P[p.subsegs['cell'], :, 1]).max(axis=1) < (78. if delta != (0., 0.) else 91.)
        checked += int(ok.sum())
        assert numpy.abs(b['w'] - p.subsegs['w'])[ok].max(initial=0.) <= 1e-11
    assert checked > 500


def test_c_oracle_vs_brute_force_on_the_full_orca1_grid(oracle):
    """the same cross-check at a size the benchmark uses: the 362 x 332 ORCA1-shaped grid of bench.py's config C3
    (120 184 curvilinear cells, displaced pole), node-to-node, closed and free transects of its synthetic workload --
    identical cell / segment / image lists, ta equal, weights to 1e-12 (away from the folded cells at the pole)"""
    import warnings
    from nemoflux_b200 import synth
    from oracle import brute_numpy
    syn = synth.make('C3')
    g = oracle.Grid(syn.points)
    checked = 0
    with warnings.catch_warnings():
        warnings.simplefilter('ignore')
        for m in (0, 1, 2, 5, 7):
            xyz = syn.transects[m]
            p = oracle.PolylineIntegral(g)
            p.computeWeights(xyz)
            b = brute_numpy.compute_weights(syn.points, xyz)
            assert numpy.array_equal(b['cell'], p.subsegs['cell']), (m, syn.kinds[m])
            assert numpy.array_equal(b['seg'], p.subsegs['seg']) and numpy.array_equal(b['img'], p.subsegs['img'])
            assert numpy.allclose(b['ta'], p.subsegs['ta'], atol=1e-13) and numpy.allclose(b['coeff'], p.subsegs['coeff'], atol=1e-12)
            ok = numpy.abs(syn.points[p.subsegs['cell'], :, 1]).max(axis=1) < 78.
            assert numpy.abs(b['w'] - p.subsegs['w'])[ok].max(initial=0.) <= 1e-12
            checked += int(ok.sum())
    assert checked > 4000


def test_map_and_list_orders(oracle):
    d = oracle.DataGen(nx=36, ny=18)
    p = oracle.PolylineIntegral(oracle.Grid(d.points()))
    p.computeWeights(tr(README_SINGULAR))          # runs along grid lines: duplicate sub-segments, coeff 0/1
    assert set(numpy.round(p.subsegs['coeff'], 12)) <= {0.0, 1.0}
    assert (p.subsegs['coeff'] == 0.0).any()
    keys, ws = p.merged_map()
    assert (numpy.diff(keys) > 0).all()
    cells, edges, w = p.emission_list()
    acc = {}
    for c, e, x in zip(cells, edges, w):
        acc[c * 4 + e] = acc.get(c * 4 + e, 0.0) + x
    assert numpy.array_equal(keys, numpy.array(sorted(acc)))
    assert numpy.array_equal(ws, numpy.array([acc[k] for k in sorted(acc)]))
    data = numpy.random.default_rng(0).standard_normal((36 * 18, 4))
    a, b = p.getIntegral(data, 'map'), p.getIntegral(data, 'list')
    assert abs(a - b) <= 1e-13 * numpy.abs(data).max() * numpy.abs(w).sum()


def test_edge_cases(oracle):
    d = oracle.DataGen()
    g = oracle.Grid(d.points())
    p = oracle.PolylineIntegral(g)
    for xyz in (numpy.zeros((0, 3)), tr([(1, 1)]), tr([(1, 1), (1, 1)]), tr([(0, 100), (10, 120)])):
        p.computeWeights(xyz)
        assert len(p.subsegs) == 0
        assert p.getIntegral(numpy.ones((648, 4))) == 0.0
    # the x-period: a transect given 360 degrees to the east gives the same weights
    a = oracle.PolylineIntegral(g)
    a.computeWeights(tr([(-100, -20), (-60, 30)]))
    b = oracle.PolylineIntegral(g)
    b.computeWeights(tr([(260, -20), (300, 30)]))
    assert numpy.array_equal(a.subsegs['cell'], b.subsegs['cell'])
    assert numpy.allclose(a.subsegs['w'], b.subsegs['w'], atol=1e-13)
    # without the period nothing is found out there
    c = oracle.PolylineIntegral(g, periodX=0.)
    c.computeWeights(tr([(260, -20), (300, 30)]))
    assert len(c.subsegs) == 0
    # row 0 south edges stay zero (field.py:219) and the west edge of column 0 is periodic (field.py:223)
    U = numpy.arange(18 * 36, dtype=float).reshape(18, 36) + 1
    iV, eU, eV = oracle.integrated_flux(U, 2 * U, numpy.ones((648, 4)))
    iV = iV.reshape(18, 36, 4)
    assert (iV[0, :, 0] == 0).all() and numpy.array_equal(iV[:, 0, 3], eU.reshape(18, 36)[:, -1])
    assert oracle.lib().orc_flux_index(0, 0, 18, 36) == -1 and oracle.lib().orc_flux_index(36, 3, 18, 36) == 71


def test_orientation_and_additivity_properties(oracle):
    """properties any line integral of a 1-form has, with random single-valued edge data: reversing the transect
    flips the sign, cutting it at a vertex splits the integral, every segment inside the grid is fully covered
    (sum of (tb - ta) * coeff = 1) -- on a curvilinear (pole-displaced) and on a rectilinear grid; inserting a vertex
    on a segment changes nothing on the rectilinear grid (on a curvilinear cell the weights integrate along the
    straight line in PARAMETER space between the sub-segment's ends, so an extra vertex changes the path)"""
    rng = numpy.random.default_rng(42)
    for delta in ((20., 30.), (0., 0.)):
        d = oracle.DataGen(nx=48, ny=24, deltaDeg=delta, ymin=-80., ymax=80., dy=160. / 24)
        g = oracle.Grid(d.points())
        data = rng.standard_normal((48 * 24, 4))
        # single valued per edge (east of c = west of c+1, north of c = south of the cell above), as C-grid fluxes are
        dd = data.reshape(24, 48, 4)
        dd[:, 1:, 3] = dd[:, :-1, 1]
        dd[:, 0, 3] = dd[:, -1, 1]
        dd[1:, :, 0] = dd[:-1, :, 2]
        scale = numpy.abs(data).max()

        def integral(pts):
            p = oracle.PolylineIntegral(g)
            p.computeWeights(tr(pts))
            return p.getIntegral(data), p

        for _ in range(12):
            k = int(rng.integers(3, 7))
            lat = 60. if delta == (0., 0.) else 45.     # the displaced grid leaves a 10 degree cap around (., +-60) uncovered
            pts = [(float(rng.uniform(-170, 170)), float(rng.uniform(-lat, lat))) for _ in range(k)]
            f, p = integral(pts)
            l1 = numpy.abs(p.emission_list()[2]).sum() * scale
            frev, _ = integral(pts[::-1])
            assert abs(f + frev) <= 1e-12 * l1
            cut = int(rng.integers(1, k - 1))
            fa, _ = integral(pts[:cut + 1])
            fb, _ = integral(pts[cut:])
            assert abs(f - (fa + fb)) <= 1e-12 * l1
            assert numpy.abs(p.segment_totals(k - 1) - 1.0).max() <= 1e-12
            if delta == (0., 0.):
                s = float(rng.uniform(0.2, 0.8))
                mid = (pts[0][0] + s * (pts[1][0] - pts[0][0]), pts[0][1] + s * (pts[1][1] - pts[0][1]))
                fins, _ = integral([pts[0], mid] + pts[1:])
                assert abs(f - fins) <= 1e-11 * l1


def _sa_grid():
    """the reference's real NEMO T grid (data/sa/T.nc, committed as tests/golden/sa_T_grid.npz): (ncell,4,3) points"""
    import os
    from conftest import GOLDEN
    g = numpy.load(os.path.join(GOLDEN, 'sa_T_grid.npz'))
    lon, lat = g['bounds_lon'].astype(numpy.float64), g['bounds_lat'].astype(numpy.float64)
    pts = numpy.zeros((100, 100, 4, 3))
    pts[..., 0], pts[..., 1] = lon, lat
    return pts.reshape(-1, 4, 3), lon, lat


def test_real_nemo_grid_transect(oracle):
    """K1/K3 of the oracle on the real ORCA025 window south of Africa with the reference's own transect
    data/sa/S3_sa.txt: every segment fully covered; with edge fluxes derived from a nodal stream function the
    integral between two grid nodes is psi(B) - psi(A), whatever the path (fluxexact.py:36-46), with the
    reference's sign convention (field.py:195-196: eU = +U*dy on the east edge, eV = -V*dx on the north edge)"""
    P, lon, lat = _sa_grid()
    og = oracle.Grid(P)
    s3 = tr([(16., -40.4), (28., -34.5), (31., -28.5), (36., -30.5)])             # data/sa/S3_sa.txt:5-8 as (lon, lat)
    p = oracle.PolylineIntegral(og)
    p.computeWeights(s3)
    assert len(p.subsegs) > 100
    assert numpy.abs(p.segment_totals(3) - 1.0).max() <= 1e-12
    # nodal stream function -> C-grid edge fluxes: east edge (SE->NE) carries psi(NE)-psi(SE), north edge (NW->NE)
    # carries -(psi(NE)-psi(NW)) before the minus sign of field.py:196, i.e. iV[:,2] = psi(NE)-psi(NW)
    def psi(x, y):
        return numpy.sin(numpy.radians(3 * x)) * (y + 45.) + 0.01 * x * y
    se, ne, nw = psi(lon[..., 1], lat[..., 1]), psi(lon[..., 2], lat[..., 2]), psi(lon[..., 3], lat[..., 3])
    iV = numpy.zeros((100, 100, 4))
    iV[..., 1] = ne - se
    iV[..., 2] = ne - nw
    iV[1:, :, 0] = iV[:-1, :, 2]
    iV[:, 1:, 3] = iV[:, :-1, 1]
    iV[0, :, 0] = psi(lon[0, :, 1], lat[0, :, 1]) - psi(lon[0, :, 0], lat[0, :, 0])
    iV[:, 0, 3] = psi(lon[:, 0, 3], lat[:, 0, 3]) - psi(lon[:, 0, 0], lat[:, 0, 0])
    rng = numpy.random.default_rng(4)
    for _ in range(6):
        ja, ia, jb, ib = (int(v) for v in rng.integers(5, 95, 4))
        a = (lon[ja, ia, 0], lat[ja, ia, 0])                    # SW nodes of two cells
        b = (lon[jb, ib, 0], lat[jb, ib, 0])
        mid = (float(rng.uniform(15., 35.)), float(rng.uniform(-39., -23.)))
        q = oracle.PolylineIntegral(og)
        q.computeWeights(tr([a, mid, b]))
        exact = psi(*b) - psi(*a)
        got = q.getIntegral(iV.reshape(-1, 4))
        assert abs(got - exact) <= 1e-10 * max(1.0, abs(exact)), (got, exact)

