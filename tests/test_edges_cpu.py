"""-m "not gpu": the float64 reference of tests/test_gpu_edges.py pinned on the CPU -- its series against the oracle's
fluxplot loop on the README C2 case, its edge fluxes against the C restatement of K2 bit for bit, its tracer of ones
against its section, its layers against its whole column, and its tile fold and window sums against plain sums."""
import numpy
import pytest

from helpers import README_C2, SF_C2, tr
from test_gpu_edges import Reference, oracle_crossings, window_sums


@pytest.fixture(scope='module')
def c2(oracle):
    nt, nz = 4, 10
    d = oracle.DataGen(nx=360, ny=180, nz=nz, nt=nt, deltaDeg=(20., 30.))
    u, v = d.uv(SF_C2)
    P = d.points()
    arc = oracle.arc_lengths(P)
    lines = [tr(README_C2), tr([(-30., -40.), (40., 20.)])]
    sub = oracle_crossings(oracle, P, lines)
    return dict(d=d, u=u, v=v, P=P, arc=arc, lines=lines, sub=sub, nt=nt, nz=nz,
                R=Reference(sub, 360, 180, arc[:, 1].copy(), arc[:, 2].copy()))


def test_reference_series_against_the_oracle(oracle, c2):
    """README C2: the reference's sum over every transect's crossings is the oracle's series within 1e-12 * sum |w f|,
    and so is its tile fold; the first transect is the documented 1.7386322852896516 * (t + 1)"""
    nt, nz, R = c2['nt'], c2['nz'], c2['R']
    th = c2['d'].thickness()
    u, v = c2['u'].reshape(nt, nz, -1), c2['v'].reshape(nt, nz, -1)
    for sverdrup in (False, True):
        sec, bar = R.section(u, v, [0, nz], th=th, sverdrup=sverdrup)
        want = oracle.flux_series(c2['P'], c2['lines'], c2['u'], c2['v'], th, sverdrup=sverdrup)
        b = R.per_transect(bar[:, 0])
        assert (b > 0).all()
        assert (numpy.abs(R.per_transect(sec[:, 0]) - want) <= 1e-12 * b).all()
        assert (numpy.abs(R.tile_fold(sec[:, 0]) - want) <= 1e-12 * b).all()
    sec, _ = R.section(u, v, [0, nz], th=th)
    assert numpy.allclose(R.per_transect(sec[:, 0])[:, 0], 1.7386322852896516 * numpy.arange(1, nt + 1), rtol=1e-11)
    # layers add up to the whole column
    lay, lbar = R.section(u, v, [0, 3, 4, nz], th=th)
    assert (numpy.abs(lay.sum(1) - sec[:, 0]) <= 1e-12 * lbar.sum(1) + 1e-300).all()


@pytest.mark.parametrize('dtype', [numpy.float64, numpy.float32])
def test_reference_edge_fluxes_against_the_c_restatement(oracle, dtype):
    """cell_fluxes (the K2 values the section gathers) equal oracle.edgeflux_step_c / _e3 bit for bit, with NaN, the
    fill marker, denormals and sverdrup"""
    nt, nz, ny, nx = 2, 5, 6, 8
    rng = numpy.random.default_rng(4)
    P = oracle.DataGen(nx=nx, ny=ny).points()
    arc = oracle.arc_lengths(P)
    a1, a2 = arc[:, 1].copy(), arc[:, 2].copy()
    u = rng.uniform(-2, 2, (nt, nz, ny * nx)).astype(dtype)
    v = rng.uniform(-2, 2, (nt, nz, ny * nx)).astype(dtype)
    u[:, 1, ::5] = numpy.nan
    v[:, 2, ::7] = -7.0
    u[:, 3, ::3] = numpy.finfo(dtype).tiny / 8
    th = rng.uniform(0.5, 30., nz)
    R = Reference(dict(cell=numpy.zeros(0, numpy.int64), w=numpy.zeros((0, 4)), offsets=numpy.zeros(1, numpy.int64)),
                  nx, ny, a1, a2)
    got = R.cell_fluxes(u, v, [0, nz], th=th, fill=-7.0, sverdrup=True, arc1=a1, arc2=a2)[:, 0]
    for t in range(nt):
        _, eU, eV = oracle.edgeflux_step_c(u[t].reshape(nz, ny, nx), v[t].reshape(nz, ny, nx), th, a1, a2, True, -7.0,
                                           want_iV=False)
        assert numpy.array_equal(got[t].view(numpy.int64), numpy.concatenate([eU, eV]).view(numpy.int64))
    e3u = rng.uniform(0.5, 30., (1, nz, ny * nx)).astype(dtype)
    e3v = rng.uniform(0.5, 30., (1, nz, ny * nx)).astype(dtype)
    e3u[0, 0, ::4] = numpy.nan
    got = R.cell_fluxes(u, v, [0, nz], e3u=e3u, e3v=e3v, fill=-7.0, arc1=a1, arc2=a2)[:, 0]
    for t in range(nt):
        eU, eV = oracle.edgeflux_step_c_e3(*(x.reshape(nz, ny, nx) for x in (u[t], v[t], e3u[0], e3v[0])), a1, a2,
                                           False, -7.0)
        assert numpy.array_equal(got[t].view(numpy.int64), numpy.concatenate([eU, eV]).view(numpy.int64))


def test_reference_tracer_tiles_and_windows(c2):
    """a tracer of ones (ref 0) gives the section bit for bit and one of 2 twice it; the tile fold of 1 ... n is the
    exact sum for every n around the tile size; window sums are sequential sums, a continued window adds to its start"""
    nt, nz, R = c2['nt'], c2['nz'], c2['R']
    th = c2['d'].thickness()
    u, v = c2['u'].reshape(nt, nz, -1), c2['v'].reshape(nt, nz, -1)
    sec, _ = R.section(u, v, [0, 2, nz], th=th)
    ones = numpy.ones((1, nz, u.shape[2]))
    assert numpy.array_equal(R.section(u, v, [0, 2, nz], th=th, tau=ones)[0].view(numpy.int64), sec.view(numpy.int64))
    assert numpy.array_equal(R.section(u, v, [0, 2, nz], th=th, tau=2 * ones)[0], 2 * sec)
    for n in (1, 31, 32, 33, 64, 65):
        F = Reference(dict(cell=numpy.zeros(n, numpy.int64), w=numpy.zeros((n, 4)),
                           offsets=numpy.array([0, n], numpy.int64)), 4, 4, numpy.ones(16), numpy.ones(16))
        assert F.tile_fold(numpy.arange(1., n + 1.))[0] == n * (n + 1) / 2
    wins = [0, 1, 3, 4]
    ws = window_sums(sec, wins)
    assert numpy.array_equal(ws[1], sec[1] + sec[2]) and numpy.array_equal(ws[0], 0.0 + sec[0])
    start = numpy.full(sec.shape[1:], 0.25)
    assert numpy.array_equal(window_sums(sec, wins, start)[0], 0.25 + sec[0])
