"""Same-box A/B of the tracer transport (fluxTracer): the [0, nz] tracer series, the per-level tracer section, the
composition the tracer series replaces (per-level edge fluxes in blocks of steps, the face tracer in torch, a product
summed over the levels and K3), the [0, nz] volume section and the plain series, alternating in one process, timed with
CUDA events.

    python tools/tracer_ab.py [--cases C3:f64:365,C3:f32:365,C4:f64:40] [--rounds 5] [--reps 1] [--out profiles/x.json]

Every round times each arm over --reps calls after one warm-up call; the median is over the rounds.  The defaults are
what profiles/r8_tracer_ab_C3_C4.json was measured with.

A case is workload:dtype:time steps (C4 with 40 steps is the one-GPU share of the 8-GPU run); level planes are padded
as bench.py pads them.  The tracer holds one value per step, level and cell (the thetao case) in the storage type of
u/v, with NaN on land and the marker 1e20 on every 97th cell (tools/classes_ab.py's class field).  The composition runs
over blocks of steps so that its per-level edge fluxes stay near 2 GB; it sums in another order than the kernel, so the
outputs are compared within 1e-12 of the sum of |w * E_k * q_k| of every entry.
"""
import argparse
import json
import os
import sys

import numpy
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from classes_ab import CFILL, class_field  # noqa: E402
from sparse_ab import gpu_info, setup  # noqa: E402


def face_tracer(tau, ny, nx):
    """(n, nz, 2 * ncell) float64 face values of tau (n, nz, ncell) in the [eU | eV] layout: eU[c] between c and its
    x-periodic east neighbour, eV[c] between c and its north neighbour (none in the top row); NaN and the marker are
    missing; the mean of two present sides, one present side, or 0"""
    n, nz = tau.shape[0], tau.shape[1]
    xs = tau.reshape(n, nz, ny, nx)
    ok = ~torch.isnan(xs) & (xs != xs.new_tensor(CFILL))                 # the marker compared in the storage type
    x = xs.double()
    x0 = torch.where(ok, x, 0.0)

    def face(b, okb):
        both = ok & okb
        return torch.where(both, 0.5 * (x0 + b), torch.where(ok, x0, torch.where(okb, b, 0.0)))
    qe = face(torch.roll(x0, -1, 3), torch.roll(ok, -1, 3))
    bn = torch.zeros_like(x0)
    okn = torch.zeros_like(ok)
    bn[:, :, :-1], okn[:, :, :-1] = x0[:, :, 1:], ok[:, :, 1:]
    qn = face(bn, okn)
    return torch.cat([qe.reshape(n, nz, -1), qn.reshape(n, nz, -1)], 2)


def composition(p, u, v, th, a1, a2, tau, ny, nx, out, block, bar=None):
    """the tracer series from per-level edge fluxes: fluxSeries(layers=range(nz + 1), eflux=) over blocks of steps,
    times the face tracer, summed over the levels, then K3 (integrate); bar: the sum of |w * E_k * q_k| per entry"""
    nt, nz = u.shape[0], u.shape[1]
    ncell = ny * nx
    levels = list(range(nz + 1))
    ef = torch.empty((block, nz, 2 * ncell), dtype=torch.float64, device=u.device)
    if bar is not None:
        sub = p.getSubsegments()
        cell = sub['cell'].astype(numpy.int64)
        j, i = cell // nx, cell % nx
        idx = numpy.stack([numpy.where(j >= 1, ncell + cell - nx, 0), cell, ncell + cell,
                           numpy.where(i >= 1, cell - 1, cell + nx - 1)], 1)
        w = numpy.where(numpy.stack([j >= 1] + [j >= 0] * 3, 1), numpy.abs(sub['w']), 0.0)
        idx_t, w_t = torch.from_numpy(idx).to(u.device), torch.from_numpy(w).to(u.device)
        tr_of = torch.from_numpy(numpy.repeat(numpy.arange(len(sub['offsets']) - 1), numpy.diff(sub['offsets']))).to(
            u.device)
    for t0 in range(0, nt, block):
        n = min(block, nt - t0)
        e = ef[:n]
        p.fluxSeries(u[t0:t0 + n], v[t0:t0 + n], th, a1, a2, layers=levels, eflux=e)
        q = face_tracer(tau[t0:t0 + n], ny, nx)
        out[t0:t0 + n] = p.integrate((e * q).sum(1))
        if bar is not None:
            g = (e * q).abs().sum(1)                                      # (n, 2 * ncell)
            per = (g[:, idx_t] * w_t).sum(-1)                              # (n, nsub)
            bar[t0:t0 + n] = torch.zeros_like(bar[t0:t0 + n]).index_add_(1, tr_of, per)
        del q
    return out


def run_case(name, dtype, nt, a):
    dev = torch.device('cuda', 0)
    syn, g, p = setup(name)
    tdt = torch.float32 if dtype == 'f32' else torch.float64
    pad = 8 if dtype == 'f32' else 4
    u, v = syn.fill_device(0, nt, dev, dtype=tdt, pad=pad)
    th, a1, a2 = (torch.from_numpy(x).to(dev) for x in (syn.thickness, syn.arc1, syn.arc2))
    nz, M, ncell, ny, nx = syn.nz, syn.ntransects, syn.ncell, syn.ny, syn.nx
    nsub = p.getNumberOfSubsegments()
    tau = class_field(u, nt, nz, ncell)
    block = max(1, min(nt, int(2e9 // (8 * nz * 2 * ncell))))
    arms = ['tracer series [0, nz]', 'tracer section per level', 'composition', 'volume section [0, nz]',
            'plain series']
    times = {m: [] for m in arms}
    comp = torch.empty((nt, M), dtype=torch.float64, device=dev)

    def call(arm, keep):
        if arm == 'tracer series [0, nz]':
            return p.fluxTracer(u, v, th, a1, a2, tau, tfill=CFILL)
        if arm == 'tracer section per level':
            keep['sec'] = p.fluxTracer(u, v, th, a1, a2, tau, tfill=CFILL, section=True)
            return None
        if arm == 'composition':
            return composition(p, u, v, th, a1, a2, tau, ny, nx, comp, block)
        if arm == 'volume section [0, nz]':
            return p.fluxSection(u, v, th, a1, a2, layers=[0, nz])
        return p.fluxSeries(u, v, th, a1, a2)
    for _ in range(a.rounds):
        for arm in arms:
            keep = {}
            call(arm, keep)                 # warm-up
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(a.reps):
                keep.pop('sec', None)
                call(arm, keep)
            e1.record()
            torch.cuda.synchronize()
            times[arm].append(e0.elapsed_time(e1) / a.reps)
            del keep                        # one per-level section alive at a time: 12.6 GB at C3 f64 x 365
            torch.cuda.empty_cache()
    got = p.fluxTracer(u, v, th, a1, a2, tau, tfill=CFILL).cpu().numpy()
    again = p.fluxTracer(u, v, th, a1, a2, tau, tfill=CFILL).cpu().numpy()
    bar = torch.empty_like(comp)
    ref = composition(p, u, v, th, a1, a2, tau, ny, nx, comp, block, bar).cpu().numpy()
    bar = bar.cpu().numpy()
    err = numpy.abs(got - ref)
    ok = bool((err <= 1e-12 * bar + 1e-300).all())
    rows = []
    base = float(numpy.median(times['volume section [0, nz]']))
    for arm in arms:
        ts = times[arm]
        med = float(numpy.median(ts))
        rows.append(dict(arm=arm, ms_median=med, ms_min=float(min(ts)), ms_max=float(max(ts)), ms_all=ts,
                         x_volume_section=med / base))
    print(f'{name} {dtype} nt={nt}: {nsub} crossings, {M} transects, composition blocks of {block} steps; '
          f'tracer series vs composition within 1e-12 * sum|terms|: {ok} '
          f'(max rel {float((err / (bar + 1e-300)).max()):.2e}); repeat bit-identical: '
          f'{bool(numpy.array_equal(got, again))}')
    for r in rows:
        print(f'  {r["arm"]:26s} median {r["ms_median"]:9.3f} ms  [{r["ms_min"]:.3f} .. {r["ms_max"]:.3f}]  '
              f'x{r["x_volume_section"]:.3f} of the [0, nz] volume section')
    del u, v, tau
    torch.cuda.empty_cache()
    return dict(workload=name, dtype=dtype, nt=nt, nsub=nsub, ntransects=M, composition_block_steps=block,
                tracer_matches_composition=ok, tracer_repeat_identical=bool(numpy.array_equal(got, again)),
                rows=rows)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--cases', default='C3:f64:365,C3:f32:365,C4:f64:40')
    ap.add_argument('--rounds', type=int, default=5)
    ap.add_argument('--reps', type=int, default=1)
    ap.add_argument('--out', default='')
    a = ap.parse_args()
    info = gpu_info()
    print(info)
    cases = [run_case(n, d, int(t), a) for n, d, t in (c.split(':') for c in a.cases.split(','))]
    print(gpu_info())
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, 'w') as f:
            json.dump(dict(gpu=info, rounds=a.rounds, reps=a.reps, cases=cases), f, indent=1)


if __name__ == '__main__':
    main()
