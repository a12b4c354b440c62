"""Same-box A/B of the class transport (fluxClasses): the one-pass class kernel with 20 classes, the composition it
replaces (the per-level fluxSection, a torch gather of the class field at every crossing's cell and an index_add), and
the per-level section alone, alternating in one process, timed with CUDA events.

    python tools/classes_ab.py [--cases C3:f64:365,C3:f32:365,C4:f64:40] [--rounds 5] [--out profiles/x.json]

A case is workload:dtype:time steps (C4 with 40 steps is the one-GPU share of the 8-GPU run); level planes are padded
as bench.py pads them.  The class field holds one value per step, level and cell (ct = nt, the thetao case) in the
storage type of u/v, with NaN on land and the marker 1e20 on a band of cells.  The composition runs over blocks of
steps so that its temporaries stay near 2 GB (the per-level section of a C3 year alone is 12.6 GB); its index_add is
not deterministic, so the outputs are compared within 1e-12 of the sum of |f| of every entry.
"""
import argparse
import json
import os
import sys

import numpy
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from sparse_ab import gpu_info, setup  # noqa: E402

CFILL = 1e20


def class_field(u, nt, nz, ncell):
    """(nt, nz, cells) with u's dtype and plane layout: 18 k / nz + 2 sin(cell / 900 + t / 10), NaN where u is NaN (land)
    and the marker on every 97th cell"""
    dev = u.device
    if u.dim() == 3:
        ld = u.stride(1)
        c = torch.empty((nt, nz, ld), dtype=u.dtype, device=dev)[:, :, :ncell]
    else:
        c = torch.empty_like(u).view(nt, nz, ncell)
    cells = torch.arange(ncell, device=dev, dtype=torch.float64)
    marked = (torch.arange(ncell, device=dev) % 97) == 0
    for t in range(nt):
        for k in range(nz):
            x = 18.0 * k / nz + 2.0 * torch.sin(cells / 900.0 + t / 10.0)
            x = torch.where(torch.isnan(u.reshape(nt, nz, ncell)[t, k].double()), float('nan'), x)
            c[t, k] = torch.where(marked, CFILL, x).to(u.dtype)
    return c


def composition(p, u, v, th, a1, a2, c, bounds, out, bar, block):
    """the classes from the per-level section: gather the class at every crossing's cell, bin it, index_add the flux"""
    nt, nz = u.shape[0], u.shape[1]
    sub = p.getSubsegments()
    cell = torch.from_numpy(sub['cell'].astype(numpy.int64)).to(u.device)
    tr_of = torch.from_numpy(numpy.repeat(numpy.arange(len(sub['offsets']) - 1), numpy.diff(sub['offsets']))).to(
        u.device)
    K, M = bounds.numel() - 1, out.shape[2]
    out.zero_()
    if bar is not None:
        bar.zero_()
    levels = list(range(nz + 1))
    for t0 in range(0, nt, block):
        n = min(block, nt - t0)
        sec = p.fluxSection(u[t0:t0 + n], v[t0:t0 + n], th, a1, a2, layers=levels)           # (n, nz, nsub)
        x = c[t0:t0 + n].reshape(n, nz, -1).index_select(2, cell).double()                   # (n, nz, nsub)
        j = torch.bucketize(x, bounds, right=True) - 1
        ok = ~torch.isnan(x) & (x != CFILL) & (j >= 0) & (j < K)
        tt = torch.arange(n, device=u.device).view(n, 1, 1)
        key = ((tt + t0) * K + j) * M + tr_of.view(1, 1, -1)
        out.view(-1).index_add_(0, key[ok], sec[ok])
        if bar is not None:
            bar.view(-1).index_add_(0, key[ok], sec[ok].abs())
        del sec, x, j, ok, key
    return out


def run_case(name, dtype, nt, a):
    dev = torch.device('cuda', 0)
    syn, g, p = setup(name)
    tdt = torch.float32 if dtype == 'f32' else torch.float64
    pad = 8 if dtype == 'f32' else 4
    u, v = syn.fill_device(0, nt, dev, dtype=tdt, pad=pad)
    th, a1, a2 = (torch.from_numpy(x).to(dev) for x in (syn.thickness, syn.arc1, syn.arc2))
    nz, M, ncell = syn.nz, syn.ntransects, syn.ncell
    nsub = p.getNumberOfSubsegments()
    c = class_field(u, nt, nz, ncell)
    bounds = numpy.linspace(-2.0, 20.0, a.classes + 1)
    bt = torch.from_numpy(bounds).to(dev)
    K = a.classes
    block = max(1, min(nt, int(2e9 // (8 * nz * max(nsub, 1)))))
    per_level = list(range(nz + 1))
    arms = ['classes', 'composition', 'section per level']
    times = {m: [] for m in arms}
    classes = torch.empty((nt, K, M), dtype=torch.float64, device=dev)
    comp = torch.empty_like(classes)

    def call(arm, keep):
        if arm == 'classes':
            return p.fluxClasses(u, v, th, a1, a2, c, bounds, cfill=CFILL)
        if arm == 'composition':
            return composition(p, u, v, th, a1, a2, c, bt, comp, None, block)
        keep['sec'] = p.fluxSection(u, v, th, a1, a2, layers=per_level, out=keep.get('sec'))
    for _ in range(a.rounds):
        for arm in arms:
            keep = {}
            call(arm, keep)                 # warm-up
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(a.reps):
                call(arm, keep)
            e1.record()
            torch.cuda.synchronize()
            times[arm].append(e0.elapsed_time(e1) / a.reps)
            del keep                        # one per-level section alive at a time: 12.6 GB at C3 f64 x 365
            torch.cuda.empty_cache()
    got = p.fluxClasses(u, v, th, a1, a2, c, bounds, cfill=CFILL).cpu().numpy()
    again = p.fluxClasses(u, v, th, a1, a2, c, bounds, cfill=CFILL).cpu().numpy()
    bar = torch.empty_like(classes)
    ref = composition(p, u, v, th, a1, a2, c, bt, comp, bar, block).cpu().numpy()
    bar = bar.cpu().numpy()
    err = numpy.abs(got - ref)
    ok = bool((err <= 1e-12 * bar + 1e-300).all())
    plain = p.fluxSeries(u, v, th, a1, a2).cpu().numpy()
    covered = float(numpy.abs(got.sum(1)).sum() / max(numpy.abs(plain).sum(), 1e-300))
    rows = []
    base = float(numpy.median(times['section per level']))
    for arm in arms:
        ts = times[arm]
        med = float(numpy.median(ts))
        rows.append(dict(arm=arm, ms_median=med, ms_min=float(min(ts)), ms_max=float(max(ts)), ms_all=ts,
                         x_section_per_level=med / base))
    print(f'{name} {dtype} nt={nt}: {nsub} crossings, {M} transects, {K} classes, composition blocks of {block} steps; '
          f'classes vs composition within 1e-12 * sum|f|: {ok} (max rel {float((err / (bar + 1e-300)).max()):.2e}); '
          f'repeat bit-identical: {bool(numpy.array_equal(got, again))}; |classes| / |plain series| = {covered:.3f}')
    for r in rows:
        print(f'  {r["arm"]:18s} median {r["ms_median"]:9.3f} ms  [{r["ms_min"]:.3f} .. {r["ms_max"]:.3f}]  '
              f'x{r["x_section_per_level"]:.3f} of the per-level section')
    del u, v, c
    torch.cuda.empty_cache()
    return dict(workload=name, dtype=dtype, nt=nt, nsub=nsub, ntransects=M, nclasses=K, composition_block_steps=block,
                classes_match_composition=ok, classes_repeat_identical=bool(numpy.array_equal(got, again)),
                rows=rows)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--cases', default='C3:f64:365,C3:f32:365,C4:f64:40')
    ap.add_argument('--classes', type=int, default=20)
    ap.add_argument('--rounds', type=int, default=5)
    ap.add_argument('--reps', type=int, default=3)
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
