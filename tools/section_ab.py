"""Same-box A/B of the transport section (fluxSection): the plain series, the per-level layered series, and the section
over [0, nz], five layers of 15 levels and one layer per level, alternating in one process, timed with CUDA events.

    python tools/section_ab.py [--cases C3:f64:365,C3:f32:365,C4:f64:40] [--rounds 5] [--out profiles/x.json]

A case is workload:dtype:time steps (C4 with 40 steps is the one-GPU share of the 8-GPU run); level planes are padded
as bench.py pads them.  Every case reports the section's byte model: the 32-byte sectors of u and v that the list
index touches (counted on the host, per level plane) times nz and nt, plus the 8 bytes of every section value written;
and the rate each section arm reaches against that model, next to the read ceiling of the sparse fused pattern
(probeReadBandwidth(groups=), C3 group list) and the dense read ceiling.  The section's crossings must add up to the
layered series of the same layering (max error relative to the transect's sum of |w * f| is printed).
"""
import argparse
import json
import os
import sys

import numpy
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from sparse_ab import gpu_info, probe_ceilings, setup  # noqa: E402


def layerings(nz):
    return {'[0, nz]': [0, nz], '5 x 15 levels': list(range(0, nz + 1, nz // 5)), 'per level': list(range(nz + 1))}


def sector_bytes(p, ny, nx, esize):
    """bytes of the distinct 32-byte sectors of one level plane of u and of v that the list index reads"""
    ncell = ny * nx
    cell = p.getSubsegments()['cell']
    j, i = cell // nx, cell % nx
    uc = numpy.concatenate([cell, numpy.where(i >= 1, cell - 1, cell + nx - 1)])
    vc = numpy.concatenate([cell, cell[j >= 1] - nx])
    assert uc.max(initial=0) < ncell and vc.max(initial=0) < ncell
    return 32 * (numpy.unique(uc * esize // 32).size + numpy.unique(vc * esize // 32).size)


def run_case(name, dtype, nt, a):
    dev = torch.device('cuda', 0)
    syn, g, p = setup(name)
    tdt = torch.float32 if dtype == 'f32' else torch.float64
    pad = 8 if dtype == 'f32' else 4
    u, v = syn.fill_device(0, nt, dev, dtype=tdt, pad=pad)
    th, a1, a2 = (torch.from_numpy(x).to(dev) for x in (syn.thickness, syn.arc1, syn.arc2))
    nz, M = syn.nz, syn.ntransects
    nsub = p.getNumberOfSubsegments()
    lays = layerings(nz)
    arms = [('series plain', 'series', None), ('series per level', 'series', lays['per level'])] + \
        [(f'section {k}', 'section', L) for k, L in lays.items()]

    def out_for(kind, L):
        if kind == 'series':
            return torch.empty((nt, M) if L is None else (nt, len(L) - 1, M), dtype=torch.float64, device=dev)
        return torch.empty((nt, len(L) - 1, nsub), dtype=torch.float64, device=dev)

    def call(kind, L, out):
        if kind == 'series':
            p.fluxSeries(u, v, th, a1, a2, out=out, layers=L)
        else:
            p.fluxSection(u, v, th, a1, a2, out=out, layers=L)
    times = {m: [] for m, _, _ in arms}
    outs = {}
    for _ in range(a.rounds):
        for mname, kind, L in arms:
            out = out_for(kind, L)          # one output alive at a time: a per-level C3 section is 12.6 GB
            call(kind, L, out)              # warm-up
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(a.reps):
                call(kind, L, out)
            e1.record()
            torch.cuda.synchronize()
            p.seriesStatus()
            times[mname].append(e0.elapsed_time(e1) / a.reps)
            if kind == 'series' or mname not in outs:
                # the section is summed per transect on the device (float64, crossing order) and kept with the series
                offs = torch.from_numpy(p.getSubsegments()['offsets']).to(dev)
                outs[mname] = out.cpu().numpy() if kind == 'series' else torch.stack(
                    [out[..., int(offs[m]):int(offs[m + 1])].sum(-1) for m in range(M)], -1).cpu().numpy()
            del out
            torch.cuda.empty_cache()
    # sums of the crossings against the layered series of the same layering
    sums = {}
    for k, L in lays.items():
        ser = p.fluxSeries(u, v, th, a1, a2, layers=L).cpu().numpy()
        sums[k] = float(numpy.abs(outs[f'section {k}'] - ser).max() / max(numpy.abs(ser).max(), 1e-300))
    esize = 4 if dtype == 'f32' else 8
    read = sector_bytes(p, syn.ny, syn.nx, esize) * nz * nt
    dense = 2 * esize * syn.ncell * nz * nt
    base = float(numpy.median(times['series plain']))
    layered = float(numpy.median(times['series per level']))
    rows = []
    for mname, kind, L in arms:
        ts = times[mname]
        med = float(numpy.median(ts))
        row = dict(arm=mname, nlayers=1 if L is None else len(L) - 1, ms_median=med, ms_min=float(min(ts)),
                   ms_max=float(max(ts)), ms_all=ts, x_plain=med / base, x_per_level_series=med / layered)
        if kind == 'section':
            written = 8 * nt * (len(L) - 1) * nsub
            row.update(model_bytes_read=read, model_bytes_written=written,
                       model_GBps=(read + written) / (med * 1e-3) / 1e9)
        rows.append(row)
    print(f'{name} {dtype} nt={nt}: {nsub} crossings; u/v sectors read per step {read / nt / 1e6:.1f} MB '
          f'(dense planes {dense / nt / 1e6:.1f} MB); max |crossing sum - layered series| / max |series|: {sums}')
    for r in rows:
        extra = f'  {r["model_GBps"]:7.1f} GB/s of the byte model' if 'model_GBps' in r else ''
        print(f'  {r["arm"]:22s} median {r["ms_median"]:9.3f} ms  [{r["ms_min"]:.3f} .. {r["ms_max"]:.3f}]  '
              f'x{r["x_plain"]:.2f} of the plain series, x{r["x_per_level_series"]:.3f} of the per-level series'
              + extra)
    del u, v
    torch.cuda.empty_cache()
    return dict(workload=name, dtype=dtype, nt=nt, nsub=nsub, ntransects=M, sector_bytes_read=read,
                dense_bytes_read=dense, crossing_sum_rel_err=sums, rows=rows)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--cases', default='C3:f64:365,C3:f32:365,C4:f64:40')
    ap.add_argument('--rounds', type=int, default=5)
    ap.add_argument('--reps', type=int, default=3)
    ap.add_argument('--probe-reps', type=int, default=5)
    ap.add_argument('--out', default='')
    a = ap.parse_args()
    info = gpu_info()
    print(info)
    dense_gbps, sparse_gbps, share = probe_ceilings(a.probe_reps)
    print(f'read ceilings: dense {dense_gbps:.1f} GB/s, C3 sparse-group pattern {sparse_gbps:.1f} GB/s '
          f'({share:.2f} of the plane)')
    cases = [run_case(n, d, int(t), a) for n, d, t in (c.split(':') for c in a.cases.split(','))]
    for c in cases:
        for r in c['rows']:
            if 'model_GBps' in r:
                r['model_over_sparse_ceiling'] = r['model_GBps'] / sparse_gbps
    print(gpu_info())
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, 'w') as f:
            json.dump(dict(gpu=info, read_ceiling_dense_GBps=dense_gbps, read_ceiling_sparse_GBps=sparse_gbps,
                           rounds=a.rounds, reps=a.reps, cases=cases), f, indent=1)


if __name__ == '__main__':
    main()
