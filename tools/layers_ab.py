"""Same-box A/B of the layered flux series (fluxSeries(layers=)): the plain series against one layer [0, nz], five layers
of 15 levels and one layer per level, alternating in one process, timed with CUDA events around fluxSeries.

    python tools/layers_ab.py [--cases C3:f64:365,C3:f32:365,C4:f64:40] [--rounds 5] [--out profiles/x.json]

A case is workload:dtype:time steps (C4 with 40 steps is the one-GPU share of the 8-GPU run); level planes are padded
as bench.py pads them.  The one-layer series must be the plain series bit for bit, and the layers must add up to it.
--split adds a torch.profiler run per case of the per-level series: the fused pass (one kernel) against the two-launch
path (K2 into HBM, then K3), whose kernel times say how much of the per-level time is K3's gathers.
"""
import argparse
import json
import os
import sys

import numpy
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from nemoflux_b200 import _lib  # noqa: E402
from sparse_ab import gpu_info, setup  # noqa: E402


def arms(nz):
    return [('plain', None), ('one layer', [0, nz]), ('5 x 15 levels', list(range(0, nz + 1, nz // 5))),
            ('per level', list(range(nz + 1)))]


def kernel_split(p, u, v, th, a1, a2, layers, nt_split):
    """CUDA time per kernel name of one per-level call on the first nt_split steps: fused, and two launches"""
    from torch.profiler import ProfilerActivity, profile
    ncell = a1.numel()
    res = {}
    us, vs = u[:nt_split], v[:nt_split]
    eflux = torch.empty((nt_split, len(layers) - 1, 2 * ncell), dtype=torch.float64, device=u.device)
    for mode, ef in (('fused', None), ('two launches', eflux)):
        p.fluxSeries(us, vs, th, a1, a2, layers=layers, eflux=ef)
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            p.fluxSeries(us, vs, th, a1, a2, layers=layers, eflux=ef)
            torch.cuda.synchronize()
        ks = {}
        for e in prof.key_averages():
            t = getattr(e, 'device_time_total', None)
            if t is None:
                t = e.cuda_time_total
            if t > 0:
                ks[e.key[:90]] = ks.get(e.key[:90], 0.0) + t / 1e3
        res[mode] = dict(nt=nt_split, kernels_ms=ks)
    del eflux
    torch.cuda.empty_cache()
    return res


def run_case(name, dtype, nt, a):
    dev = torch.device('cuda', 0)
    syn, g, p = setup(name)
    tdt = torch.float32 if dtype == 'f32' else torch.float64
    pad = 8 if dtype == 'f32' else 4
    u, v = syn.fill_device(0, nt, dev, dtype=tdt, pad=pad)
    th, a1, a2 = (torch.from_numpy(x).to(dev) for x in (syn.thickness, syn.arc1, syn.arc2))
    modes = arms(syn.nz)
    outs = {m: torch.empty((nt, syn.ntransects) if L is None else (nt, len(L) - 1, syn.ntransects), dtype=torch.float64,
                           device=dev) for m, L in modes}
    times = {m: [] for m, _ in modes}
    for _ in range(a.rounds):
        for mname, L in modes:
            p.fluxSeries(u, v, th, a1, a2, out=outs[mname], layers=L)          # warm-up
            torch.cuda.synchronize()
            assert _lib.get_option(_lib.NFX_OPT_LAST_SERIES_PATH) == 1
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(a.reps):
                p.fluxSeries(u, v, th, a1, a2, out=outs[mname], layers=L)
            e1.record()
            torch.cuda.synchronize()
            p.seriesStatus()
            times[mname].append(e0.elapsed_time(e1) / a.reps)
    res = {m: outs[m].cpu().numpy() for m, _ in modes}
    plain = res['plain']
    scale = float(numpy.abs(plain).max())
    one_same = bool(numpy.array_equal(res['one layer'][:, 0], plain))
    sums = {m: float(numpy.abs(res[m].sum(axis=1) - plain).max() / scale) for m, L in modes if L is not None}
    rows = []
    base = float(numpy.median(times['plain']))
    for mname, L in modes:
        ts = times[mname]
        med = float(numpy.median(ts))
        rows.append(dict(arm=mname, nlayers=1 if L is None else len(L) - 1, ms_median=med, ms_min=float(min(ts)),
                         ms_max=float(max(ts)), ms_all=ts, x_plain=med / base))
    print(f'{name} {dtype} nt={nt}: one layer == plain bit for bit: {one_same}; '
          f'max |sum of layers - plain| / max |plain|: {sums}')
    for r in rows:
        print(f'  {r["arm"]:14s} median {r["ms_median"]:9.3f} ms  [{r["ms_min"]:.3f} .. {r["ms_max"]:.3f}]  '
              f'x{r["x_plain"]:.3f} of the plain pass')
    split = None
    if a.split:
        split = kernel_split(p, u, v, th, a1, a2, modes[-1][1], min(nt, a.split_steps))
        for mode, d in split.items():
            print(f'  per level, {mode} ({d["nt"]} steps): ' +
                  ', '.join(f'{k}: {t:.3f} ms' for k, t in sorted(d['kernels_ms'].items(), key=lambda kv: -kv[1])[:4]))
    del u, v, outs
    torch.cuda.empty_cache()
    return dict(workload=name, dtype=dtype, nt=nt, one_layer_bit_identical=one_same, layer_sum_rel_err=sums, rows=rows,
                per_level_kernel_split=split)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--cases', default='C3:f64:365,C3:f32:365,C4:f64:40')
    ap.add_argument('--rounds', type=int, default=5)
    ap.add_argument('--reps', type=int, default=3)
    ap.add_argument('--split', action='store_true', help='torch.profiler kernel split of the per-level series')
    ap.add_argument('--split-steps', type=int, default=40)
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
