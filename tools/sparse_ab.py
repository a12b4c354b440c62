"""Same-box A/B of the fused flux-series pass: dense (every column of u, v) against sparse (only the column groups the
transects read, NFX_OPT_SPARSE_COLUMNS), alternating in one process, with the series compared bit for bit.

    python tools/sparse_ab.py [--cases C3:f64:365,C3:f32:365,C4:f64:40,C5:f64:8] [--rounds 5] [--out profiles/x.json]

A case is workload:dtype:time steps; C4 with 40 and C5 with 8 steps are the one-GPU shares of the 8-GPU runs.  Level
planes are padded as bench.py pads them (32-byte rows).  Besides the times it reports the bytes the column groups
cover, and the read-only ceilings of the device: nfx_probe_read_bandwidth (every column) and its group-list variant
walked with the C3 float64 group list, the access pattern of the sparse pass on the flagship workload.
"""
import argparse
import json
import os
import subprocess
import sys

import numpy
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from nemoflux_b200 import _lib, nemoflux_gpu, synth  # noqa: E402


def gpu_info():
    info = dict(torch_name=torch.cuda.get_device_name(0))
    try:
        q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.sm,clocks.max.sm', '--format=csv,noheader'],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        info['nvidia_smi'] = q[0] if q else ''
    except (OSError, subprocess.SubprocessError) as e:
        info['nvidia_smi'] = f'unavailable: {e}'
    return info


def setup(name):
    syn = synth.make(name)
    g = nemoflux_gpu.Grid()
    g.setPoints(syn.points)
    g.setCGridShape(syn.ny, syn.nx)
    p = nemoflux_gpu.PolylineIntegral()
    p.build(g)
    p.computeWeights(syn.transects)
    return syn, g, p


def probe_ceilings(reps):
    """(dense GB/s, sparse GB/s, share of the plane's vectors) with the C3 float64 group list (vec 4, one panel)"""
    syn, g, p = setup('C3')
    offs, grp = p.getColumnGroups('float64', 'map', 4)
    assert offs.size == 2, 'C3 is one panel'
    dev = torch.device('cuda', 0)
    buf = torch.empty(int(9.4e9) // 8, dtype=torch.float64, device=dev)
    dense = nemoflux_gpu.probeReadBandwidth(buf, reps=reps)
    sparse = nemoflux_gpu.probeReadBandwidth(buf, reps=reps, groups=torch.from_numpy(grp).to(dev))
    del buf
    torch.cuda.empty_cache()
    return dense, sparse, grp.size / ((syn.ncell + 3) // 4)


def run_case(name, dtype, nt, a, ceil):
    dev = torch.device('cuda', 0)
    syn, g, p = setup(name)
    tdt = torch.float32 if dtype == 'f32' else torch.float64
    esize = 4 if dtype == 'f32' else 8
    pad = 8 if dtype == 'f32' else 4
    u, v = syn.fill_device(0, nt, dev, dtype=tdt, pad=pad)
    th, a1, a2 = (torch.from_numpy(x).to(dev) for x in (syn.thickness, syn.arc1, syn.arc2))
    out = torch.empty((nt, syn.ntransects), dtype=torch.float64, device=dev)
    # the pass's vector width: 256-bit rows for float64, 128-bit for float32 (default fused shape 45)
    vec = 4
    offs, grp = p.getColumnGroups('float32' if dtype == 'f32' else 'float64', 'map', vec)
    dense_bytes = 2.0 * esize * syn.nz * syn.ncell * nt
    sparse_bytes = 2.0 * esize * syn.nz * vec * grp.size * nt
    modes = [('dense', {_lib.NFX_OPT_SPARSE_COLUMNS: 0}), ('sparse', {_lib.NFX_OPT_SPARSE_COLUMNS: 2})]
    for mb in a.ring_max_mb:
        modes.append((f'sparse ring<={mb}MB', {_lib.NFX_OPT_SPARSE_COLUMNS: 2, _lib.NFX_OPT_RING_MAX_MB: mb}))
    times = {m: [] for m, _ in modes}
    ref, same = None, True
    for _ in range(a.rounds):
        for mname, opts in modes:
            full = {_lib.NFX_OPT_SPARSE_COLUMNS: 1, _lib.NFX_OPT_RING_MAX_MB: 0}
            full.update(opts)
            for k, val in full.items():
                _lib.set_option(k, val)
            p.fluxSeries(u, v, th, a1, a2, out=out)          # warm-up (builds the group list on the first call)
            torch.cuda.synchronize()
            assert _lib.get_option(_lib.NFX_OPT_LAST_SERIES_PATH) == 1
            assert _lib.get_option(_lib.NFX_OPT_LAST_SERIES_SPARSE) == (0 if mname == 'dense' else 1)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(a.reps):
                p.fluxSeries(u, v, th, a1, a2, out=out)
            e1.record()
            torch.cuda.synchronize()
            p.seriesStatus()
            times[mname].append(e0.elapsed_time(e1) / a.reps)
            res = out.cpu().numpy().copy()
            if ref is None:
                ref = res
            same = same and bool(numpy.array_equal(res, ref, equal_nan=True))
    _lib.set_option(_lib.NFX_OPT_SPARSE_COLUMNS, 1)
    _lib.set_option(_lib.NFX_OPT_RING_MAX_MB, 0)
    rows = []
    for mname, ts in times.items():
        med = float(numpy.median(ts))
        nb = dense_bytes if mname == 'dense' else sparse_bytes
        rate = nb / med / 1e6
        ceiling = ceil['dense_gbs'] if mname == 'dense' else ceil['sparse_gbs']
        rows.append(dict(mode=mname, ms_median=med, ms_min=float(min(ts)), ms_max=float(max(ts)), ms_all=ts,
                         bytes=nb, gbs=rate, frac_of_probe=rate / ceiling))
    d = rows[0]['ms_median']
    print(f'{name} {dtype} nt={nt}: groups cover {grp.size * vec / syn.ncell:.3f} of the columns '
          f'({len(offs) - 1} panels), series identical: {same}')
    for r in rows:
        print(f'  {r["mode"]:20s} median {r["ms_median"]:9.3f} ms  [{r["ms_min"]:.3f} .. {r["ms_max"]:.3f}]  '
              f'x{d / r["ms_median"]:.3f}  {r["gbs"]:7.0f} GB/s over its bytes = {r["frac_of_probe"]:.3f} of its probe')
    del u, v
    torch.cuda.empty_cache()
    return dict(workload=name, dtype=dtype, nt=nt, vec=vec, npanels=len(offs) - 1, ngroups=int(grp.size),
                group_share=grp.size * vec / syn.ncell, series_bit_identical=same, rows=rows,
                speedup=d / rows[1]['ms_median'])


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--cases', default='C3:f64:365,C3:f32:365,C4:f64:40,C5:f64:8')
    ap.add_argument('--rounds', type=int, default=5)
    ap.add_argument('--reps', type=int, default=3)
    ap.add_argument('--ring-max-mb', default='', help='extra sparse modes with these NFX_OPT_RING_MAX_MB values, e.g. 32,48')
    ap.add_argument('--out', default='')
    a = ap.parse_args()
    a.ring_max_mb = [int(x) for x in a.ring_max_mb.split(',') if x]
    info = gpu_info()
    print(info)
    dense, sparse, share = probe_ceilings(5)
    ceil = dict(dense_gbs=dense, sparse_gbs=sparse, sparse_pattern='C3 float64 group list, vec 4',
                sparse_pattern_share=share)
    print(f'read-only probe: every column {dense:.0f} GB/s, C3 group list ({share:.3f} of the vectors) {sparse:.0f} GB/s '
          f'= {sparse / dense:.3f} of the dense rate')
    cases = []
    for c in a.cases.split(','):
        name, dtype, nt = c.split(':')
        cases.append(run_case(name, dtype, int(nt), a, ceil))
    print(gpu_info())
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, 'w') as f:
            json.dump(dict(gpu=info, probe=ceil, rounds=a.rounds, reps=a.reps, cases=cases), f, indent=1)


if __name__ == '__main__':
    main()
