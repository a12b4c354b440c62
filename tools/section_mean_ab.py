"""Same-box A/B of the time-mean transport section (fluxSection(windows=)) against the per-step section, alternating
in one process, timed with CUDA events.

    python tools/section_mean_ab.py [--cases C3:f64:365,C3:f32:365,C4:f64:40] [--rounds 3] [--out profiles/x.json]

A case is workload:dtype:time steps (C4 with 40 steps is the one-GPU share of the 8-GPU run); level planes are padded
as bench.py pads them.  For each layering ([0, nz], five layers of 15 levels, one layer per level) the arms are the
per-step section and the windowed section with windows of 1 step, 30 steps and the whole record.  Every windowed
output is checked against the per-step output of the same process averaged on the device with the definition (a
sequential float64 sum over the window's steps from +0, then one division): bit_identical must hold.  The byte model
is the section's: the 32-byte sectors of u and v the list index touches per level plane (section_ab.sector_bytes) times
nz and nt, plus 8 bytes per value written.  The device memory of the host entry point (two slots of the windows a chunk
of the default size touches) is stated next to nt * nlayers * nsub, the output the per-step host entry point stages.
"""
import argparse
import json
import os
import sys

import numpy
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from sparse_ab import gpu_info, setup  # noqa: E402
from section_ab import layerings, sector_bytes  # noqa: E402


def windows_of(nt, n):
    return list(range(0, nt, n)) + [nt]


def device_mean(sec, bounds):
    """the definition on the device: acc = +0, acc = acc + sec[t] in ascending t, then acc / length"""
    out = torch.empty((len(bounds) - 1,) + tuple(sec.shape[1:]), dtype=torch.float64, device=sec.device)
    for w in range(len(bounds) - 1):
        acc = torch.zeros(sec.shape[1:], dtype=torch.float64, device=sec.device)
        for t in range(bounds[w], bounds[w + 1]):
            acc = acc + sec[t]
        out[w] = acc / torch.full((1,), float(bounds[w + 1] - bounds[w]), dtype=torch.float64, device=sec.device)
    return out


def host_staging_bytes(nt, bounds, step_bytes, row_bytes):
    """device bytes of the window staging of nfx_flux_section_window_sums_host at the default chunk size (256 MB per
    variable and slot, as host_pipeline picks it): two slots of the most windows a chunk touches"""
    cs = min(max(1, (256 << 20) // step_bytes), nt)
    b = numpy.asarray(bounds)
    most = 1
    for t0 in range(0, nt, cs):
        n = min(cs, nt - t0)
        wa = int(numpy.searchsorted(b, t0, 'right')) - 1
        wb = int(numpy.searchsorted(b, t0 + n, 'left'))
        most = max(most, wb - wa)
    return 2 * most * row_bytes, cs


def run_case(name, dtype, nt, a):
    dev = torch.device('cuda', 0)
    syn, g, p = setup(name)
    tdt = torch.float32 if dtype == 'f32' else torch.float64
    pad = 8 if dtype == 'f32' else 4
    u, v = syn.fill_device(0, nt, dev, dtype=tdt, pad=pad)
    th, a1, a2 = (torch.from_numpy(x).to(dev) for x in (syn.thickness, syn.arc1, syn.arc2))
    nz = syn.nz
    nsub = p.getNumberOfSubsegments()
    lays = layerings(nz)
    wins = {'1 step': windows_of(nt, 1), '30 steps': windows_of(nt, 30), 'whole record': [0, nt]}
    esize = 4 if dtype == 'f32' else 8
    read = sector_bytes(p, syn.ny, syn.nx, esize) * nz * nt
    arms = []
    for lk, L in lays.items():
        arms.append((f'section {lk}', lk, L, None))
        arms += [(f'mean {lk} / {wk}', lk, L, W) for wk, W in wins.items()]
    outs = {}
    for mname, lk, L, W in arms:
        shape = (nt if W is None else len(W) - 1, len(L) - 1, nsub)
        outs[mname] = torch.empty(shape, dtype=torch.float64, device=dev)

    def call(L, W, out):
        if W is None:
            p.fluxSection(u, v, th, a1, a2, out=out, layers=L)
        else:
            p.fluxSection(u, v, th, a1, a2, out=out, layers=L, windows=W)
    times = {m[0]: [] for m in arms}
    for _ in range(a.rounds):
        for mname, lk, L, W in arms:
            out = outs[mname]
            call(L, W, out)                 # warm-up
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(a.reps):
                call(L, W, out)
            e1.record()
            torch.cuda.synchronize()
            times[mname].append(e0.elapsed_time(e1) / a.reps)
    rows, checks = [], {}
    for mname, lk, L, W in arms:
        ts = times[mname]
        med = float(numpy.median(ts))
        base = float(numpy.median(times[f'section {lk}']))
        nvals = (nt if W is None else len(W) - 1) * (len(L) - 1) * nsub
        row = dict(arm=mname, layering=lk, nlayers=len(L) - 1, nwindows=None if W is None else len(W) - 1,
                   ms_median=med, ms_min=float(min(ts)), ms_max=float(max(ts)), ms_all=ts, x_per_step_section=med / base,
                   model_bytes_read=read, model_bytes_written=8 * nvals,
                   model_GBps=(read + 8 * nvals) / (med * 1e-3) / 1e9)
        if W is not None:
            ref = device_mean(outs[f'section {lk}'], W)
            got = outs[mname]
            same = bool(torch.equal(got, ref) and torch.equal(torch.signbit(got), torch.signbit(ref)))
            row['bit_identical'] = same
            row['max_abs_diff'] = float((got - ref).abs().max())
            checks[mname] = same
            del ref
            row_bytes = 8 * (len(L) - 1) * nsub
            stage, cs = host_staging_bytes(nt, W, esize * nz * syn.ncell, row_bytes)
            row.update(host_staging_bytes=stage, host_chunk_steps=cs, per_step_output_bytes=8 * nt * (len(L) - 1) * nsub)
        rows.append(row)
    print(f'{name} {dtype} nt={nt}: {nsub} crossings; u/v sectors read per step {read / nt / 1e6:.1f} MB')
    for r in rows:
        extra = ''
        if r['nwindows'] is not None:
            extra = (f'  bits {"identical" if r["bit_identical"] else "DIFFER"}; host staging '
                     f'{r["host_staging_bytes"] / 1e6:.1f} MB vs {r["per_step_output_bytes"] / 1e6:.1f} MB per-step')
        print(f'  {r["arm"]:34s} median {r["ms_median"]:9.3f} ms  [{r["ms_min"]:.3f} .. {r["ms_max"]:.3f}]  '
              f'x{r["x_per_step_section"]:.2f} of the per-step section  {r["model_GBps"]:7.1f} GB/s' + extra)
    del u, v, outs
    torch.cuda.empty_cache()
    return dict(workload=name, dtype=dtype, nt=nt, nsub=nsub, sector_bytes_read=read, all_bit_identical=all(
        checks.values()), rows=rows)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--cases', default='C3:f64:365,C3:f32:365,C4:f64:40')
    ap.add_argument('--rounds', type=int, default=3)
    ap.add_argument('--reps', type=int, default=3)
    ap.add_argument('--out', default='')
    a = ap.parse_args()
    info = gpu_info()
    print(info)
    cases = [run_case(n, d, int(t), a) for n, d, t in (c.split(':') for c in a.cases.split(','))]
    print(gpu_info())
    ok = all(c['all_bit_identical'] for c in cases)
    print('windowed outputs bit-identical to the averaged per-step outputs:', ok)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, 'w') as f:
            json.dump(dict(gpu=info, rounds=a.rounds, reps=a.reps, cases=cases), f, indent=1)
    return 0 if ok else 1


if __name__ == '__main__':
    sys.exit(main())
