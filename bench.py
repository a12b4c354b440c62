#!/usr/bin/env python
"""bench.py -- transect-flux throughput on synthetic ORCA-shaped data (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload auto|C3|C4|C5] [--dtype f64|f32] [--impl reference]
                    [--dump-outputs DIR]

One "step" = one pass of the hot path (K2 edge-flux assembly + K3 batched transect reduction, plus the NCCL
allgather of the flux series when N > 1) over the whole time series of the workload.

Workloads (BASELINE.json configs; `--workload auto`, the default, picks by N):
  N = 1   C3: ORCA1-shaped 362x332x75, 365 daily steps, 64 transects, all resident in HBM (52.6 GB).
  N >= 2  C4: ORCA025-shaped 1442x1021x75, 365 steps, 256 transects, STRONG scaling: the 365 steps are sharded by
          time over the ranks (fluxplot.py:51-59 carries no state between time steps), no u/v data crosses NVLink,
          the only collective is the allgather of the per-rank (nt_r, M) series.  Where a rank's shard exceeds HBM
          (N = 2: 323 GB) the rank holds a resident chunk, runs the pass per chunk and regenerates the next chunk
          OUTSIDE the timed region; the step time is the sum over the chunk passes of the max-over-ranks CUDA-event
          time (every chunk pass is bracketed by a barrier + synchronize).
  N = 8   additionally `target_c5`: BASELINE's target config C5 (ORCA12-shaped 4322x3059x75, 73 snapshots, 1024
          transects) in a second pass of the same run, sharded at (time step, panel) granularity (--balance).

Rank 0 prints ONE JSON line.  `value` = cell*level*timesteps per second with u, v resident in HBM; `e2e` = the same
metric through PolylineIntegral.fluxSeries() on pinned HOST arrays (H2D copies of u, v and the D2H copy of the series
inside the timed region; at N > 1 the host-fed time steps are apportioned by each rank's measured H2D rate);
`roofline` is for the fused K2+K3 pass, the dominant kernel: algorithmic bytes = 2*sizeof(dtype)*nz per cell and time
step (SURVEY.md 8d) over the CUDA-event duration of its launches; `cpu_baseline` times the CPU oracle on a bounded
sample (rank 0, N = 1).  Every line carries oracle parity: K1 lists bit for bit, flux error on one time step per rank.

--impl reference runs the reference's CPU path (numpy restatement of field.py:145-234 + the C restatement of mint's
getIntegral; the reference itself cannot run here: mint/xarray are absent) on a bounded sample of the same workload,
with the same `config` dict as the GPU arm.
"""
import argparse
import json
import math
import os
import subprocess
import sys
import tempfile
import time

import numpy

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = 'transect-flux cell*level*timesteps/sec'
UNIT = 'cell*level*timesteps/s'


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=20)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='b200', choices=['b200', 'reference'])
    ap.add_argument('--workload', default='auto', help='auto: C3 at N=1, C4 (strong, time-sharded) at N>=2')
    ap.add_argument('--nt-local', type=int, default=0, help='weak scaling: time steps resident per rank')
    ap.add_argument('--nt-total', type=int, default=0, help='strong scaling: shard this many time steps over the ranks')
    ap.add_argument('--balance', action='store_true',
                    help='shard at (time step, panel of cells) granularity so that every rank gets the same number of '
                         'batches (73 snapshots over 8 GPUs: 9.125 steps each instead of 10,9,..,9); single chunk only')
    ap.add_argument('--no-rate-balance', action='store_true',
                    help='--balance: equal batch counts per rank instead of counts proportional to the measured rates')
    ap.add_argument('--dtype', default='f64', choices=['f64', 'f32'], help='storage type of uo/vo (compute is f64)')
    ap.add_argument('--e2e-steps', type=int, default=0, help='time steps of the host-buffer (e2e) sample, all ranks together')
    ap.add_argument('--cpu-steps', type=int, default=0, help='time steps of the cpu_baseline / reference-arm sample')
    ap.add_argument('--no-cpu', action='store_true', help='skip cpu_baseline (parity against the oracle still runs)')
    ap.add_argument('--no-parity', action='store_true')
    ap.add_argument('--no-e2e', action='store_true')
    ap.add_argument('--no-target', action='store_true', help='N = 8: skip the target_c5 pass')
    ap.add_argument('--target-steps', type=int, default=10)
    ap.add_argument('--hbm-reserve-gb', type=float, default=8.0, help='HBM kept free of u/v when sizing resident chunks')
    ap.add_argument('--max-chunk-steps', type=int, default=0, help='cap the resident chunk (tests the chunked path)')
    ap.add_argument('--k2-variant', type=int, default=0)
    ap.add_argument('--k2-unroll', type=int, default=0)
    ap.add_argument('--k2-block', type=int, default=0)
    ap.add_argument('--order', default='map', choices=['map', 'list'])
    ap.add_argument('--classic', action='store_true',
                    help='K2 -> eflux in HBM -> K3 as two launches (default: the fused pass that keeps eflux in L2)')
    ap.add_argument('--ring-slot-mb', type=int, default=0)
    ap.add_argument('--no-pad', action='store_true',
                    help='store u/v densely; default: level planes padded to 32 bytes when ncell*itemsize is not')
    ap.add_argument('--dump-outputs', metavar='DIR', default='',
                    help='after the timed steps, write what the last step computed (the flux series) as DIR/<name>.npy')
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    return args


DUMP_BUDGET_BYTES = 64 << 20


def dump_outputs(path, arrays):
    """--dump-outputs: every array as float64 <path>/<name>.npy.  The inputs are a function of the arguments only
    (synth.py is seeded), so two builds run with the same arguments can be compared file for file.  Should the total
    pass 64 MB, every array keeps the same fixed stride of its rows (time steps)."""
    os.makedirs(path, exist_ok=True)
    stride = max(1, math.ceil(sum(a.size * 8 for a in arrays.values()) / DUMP_BUDGET_BYTES))
    for name, a in arrays.items():
        numpy.save(os.path.join(path, name + '.npy'), numpy.ascontiguousarray(a[::stride], numpy.float64))


def pick_workload(args, world):
    """(name, nt_total, scaling): BASELINE config for this N, or what the flags ask for"""
    from nemoflux_b200 import synth
    name = args.workload
    if name == 'auto':
        name = 'C3' if world == 1 else 'C4'
    nt = synth.CONFIGS[name]['nt']
    if args.nt_local > 0:
        return name, args.nt_local * world, 'weak'
    if args.nt_total > 0:
        return name, args.nt_total, 'strong'
    if world == 1:
        return name, nt, 'weak'
    return name, nt, 'strong'


def make_config(name, cfg, world, dtype, nt_total, scaling, balance=False):
    """the `config` of the JSON line: a function of (workload, N, dtype) only, so that both arms print the same dict"""
    esize = 8 if dtype == 'f64' else 4
    units = cfg['nx'] * cfg['ny'] * cfg['nz']
    from nemoflux_b200 import dist as nfx_dist
    return {'workload': f'{name}: {cfg["label"]}, {nt_total} time steps, {cfg["ntransects"]} transects, u/v stored {dtype}',
            'nx': cfg['nx'], 'ny': cfg['ny'], 'nz': cfg['nz'], 'nt_total': nt_total, 'transects': cfg['ntransects'],
            'storage_dtype': dtype, 'n_gpus': world,
            'sharding': ('(time step, panel of cells) batches, balanced' if balance else
                         f'time steps {nfx_dist.shard_counts(nt_total, world)}') + f' over {world} GPU(s), {scaling} scaling',
            'l2_policy': f'no flush: every pass streams {2 * esize * units * nt_total / world / 1e9:.1f} GB per GPU '
                         f'through a 126 MB L2'}


# ---------------------------------------------------------------------------------------------------
class ClockSampler(object):
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)"""
    Q = ('timestamp,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,'
         'clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,'
         'clocks_event_reasons.sw_power_cap')

    def __init__(self, index):
        self.index = index
        self.proc = None
        self.path = None

    def start(self):
        try:
            fd, self.path = tempfile.mkstemp(suffix='.csv')
            os.close(fd)
            self.proc = subprocess.Popen(['nvidia-smi', f'--query-gpu={self.Q}', '--format=csv,noheader,nounits',
                                          '-lms', '50', '-i', str(self.index)],
                                         stdout=open(self.path, 'w'), stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None
            return
        t0 = time.time()            # nvidia-smi takes a few 100 ms to print its first sample: wait for it, so that a
        while time.time() - t0 < 3.0:   # short timed region (float32 storage: 0.2 s) is not over before it starts
            try:
                if os.path.getsize(self.path) > 0:
                    break
            except OSError:
                break
            time.sleep(0.02)

    def stop(self, t_begin=None, t_end=None):
        """median SM clock / reasons of the samples taken between t_begin and t_end (time.time()); when the timed
        region is shorter than the sampling period, of the samples under load around it"""
        import datetime
        out = dict(sm_mhz=None, sm_max_mhz=None, reasons=[], samples=0)
        if self.proc is None:
            return out
        time.sleep(0.12)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        rows = []
        try:
            for line in open(self.path):
                f = [x.strip() for x in line.split(',')]
                if len(f) < 9:
                    continue
                try:
                    ts = datetime.datetime.strptime(f[0], '%Y/%m/%d %H:%M:%S.%f').timestamp()
                    rows.append((ts, float(f[1]), float(f[2]), float(f[3]), f[5:9]))
                except ValueError:
                    continue
            os.unlink(self.path)
        except Exception:
            pass
        if not rows:
            return out
        sel = [r for r in rows if t_begin is not None and t_begin - 0.05 <= r[0] <= t_end + 0.05]
        window = 'timed region'
        pmax = max(r[3] for r in rows)
        busy = [r for r in sel if r[3] >= 0.6 * pmax]
        if len(busy) >= 2:      # a chunked step regenerates data between passes: keep the samples under load
            sel = busy
        if len(sel) < 2:      # fall back to the samples under load (power above idle) of the whole run
            sel = [r for r in rows if r[3] >= 0.6 * pmax] or rows
            window = 'samples under load (warm-up + timed region)'
        reasons = set()
        for r in sel:
            for name, val in zip(('hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap'), r[4]):
                if val.lower().startswith('active'):
                    reasons.add(name)
        out.update(sm_mhz=float(numpy.median([r[1] for r in sel])), sm_max_mhz=float(max(r[2] for r in sel)),
                   reasons=sorted(reasons), samples=len(sel), window=window,
                   power_w_max=float(max(r[3] for r in sel)))
        return out


# ---------------------------------------------------------------------------------------------------
def cpu_reference_pass(O, syn, plis, fields, order, use_c=False):
    """the reference's per-time-step compute on the host; fields = [(u, v) (nz,ny,nx) per time step], already
    in memory (the reference reads them from NetCDF, field.py:149 -- I/O is not timed); returns (seconds, series)"""
    arc = numpy.zeros((syn.ncell, 4))
    arc[:, 1], arc[:, 2] = syn.arc1, syn.arc2
    out = numpy.zeros((len(fields), len(plis)))
    t0 = time.perf_counter()
    for n, (u, v) in enumerate(fields):
        if use_c:
            iV, _, _ = O.edgeflux_step_c(u, v, syn.thickness, syn.arc1, syn.arc2, False)
        else:
            U = O.read_field(u, syn.thickness)             # field.py:145-163
            V = O.read_field(v, syn.thickness)
            iV, _, _ = O.integrated_flux(U, V, arc, False)  # field.py:183-234
        for m, p in enumerate(plis):                       # fluxplot.py:55-57
            out[n, m] = p.getIntegral(iV, order)
    return time.perf_counter() - t0, out


def build_oracle_plis(O, syn):
    g = O.Grid(syn.points)
    plis = []
    for xyz in syn.transects:
        p = O.PolylineIntegral(g, 360.)
        p.computeWeights(xyz)
        plis.append(p)
    return g, plis


def all_host_threads():
    try:        # torchrun exports OMP_NUM_THREADS=1: give the BLAS behind numpy.tensordot all host threads back
        from threadpoolctl import threadpool_limits
        threadpool_limits(limits=os.cpu_count())
    except Exception:
        pass


def default_cpu_steps(args, syn):
    if args.cpu_steps > 0:
        return args.cpu_steps
    return max(1, min(24, int(5.2e9 // (16 * syn.units_per_step()))))     # C3: 24 steps, C4: 2, C5: 1


def run_reference(args):
    """--impl reference: CPU path on the host cores (rank 0 only)"""
    rank = int(os.environ.get('RANK', '0'))
    world = int(os.environ.get('WORLD_SIZE', str(args.gpus)))
    if rank != 0:
        return
    from nemoflux_b200 import synth
    from oracle import oracle as O
    O.lib()
    cores = os.cpu_count()
    all_host_threads()
    name, nt_total, scaling = pick_workload(args, world)
    syn = synth.make(name)
    g, plis = build_oracle_plis(O, syn)
    sample = min(default_cpu_steps(args, syn), nt_total)
    npdt = numpy.float64 if args.dtype == 'f64' else numpy.float32
    fields = [syn.uv_host(t, dtype=npdt) for t in range(sample)]
    for _ in range(max(args.warmup, 0)):
        cpu_reference_pass(O, syn, plis, fields[:1], args.order)
    times = []
    for _ in range(args.steps):
        dt, series = cpu_reference_pass(O, syn, plis, fields, args.order)
        times.append(dt)
    dt = float(numpy.mean(times))
    units = syn.units_per_step() * sample
    value = units / dt
    line = {
        'impl': 'reference', 'metric': METRIC, 'value': value, 'unit': UNIT, 'n_gpus': world, 'steps': args.steps,
        'warmup': args.warmup, 'ms_per_step': 1e3 * dt, 'higher_is_better': True, 'scaling': scaling,
        'vs_baseline': None, 'dtype': args.dtype, 'data': 'synthetic',
        'config': make_config(name, synth.CONFIGS[name], world, args.dtype, nt_total, scaling, args.balance),
        'cpu_baseline': {'value': value, 'unit': UNIT, 'cores': cores, 'kind': 'port',
                         'sample': f'{sample} of {nt_total} time steps of {name} ({units:.3e} units) per step, rank 0 only; '
                                   f'numpy restatement of field.py:145-234 (BLAS threads default) + C getIntegral per '
                                   f'transect'},
        'e2e': {'value': value, 'unit': UNIT, 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
        'gpu_launches': 0,
    }
    print(json.dumps(line), flush=True)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {'flux_series': series})


# ---------------------------------------------------------------------------------------------------
class Ctx(object):
    """process-wide state of the GPU arm"""

    def __init__(self):
        import torch
        import torch.distributed as dist
        self.torch, self.dist = torch, dist
        self.world = int(os.environ.get('WORLD_SIZE', '1'))
        self.rank = int(os.environ.get('RANK', '0'))
        self.local_rank = int(os.environ.get('LOCAL_RANK', '0'))
        assert torch.cuda.is_available(), 'bench.py needs a CUDA device (no CPU fallback)'
        torch.cuda.set_device(self.local_rank)
        self.dev = torch.device('cuda', self.local_rank)
        self.cpu_binding = 0
        if self.world > 1:
            os.environ.setdefault('MASTER_ADDR', '127.0.0.1')
            dist.init_process_group('nccl', device_id=self.dev)
            # one process per GPU: keep the rank (and the pinned host buffers of the e2e leg) on the CPUs next to its
            # GPU.  No effect where NVML reports no affinity (single-node VMs, profiles/r1_numa_probe8.md)
            from nemoflux_b200 import dist as _nd
            self.cpu_binding = _nd.bind_to_gpu_cpus(self.local_rank)

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def allreduce(self, values, op='max'):
        """elementwise max / min / sum over ranks of a list of floats"""
        t = self.torch.tensor([float(x) for x in values], dtype=self.torch.float64, device=self.dev)
        if self.world > 1:
            ops = {'max': self.dist.ReduceOp.MAX, 'min': self.dist.ReduceOp.MIN, 'sum': self.dist.ReduceOp.SUM}
            self.dist.all_reduce(t, op=ops[op])
        return [float(x) for x in t.cpu()]

    def allgather_floats(self, value):
        t = self.torch.tensor([float(value)], dtype=self.torch.float64, device=self.dev)
        if self.world == 1:
            return [float(value)]
        out = self.torch.empty(self.world, dtype=self.torch.float64, device=self.dev)
        self.dist.all_gather_into_tensor(out, t)
        return [float(x) for x in out.cpu()]


class Workload(object):
    """grid, locator, K1 weights and metric arrays of one BASELINE config on this rank's GPU"""

    def __init__(self, cx, name):
        from nemoflux_b200 import nemoflux_gpu, synth
        torch = cx.torch
        self.name = name
        self.syn = syn = synth.make(name)
        self.grid = nemoflux_gpu.Grid()
        self.grid.setPoints(syn.points)
        self.grid.setCGridShape(syn.ny, syn.nx)
        self.pli = nemoflux_gpu.PolylineIntegral()
        torch.cuda.synchronize()
        tk = time.perf_counter()
        self.pli.build(self.grid, periodX=360.)
        torch.cuda.synchronize()
        self.t_locator = time.perf_counter() - tk
        self.pli.computeWeights(syn.transects)      # first call: sizes the scratch arena (cudaMalloc) -- not the K1 time
        torch.cuda.synchronize()
        tk = time.perf_counter()
        self.pli.computeWeights(syn.transects)
        torch.cuda.synchronize()
        self.t_k1 = time.perf_counter() - tk
        self.thickness = torch.from_numpy(syn.thickness).to(cx.dev)
        self.arc1 = torch.from_numpy(syn.arc1).to(cx.dev)
        self.arc2 = torch.from_numpy(syn.arc2).to(cx.dev)
        self.M = syn.ntransects


def plan_chunks(cx, args, nt_local, step_bytes):
    """resident chunks of this rank's shard: [(offset, n)], the same number of chunks on every rank"""
    free, _total = cx.torch.cuda.mem_get_info(cx.dev)
    fit = max(1, int((free - args.hbm_reserve_gb * 1e9) // step_bytes))
    if args.max_chunk_steps > 0:
        fit = min(fit, args.max_chunk_steps)
    n = max(1, math.ceil(nt_local / fit))
    n = int(cx.allreduce([n], 'max')[0])
    base, rem = divmod(nt_local, n)
    chunks, off = [], 0
    for i in range(n):
        c = base + (1 if i < rem else 0)
        chunks.append((off, c))
        off += c
    return chunks, fit


def alloc_uv(cx, syn, cap, tdtype, pad):
    """u, v device buffers for `cap` time steps; padded level planes -> (cap, nz, ncell) views with stride(1) = ld"""
    torch = cx.torch
    if pad and syn.ncell % pad != 0:
        ld = (syn.ncell + pad - 1) // pad * pad
        bu = torch.zeros((cap, syn.nz, ld), dtype=tdtype, device=cx.dev)
        bv = torch.zeros((cap, syn.nz, ld), dtype=tdtype, device=cx.dev)
        return bu[:, :, :syn.ncell], bv[:, :, :syn.ncell], ld
    bu = torch.empty((cap, syn.nz, syn.ny, syn.nx), dtype=tdtype, device=cx.dev)
    bv = torch.empty((cap, syn.nz, syn.ny, syn.nx), dtype=tdtype, device=cx.dev)
    return bu, bv, syn.ncell


def run_passes(cx, args, wl, nt_total, t0_rank, nt_local, counts, steps, warmup, bal=None, sampler=None):
    """warm-up + `steps` timed passes over this rank's shard; returns a dict of timings and the gathered series"""
    from nemoflux_b200 import _lib, nemoflux_gpu
    from nemoflux_b200 import dist as nfx_dist
    torch, dist = cx.torch, cx.dist
    syn, pli, M = wl.syn, wl.pli, wl.M
    world = cx.world
    esize = 8 if args.dtype == 'f64' else 4
    tdtype = torch.float64 if args.dtype == 'f64' else torch.float32
    pad = 0 if args.no_pad else (4 if args.dtype == 'f64' else 8)
    ld_est = (syn.ncell + pad - 1) // pad * pad if pad else syn.ncell
    step_bytes = 2 * esize * syn.nz * ld_est
    chunks, fit = plan_chunks(cx, args, nt_local, step_bytes)
    nchunks = len(chunks)
    assert bal is None or nchunks == 1, '--balance needs the whole shard resident'
    cap = max(c for _, c in chunks)
    u, v, ld = alloc_uv(cx, syn, max(cap, 1), tdtype, pad)
    cmax = max(max(counts), 1)
    eflux = torch.empty((cap, 2 * syn.ncell), dtype=torch.float64, device=cx.dev) if args.classic else None
    series_pad = torch.zeros((cmax, M), dtype=torch.float64, device=cx.dev)       # padded to the largest shard
    gathered = torch.empty((world * cmax, M), dtype=torch.float64, device=cx.dev) if world > 1 else None
    full_series = None
    shards_all = [nfx_dist.shard_batches(nt_total, bal['npanels'], world, r, bal.get('weights')) for r in range(world)] if bal else None
    combine_idx = None
    if bal is not None:
        # row r*cmax + k of the gathered blocks is time step t_first_r + k (rows past a rank's last step go to a spare row)
        idx = numpy.full(world * cmax, nt_total, numpy.int64)
        for r, sh in enumerate(shards_all):
            idx[r * cmax:r * cmax + sh['nt_touched']] = sh['t_first'] + numpy.arange(sh['nt_touched'])
        combine_idx = torch.from_numpy(idx).to(cx.dev)
        full_series = torch.zeros((nt_total + 1, M), dtype=torch.float64, device=cx.dev)
    resident = [-1]

    def load_chunk(ci):
        if resident[0] == ci:
            return
        off, n = chunks[ci]
        if n:
            syn.fill_device(t0_rank + off, n, cx.dev, tdtype, out=(u[:n], v[:n]))
        resident[0] = ci

    def chunk_pass(ci, ev=None):
        off, n = chunks[ci]
        if ev is not None:
            ev[0].record()
        if n:
            out = series_pad[off:off + n]
            if args.classic:
                nemoflux_gpu.edgeFluxAssemble(u[:n], v[:n], wl.thickness, wl.arc1, wl.arc2, out=eflux[:n])    # K2
                pli.integrate(eflux[:n], order=args.order, out=out)                                            # K3
            elif bal is not None:    # this rank's batch range, partial sums; combined after the allgather
                pli.fluxSeries(u[:n], v[:n], wl.thickness, wl.arc1, wl.arc2, order=args.order, out=out,
                               batch_range=(bal['b0'], bal['b1']))
            else:   # the public call: K2 + K3 batches, edge fluxes kept in an L2-resident ring
                pli.fluxSeries(u[:n], v[:n], wl.thickness, wl.arc1, wl.arc2, order=args.order, out=out)
        if ev is not None:
            ev[1].record()

    def gather():
        if world == 1:
            return series_pad
        dist.all_gather_into_tensor(gathered, series_pad)
        if bal is not None:
            # a time step shared by two ranks: the sum of its two partial rows (two addends: the order cannot matter)
            full_series.zero_()
            full_series.index_add_(0, combine_idx, gathered)
            return full_series[:nt_total]
        return gathered

    def step(evs=None, eg=None):
        """one pass over the whole shard.  evs[ci] = (begin, end) events of chunk ci, eg = event after the allgather"""
        for ci in range(nchunks):
            if nchunks > 1:
                load_chunk(ci)                         # regenerate the chunk: outside the timed region
                cx.barrier()
            chunk_pass(ci, None if evs is None else evs[ci])
            if ci == nchunks - 1:
                out = gather()
                if eg is not None:
                    eg.record()
            if nchunks > 1:
                cx.barrier()
        return out

    load_chunk(0)
    for _ in range(max(warmup, 3)):
        step()
    cx.barrier()
    mk = lambda: torch.cuda.Event(enable_timing=True)   # noqa: E731
    evs = [[(mk(), mk()) for _ in range(nchunks)] for _ in range(steps)]
    egs = [mk() for _ in range(steps)]
    e_beg, e_end = mk(), mk()
    launches0 = _lib.launch_count()
    if nchunks > 1:
        load_chunk(0)
    cx.barrier()
    t_wall0 = time.time()
    e_beg.record()
    for i in range(steps):
        out = step(evs[i], egs[i])
    e_end.record()
    cx.barrier()
    t_wall1 = time.time()
    launches = _lib.launch_count() - launches0
    # per (step, chunk): pass time; the last chunk's section also holds the allgather
    sect = numpy.zeros((steps, nchunks))
    k2 = numpy.zeros((steps, nchunks))
    for i in range(steps):
        for ci in range(nchunks):
            k2[i, ci] = evs[i][ci][0].elapsed_time(evs[i][ci][1])
            sect[i, ci] = k2[i, ci]
        sect[i, -1] = evs[i][-1][0].elapsed_time(egs[i])
    if nchunks == 1:
        # back-to-back passes bracketed once: the whole interval, max over ranks
        total_ms = cx.allreduce([e_beg.elapsed_time(e_end)], 'max')[0]
    else:
        # barrier-separated sections: a section lasts as long as its slowest rank
        smax = numpy.array(cx.allreduce(sect.reshape(-1), 'max')).reshape(sect.shape)
        total_ms = float(smax.sum())
    k2_ms_step = float(k2.sum() / steps)                           # this rank, per step (sum over its chunk launches)
    gather_ms = float((sect[:, -1] - k2[:, -1]).mean())
    final = out.cpu().numpy().copy()
    if world > 1 and bal is None:                                  # drop the padding of the shorter shards
        final = numpy.concatenate([final[r * cmax:r * cmax + counts[r]] for r in range(world)], 0)
    elif world == 1:
        final = final[:nt_local]
    own = series_pad[:nt_local].cpu().numpy().copy()
    return dict(total_ms=total_ms, ms_per_step=total_ms / steps, k2_ms_step=k2_ms_step, gather_ms=gather_ms,
                launches=int(launches), series=final, own_series=own, chunks=chunks, fit=fit, u=u, v=v, ld=ld,
                resident_chunk=resident[0], t_wall=(t_wall0, t_wall1), padded=(u.dim() == 3),
                fused=(not args.classic) and _lib.get_option(_lib.NFX_OPT_LAST_SERIES_PATH) == 1)


def roofline_of(args, wl, res, nt_local, bal, peaks, read_ceiling):
    esize = 8 if args.dtype == 'f64' else 4
    syn = wl.syn
    units = syn.units_per_step()
    nlaunch = sum(1 for _, c in res['chunks'] if c > 0) or 1
    bytes_step = 2.0 * esize * units * nt_local                    # this rank, one pass over its shard
    if bal is not None:
        bytes_step = 2.0 * esize * units * (bal['b1'] - bal['b0']) / bal['npanels']
    achieved = bytes_step / max(res['k2_ms_step'], 1e-9) / 1e6
    peak = float(peaks.get('hbm_gbs', 6650.0))
    fused = res['fused']
    rl = {'bound': 'hbm',
          'kernel': 'k2_edgeflux_ldg + k3_integrate (two launches)' if not fused else
                    'k23_fused (persistent K2+K3; algorithmic bytes = the u/v stream)',
          'achieved': achieved, 'peak': peak, 'unit': 'GB/s', 'frac': achieved / peak, 'traffic': None,
          'peak_source': 'MEASURED_PEAKS.json hbm_gbs (of measured; a COPY rate, reads + writes)' if peaks
                         else 'fallback 6650 GB/s (of fallback)',
          'algorithmic_bytes_per_launch': bytes_step / nlaunch, 'launches_per_step': nlaunch,
          'kernel_ms_per_launch': res['k2_ms_step'] / nlaunch, 'frac_of_nominal_8TBs': achieved / 8000.0}
    if read_ceiling:
        # the pass only reads: its ceiling is the read-only rate of the same access pattern, measured on THIS device
        # by nfx_probe_read_bandwidth right before the timed region
        rl['read_only_ceiling_gbs'] = read_ceiling
        rl['frac_of_read_only_ceiling'] = achieved / read_ceiling
        rl['read_only_ceiling_source'] = 'nfx_probe_read_bandwidth on this device, this run (best of 5)'
    tr_path = os.path.join(ROOT, 'profiles', 'k2_traffic.json')
    if os.path.exists(tr_path):
        try:
            tr = json.load(open(tr_path))
            key = f'{wl.name}_{args.dtype}' + ('_fused' if fused else '')
            if key in tr:    # ncu dram bytes per launch were measured on a reduced nt: scale per time step
                rl['traffic'] = tr[key]['dram_bytes_per_timestep'] * bytes_step / (2.0 * esize * units) / nlaunch
                rl['traffic_source'] = tr[key].get('source', 'profiles/')
        except Exception:
            pass
    return rl


def parity_check(cx, args, wl, res, t0_rank, nt_local):
    """every rank: K1 lists bit for bit against the C oracle (all transects) and the flux of ONE of its own time
    steps against the oracle's edge fluxes summed over the oracle's weight map; reduced over ranks"""
    from oracle import oracle as O
    torch = cx.torch
    syn, pli = wl.syn, wl.pli
    O.lib()
    tk = time.perf_counter()
    _, oplis = build_oracle_plis(O, syn)
    t_k1_cpu = time.perf_counter() - tk
    sub = pli.getSubsegments()
    ok, nsub = True, 0
    for m, op in enumerate(oplis):
        a, b = sub['offsets'][m], sub['offsets'][m + 1]
        o = op.subsegs
        ok = ok and (b - a == len(o)) and numpy.array_equal(sub['cell'][a:b], o['cell']) and \
            numpy.array_equal(sub['w'][a:b].view(numpy.int64), o['w'].view(numpy.int64))
        nsub += len(o)
    del sub
    err, scale_max, checked = 0.0, 0.0, 0
    if nt_local > 0:
        # the first time step of the chunk that is still resident on this rank
        off, n = res['chunks'][res['resident_chunk']]
        step_host_bytes = 2 * 8 * syn.units_per_step() * 1.7          # u, v (+ iV and temporaries)
        try:
            import psutil
            avail = psutil.virtual_memory().available
        except Exception:
            avail = 64e9
        group = int(max(1, min(cx.world, (0.5 * avail) // step_host_bytes)))
        for rnd in range(math.ceil(cx.world / group)):
            if rnd == cx.rank // group and n > 0:
                uh = res['u'][0].reshape(syn.nz, -1)[:, :syn.ncell].cpu().numpy().reshape(syn.nz, syn.ny, syn.nx)
                vh = res['v'][0].reshape(syn.nz, -1)[:, :syn.ncell].cpu().numpy().reshape(syn.nz, syn.ny, syn.nx)
                iV, _, _ = O.edgeflux_step_c(uh, vh, syn.thickness, syn.arc1, syn.arc2, False)
                del uh, vh
                f = iV.reshape(-1)
                row = res['series'][t0_rank + off]     # the gathered series: complete also where ranks share a time step
                for m, op in enumerate(oplis):
                    keys, ws = op.merged_map()
                    sc = float(numpy.abs(ws * f[keys]).sum())
                    cpu = op.getIntegral(iV, args.order)
                    err = max(err, abs(row[m] - cpu) / max(sc, 1e-300))
                    scale_max = max(scale_max, sc)
                del iV, f
                checked = 1
            if cx.world > 1:
                cx.dist.barrier()
    red = cx.allreduce([err, 0.0 if ok else 1.0], 'max')
    nchk = cx.allreduce([checked], 'sum')[0]
    torch.cuda.synchronize()
    return {'edge_lists_bit_exact': red[1] == 0.0, 'subsegments': int(nsub),
            'flux_max_rel_err_vs_oracle': red[0], 'flux_checked_steps': int(nchk),
            'flux_check': 'one time step per rank (the first of its resident chunk): |F_gpu - F_oracle| / sum|w f|, '
                          'max over transects and ranks; bar 1e-12',
            'k1_seconds_cpu': t_k1_cpu}, oplis


def property_parity(syn, series, nt_total, M):
    """size-independent properties of the full gathered series: linear in (t+1); closed loops and node-to-node
    transects equal the analytic value (fluxexact.py:36-46)"""
    out = {}
    tfac = numpy.arange(1, nt_total + 1, dtype=numpy.float64)[:, None]
    out['linear_in_time_max_rel'] = float(numpy.abs(series - series[0:1] * tfac).max() /
                                          max(numpy.abs(series).max(), 1e-300))
    exact_err = 0.0
    for m in range(M):
        ex = syn.exact_flux(m, 0)
        if ex is not None:
            exact_err = max(exact_err, abs(series[0, m] - ex))
    out['exact_transects_max_abs_err_t0'] = float(exact_err)
    out['series_abs_max_t0'] = float(numpy.abs(series[0]).max())
    out['all_finite'] = bool(numpy.isfinite(series).all())
    return out


def e2e_legs(cx, args, wl):
    """host buffers through the public API: every rank streams its own time steps from pinned host memory.
    Three legs on the same sample of E time steps: equal shards (f64), shards apportioned by the measured H2D rate
    (f64, the headline) and the same with float32 storage."""
    from nemoflux_b200 import dist as nfx_dist
    torch, dist = cx.torch, cx.dist
    syn, pli, M = wl.syn, wl.pli, wl.M
    world, rank = cx.world, cx.rank
    units = syn.units_per_step()
    step_bytes = 16 * units
    if args.e2e_steps > 0:
        E = args.e2e_steps
    else:   # about 3.5 GB (C3) .. 9 GB (C4: 5 time steps) of pinned memory per rank on average: enough steps to apportion
        E = world * max(1, min(24, int(round(8.9e9 / step_bytes)))) if world > 1 else max(1, min(24, int(5.2e9 // step_bytes)))
    rate = nfx_dist.measure_h2d_rate(cx.dev)
    rates = cx.allgather_floats(rate)
    eq_counts = nfx_dist.shard_counts(E, world)
    rt_counts = nfx_dist.apportion_by_rate(E, rates) if world > 1 else [E]
    cap = max(eq_counts[rank], rt_counts[rank], 1)
    th_h, a1_h, a2_h = syn.thickness, syn.arc1, syn.arc2
    du, dv, _ = alloc_uv(cx, syn, cap, torch.float64, 0)
    hu = torch.empty((cap, syn.nz, syn.ny, syn.nx), dtype=torch.float64).pin_memory()
    hv = torch.empty_like(hu).pin_memory()
    reps = max(3, min(args.steps, 5))
    out = {'h2d_probe_gbs_per_rank': rates, 'sample_time_steps': E}
    gathered = {}

    def leg(name, counts, tdtype):
        t0, n = nfx_dist.blocks_from_counts(counts)[rank]
        esz = 8 if tdtype == torch.float64 else 4
        a, b = hu, hv
        if n:
            syn.fill_device(t0, n, cx.dev, torch.float64, out=(du[:n], dv[:n]))
            if tdtype == torch.float64:
                hu[:n].copy_(du[:n])
                hv[:n].copy_(dv[:n])
            else:
                a = torch.empty((cap, syn.nz, syn.ny, syn.nx), dtype=tdtype).pin_memory()
                b = torch.empty_like(a).pin_memory()
                a[:n].copy_(du[:n].to(tdtype))
                b[:n].copy_(dv[:n].to(tdtype))
        torch.cuda.synchronize()
        s = numpy.zeros((0, M))
        for _ in range(2):
            if n:
                s = pli.fluxSeries(a[:n], b[:n], th_h, a1_h, a2_h, order=args.order)
        cx.barrier()
        tk = time.perf_counter()
        for _ in range(reps):
            if n:
                s = pli.fluxSeries(a[:n], b[:n], th_h, a1_h, a2_h, order=args.order)   # blocking: result on the host
        dt_own = (time.perf_counter() - tk) / reps
        dt = cx.allreduce([dt_own], 'max')[0]
        same = True
        if n and tdtype == torch.float64:     # the device path on the same device data gives the same bits
            sd = pli.fluxSeries(du[:n], dv[:n], wl.thickness, wl.arc1, wl.arc2, order=args.order).cpu().numpy()
            same = bool(numpy.array_equal(sd, s))
        same = cx.allreduce([0.0 if same else 1.0], 'max')[0] == 0.0
        # gather the E x M series of the leg on every rank (padded blocks)
        cm = max(max(counts), 1)
        blk = torch.zeros((cm, M), dtype=torch.float64, device=cx.dev)
        if n:
            blk[:n] = torch.from_numpy(numpy.ascontiguousarray(s)).to(cx.dev)
        if world > 1:
            g = torch.empty((world * cm, M), dtype=torch.float64, device=cx.dev)
            dist.all_gather_into_tensor(g, blk)
            g = g.cpu().numpy()
            gathered[name] = numpy.concatenate([g[r * cm:r * cm + counts[r]] for r in range(world)], 0)
        else:
            gathered[name] = blk[:n].cpu().numpy()
        h2d = 2 * units * esz * E + (8 * (syn.nz + 2 * syn.ncell)) * sum(1 for c in counts if c)
        return {'value': units * E / dt, 'unit': UNIT, 'h2d_bytes_per_step': int(h2d), 'd2h_bytes_per_step': int(E * M * 8),
                'ms_per_step': 1e3 * dt, 'time_steps_per_rank': counts, 'h2d_gbs_aggregate': h2d / dt / 1e9,
                'h2d_gbs_this_rank': (2 * units * esz * n) / max(dt_own, 1e-9) / 1e9,
                'equals_device_path_bits': same, 'storage_dtype': 'f64' if esz == 8 else 'f32'}

    eq = leg('equal', eq_counts, torch.float64)
    if world > 1:
        rt = leg('rate', rt_counts, torch.float64)
        rt['series_bit_equal_to_equal_shards'] = bool(numpy.array_equal(gathered['equal'], gathered['rate']))
        rt['equal_shards'] = {k: eq[k] for k in ('value', 'ms_per_step', 'time_steps_per_rank', 'h2d_gbs_aggregate')}
        head = rt
    else:
        head = eq
    head['sample'] = (f'{E} time steps of {wl.name} over {world} rank(s) from pinned host memory per call of '
                      f'PolylineIntegral.fluxSeries (C ABI nfx_flux_series_host: double-buffered H2D + fused K2+K3 + '
                      f'D2H of the series), wall clock, max over ranks' +
                      ('; time steps apportioned by the H2D rate measured per rank at start' if world > 1 else ''))
    f32 = leg('f32', rt_counts, torch.float32)
    ref = gathered['rate' if world > 1 else 'equal']
    f32['max_rel_diff_to_f64_storage'] = float(numpy.abs(gathered['f32'] - ref).max() / max(numpy.abs(ref).max(), 1e-300))
    out['e2e'] = head
    out['e2e_f32'] = f32
    del hu, hv, du, dv
    torch.cuda.empty_cache()
    return out


def measure_read_ceiling(cx, res):
    """read-only ceiling of this device, on the (already allocated) u buffer; None when the buffer is too small"""
    from nemoflux_b200 import nemoflux_gpu
    try:
        base = res['u']._base if res['u']._base is not None else res['u']
        if base.numel() * base.element_size() < 10e9:
            return None
        return float(nemoflux_gpu.probeReadBandwidth(base, reps=5))
    except Exception as e:   # a measurement aid: never fail the bench over it
        sys.stderr.write(f'read ceiling probe failed: {e}\n')
        return None


def run_config(cx, args, name, nt_total, scaling, steps, warmup, balance, with_e2e, with_cpu, sampler=None):
    """one BASELINE config end to end on all ranks; returns rank 0's result dict (None elsewhere)"""
    from nemoflux_b200 import _lib, synth
    from nemoflux_b200 import dist as nfx_dist
    torch = cx.torch
    world, rank = cx.world, cx.rank
    wl = Workload(cx, name)
    syn, M = wl.syn, wl.M
    esize = 8 if args.dtype == 'f64' else 4
    if scaling == 'weak':
        nt_local = nt_total // world
        counts = [nt_local] * world
        t0_rank = rank * nt_local
    else:
        counts = nfx_dist.shard_counts(nt_total, world)
        t0_rank, nt_local = nfx_dist.shard_time(nt_total, world, rank)
    bal = None
    rate_weights = None
    if balance and world > 1:
        npanels, _pc = wl.pli.getNumberOfPanels(args.dtype)
        _lib.set_option(_lib.NFX_OPT_FAST_SERIES, 2)

        def shard(weights):
            b = nfx_dist.shard_batches(nt_total, npanels, world, rank, weights)
            b['npanels'], b['weights'] = npanels, weights
            cnt = [nfx_dist.shard_batches(nt_total, npanels, world, r, weights)['nt_touched'] for r in range(world)]
            return b, cnt
        bal, counts = shard(None)
        if not args.no_rate_balance:
            # the GPUs of one box differ by a few per cent in sustained rate (shared power budget): time a few passes
            # with equal shares, then cut the batch space in proportion to each rank's measured rate (outside the
            # timed region, like the H2D probe of the e2e leg)
            probe = run_passes(cx, args, wl, nt_total, bal['t_first'], bal['nt_touched'], counts, 3, 3, bal)
            own_batches = bal['b1'] - bal['b0']
            rate = own_batches / max(probe['k2_ms_step'], 1e-9)
            probe.clear()
            torch.cuda.empty_cache()
            rates = cx.allgather_floats(rate)
            rate_weights = [r / max(rates) for r in rates]
            bal, counts = shard(rate_weights)
        t0_rank, nt_local = bal['t_first'], bal['nt_touched']
    res = run_passes(cx, args, wl, nt_total, t0_rank, nt_local, counts, steps, warmup, bal)
    clocks = None
    if sampler is not None and rank == 0:
        clocks = sampler.stop(*res['t_wall'])
    if bal is not None:
        _lib.set_option(_lib.NFX_OPT_FAST_SERIES, 1)
    read_ceiling = measure_read_ceiling(cx, res)
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, 'MEASURED_PEAKS.json')))
    except Exception:
        pass
    roofline = roofline_of(args, wl, res, nt_local, bal, peaks, read_ceiling)
    # the slowest rank's kernel time sets the step: report the min achieved rate over ranks beside rank 0's
    roofline['achieved_min_over_ranks'] = cx.allreduce([roofline['achieved']], 'min')[0]
    status = wl.pli.seriesStatus()
    parity = {'series_status': status}
    oplis = None
    if not args.no_parity:
        p, oplis = parity_check(cx, args, wl, res, t0_rank, nt_local)
        parity.update(p)
    # free the resident u/v before the host-fed legs
    series, chunks, fit, padded, ld = res['series'], res['chunks'], res['fit'], res['padded'], res['ld']
    units_step_all = syn.units_per_step() * nt_total
    ms_per_step = res['ms_per_step']
    keep = {k: res[k] for k in ('k2_ms_step', 'gather_ms', 'launches', 'fused')}
    res.clear()
    torch.cuda.empty_cache()
    e2e = e2e_legs(cx, args, wl) if with_e2e else None
    if rank != 0:
        return None
    parity.update(property_parity(syn, series, nt_total, M))
    if e2e is not None:
        parity['e2e_equals_device'] = bool(e2e['e2e']['equals_device_path_bits'])
    cpu = None
    if with_cpu and world == 1 and oplis is not None:
        from oracle import oracle as O
        nc = min(default_cpu_steps(args, syn), nt_total)
        fields = [syn.uv_host(t) for t in range(nc)]
        all_host_threads()
        cpu_reference_pass(O, syn, oplis, fields[:1], args.order)          # warm-up
        dt_np, _ = cpu_reference_pass(O, syn, oplis, fields, args.order)
        dt_c, _ = cpu_reference_pass(O, syn, oplis, fields, args.order, use_c=True)
        units = syn.units_per_step() * nc
        cpu = {'value': units / dt_np, 'unit': UNIT, 'cores': os.cpu_count(), 'kind': 'port',
               'sample': f'{nc} of {nt_total} time steps of {name} ({units:.3e} units): numpy restatement '
                         f'of field.py:145-234 (OpenBLAS threads default) + C getIntegral per transect',
               'value_c_openmp': units / dt_c, 'c_openmp_threads': O.lib().orc_num_threads()}
    out = {
        'value': units_step_all / (ms_per_step * 1e-3), 'ms_per_step': ms_per_step, 'scaling': scaling,
        'config': make_config(name, synth.CONFIGS[name], world, args.dtype, nt_total, scaling, bal is not None),
        'details': {
            'nt_per_gpu': counts, 'resident_chunks_per_gpu': [c for _, c in chunks], 'chunk_fit_steps': fit,
            'chunking': ('whole shard resident in HBM' if len(chunks) == 1 else
                         f'{len(chunks)} resident chunks per rank, regenerated on the device between chunk passes outside '
                         f'the timed region; step time = sum over chunk passes of the max-over-ranks CUDA-event time'),
            'device_layout': f'(nt, nz, ld={ld}) level planes padded to 32 B' if padded else '(nt, nz, ny, nx) dense',
            'batch_shares_by_measured_rate': rate_weights,
            'summation_order': args.order, 'allgather_ms': keep['gather_ms'],
            'pass': 'classic: K2 -> eflux in HBM -> K3 (two launches)' if args.classic else
                    'PolylineIntegral.fluxSeries (nfx_flux_series, eflux=NULL): fused persistent K2+K3 with the edge '
                    'fluxes in an L2-resident ring' + ('' if keep['fused'] else ' -- NOT taken: two launches')},
        'hbm_gbs_aggregate': 2.0 * esize * units_step_all / (ms_per_step * 1e-3) / 1e9,
        'roofline': roofline, 'clocks': clocks, 'gpu_launches': keep['launches'],
        'one_off': {'locator_s': wl.t_locator, 'k1_compute_weights_s': wl.t_k1},
        'parity': parity, 'series': series,
    }
    if e2e is not None:
        out['e2e'] = e2e['e2e']
        out['e2e_f32'] = e2e['e2e_f32']
        out['h2d_probe_gbs_per_rank'] = e2e['h2d_probe_gbs_per_rank']
    if cpu is not None:
        out['cpu_baseline'] = cpu
    return out


def run_b200(args):
    from nemoflux_b200 import _lib
    cx = Ctx()
    world, rank = cx.world, cx.rank
    if args.k2_variant:
        _lib.set_option(_lib.NFX_OPT_K2_VARIANT, args.k2_variant)
    if args.k2_unroll:
        _lib.set_option(_lib.NFX_OPT_K2_UNROLL, args.k2_unroll)
    if args.k2_block:
        _lib.set_option(_lib.NFX_OPT_K2_BLOCK, args.k2_block)
    if args.ring_slot_mb:
        _lib.set_option(_lib.NFX_OPT_RING_SLOT_MB, args.ring_slot_mb)
    name, nt_total, scaling = pick_workload(args, world)
    sampler = ClockSampler(cx.local_rank)
    if rank == 0:
        sampler.start()
    main = run_config(cx, args, name, nt_total, scaling, args.steps, args.warmup, args.balance,
                      with_e2e=not args.no_e2e, with_cpu=not args.no_cpu, sampler=sampler)
    outputs = {'flux_series': main.pop('series')} if rank == 0 else None
    target = None
    if world == 8 and args.workload == 'auto' and not args.no_target:
        # BASELINE's target: ORCA12 x 73 snapshots x 1024 transects on 8 GPUs, balanced (time step, panel) sharding
        cx.torch.cuda.empty_cache()
        tsampler = ClockSampler(cx.local_rank)
        if rank == 0:
            tsampler.start()
        t = run_config(cx, args, 'C5', 73, 'strong', max(3, min(args.steps, args.target_steps)), 3, True,
                       with_e2e=False, with_cpu=False, sampler=tsampler)
        if rank == 0:
            outputs['target_c5_flux_series'] = t.pop('series')
            rl = t['roofline']
            target = {'workload': t['config']['workload'], 'ms': t['ms_per_step'], 'value': t['value'], 'unit': UNIT,
                      'steps': max(3, min(args.steps, args.target_steps)), 'warmup': 3,
                      'hbm_gbs_aggregate': t['hbm_gbs_aggregate'],
                      'frac_of_nominal': t['hbm_gbs_aggregate'] / (8 * 8000.0),
                      'frac_of_measured_copy_peak': t['hbm_gbs_aggregate'] / (8 * rl['peak']),
                      'north_star_bar': '>= 0.70 of aggregate HBM roofline', 'config': t['config'],
                      'details': t['details'], 'roofline': rl, 'parity': t['parity'], 'clocks': t['clocks'],
                      'one_off': t['one_off'], 'gpu_launches': t['gpu_launches']}
    if rank == 0:
        line = {'metric': METRIC, 'value': main['value'], 'unit': UNIT, 'n_gpus': world, 'steps': args.steps,
                'warmup': max(args.warmup, 3), 'ms_per_step': main['ms_per_step'], 'higher_is_better': True,
                'scaling': main['scaling'], 'vs_baseline': None, 'dtype': args.dtype, 'data': 'synthetic'}
        for k, v in main.items():
            if k not in line:
                line[k] = v
        line['cpus_bound_per_rank'] = cx.cpu_binding
        if target is not None:
            line['target_c5'] = target
        print(json.dumps(line), flush=True)
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, outputs)
    if world > 1:
        cx.dist.barrier()
        cx.dist.destroy_process_group()


def main():
    args = parse_args()
    if args.impl == 'reference':
        run_reference(args)
    else:
        run_b200(args)


if __name__ == '__main__':
    main()
