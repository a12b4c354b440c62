"""Fraction of the u/v stream the transects of a synth workload read (CPU, C oracle K1).
    python tools/column_coverage.py C3|C4|C5|tiny|small     (NFX_REPO = repository root, default .)"""
import sys, time, numpy
import os; sys.path.insert(0, os.environ.get('NFX_REPO', '.'))
from nemoflux_b200 import synth
from oracle import oracle as O
name = sys.argv[1]
t0 = time.time()
syn = synth.make(name)
g = O.Grid(syn.points)
nx, ny, nc = syn.nx, syn.ny, syn.ncell
ucols = numpy.zeros(nc, bool); vcols = numpy.zeros(nc, bool)
nent = 0; nsub = 0
for xyz in syn.transects:
    p = O.PolylineIntegral(g, 360.); p.computeWeights(xyz)
    keys, ws = p.merged_map(); nent += len(keys); nsub += len(p.subsegs)
    c = keys // 4; e = keys % 4; j = c // nx; i = c % nx
    ucols[c[e == 1]] = True
    w = e == 3; ucols[j[w] * nx + (i[w] - 1) % nx] = True
    vcols[c[e == 2]] = True
    s = (e == 0) & (j > 0); vcols[(j[s] - 1) * nx + i[s]] = True
print(name, 'ncell', nc, 'transects', syn.ntransects, 'subsegs', nsub, 'map entries', nent, 'secs', round(time.time()-t0,1))
for lab, cols in (('u', ucols), ('v', vcols)):
    print(f' {lab}: columns {cols.sum()} = {cols.mean():.4f} of the plane')
for esz, dt in ((8, 'f64'), (4, 'f32')):
    ld = (nc + 8191)//8192*8192
    for gran in (32, 64, 128, 256, 1024, 4096, 8192, 32768):
        per = gran // esz
        tot = 0; used = 0
        for cols in (ucols, vcols):
            pad = numpy.zeros(ld, bool); pad[:nc] = cols
            blk = pad.reshape(-1, per).any(1)
            nb = -(-nc // per)
            tot += nb; used += blk[:nb].sum()
        print(f' {dt} {gran:3d}B blocks touched: {used/tot:.4f} of the u+v stream')
for gran in (32, 64):
    per = gran // 8
    pad = numpy.zeros((nc + 8191)//8192*8192, bool); pad[:nc] = ucols | vcols
    print(f" union u|v f64 {gran}B blocks: {pad.reshape(-1, per).any(1)[:-(-nc // per)].mean():.4f}")
# row runs: how contiguous are touched columns
runs = numpy.diff(numpy.concatenate([[0], ucols.astype(int), [0]]))
print(' u runs of touched columns:', (runs == 1).sum(), 'mean length', ucols.sum() / max((runs == 1).sum(), 1))
