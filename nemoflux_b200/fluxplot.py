"""fluxplot -- drop-in for nemoflux/fluxplot.py: flux time series of every transect (same flags).

    python -m nemoflux_b200.fluxplot -t T.nc -u U.nc -v V.nc -i "../data/nz/S*.txt" [-s] [--output series.csv]
        [--layers "0,10,35,75" | --depthLayers "0,200,1000,6000" | --classField NAME[:FILE] --classBounds=b0,b1,...]
        [--section section.nc] [--timeMean N|month|year] [--tracer NAME[:FILE] [--tracerRef R]]

The reference loops ``for itime: fld.update(); for pli: pli.getIntegral(...)`` (fluxplot.py:51-59); here the
whole (nt, M) series comes from Field.fluxSeries() (K2+K3 over chunks of time steps).  The series is printed
and optionally written as CSV; it is plotted only when matplotlib is importable and --plot is given.
--layers (model-level boundaries) or --depthLayers (depths in metres, snapped to the nearest level interfaces) split
every transect's flux by depth: one column per (transect, layer), transect-major, headed label[top-bottom m] with the
interfaces that were integrated.
--section FILE.nc also writes the transport section (Field.fluxSection): the flux across every cell crossing of every
transect per layer (the layers of --layers / --depthLayers, else one per level) as a NetCDF classic (64-bit offset)
file, see writeSection.
--classField NAME[:FILE] --classBounds=b0,b1,... split every transect's flux by the class of a T-grid variable
(thetao, so, sigma0...; from the T file unless FILE is given): one column per (transect, class), headed
label[b_j–b_{j+1}), the water with b_j <= value < b_{j+1} (Field.fluxClasses).  Not combined with --layers /
--depthLayers.
--tracer NAME[:FILE] [--tracerRef R] weights every transect's flux by a T-grid tracer (thetao, so...; from the T file
unless FILE is given) taken at the C-grid faces, minus R (default 0): the heat, salt or freshwater it carries
(Field.fluxTracer), in tracer units x flux units.  One column per transect, or per (transect, layer) with --layers /
--depthLayers, headed label[NAME] or label[NAME top-bottom m].  Not combined with --classField or --section.
--timeMean N|month|year averages over windows of N steps, or of the steps of each calendar month / year
(timeobj.timeWindows): the printed and CSV series become window means (windowMeans), one row per window labelled
first/last (the dates of its first and last step), and the --section file holds window means computed on the device
(Field.fluxSection(windows=)) with time_bnds and cell_methods = "time: mean".
"""
import argparse
import os

import numpy

from . import ncio
from .field import Field
from .fluxviz import parseTransects
from .timeobj import timeWindows


def parseList(text, kind=float):
    """'0,200,1000' -> [0.0, 200.0, 1000.0] (kind=int: integers only)"""
    try:
        vals = [kind(x) for x in text.replace(' ', '').split(',') if x != '']
    except ValueError:
        raise argparse.ArgumentTypeError(f'expected a comma-separated list of {kind.__name__} values, got {text!r}')
    if len(vals) < 2:
        raise argparse.ArgumentTypeError(f'expected at least two boundaries, got {text!r}')
    return vals


def parseTimeMean(text):
    """'--timeMean' value: a number of steps >= 1, 'month' or 'year'"""
    t = text.strip().lower()
    if t in ('month', 'year'):
        return t
    if t.isdigit() and int(t) >= 1:
        return int(t)
    raise argparse.ArgumentTypeError(f"expected a number of steps >= 1, 'month' or 'year', got {text!r}")


def windowMeans(x, bounds):
    """(K, ...) means over the windows [b_w, b_{w+1}) of the first axis of x: the sum in ascending step order from
    +0, divided by the window's length (the definition of fluxSection(windows=))"""
    x = numpy.asarray(x, numpy.float64)
    out = numpy.empty((len(bounds) - 1,) + x.shape[1:])
    for w in range(len(bounds) - 1):
        acc = numpy.zeros(x.shape[1:])
        for t in range(bounds[w], bounds[w + 1]):
            acc = acc + x[t]
        out[w] = acc / (bounds[w + 1] - bounds[w])
    return out


def classLabels(labels, bounds):
    """column headings of a class series, transect-major: label[b_j–b_{j+1})"""
    return [f'{lab}[{b0:g}–{b1:g})' for lab in labels for b0, b1 in zip(bounds[:-1], bounds[1:])]


def tracerLabels(labels, name, iface=None, layers=None):
    """column headings of a tracer series, transect-major: label[NAME], or label[NAME top-bottom m] per layer"""
    if layers is None:
        return [f'{lab}[{name}]' for lab in labels]
    return [f'{lab}[{name} {iface[k0]:g}-{iface[k1]:g} m]' for lab in labels for k0, k1 in zip(layers[:-1], layers[1:])]


def writeSection(path, fld, layers, units, windows=None):
    """transport(time, layer, crossing) of fld.fluxSection(layers) with the crossings' geometry
    (PolylineIntegral.getSectionGeometry), layer_top / layer_bottom in metres, transect_offsets and time (the record
    dimension: only one record has to fit the 4 GB of the classic 64-bit-offset format).  Returns the number of
    crossings.
    windows (step bounds, see timeobj.timeWindows): window means instead, cell_methods = "time: mean"; time is the mean
    of the window's time values and time_bnds (time, 2) its extent: from the time variable's bounds variable (NEMO's
    time_centered_bounds) when the file has one, else the first and last time stamps."""
    lev = list(range(fld.nz + 1)) if layers is None else list(layers)
    sec = fld.fluxSection(layers=lev) if windows is None else fld.fluxSection(layers=lev, windows=windows)
    geo = fld.pli.getSectionGeometry()
    iface = fld.layerInterfaces()
    nsub = sec.shape[2]
    w = ncio.Writer(path, classic=True)
    w.createDimension('time', None)
    w.createDimension('layer', len(lev) - 1)
    w.createDimension('crossing', nsub)
    w.createDimension('transect_edge', geo['offsets'].size)
    tv = fld.timeObj.getValues() if fld.timeObj.getSize() == fld.nt else numpy.arange(fld.nt)
    tattrs = {k: v for k, v in (('units', fld.timeObj.units), ('calendar', fld.timeObj.calendar)) if v} \
        if fld.timeObj.getSize() == fld.nt else {'long_name': 'time index'}
    tv = numpy.asarray(tv, numpy.float64)
    tattrs_sec = {'units': units, 'long_name': 'flux across the cell crossing, per layer of model levels'}
    if windows is not None:
        b = list(windows)
        bnds = fld.timeObj.getBounds() if fld.timeObj.getSize() == fld.nt else None
        lo = numpy.array([bnds[b0, 0] if bnds is not None else tv[b0] for b0 in b[:-1]], numpy.float64)
        hi = numpy.array([bnds[b1 - 1, 1] if bnds is not None else tv[b1 - 1] for b1 in b[1:]], numpy.float64)
        tv = numpy.array([tv[b0:b1].mean() for b0, b1 in zip(b[:-1], b[1:])], numpy.float64)
        tattrs = dict(tattrs, bounds='time_bnds')
        tattrs_sec['cell_methods'] = 'time: mean'
        w.createDimension('nv', 2)
    w.createVariable('time', 'f8', ('time',), attrs=tattrs, data=tv)
    if windows is not None:
        w.createVariable('time_bnds', 'f8', ('time', 'nv'), data=numpy.stack([lo, hi], 1))
    w.createVariable('transport', 'f8', ('time', 'layer', 'crossing'), data=sec, attrs=tattrs_sec)
    w.createVariable('layer_top', 'f8', ('layer',), attrs={'units': 'm'}, data=iface[lev[:-1]])
    w.createVariable('layer_bottom', 'f8', ('layer',), attrs={'units': 'm'}, data=iface[lev[1:]])
    w.createVariable('transect_offsets', 'i4', ('transect_edge',), data=geo['offsets'].astype(numpy.int32))
    for name, unit in (('transect', ''), ('segment', ''), ('cell_j', ''), ('cell_i', ''), ('lon0', 'degrees_east'),
                       ('lat0', 'degrees_north'), ('lon1', 'degrees_east'), ('lat1', 'degrees_north'),
                       ('length_km', 'km'), ('distance_km', 'km')):
        a = geo[name]
        kind = 'i4' if a.dtype.kind in 'iu' else 'f8'
        w.createVariable(name, kind, ('crossing',), attrs={'units': unit} if unit else None, data=a.astype(kind))
    w.close()
    return nsub


def main(argv=None):
    ap = argparse.ArgumentParser(description='Flux time series')
    ap.add_argument('-t', '--tFile', required=True)
    ap.add_argument('-u', '--uFile', required=True)
    ap.add_argument('-v', '--vFile', required=True)
    ap.add_argument('-l', '--lonLatPoints', default='')
    ap.add_argument('-i', '--iFiles', default='')
    ap.add_argument('-s', '--sverdrup', action='store_true')
    ap.add_argument('-o', '--output', default='', help='write the series as CSV (time, one column per transect)')
    ap.add_argument('--plot', action='store_true')
    ap.add_argument('--meshFile', default='', help='optional mesh_mask file: e3u_0/e3v_0 (and e2u/e1v) scale factors')
    lay = ap.add_mutually_exclusive_group()
    lay.add_argument('--layers', type=lambda x: parseList(x, int), default=None,
                     help='flux per layer of model levels: level boundaries "0,10,35,75"')
    lay.add_argument('--depthLayers', type=parseList, default=None,
                     help='flux per depth range: depths in metres "0,200,1000,6000", snapped to level interfaces')
    lay.add_argument('--classField', default=None,
                     help='flux per class of a T-grid variable: NAME or NAME:FILE (default file: the T file)')
    ap.add_argument('--classBounds', type=parseList, default=None,
                    help='class bounds of --classField, ascending, -inf/inf allowed: --classBounds=-2,0,4,10,inf')
    ap.add_argument('--section', default='',
                    help='write the transport section (flux per cell crossing and layer) to this NetCDF file')
    ap.add_argument('--timeMean', type=parseTimeMean, default=None,
                    help='average over windows of N steps, or per calendar month / year: N|month|year')
    ap.add_argument('--tracer', default=None,
                    help='transport of a T-grid tracer at the cell faces: NAME or NAME:FILE (default file: the T file)')
    ap.add_argument('--tracerRef', type=float, default=None,
                    help='reference value subtracted from the tracer (default 0): --tracerRef=34.8')
    a = ap.parse_args(argv)
    if a.tracerRef is not None and a.tracer is None:
        ap.error('--tracerRef needs --tracer')
    if a.tracer is not None and (a.classField is not None or a.section):
        ap.error('--tracer cannot be combined with --classField or --section')
    if (a.classField is None) != (a.classBounds is None):
        ap.error('--classField and --classBounds go together')
    pts, names = parseTransects(a.lonLatPoints, a.iFiles)
    print(f'target points:\n {pts}')
    fld = Field(a.tFile, a.uFile, a.vFile, pts, a.sverdrup, meshFile=a.meshFile or None)
    layers = fld.levelsForDepths(a.depthLayers) if a.depthLayers is not None else a.layers
    if a.classField is not None:
        var, _, cfile = a.classField.partition(':')
        series = fld.fluxClasses(var, a.classBounds, file=cfile or None)
    elif a.tracer is not None:
        tvar, _, tfile = a.tracer.partition(':')
        series = fld.fluxTracer(tvar, file=tfile or None, ref=a.tracerRef or 0.0, layers=layers)
    else:
        series = fld.fluxSeries(layers=layers)
    timeVals = [fld.timeObj.getTimeAsDate(i) for i in range(fld.nt)]
    windows = None
    if a.timeMean is not None:
        windows = timeWindows(fld.timeObj, fld.nt, a.timeMean)
        series = windowMeans(series, windows)
        timeVals = [f'{timeVals[b0]}/{timeVals[b1 - 1]}' for b0, b1 in zip(windows[:-1], windows[1:])]
    units = 'Sv' if a.sverdrup else 'A m^2/s'
    labels = [os.path.basename(n) for n in names]
    rows = series
    if a.tracer is not None:
        units = f'{tvar} x {units}'
        labels = tracerLabels(labels, tvar, fld.layerInterfaces() if layers is not None else None, layers)
        if layers is not None:
            rows = numpy.asarray(series).transpose(0, 2, 1).reshape(len(series), -1)   # (time, transect-major layers)
    elif layers is not None:
        iface = fld.layerInterfaces()
        labels = [f'{lab}[{iface[k0]:g}-{iface[k1]:g} m]' for lab in labels for k0, k1 in zip(layers[:-1], layers[1:])]
        rows = numpy.asarray(series).transpose(0, 2, 1).reshape(len(series), -1)   # (time, transect-major layers)
    elif a.classField is not None:
        labels = classLabels(labels, a.classBounds)
        rows = numpy.asarray(series).transpose(0, 2, 1).reshape(len(series), -1)   # (time, transect-major classes)
    print('time,' + ','.join(labels) + f'   [{units}]')
    for t, row in zip(timeVals, rows):
        print(f'{t},' + ','.join(f'{x:.15g}' for x in row))
    if a.section:
        nsub = writeSection(a.section, fld, layers, units, windows)
        print(f'section: {nsub} crossings written to {a.section}')
    if a.output:
        with open(a.output, 'w', encoding='utf-8') as f:
            f.write('time,' + ','.join(labels) + '\n')
            for t, row in zip(timeVals, rows):
                f.write(f'{t},' + ','.join(repr(float(x)) for x in row) + '\n')
    if a.plot:
        try:
            import matplotlib.pyplot as plt
        except ImportError:
            print('matplotlib is not installed: no plot')
        else:
            lineTypes = ['b-', 'm--', 'c-.', 'r:', 'g-', 'k--']
            for i in range(rows.shape[1]):
                plt.plot(timeVals, rows[:, i], lineTypes[i % len(lineTypes)])
            if len(labels) > 1:
                plt.legend(labels)
            plt.title('Water flow')
            plt.ylabel(units)
            plt.show()
    return numpy.asarray(series)


if __name__ == '__main__':
    main()
