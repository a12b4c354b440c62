"""nemoflux_gpu -- the B200 replacement for the pieces of ``mint`` nemoflux uses, plus the batched
transect-flux path.

Mirrors the reference's operator interface (same method names, argument meaning and error behaviour):

    reference (mint)                                  here
    ------------------------------------------------  ------------------------------------------------
    g = mint.Grid(); g.setPoints(points)              g = Grid(); g.setPoints(points)   horizgrid.py:23-24
    g.getNumberOfCells()                              g.getNumberOfCells()              horizgrid.py:30
    p = mint.PolylineIntegral(); p.setGrid(g)         p = PolylineIntegral(); p.setGrid(g)    field.py:45-46
    p.buildLocator(numCellsPerBucket=128,             p.buildLocator(...)  (or p.build(g))    field.py:47
                   periodX=360., enableFolding=False)
    p.computeWeights(xyz, counterclock=False)         p.computeWeights(xyz, counterclock=False) field.py:48
    p.getIntegral(data, mint.CELL_BY_CELL_DATA)       p.getIntegral(data, CELL_BY_CELL_DATA)  field.py:102
                                                      p.computeIntegral(edgeData)  (same thing)

New, batched (what the fluxplot.py:51-59 loop does, for all transects and time steps at once):

    p.computeWeights([xyz0, xyz1, ...])      many transects, one locator
    p.fluxSeries(u, v, thickness, arc1, arc2, sverdrup) -> (nt, M)

All compute runs in libnemoflux_gpu.so (hand-written sm_100a CUDA) through ctypes; torch only owns
device buffers and streams.  There is no CPU fallback.
"""
import ctypes

import numpy

from . import _lib
from ._lib import NFX_CELL_BY_CELL_DATA as CELL_BY_CELL_DATA  # noqa: F401  (mint.CELL_BY_CELL_DATA)

_ORDERS = {'list': _lib.NFX_ORDER_LIST, 'map': _lib.NFX_ORDER_MAP}


def _torch():
    import torch
    return torch


def _np_ptr(a):
    return ctypes.c_void_p(a.ctypes.data)


def _t_ptr(t):
    return ctypes.c_void_p(t.data_ptr())


def _stream_ptr():
    return ctypes.c_void_p(_torch().cuda.current_stream().cuda_stream)


def _dtype_code(dtype_name):
    if dtype_name in ('float64', 'torch.float64'):
        return _lib.NFX_F64
    if dtype_name in ('float32', 'torch.float32'):
        return _lib.NFX_F32
    raise TypeError(f'uo/vo must be float64 or float32, got {dtype_name}')


class Grid(object):
    """mint.Grid: an unstructured collection of quads, 4 private vertices per cell"""

    def __init__(self):
        self._h = ctypes.c_void_p()
        _lib.call('nfx_grid_new', ctypes.byref(self._h))
        self._points = None
        self._cgrid = None

    def __del__(self):
        try:
            if self._h:
                _lib.load().nfx_grid_del(ctypes.byref(self._h))
        except Exception:
            pass

    def setPoints(self, points):
        """points: (ncells, 4, 3) float64, vertices SW, SE, NE, NW as (lon deg, lat deg, ignored)"""
        pts = numpy.ascontiguousarray(points, numpy.float64)
        if pts.ndim != 3 or pts.shape[1:] != (4, 3):
            raise ValueError(f'points must have shape (ncells, 4, 3), got {pts.shape}')
        _lib.call('nfx_grid_set_points', ctypes.byref(self._h), pts.shape[0], _np_ptr(pts))
        self._points = pts

    def setCGridShape(self, ny, nx):
        """structured shape behind the cell ids (cell = j*nx + i); enables the compact flux layout"""
        _lib.call('nfx_grid_set_cgrid_shape', ctypes.byref(self._h), int(ny), int(nx))
        self._cgrid = (int(ny), int(nx))

    def getNumberOfCells(self):
        n = ctypes.c_int64()
        _lib.call('nfx_grid_get_num_cells', ctypes.byref(self._h), ctypes.byref(n))
        return n.value

    def getPoints(self):
        return self._points

    def arcLengths(self, out=None):
        """(ncells, 4) cuda tensor of unit-sphere edge lengths computed on the device with the well-conditioned
        haversine form.  Not the parity path: the reference's arccos formula (geo.getArcLengthArray) carries rounding
        noise of ~1e-16/arc, so reproducing it to 1e-12 needs the host formula (nemoflux_b200.geo.cellArcLengths)."""
        torch = _torch()
        n = self.getNumberOfCells()
        if out is None:
            out = torch.empty((n, 4), dtype=torch.float64, device='cuda')
        _require_cuda(out, torch.float64, 'out')
        with torch.cuda.device(out.device):
            _lib.call('nfx_grid_arc_lengths', ctypes.byref(self._h), _t_ptr(out), _stream_ptr())
        return out


class PolylineIntegral(object):
    """mint.PolylineIntegral for one transect or a batch of transects sharing one locator"""

    def __init__(self):
        self._h = ctypes.c_void_p()
        _lib.call('nfx_pli_new', ctypes.byref(self._h))
        self._grid = None
        self._batched = False
        self._polylines = []

    def __del__(self):
        try:
            if self._h:
                _lib.load().nfx_pli_del(ctypes.byref(self._h))
        except Exception:
            pass

    # -- mint interface -----------------------------------------------------------------------------
    def setGrid(self, grid):
        if not isinstance(grid, Grid):
            raise TypeError('setGrid expects a nemoflux_gpu.Grid')
        _lib.call('nfx_pli_set_grid', ctypes.byref(self._h), grid._h)
        self._grid = grid

    def buildLocator(self, numCellsPerBucket=128, periodX=360., enableFolding=False):
        _lib.call('nfx_pli_build_locator', ctypes.byref(self._h), int(numCellsPerBucket), float(periodX),
                  int(bool(enableFolding)))

    def build(self, grid, periodX=360.):
        """setGrid + buildLocator, once per grid; every transect shares the locator"""
        self.setGrid(grid)
        self.buildLocator(numCellsPerBucket=128, periodX=periodX, enableFolding=False)

    def computeWeights(self, xyz, counterclock=False):
        """xyz: one polyline (npoints, 3), or a sequence of polylines [(n0,3), (n1,3), ...]"""
        try:
            single = numpy.asarray(xyz, numpy.float64).ndim == 2
        except ValueError:      # ragged sequence of polylines
            single = False
        lines = [xyz] if single else list(xyz)
        arrs = []
        for ln in lines:
            a = numpy.ascontiguousarray(ln, numpy.float64)
            if a.ndim != 2 or a.shape[1] != 3:
                raise ValueError(f'a polyline must have shape (npoints, 3), got {a.shape}')
            arrs.append(a)
        offsets = numpy.zeros(len(arrs) + 1, numpy.int32)
        for i, a in enumerate(arrs):
            offsets[i + 1] = offsets[i] + a.shape[0]
        allpts = numpy.concatenate(arrs, axis=0) if arrs else numpy.zeros((0, 3))
        allpts = numpy.ascontiguousarray(allpts, numpy.float64)
        _lib.call('nfx_pli_compute_weights_batch', ctypes.byref(self._h), len(arrs), _np_ptr(offsets),
                  _np_ptr(allpts), int(bool(counterclock)))
        self._batched = not single
        self._polylines = [a.copy() for a in arrs]      # for getSectionGeometry
        return 0

    def getIntegral(self, data, placement=CELL_BY_CELL_DATA, order='map'):
        """data: (ncells, 4) float64 host array.  One transect -> float; a batch -> (M,) array"""
        d = numpy.ascontiguousarray(data, numpy.float64)
        ncell = self._grid.getNumberOfCells() if self._grid else -1
        if d.size != ncell * 4:
            raise ValueError(f'data must hold ncells*4 = {ncell * 4} values, got {d.size}')
        m = self.getNumberOfTransects()
        res = numpy.zeros(max(m, 1), numpy.float64)
        _lib.call('nfx_pli_get_integrals', ctypes.byref(self._h), _np_ptr(d), int(placement), _ORDERS[order],
                  _np_ptr(res))
        if self._batched:
            return res[:m]
        return float(res[0])

    computeIntegral = getIntegral

    # -- inspection -----------------------------------------------------------------------------------
    def getNumberOfTransects(self):
        n = ctypes.c_int()
        _lib.call('nfx_pli_get_num_transects', ctypes.byref(self._h), ctypes.byref(n))
        return n.value

    def getSubsegments(self):
        """dict of arrays in emission order (transect, segment, ta, cell, image) + 'offsets' (M+1)"""
        n = ctypes.c_int64()
        _lib.call('nfx_pli_get_num_subsegments', ctypes.byref(self._h), ctypes.byref(n))
        n = n.value
        m = self.getNumberOfTransects()
        out = dict(offsets=numpy.zeros(m + 1, numpy.int64), cell=numpy.zeros(n, numpy.int64),
                   seg=numpy.zeros(n, numpy.int32), img=numpy.zeros(n, numpy.int32), ta=numpy.zeros(n),
                   tb=numpy.zeros(n), coeff=numpy.zeros(n), xia=numpy.zeros((n, 2)), xib=numpy.zeros((n, 2)),
                   w=numpy.zeros((n, 4)))
        _lib.call('nfx_pli_get_subsegments', ctypes.byref(self._h),
                  *[_np_ptr(out[k]) for k in ('offsets', 'cell', 'seg', 'img', 'ta', 'tb', 'coeff', 'xia', 'xib', 'w')])
        return out

    def getWeights(self, transect=0):
        """(cellIds, edgeIndices, weights) of one transect, 4 entries per sub-segment, emission order"""
        s = self.getSubsegments()
        a, b = s['offsets'][transect], s['offsets'][transect + 1]
        cells = numpy.repeat(s['cell'][a:b], 4)
        edges = numpy.tile(numpy.arange(4, dtype=numpy.int32), b - a)
        return cells, edges, s['w'][a:b].reshape(-1).copy()

    def getMap(self):
        """mint's std::map view: dict(offsets (M+1), keys = cell*4+edge ascending per transect, w)"""
        n = ctypes.c_int64()
        _lib.call('nfx_pli_get_map_size', ctypes.byref(self._h), ctypes.byref(n))
        m = self.getNumberOfTransects()
        out = dict(offsets=numpy.zeros(m + 1, numpy.int64), keys=numpy.zeros(n.value, numpy.int64),
                   w=numpy.zeros(n.value))
        _lib.call('nfx_pli_get_map', ctypes.byref(self._h), _np_ptr(out['offsets']), _np_ptr(out['keys']),
                  _np_ptr(out['w']))
        return out

    # -- batched device path ----------------------------------------------------------------------------
    def integrate(self, eflux, order='map', out=None):
        """K3: eflux cuda tensor (nt, 2*ncell) float64 -> (nt, M) cuda tensor"""
        torch = _torch()
        _require_cuda(eflux, torch.float64, 'eflux')
        nt = eflux.shape[0]
        m = self.getNumberOfTransects()
        if out is None:
            out = torch.empty((nt, m), dtype=torch.float64, device=eflux.device)
        with torch.cuda.device(eflux.device):
            _lib.call('nfx_pli_integrate', ctypes.byref(self._h), _t_ptr(eflux), nt, _ORDERS[order], _t_ptr(out),
                      _stream_ptr())
        return out

    def integrateCellByCell(self, data, order='map', out=None):
        """data cuda tensor (nt, ncell, 4) float64 -> (nt, M) cuda tensor (getIntegral for every step)"""
        torch = _torch()
        _require_cuda(data, torch.float64, 'data')
        nt = data.shape[0]
        m = self.getNumberOfTransects()
        if out is None:
            out = torch.empty((nt, m), dtype=torch.float64, device=data.device)
        with torch.cuda.device(data.device):
            _lib.call('nfx_pli_get_integrals_device', ctypes.byref(self._h), _t_ptr(data), nt, _ORDERS[order],
                      _t_ptr(out), _stream_ptr())
        return out

    def getNumberOfPanels(self, dtype='float64'):
        """(npanels, panel_cells) of the fused pass for uo/vo stored as `dtype` ('float64' | 'float32' | 'f64' | 'f32'):
        batches are (time step, panel) pairs, see fluxSeries(batch_range=)"""
        code = _lib.NFX_F32 if str(dtype) in ('float32', 'f32', 'torch.float32') else _lib.NFX_F64
        n, pc = ctypes.c_int(), ctypes.c_int64()
        _lib.call('nfx_pli_get_num_panels_dtype', ctypes.byref(self._h), code, ctypes.byref(n), ctypes.byref(pc))
        return n.value, pc.value

    def getColumnGroups(self, dtype='float64', order='map', vec=4):
        """(panel_offsets (npanels+1), groups) int64/int32 numpy arrays: the column groups the sparse fused pass loads for
        uo/vo of `dtype` -- per panel q, groups[panel_offsets[q]:panel_offsets[q+1]] ascending, group g = columns
        [g*vec, g*vec+vec) of the panel in which a transect reads eU or eV"""
        code = _lib.NFX_F32 if str(dtype) in ('float32', 'f32', 'torch.float32') else _lib.NFX_F64
        npanels = self.getNumberOfPanels(dtype)[0]
        offs = numpy.zeros(npanels + 1, numpy.int64)
        n = ctypes.c_int64()
        _lib.call('nfx_pli_get_column_groups', ctypes.byref(self._h), code, _ORDERS[order], int(vec), _np_ptr(offs),
                  None, ctypes.byref(n))
        groups = numpy.zeros(max(n.value, 1), numpy.int32)
        _lib.call('nfx_pli_get_column_groups', ctypes.byref(self._h), code, _ORDERS[order], int(vec), None,
                  _np_ptr(groups), ctypes.byref(n))
        return offs, groups[:n.value]

    def seriesStatus(self):
        """Synchronise the current stream and raise NemofluxGpuError if a fused K2+K3 pass launched on this handle
        aborted (its series is NaN); returns 0 otherwise.  The device-path fluxSeries is asynchronous: call this
        before trusting a series that never leaves the device (a later fluxSeries call on the handle also reports it)."""
        st = ctypes.c_int()
        _lib.call('nfx_pli_series_status', ctypes.byref(self._h), _stream_ptr(), ctypes.byref(st))
        return st.value

    def fluxSeries(self, u, v, thickness, arc1, arc2, sverdrup=False, fill=float('nan'), order='map', eflux=None,
                   out=None, chunk_steps=0, batch_range=None, e3u=None, e3v=None, layers=None):
        """flux time series of every transect: (nt, M).

        u, v: (nt, nz, ny, nx) [or (nz, ny, nx)] float64/float32, either cuda tensors (device path: K2+K3 on
        the current stream, returns a cuda tensor) or host numpy arrays / CPU tensors (streams time chunks
        through double-buffered device staging, returns a numpy array; big-endian numpy arrays -- a NetCDF classic
        file as memory-mapped -- are uploaded as stored and byte-swapped on the device).  thickness (nz),
        arc1/arc2 (ncell) on the same side as u, v.  Needs Grid.setCGridShape before computeWeights.

        batch_range=(b0, b1) (device tensors only): run only the batches b = t*npanels + q in [b0, b1) and return
        PARTIAL sums -- the building block of the balanced multi-GPU sharding in nemoflux_b200.dist.

        e3u, e3v: per-column vertical scale factors, (1 or nt, nz, cells) with the dtype and plane layout of
        uo/vo (with host uo/vo: CUDA tensors uploaded once by the caller -- a mesh_mask's e3u_0/e3v_0 -- or host
        arrays in the byte order of uo/vo, streamed with them when they hold nt time steps); they replace the 1-D thickness (SURVEY 8f rank 4; fused pass with eflux=None when the
        policy of nfx_flux_series_e3 allows, else two launches).

        layers: ascending model-level boundaries [l0 < l1 < ... < lN] with 0 <= l0 and lN <= nz -> the series is
        (nt, N, M): [t, i, m] is transect m's flux at step t restricted to the levels [l_i, l_{i+1}) -- bit for bit the
        series with the thickness (or e3u/e3v) zeroed outside the layer, on finite data.  uo/vo are read once whatever
        the layering; eflux, if given, is (nt, N, 2*ncell).  Not combined with batch_range."""
        torch = _torch()
        lev = _layer_levels(layers)
        if lev is not None and batch_range is not None:
            raise ValueError('batch_range and layers cannot be combined')
        if isinstance(u, torch.Tensor) and u.is_cuda:
            return self._flux_series_device(u, v, thickness, arc1, arc2, sverdrup, fill, order, eflux, out, batch_range,
                                            e3u, e3v, lev)
        if batch_range is not None:
            raise ValueError('batch_range needs CUDA tensors')
        return self._flux_series_host(u, v, thickness, arc1, arc2, sverdrup, fill, order, chunk_steps, e3u, e3v, lev)

    def fluxSection(self, u, v, thickness, arc1, arc2, sverdrup=False, fill=float('nan'), layers=None, out=None,
                    chunk_steps=0, e3u=None, e3v=None, windows=None):
        """transport section: the flux across every sub-segment (cell crossing) of every transect, per layer of model
        levels and time step -> (nt, N, nsub), float64.  getSubsegments()['offsets'] splits the last axis by transect
        (emission order), getSectionGeometry() places every crossing along its transect.

        Arguments as fluxSeries: CUDA tensors (device path, returns a CUDA tensor on the current stream; padded planes
        and e3u/e3v of 1 or nt steps) or host arrays (chunked through the host-buffer pipeline, native or big-endian,
        returns numpy).  layers: level boundaries [l0 < ... < lN] as in fluxSeries; None = one layer per level.

        [t, i, s] = ((w0*E[idx0] + w1*E[idx1]) + w2*E[idx2]) + w3*E[idx3] over the 4 edge entries of sub-segment s, with
        E the layer-i edge flux fluxSeries(layers=, eflux=) writes, bit for bit; a transect's crossings add up to its
        layered series to rounding.

        windows: step boundaries [b0 < b1 < ... < bK] (0 <= b0, bK <= nt) -> the time mean over every window of steps
        [b_w, b_{w+1}), (K, N, nsub) (out: CUDA float64 of that shape).  The sum of the window is taken in ascending
        step order from +0 (a one-step window of -0 gives +0), every add rounded on its own, then divided by the
        window's length: numpy reproduces it bit for bit from the per-step section with a sequential loop over t.  Steps
        outside [b0, bK) are not read.  The memory is that of the K windows, whatever nt; see sectionWindowSums."""
        wins = _window_bounds(windows)
        if wins is None:
            return self._section(u, v, thickness, arc1, arc2, sverdrup, fill, layers, out, chunk_steps, e3u, e3v)
        sums = self.sectionWindowSums(u, v, thickness, arc1, arc2, wins, sverdrup=sverdrup, fill=fill, layers=layers,
                                      sums=out, chunk_steps=chunk_steps, e3u=e3u, e3v=e3v)
        lengths = numpy.diff(wins).astype(numpy.float64)
        if isinstance(sums, numpy.ndarray):
            sums /= lengths[:, None, None]
            return sums
        # a CUDA tensor of lengths, not a Python scalar: torch divides by a host scalar through its reciprocal
        return sums.div_(_torch().from_numpy(lengths).to(sums.device).view(-1, 1, 1))

    def sectionWindowSums(self, u, v, thickness, arc1, arc2, windows, sverdrup=False, fill=float('nan'), layers=None,
                          sums=None, continue_first=False, chunk_steps=0, e3u=None, e3v=None):
        """sums over windows of time steps of fluxSection(layers=): (K, N, nsub) float64, window w the steps
        [b_w, b_{w+1}) of the steps passed, added in ascending step order from +0.  fluxSection(windows=) divides these
        by the window lengths.  sums: the output (CUDA tensor for CUDA inputs, C-contiguous float64 numpy array for
        host inputs; None = a new one).  continue_first: window 0 continues the partial sums already in sums[0], so a
        record read in blocks of steps (a window split over several calls, in step order) gives the bits of one call."""
        torch = _torch()
        wins = _window_bounds(windows)
        if wins is None:
            raise ValueError('windows is required')
        lev = _layer_levels(layers)
        nsub = self.getNumberOfSubsegments()
        if isinstance(u, torch.Tensor) and u.is_cuda:
            u, v, nt, nz, ncell, ld, lev = self._section_device_inputs(u, v, thickness, arc1, arc2, e3u, e3v, lev)
            use_e3 = e3u is not None or e3v is not None
            e3_nt = _check_e3(e3u, e3v, u, nt, nz, ncell, ld) if use_e3 and nt else 0
            shape = (wins.size - 1, lev.size - 1, nsub)
            if sums is None:
                sums = (torch.zeros if continue_first else torch.empty)(shape, dtype=torch.float64, device=u.device)
            _require_cuda(sums, torch.float64, 'out')
            if tuple(sums.shape) != shape or not sums.is_contiguous():
                raise ValueError(f'out must be a contiguous CUDA tensor of shape (K, nlayers, nsub) = {shape}')
            ptr = lambda t: _t_ptr(t) if t is not None and t.numel() else None   # noqa: E731
            with torch.cuda.device(u.device):
                _lib.call('nfx_flux_section_window_sums', ctypes.byref(self._h), ptr(u), ptr(v), ptr(e3u), ptr(e3v),
                          _dtype_code(str(u.dtype)), e3_nt, None if use_e3 else _t_ptr(thickness), _t_ptr(arc1),
                          _t_ptr(arc2), nt, nz, ld, lev.size - 1, _np_ptr(lev), int(bool(sverdrup)), float(fill),
                          wins.size - 1, _np_ptr(wins), int(bool(continue_first)), ptr(sums), _stream_ptr())
            return sums
        keep = (u, v, e3u, e3v)  # keep pinned tensors alive while numpy views are in use
        h = _host_inputs(u, v, thickness, arc1, arc2, e3u, e3v)
        lev = numpy.arange(h.nz + 1, dtype=numpy.int32) if lev is None else lev
        shape = (wins.size - 1, lev.size - 1, nsub)
        if sums is None:
            sums = numpy.zeros(shape, numpy.float64)
        if not isinstance(sums, numpy.ndarray) or sums.dtype != numpy.float64 or sums.shape != shape or \
                not sums.flags.c_contiguous or not sums.flags.writeable:
            raise ValueError(f'out must be a C-contiguous float64 numpy array of shape (K, nlayers, nsub) = {shape}')
        pu, pv, e3_nt, on_device = h.e3 if h.e3 is not None else (None, None, 0, False)
        _lib.call('nfx_flux_section_window_sums_host', ctypes.byref(self._h), _np_ptr(h.u), _np_ptr(h.v), pu, pv,
                  h.code, e3_nt, int(on_device), None if h.th is None else _np_ptr(h.th), _np_ptr(h.a1), _np_ptr(h.a2),
                  h.nt, h.nz, lev.size - 1, _np_ptr(lev), int(bool(sverdrup)), float(fill), wins.size - 1,
                  _np_ptr(wins), int(bool(continue_first)), int(chunk_steps), _np_ptr(sums))
        del keep
        return sums

    def fluxClasses(self, u, v, thickness, arc1, arc2, cfield, bounds, cfill=float('nan'), sverdrup=False,
                    fill=float('nan'), e3u=None, e3v=None, chunk_steps=0):
        """class transport: the flux across every transect binned by a T-grid field (temperature, salinity, density...)
        -> (nt, K, M) float64: [t, j, m] is transect m's flux at step t carried by the levels of its crossings whose
        class value lies in [b_j, b_{j+1}).

        Arguments as fluxSection (CUDA tensors on the current stream, or host arrays through the chunk pipeline), plus:
        cfield, the class field at the T points, with the dtype, byte order and plane layout of uo/vo, (1 or nt, nz,
        ...) (a (nz, ny, nx) field is time-invariant); cfill its missing-value marker (compared in the storage type;
        NaN = none); bounds, K + 1 strictly ascending class bounds (1 <= K <= 96, +-inf allowed, no NaN).

        Every level k of crossing s adds fluxSection(layers=range(nz + 1))[t, k, s] to the class of
        c = cfield[t or 0, k, cell(s)]; NaN, cfill, c < b0 and c >= bK count nowhere.  The sum order is fixed (per
        crossing ascending levels, 32-crossing tiles by a fixed tree, tiles in order): the bits depend only on the
        inputs, whatever chunk_steps, the byte order or the side of the inputs."""
        torch = _torch()
        b = numpy.ascontiguousarray(_to_numpy(bounds), numpy.float64).reshape(-1)
        if b.size < 2:
            raise ValueError(f'bounds must hold at least 2 class bounds, got {b.size}')
        m = self.getNumberOfTransects()
        nsub = self.getNumberOfSubsegments()
        if isinstance(u, torch.Tensor) and u.is_cuda:
            u, v, nt, nz, ncell, ld = self._device_inputs(u, v, thickness, arc1, arc2, e3u, e3v)
            use_e3 = e3u is not None or e3v is not None
            cfield, c_nt = _class_field_device(cfield, u, nt, nz, ncell, ld)
            out = torch.zeros((nt, b.size - 1, m), dtype=torch.float64, device=u.device)
            if nt == 0 or nsub == 0:        # nothing to compute: no launch (empty tensors have no device address)
                return out
            e3_nt = _check_e3(e3u, e3v, u, nt, nz, ncell, ld) if use_e3 else 0
            ptr = lambda t: _t_ptr(t) if t is not None else None   # noqa: E731
            with torch.cuda.device(u.device):
                _lib.call('nfx_flux_classes', ctypes.byref(self._h), _t_ptr(u), _t_ptr(v), ptr(e3u), ptr(e3v),
                          _dtype_code(str(u.dtype)), e3_nt, None if use_e3 else _t_ptr(thickness), _t_ptr(arc1),
                          _t_ptr(arc2), nt, nz, ld, _t_ptr(cfield), c_nt, float(cfill), b.size - 1, _np_ptr(b),
                          int(bool(sverdrup)), float(fill), _t_ptr(out), _stream_ptr())
            return out
        keep = (u, v, e3u, e3v)  # keep pinned tensors alive while numpy views are in use
        h = _host_inputs(u, v, thickness, arc1, arc2, e3u, e3v)
        c = _class_field_host(cfield, h)
        res = numpy.zeros((h.nt, b.size - 1, m), numpy.float64)
        pu, pv, e3_nt, on_device = h.e3 if h.e3 is not None else (None, None, 0, False)
        _lib.call('nfx_flux_classes_host', ctypes.byref(self._h), _np_ptr(h.u), _np_ptr(h.v), pu, pv, h.code, e3_nt,
                  int(on_device), None if h.th is None else _np_ptr(h.th), _np_ptr(h.a1), _np_ptr(h.a2), h.nt, h.nz,
                  _np_ptr(c), c.shape[0], float(cfill), b.size - 1, _np_ptr(b), int(bool(sverdrup)), float(fill),
                  int(chunk_steps), _np_ptr(res))
        del keep
        return res

    def fluxTracer(self, u, v, thickness, arc1, arc2, tracer, ref=0.0, tfill=float('nan'), layers=None, section=False,
                   sverdrup=False, fill=float('nan'), e3u=None, e3v=None, chunk_steps=0):
        """tracer transport: the flux across every transect weighted by a tracer (temperature, salinity...) taken at
        the C-grid face of every edge -> float64, (nt, M) for layers=None and (nt, N, M) otherwise, as fluxSeries; with
        section=True the value of every crossing, (nt, N, nsub), one layer per level by default, as fluxSection.

        Arguments as fluxSection (CUDA tensors on the current stream, or host arrays through the chunk pipeline), plus:
        tracer, at the T points, with the dtype, byte order and plane layout of uo/vo, (1 or nt, nz, ...) (a (nz, ny,
        nx) tracer is time-invariant); tfill its missing-value marker (compared in the storage type; NaN is always
        missing); ref a reference value subtracted from the face value.

        The face of an edge lies between two T cells (E: c and east(c), W: west(c) and c, N: c and north(c), none in
        the top row, S: south(c) and c; x-periodic); its value at level k is 0.5 * (tau_a + tau_b) - ref with both
        sides present, tau - ref with one, 0 with none.  Every level term of fluxSection's edge sums is multiplied by
        it: with tracer == 1 and ref == 0 the section is fluxSection's bit for bit.  The series folds the crossings of
        a transect as fluxClasses does (32-crossing tiles by a fixed tree, tiles in order): the bits depend only on the
        inputs, whatever chunk_steps, the byte order or the side of the inputs.  Units: tracer units x flux units."""
        torch = _torch()
        lev = _layer_levels(layers)
        m = self.getNumberOfTransects()
        nsub = self.getNumberOfSubsegments()
        width = nsub if section else m

        def levels(nz):
            if lev is not None:
                return lev
            return numpy.arange(nz + 1, dtype=numpy.int32) if section else numpy.array([0, nz], numpy.int32)

        def shaped(x):          # (nt, M) for a series without layers
            return x if section or lev is not None else x.reshape(x.shape[0], m)
        if isinstance(u, torch.Tensor) and u.is_cuda:
            u, v, nt, nz, ncell, ld = self._device_inputs(u, v, thickness, arc1, arc2, e3u, e3v)
            use_e3 = e3u is not None or e3v is not None
            tracer, tr_nt = _class_field_device(tracer, u, nt, nz, ncell, ld, 'tracer')
            lv = levels(nz)
            out = torch.zeros((nt, lv.size - 1, width), dtype=torch.float64, device=u.device)
            if nt == 0 or nsub == 0:        # nothing to compute: no launch (empty tensors have no device address)
                return shaped(out)
            e3_nt = _check_e3(e3u, e3v, u, nt, nz, ncell, ld) if use_e3 else 0
            ptr = lambda t: _t_ptr(t) if t is not None else None   # noqa: E731
            with torch.cuda.device(u.device):
                _lib.call('nfx_flux_tracer', ctypes.byref(self._h), _t_ptr(u), _t_ptr(v), ptr(e3u), ptr(e3v),
                          _dtype_code(str(u.dtype)), e3_nt, None if use_e3 else _t_ptr(thickness), _t_ptr(arc1),
                          _t_ptr(arc2), nt, nz, ld, _t_ptr(tracer), tr_nt, float(tfill), float(ref), lv.size - 1,
                          _np_ptr(lv), int(bool(sverdrup)), float(fill), None if section else _t_ptr(out),
                          _t_ptr(out) if section else None, _stream_ptr())
            return shaped(out)
        keep = (u, v, e3u, e3v)  # keep pinned tensors alive while numpy views are in use
        h = _host_inputs(u, v, thickness, arc1, arc2, e3u, e3v)
        c = _class_field_host(tracer, h, 'tracer')
        lv = levels(h.nz)
        res = numpy.zeros((h.nt, lv.size - 1, width), numpy.float64)
        pu, pv, e3_nt, on_device = h.e3 if h.e3 is not None else (None, None, 0, False)
        _lib.call('nfx_flux_tracer_host', ctypes.byref(self._h), _np_ptr(h.u), _np_ptr(h.v), pu, pv, h.code, e3_nt,
                  int(on_device), None if h.th is None else _np_ptr(h.th), _np_ptr(h.a1), _np_ptr(h.a2), h.nt, h.nz,
                  _np_ptr(c), c.shape[0], float(tfill), float(ref), lv.size - 1, _np_ptr(lv), int(bool(sverdrup)),
                  float(fill), int(chunk_steps), None if section else _np_ptr(res), _np_ptr(res) if section else None)
        del keep
        return shaped(res)

    def _section_device_inputs(self, u, v, thickness, arc1, arc2, e3u, e3v, lev):
        """checks of the CUDA inputs of fluxSection / sectionWindowSums -> (u, v, nt, nz, ncell, ld, levels), the
        levels of one layer per level when lev is None"""
        u, v, nt, nz, ncell, ld = self._device_inputs(u, v, thickness, arc1, arc2, e3u, e3v)
        lev = numpy.arange(nz + 1, dtype=numpy.int32) if lev is None else lev
        return u, v, nt, nz, ncell, ld, lev

    def _section(self, u, v, thickness, arc1, arc2, sverdrup, fill, layers, out, chunk_steps, e3u, e3v):
        torch = _torch()
        lev = _layer_levels(layers)
        nsub = self.getNumberOfSubsegments()
        if isinstance(u, torch.Tensor) and u.is_cuda:
            u, v, nt, nz, ncell, ld, lev = self._section_device_inputs(u, v, thickness, arc1, arc2, e3u, e3v, lev)
            use_e3 = e3u is not None or e3v is not None
            shape = (nt, lev.size - 1, nsub)
            if out is None:
                out = torch.empty(shape, dtype=torch.float64, device=u.device)
            _require_cuda(out, torch.float64, 'out')
            if out.numel() != nt * (lev.size - 1) * nsub:
                raise ValueError(f'out must hold nt*nlayers*nsub = {nt * (lev.size - 1) * nsub} values')
            if nt == 0 or nsub == 0:        # nothing to compute: no launch (empty tensors have no device address)
                return out
            e3_nt = _check_e3(e3u, e3v, u, nt, nz, ncell, ld) if use_e3 else 0
            ptr = lambda t: _t_ptr(t) if t is not None else None   # noqa: E731
            with torch.cuda.device(u.device):
                _lib.call('nfx_flux_section', ctypes.byref(self._h), _t_ptr(u), _t_ptr(v), ptr(e3u), ptr(e3v),
                          _dtype_code(str(u.dtype)), e3_nt, None if use_e3 else _t_ptr(thickness), _t_ptr(arc1),
                          _t_ptr(arc2), nt, nz, ld, lev.size - 1, _np_ptr(lev), int(bool(sverdrup)), float(fill),
                          _t_ptr(out), _stream_ptr())
            return out
        if out is not None:
            raise ValueError('out is for CUDA inputs; host inputs return a new numpy array')
        keep = (u, v, e3u, e3v)  # keep pinned tensors alive while numpy views are in use
        h = _host_inputs(u, v, thickness, arc1, arc2, e3u, e3v)
        lev = numpy.arange(h.nz + 1, dtype=numpy.int32) if lev is None else lev
        res = numpy.zeros((h.nt, lev.size - 1, nsub), numpy.float64)
        pu, pv, e3_nt, on_device = h.e3 if h.e3 is not None else (None, None, 0, False)
        _lib.call('nfx_flux_section_host', ctypes.byref(self._h), _np_ptr(h.u), _np_ptr(h.v), pu, pv, h.code, e3_nt,
                  int(on_device), None if h.th is None else _np_ptr(h.th), _np_ptr(h.a1), _np_ptr(h.a2), h.nt, h.nz,
                  lev.size - 1, _np_ptr(lev), int(bool(sverdrup)), float(fill), int(chunk_steps), _np_ptr(res))
        del keep
        return res

    def getNumberOfSubsegments(self):
        n = ctypes.c_int64()
        _lib.call('nfx_pli_get_num_subsegments', ctypes.byref(self._h), ctypes.byref(n))
        return n.value

    def getSectionGeometry(self):
        """where every crossing of fluxSection lies, host numpy arrays per sub-segment (emission order):
        transect, segment (index of the polyline segment), cell_j / cell_i (cell = j*nx + i), lon0/lat0 and lon1/lat1
        (degrees: the crossing's end points on the polyline passed to computeWeights, x-period image shift undone),
        length_km (great-circle distance between the end points) and distance_km (of the crossing's midpoint from the
        transect's start: the great-circle lengths of the earlier segments plus the great-circle distance from the
        segment's start to the midpoint); plus offsets (M+1), as getSubsegments.  Distances are on a sphere of radius
        6371 km.  Where a transect runs along a grid line the two cells beside it both hold the crossing, with
        duplicity coefficients getSubsegments()['coeff'] that add up to 1."""
        if self._grid is None or self._grid._cgrid is None:
            raise RuntimeError('getSectionGeometry needs Grid.setCGridShape before computeWeights')
        return sectionGeometry(self.getSubsegments(), self._polylines, self._grid._cgrid[1])

    def _device_inputs(self, u, v, thickness, arc1, arc2, e3u, e3v):
        """checks of the CUDA-tensor inputs of fluxSeries / fluxSection -> (u, v, nt, nz, ncell, ld), u and v with a
        time axis"""
        torch = _torch()
        ncells = self._grid.getNumberOfCells() if self._grid is not None else -1
        if u.dim() == 3 and u.shape[2] != ncells and u.shape[1] * u.shape[2] == ncells:
            u, v = u.unsqueeze(0), v.unsqueeze(0)          # (z, y, x): one time step (field.py:130)
        for name, t in (('u', u), ('v', v)):
            if not isinstance(t, torch.Tensor) or not t.is_cuda:
                raise TypeError(f'{name} must be a CUDA tensor (there is no CPU fallback)')
        if u.dtype != v.dtype or u.shape != v.shape or u.stride() != v.stride():
            raise ValueError('uo and vo must have the same dtype, shape and strides')
        nt, nz, ncell, ld = _plane_layout(u, 'uo')
        if ncell != ncells:
            raise ValueError(f'uo has {ncell} cells per level, the grid has {ncells}')
        use_e3 = e3u is not None or e3v is not None
        checks = [('arc1', arc1, ncell), ('arc2', arc2, ncell)] + ([] if use_e3 else [('thickness', thickness, nz)])
        for name, t, n in checks:
            _require_cuda(t, torch.float64, name)
            if t.numel() != n:
                raise ValueError(f'{name} must hold {n} values, got {t.numel()}')
        return u, v, nt, nz, ncell, ld

    def _flux_series_device(self, u, v, thickness, arc1, arc2, sverdrup, fill, order, eflux, out, batch_range=None,
                            e3u=None, e3v=None, lev=None):
        torch = _torch()
        u, v, nt, nz, ncell, ld = self._device_inputs(u, v, thickness, arc1, arc2, e3u, e3v)
        use_e3 = e3u is not None or e3v is not None
        m = self.getNumberOfTransects()
        shape = (nt, m) if lev is None else (nt, lev.size - 1, m)
        if nt == 0 or m == 0:       # nothing to integrate: no launch (empty tensors have no device address)
            return out if out is not None else torch.zeros(shape, dtype=torch.float64, device=u.device)
        if lev is not None:
            e3_nt = _check_e3(e3u, e3v, u, nt, nz, ncell, ld) if use_e3 else 0
            if eflux is not None:
                _require_cuda(eflux, torch.float64, 'eflux')
                if eflux.numel() != nt * (lev.size - 1) * 2 * ncell:
                    raise ValueError(f'eflux must hold nt*nlayers*2*ncell = {nt * (lev.size - 1) * 2 * ncell} values')
            if out is None:
                out = torch.empty(shape, dtype=torch.float64, device=u.device)
            _require_cuda(out, torch.float64, 'out')
            if out.numel() != nt * (lev.size - 1) * m:
                raise ValueError(f'out must hold nt*nlayers*M = {nt * (lev.size - 1) * m} values')
            ptr = lambda t: _t_ptr(t) if t is not None else None   # noqa: E731
            with torch.cuda.device(u.device):
                _lib.call('nfx_flux_series_layers', ctypes.byref(self._h), _t_ptr(u), _t_ptr(v), ptr(e3u), ptr(e3v),
                          _dtype_code(str(u.dtype)), e3_nt, None if use_e3 else _t_ptr(thickness), _t_ptr(arc1),
                          _t_ptr(arc2), nt, nz, ld, lev.size - 1, _np_ptr(lev), int(bool(sverdrup)), float(fill),
                          _ORDERS[order], ptr(eflux), _t_ptr(out), _stream_ptr())
            return out
        if use_e3:
            e3_nt = _check_e3(e3u, e3v, u, nt, nz, ncell, ld)
            if eflux is not None:
                _require_cuda(eflux, torch.float64, 'eflux')
            if out is None:
                out = torch.empty((nt, m), dtype=torch.float64, device=u.device)
            if batch_range is not None:
                if eflux is not None:
                    raise ValueError('batch_range and eflux cannot be combined')
                with torch.cuda.device(u.device):
                    _lib.call('nfx_flux_series_range_e3', ctypes.byref(self._h), _t_ptr(u), _t_ptr(v), _t_ptr(e3u),
                              _t_ptr(e3v), _dtype_code(str(u.dtype)), e3_nt, _t_ptr(arc1), _t_ptr(arc2), nt, nz, ld,
                              int(bool(sverdrup)), float(fill), _ORDERS[order], int(batch_range[0]), int(batch_range[1]),
                              _t_ptr(out), _stream_ptr())
                return out
            with torch.cuda.device(u.device):
                _lib.call('nfx_flux_series_e3', ctypes.byref(self._h), _t_ptr(u), _t_ptr(v), _t_ptr(e3u), _t_ptr(e3v),
                          _dtype_code(str(u.dtype)), e3_nt, _t_ptr(arc1), _t_ptr(arc2), nt, nz, ld, int(bool(sverdrup)),
                          float(fill), _ORDERS[order], _t_ptr(eflux) if eflux is not None else None, _t_ptr(out),
                          _stream_ptr())
            return out
        if eflux is not None:       # the caller wants the (nt, 2*ncell) edge fluxes too: classic K2 -> HBM -> K3
            _require_cuda(eflux, torch.float64, 'eflux')
            if eflux.numel() != nt * 2 * ncell:
                raise ValueError(f'eflux must hold nt*2*ncell = {nt * 2 * ncell} values')
        if out is None:
            out = torch.empty((nt, m), dtype=torch.float64, device=u.device)
        if batch_range is not None:
            if eflux is not None:
                raise ValueError('batch_range and eflux cannot be combined')
            with torch.cuda.device(u.device):
                _lib.call('nfx_flux_series_range', ctypes.byref(self._h), _t_ptr(u), _t_ptr(v), _dtype_code(str(u.dtype)),
                          _t_ptr(thickness), _t_ptr(arc1), _t_ptr(arc2), nt, nz, ld, int(bool(sverdrup)), float(fill),
                          _ORDERS[order], int(batch_range[0]), int(batch_range[1]), _t_ptr(out), _stream_ptr())
            return out
        with torch.cuda.device(u.device):
            # eflux NULL -> the fast path: edge fluxes stay in an L2-resident ring between K2 and K3
            _lib.call('nfx_flux_series_ld', ctypes.byref(self._h), _t_ptr(u), _t_ptr(v), _dtype_code(str(u.dtype)),
                      _t_ptr(thickness), _t_ptr(arc1), _t_ptr(arc2), nt, nz, ld, int(bool(sverdrup)), float(fill),
                      _ORDERS[order], _t_ptr(eflux) if eflux is not None else None, _t_ptr(out), _stream_ptr())
        return out

    def _flux_series_host(self, u, v, thickness, arc1, arc2, sverdrup, fill, order, chunk_steps, e3u=None, e3v=None,
                          lev=None):
        keep = (u, v, e3u, e3v)  # keep pinned tensors alive while numpy views are in use
        h = _host_inputs(u, v, thickness, arc1, arc2, e3u, e3v)
        u, v, code, nt, nz, a1, a2 = h.u, h.v, h.code, h.nt, h.nz, h.a1, h.a2
        m = self.getNumberOfTransects()
        out = numpy.zeros((nt, m) if lev is None else (nt, lev.size - 1, m), numpy.float64)
        if h.e3 is not None:
            pu, pv, e3_nt, on_device = h.e3
            if lev is not None:
                _lib.call('nfx_flux_series_layers_host', ctypes.byref(self._h), _np_ptr(u), _np_ptr(v), pu, pv, code,
                          e3_nt, int(on_device), None, _np_ptr(a1), _np_ptr(a2), nt, nz, lev.size - 1, _np_ptr(lev),
                          int(bool(sverdrup)), float(fill), _ORDERS[order], int(chunk_steps), _np_ptr(out))
                del keep
                return out
            _lib.call('nfx_flux_series_host_e3', ctypes.byref(self._h), _np_ptr(u), _np_ptr(v), pu, pv, code, e3_nt,
                      int(on_device), _np_ptr(a1), _np_ptr(a2), nt, nz, int(bool(sverdrup)), float(fill), _ORDERS[order],
                      int(chunk_steps), _np_ptr(out))
            del keep
            return out
        th = h.th
        if lev is not None:
            _lib.call('nfx_flux_series_layers_host', ctypes.byref(self._h), _np_ptr(u), _np_ptr(v), None, None, code, 0, 0,
                      _np_ptr(th), _np_ptr(a1), _np_ptr(a2), nt, nz, lev.size - 1, _np_ptr(lev), int(bool(sverdrup)),
                      float(fill), _ORDERS[order], int(chunk_steps), _np_ptr(out))
            del keep
            return out
        _lib.call('nfx_flux_series_host', ctypes.byref(self._h), _np_ptr(u), _np_ptr(v), code,
                  _np_ptr(th), _np_ptr(a1), _np_ptr(a2), nt, nz, int(bool(sverdrup)), float(fill), _ORDERS[order],
                  int(chunk_steps), _np_ptr(out))
        del keep
        return out


class VectorInterp(object):
    """mint.VectorInterp (field.py:90-95,119-120): vectors of the edge-flux field at arbitrary points"""

    def __init__(self):
        self._h = ctypes.c_void_p()
        _lib.call('nfx_vinterp_new', ctypes.byref(self._h))
        self._grid = None
        self._npts = 0

    def __del__(self):
        try:
            if self._h:
                _lib.load().nfx_vinterp_del(ctypes.byref(self._h))
        except Exception:
            pass

    def setGrid(self, grid):
        if not isinstance(grid, Grid):
            raise TypeError('setGrid expects a nemoflux_gpu.Grid')
        _lib.call('nfx_vinterp_set_grid', ctypes.byref(self._h), grid._h)
        self._grid = grid

    def buildLocator(self, numCellsPerBucket=128, periodX=360., enableFolding=False):
        _lib.call('nfx_vinterp_build_locator', ctypes.byref(self._h), int(numCellsPerBucket), float(periodX),
                  int(bool(enableFolding)))

    def findPoints(self, points, tol2=1.e-12):
        """points (n, 3) lon, lat, ignored; returns the number of points that are in no cell"""
        pts = numpy.ascontiguousarray(points, numpy.float64)
        if pts.ndim != 2 or pts.shape[1] != 3:
            raise ValueError(f'points must have shape (npoints, 3), got {pts.shape}')
        bad = ctypes.c_int64()
        _lib.call('nfx_vinterp_find_points', ctypes.byref(self._h), pts.shape[0], _np_ptr(pts), float(tol2),
                  ctypes.byref(bad))
        self._npts = pts.shape[0]
        return bad.value

    def getCells(self):
        """(cell ids (-1 = not found), parametric coordinates (n, 2)) of the points of the last findPoints"""
        cell = numpy.zeros(self._npts, numpy.int64)
        xi = numpy.zeros((self._npts, 2))
        if self._npts:
            _lib.call('nfx_vinterp_get_cells', ctypes.byref(self._h), _np_ptr(cell), _np_ptr(xi))
        return cell, xi

    def getFaceVectors(self, data, placement=CELL_BY_CELL_DATA):
        """data (ncells, 4) host array of edge fluxes (S, E, N, W) -> (n, 3) vectors"""
        d = numpy.ascontiguousarray(data, numpy.float64)
        ncell = self._grid.getNumberOfCells() if self._grid else -1
        if d.size != ncell * 4:
            raise ValueError(f'data must hold ncells*4 = {ncell * 4} values, got {d.size}')
        vec = numpy.zeros((self._npts, 3))
        if self._npts:
            _lib.call('nfx_vinterp_get_face_vectors', ctypes.byref(self._h), _np_ptr(d), int(placement), _np_ptr(vec))
        return vec


def _to_numpy(x):
    torch = _torch()
    if isinstance(x, torch.Tensor):
        return x.detach().cpu().numpy()
    return numpy.asarray(x)


def sectionGeometry(sub, polylines, nx):
    """PolylineIntegral.getSectionGeometry from its pieces: sub = getSubsegments() (offsets, cell, seg, ta, tb), the
    polylines (npoints, >= 2) of lon/lat degrees in transect order, nx = cells per grid row"""
    offs = numpy.asarray(sub['offsets'], numpy.int64)
    n = int(offs[-1]) if offs.size else 0
    transect = numpy.repeat(numpy.arange(offs.size - 1, dtype=numpy.int32), numpy.diff(offs))
    seg = numpy.asarray(sub['seg'], numpy.int64)
    cell = numpy.asarray(sub['cell'], numpy.int64)
    p0 = numpy.zeros((n, 2))
    d = numpy.zeros((n, 2))
    start_km = numpy.zeros(n)          # distance of the segment's start from the transect's start
    for m, pts in enumerate(polylines):
        a, b = offs[m], offs[m + 1]
        if a == b:
            continue
        ll = numpy.asarray(pts, numpy.float64)[:, :2]
        cum = numpy.concatenate([[0.], numpy.cumsum(_great_circle_km(ll[:-1], ll[1:]))])
        sm = seg[a:b]
        p0[a:b] = ll[sm]
        d[a:b] = ll[sm + 1] - ll[sm]
        start_km[a:b] = cum[sm]
    ta, tb = numpy.asarray(sub['ta'], numpy.float64), numpy.asarray(sub['tb'], numpy.float64)
    e0 = p0 + ta[:, None] * d
    e1 = p0 + tb[:, None] * d
    mid = p0 + (0.5 * (ta + tb))[:, None] * d
    return dict(offsets=offs, transect=transect, segment=numpy.asarray(sub['seg'], numpy.int32), cell_j=cell // nx,
                cell_i=cell % nx, lon0=e0[:, 0], lat0=e0[:, 1], lon1=e1[:, 0], lat1=e1[:, 1],
                length_km=_great_circle_km(e0, e1), distance_km=start_km + _great_circle_km(p0, mid))


def _great_circle_km(a, b):
    """great-circle distance in km on a sphere of radius 6371 km between (n, 2) lon/lat points in degrees (haversine)"""
    a, b = numpy.radians(numpy.asarray(a, numpy.float64)), numpy.radians(numpy.asarray(b, numpy.float64))
    h = numpy.sin(0.5 * (b[..., 1] - a[..., 1])) ** 2 + \
        numpy.cos(a[..., 1]) * numpy.cos(b[..., 1]) * numpy.sin(0.5 * (b[..., 0] - a[..., 0])) ** 2
    return 2. * 6371. * numpy.arcsin(numpy.sqrt(numpy.clip(h, 0., 1.)))


class _HostInputs(object):
    pass


def _host_inputs(u, v, thickness, arc1, arc2, e3u, e3v):
    """checks of the host-array inputs of fluxSeries / fluxSection: u, v (C-contiguous, with a time axis), the dtype
    code (| NFX_BIG_ENDIAN for big-endian bytes), nt, nz, arc1/arc2 as float64 arrays, and either th (the thickness)
    or e3 = (pointer of e3u, pointer of e3v, e3_nt, on_device).  The arrays must stay alive for the call."""
    torch = _torch()
    if isinstance(u, torch.Tensor):
        u, v = u.numpy(), v.numpy()
    u = numpy.asarray(u)
    v = numpy.asarray(v)
    if u.ndim == 3:
        u, v = u[None], v[None]
    if u.ndim != 4 or u.shape != v.shape or u.dtype != v.dtype:
        raise ValueError("uo/vo shape does not match (t, z, y, x) or (z, y, x)")
    code = _dtype_code(u.dtype.newbyteorder('=').name)
    if not u.dtype.isnative:        # bytes as stored in a NetCDF classic file: swapped on the device
        code |= _lib.NFX_BIG_ENDIAN
    if not (u.flags.c_contiguous and v.flags.c_contiguous):
        u, v = numpy.ascontiguousarray(u), numpy.ascontiguousarray(v)
    nt, nz, ny, nx = u.shape
    ncell = ny * nx
    a1 = numpy.ascontiguousarray(_to_numpy(arc1), numpy.float64).reshape(-1)
    a2 = numpy.ascontiguousarray(_to_numpy(arc2), numpy.float64).reshape(-1)
    if a1.size != ncell or a2.size != ncell:
        raise ValueError('arc1/arc2 sizes do not match uo')
    h = _HostInputs()
    h.u, h.v, h.code, h.nt, h.nz, h.a1, h.a2, h.e3, h.th = u, v, code, nt, nz, a1, a2, None, None
    if e3u is not None or e3v is not None:
        if e3u is None or e3v is None:
            raise ValueError('e3u and e3v go together')
        on_device = isinstance(e3u, torch.Tensor) and e3u.is_cuda
        if on_device:
            if not (isinstance(e3v, torch.Tensor) and e3v.is_cuda):
                raise ValueError('e3u and e3v must live on the same side')
            want = torch.float64 if u.dtype.itemsize == 8 else torch.float32
            for name, t in (('e3u', e3u), ('e3v', e3v)):
                if t.dtype != want or not t.is_contiguous():
                    raise ValueError(f'{name} must be a contiguous CUDA tensor of the dtype of uo')
            pu, pv = _t_ptr(e3u), _t_ptr(e3v)
            # the host path runs on the handle's own streams: whatever produced e3u/e3v on the caller's stream
            # must be complete before they are read there
            torch.cuda.current_stream(e3u.device).synchronize()
        else:
            e3u, e3v = (numpy.asarray(x.numpy() if isinstance(x, torch.Tensor) else x) for x in (e3u, e3v))
            for name, x in (('e3u', e3u), ('e3v', e3v)):
                if x.dtype != u.dtype:
                    raise ValueError(f'{name} must have the dtype and byte order of uo ({u.dtype}), got {x.dtype}')
            e3u, e3v = numpy.ascontiguousarray(e3u), numpy.ascontiguousarray(e3v)
            pu, pv = _np_ptr(e3u), _np_ptr(e3v)
            h.keep_e3 = (e3u, e3v)
        n3 = int(e3u.numel() if on_device else e3u.size)
        if tuple(e3u.shape) != tuple(e3v.shape) or n3 not in (nz * ncell, nt * nz * ncell):
            raise ValueError('e3u/e3v must hold (1 or nt, nz, ny*nx) values of the same shape')
        h.e3 = (pu, pv, n3 // (nz * ncell), on_device)
        return h
    h.th = numpy.ascontiguousarray(_to_numpy(thickness), numpy.float64)
    if h.th.size != nz:
        raise ValueError('thickness size does not match uo')
    return h


def _layer_levels(layers):
    """layers -> contiguous int32 array of level boundaries (None stays None).  Only the form is checked here; the
    library rejects boundaries that are not strictly ascending inside [0, nz]."""
    if layers is None:
        return None
    a = numpy.asarray(_to_numpy(layers))
    if a.ndim != 1 or a.size < 2:
        raise ValueError(f'layers must be a 1-D sequence of at least 2 level boundaries, got shape {a.shape}')
    if a.dtype.kind not in 'iu' and not (a.dtype.kind == 'f' and numpy.all(a == numpy.round(a))):
        raise ValueError('layers must hold integer level indices')
    if numpy.any(numpy.abs(a) > 2 ** 31 - 1):
        raise ValueError('layers: level index out of range')
    return numpy.ascontiguousarray(a, numpy.int32)


def _window_bounds(windows):
    """windows -> contiguous int32 array of step boundaries (None stays None).  Only the form is checked here; the
    library rejects boundaries that are not strictly ascending inside [0, nt]."""
    if windows is None:
        return None
    a = numpy.asarray(_to_numpy(windows))
    if a.ndim != 1 or a.size < 2:
        raise ValueError(f'windows must be a 1-D sequence of at least 2 step boundaries, got shape {a.shape}')
    if a.dtype.kind not in 'iu' and not (a.dtype.kind == 'f' and numpy.all(a == numpy.round(a))):
        raise ValueError('windows must hold integer step indices')
    if numpy.any(numpy.abs(a) > 2 ** 31 - 1):
        raise ValueError('windows: step index out of range')
    return numpy.ascontiguousarray(a, numpy.int32)


def _plane_layout(t, name, ncell_expected=None):
    """(nt, nz, ncell, ld) of a uo/vo device tensor: (nt, nz, ny, nx) contiguous, or (nt, nz, ncell) whose level
    planes are padded in memory (stride(1) = ld >= ncell, stride(2) = 1, stride(0) = nz*ld)"""
    if t.dim() == 4:
        if not t.is_contiguous():
            raise ValueError(f'{name} must be contiguous')
        nt, nz = t.shape[0], t.shape[1]
        ncell = t.shape[2] * t.shape[3]
        return nt, nz, ncell, ncell
    if t.dim() == 3:
        nt, nz, ncell = t.shape
        ld = t.stride(1) if nz > 1 else (t.stride(0) if nt > 1 else ncell)
        ok = t.stride(2) == 1 and ld >= ncell and (nt == 1 or t.stride(0) == nz * ld) and (nz == 1 or t.stride(1) == ld)
        if not ok:
            raise ValueError(f'{name}: unsupported strides {t.stride()} for shape {tuple(t.shape)}')
        return nt, nz, ncell, ld
    raise ValueError(f"{name} shape does not match (t, z, y, x) or (t, z, ncell)")


def _check_e3(e3u, e3v, u, nt, nz, ncell, ld):
    """e3u/e3v: same dtype and plane layout as u, 1 or nt time steps; returns e3_nt"""
    torch = _torch()
    if e3u is None or e3v is None:
        raise ValueError('e3u and e3v go together')
    for name, t in (('e3u', e3u), ('e3v', e3v)):
        if not isinstance(t, torch.Tensor) or not t.is_cuda or t.dtype != u.dtype:
            raise TypeError(f'{name} must be a CUDA tensor with the dtype of uo/vo')
        ent, enz, encell, eld = _plane_layout(t, name)
        # the kernels step levels by ld and time steps by nz * ld, the layout of uo/vo
        if (enz, encell) != (nz, ncell) or ent not in (1, nt) or (eld != ld and enz > 1) or \
                (ent > 1 and t.stride(0) != nz * ld):
            raise ValueError(f'{name} must be (1 or nt, nz, cells) with the plane layout of uo/vo')
    if e3u.shape[0] != e3v.shape[0]:
        raise ValueError('e3u and e3v must hold the same number of time steps')
    return int(e3u.shape[0])


def _class_field_device(c, u, nt, nz, ncell, ld, name='cfield'):
    """a T-grid field next to uo/vo on the device (the class field of fluxClasses, the tracer of fluxTracer): a CUDA
    tensor with the dtype and plane layout of uo, (1 or nt, nz, ny, nx), (1 or nt, nz, cells) or (nz, ny, nx) -> (c with
    a time axis, its number of time steps)"""
    torch = _torch()
    if not isinstance(c, torch.Tensor) or not c.is_cuda or c.dtype != u.dtype:
        raise TypeError(f'{name} must be a CUDA tensor with the dtype of uo/vo')
    if c.dim() == 3 and c.shape[0] == nz and c.shape[1] * c.shape[2] == ncell and c.shape[2] != ncell:
        c = c.unsqueeze(0)                                  # (z, y, x): time-invariant
    cnt, cnz, cncell, cld = _plane_layout(c, name)
    # the kernel steps levels by ld and time steps by nz * ld, the layout of uo/vo
    if (cnz, cncell) != (nz, ncell) or cnt not in (1, nt) or (cld != ld and cnz > 1) or \
            (cnt > 1 and c.stride(0) != nz * ld):
        raise ValueError(f'{name} must be (1 or nt, nz, cells) with the plane layout of uo/vo')
    return c, int(cnt)


def _class_field_host(c, h, name='cfield'):
    """the same next to host uo/vo (h: _host_inputs): the dtype and byte order of uo, (1 or nt, nz, ny, nx),
    (1 or nt, nz, ny*nx) or (nz, ny, nx) -> C-contiguous (1 or nt, nz, ny, nx)"""
    torch = _torch()
    c = numpy.asarray(c.numpy() if isinstance(c, torch.Tensor) else c)
    if c.dtype != h.u.dtype:
        raise ValueError(f'{name} must have the dtype and byte order of uo ({h.u.dtype}), got {c.dtype}')
    nz, ny, nx = h.u.shape[1:]
    if c.ndim == 3 and c.shape == (nz, ny, nx):
        c = c[None]
    if c.ndim == 3:
        c = c.reshape(c.shape[0], c.shape[1], ny, nx) if c.shape[2] == ny * nx else c
    if c.ndim != 4 or c.shape[1:] != (nz, ny, nx) or c.shape[0] not in (1, h.nt):
        raise ValueError(f'{name} must be (1 or nt, nz, ny, nx) or (nz, ny, nx), got shape {c.shape}')
    return numpy.ascontiguousarray(c)


def _require_cuda(t, dtype, name):
    torch = _torch()
    if not isinstance(t, torch.Tensor) or not t.is_cuda:
        raise TypeError(f'{name} must be a CUDA tensor (there is no CPU fallback)')
    if t.dtype != dtype:
        raise TypeError(f'{name} must have dtype {dtype}, got {t.dtype}')
    if not t.is_contiguous():
        raise ValueError(f'{name} must be contiguous')


# -- K2 as a free function (Field.readField + Field.computeIntegratedFlux for many time steps) ------------
def edgeFluxAssemble(u, v, thickness, arc1, arc2, sverdrup=False, fill=float('nan'), out=None, e3u=None, e3v=None):
    """u, v cuda (nt, nz, ny, nx) or (nt, nz, ncell) (level planes may be padded in memory, see _plane_layout);
    returns eflux cuda (nt, 2*ncell): [eU | eV] signed"""
    torch = _torch()
    for name, t in (('u', u), ('v', v)):
        if not isinstance(t, torch.Tensor) or not t.is_cuda:
            raise TypeError(f'{name} must be a CUDA tensor (there is no CPU fallback)')
    if u.dtype != v.dtype or u.shape != v.shape or u.stride() != v.stride():
        raise ValueError('u and v must have the same dtype, shape and strides')
    nt, nz, ncell, ld = _plane_layout(u, 'u')
    use_e3 = e3u is not None or e3v is not None
    checks = [('arc1', arc1, ncell), ('arc2', arc2, ncell)] + ([] if use_e3 else [('thickness', thickness, nz)])
    for name, t, n in checks:
        _require_cuda(t, torch.float64, name)
        if t.numel() != n:
            raise ValueError(f'{name} must hold {n} values, got {t.numel()}')
    if out is None:
        out = torch.empty((nt, 2 * ncell), dtype=torch.float64, device=u.device)
    if use_e3:      # per-column vertical scale factors replace the 1-D thickness (which is ignored)
        e3_nt = _check_e3(e3u, e3v, u, nt, nz, ncell, ld)
        with torch.cuda.device(u.device):
            _lib.call('nfx_edgeflux_assemble_e3', _t_ptr(u), _t_ptr(v), _t_ptr(e3u), _t_ptr(e3v),
                      _dtype_code(str(u.dtype)), e3_nt, _t_ptr(arc1), _t_ptr(arc2), nt, nz, ncell, ld,
                      int(bool(sverdrup)), float(fill), _t_ptr(out), _stream_ptr())
        return out
    with torch.cuda.device(u.device):
        _lib.call('nfx_edgeflux_assemble_ld', _t_ptr(u), _t_ptr(v), _dtype_code(str(u.dtype)), _t_ptr(thickness),
                  _t_ptr(arc1), _t_ptr(arc2), nt, nz, ncell, ld, int(bool(sverdrup)), float(fill), _t_ptr(out),
                  _stream_ptr())
    return out


def edgeFluxToCellByCell(eflux, ny, nx, out=None):
    """compact (nt, 2*ncell) -> mint's (nt, ncell, 4) integratedVelocity layout (field.py:209-223)"""
    torch = _torch()
    _require_cuda(eflux, torch.float64, 'eflux')
    nt = eflux.shape[0]
    if eflux.shape[1] != 2 * ny * nx:
        raise ValueError('eflux must be (nt, 2*ny*nx)')
    if out is None:
        out = torch.empty((nt, ny * nx, 4), dtype=torch.float64, device=eflux.device)
    with torch.cuda.device(eflux.device):
        _lib.call('nfx_edgeflux_to_cell_by_cell', _t_ptr(eflux), nt, ny, nx, _t_ptr(out), _stream_ptr())
    return out


def h5DecodeChunks(comp, in_off, in_size, filters, chunk_dims, dst, chunk_start, swap_bytes=False):
    """chunked NetCDF-4 / HDF5 data decoded on the device (C ABI nfx_h5_decode_chunks): comp = cuda uint8 tensor with
    the chunks as stored in the file (chunk c at byte in_off[c], a multiple of 16, in_size[c] bytes), filters = bit mask
    of NFX_H5_DEFLATE / SHUFFLE / FLETCHER32, chunk_dims = extents of a chunk, dst = dense cuda tensor the chunks are
    placed into (its shape has the rank of chunk_dims), chunk_start (nchunks, rank) = index in dst of every chunk's first
    element.  Returns the per-chunk status array (all 0); raises NemofluxGpuError when a chunk is not a valid stream."""
    torch = _torch()
    if not (isinstance(comp, torch.Tensor) and comp.is_cuda and comp.dtype == torch.uint8 and comp.is_contiguous()):
        raise TypeError('comp must be a contiguous CUDA uint8 tensor')
    if not (isinstance(dst, torch.Tensor) and dst.is_cuda and dst.is_contiguous() and dst.device == comp.device):
        raise TypeError('dst must be a contiguous CUDA tensor on the device of comp')
    off = numpy.ascontiguousarray(in_off, numpy.int64).reshape(-1)
    size = numpy.ascontiguousarray(in_size, numpy.int64).reshape(-1)
    cdims = numpy.ascontiguousarray(chunk_dims, numpy.int64).reshape(-1)
    rank = cdims.size
    if dst.dim() != rank:
        raise ValueError(f'dst has {dst.dim()} dimensions, the chunks {rank}')
    ddims = numpy.array(dst.shape, numpy.int64)
    start = numpy.ascontiguousarray(chunk_start, numpy.int64).reshape(-1, rank)
    if not (off.size == size.size == start.shape[0]):
        raise ValueError('in_off, in_size and chunk_start must describe the same number of chunks')
    status = numpy.zeros(max(off.size, 1), numpy.int32)
    with torch.cuda.device(comp.device):
        _lib.call('nfx_h5_decode_chunks', _t_ptr(comp), int(comp.numel()), int(off.size), _np_ptr(off), _np_ptr(size),
                  int(filters), int(dst.element_size()), rank, _np_ptr(cdims), _np_ptr(ddims), _np_ptr(start),
                  int(bool(swap_bytes)), _t_ptr(dst), _np_ptr(status), _stream_ptr())
    return status[:off.size]


class H5DeviceReader(object):
    """Blocks of chunked (deflate / shuffle) HDF5 variables read straight onto the GPU: the COMPRESSED chunks are
    copied from the memory-mapped files into a pinned staging buffer, cross PCIe as stored and are inflated, unshuffled
    and placed by nfx_h5_decode_chunks -- the decompression the reference leaves to one host thread inside
    netCDF4 / HDF5 (field.py:22-35, 149; subsetNEMO.py:78 writes zlib=True).

        rd = H5DeviceReader(ds, device)            # ds: nemoflux_b200.h5lite.Dataset, chunked
        block = rd.read(starts, stops)             # cuda tensor of shape stops - starts, native byte order
        rd = H5DeviceReader([ds_u, ds_v], device)  # variables of one shape / chunking / type: ONE decode launch for
        u, v = rd.read(starts, stops)              # both (twice the chunks in flight), block[0], block[1]
    """

    def __init__(self, ds, device, workers=0):
        torch = _torch()
        self.many = isinstance(ds, (list, tuple))
        self.dss = list(ds) if self.many else [ds]
        self.ds = self.dss[0]
        self.device = torch.device(device)
        self.flags = self.ds.device_filter_flags()
        for d in self.dss:
            if d.chunk_dims is None or d.device_filter_flags() is None:
                raise ValueError(f'{d.name}: not a chunked variable with a [shuffle,] [deflate,] [fletcher32] pipeline')
            if d.dtype.kind != 'f' or d.dtype.itemsize not in (4, 8):
                raise ValueError(f'{d.name}: float32 / float64 variables only')
            if (d.shape, d.chunk_dims, d.dtype, [f[0] for f in d._filters]) != \
                    (self.ds.shape, self.ds.chunk_dims, self.ds.dtype, [f[0] for f in self.ds._filters]):
                raise ValueError('variables decoded together must share shape, chunking, type and filters')
        self.tdtype = torch.float32 if self.ds.dtype.itemsize == 4 else torch.float64
        self.swap = not self.ds.dtype.isnative
        import os as _os
        # file -> pinned copies: plain memcpy's that release the GIL; all but a few of the cores this process may use
        self.workers = max(1, int(workers)) if workers else max(4, min(16, len(_os.sched_getaffinity(0)) - 3))
        self._pinned = None
        self._dev = [None, None]
        self._slot = 0
        self._last_ready = None
        self._copy_stream = None
        self.bytes_compressed = 0          # running totals, for the caller's report
        self.bytes_decoded = 0

    def stage(self, starts, stops):
        """host half: the chunks under [starts, stops) copied into the pinned staging buffer; returns the plan the
        device half (decode) takes.  Runs without the GIL for the copies, so a reader thread can prepare block i + 1
        while block i is decoded."""
        torch = _torch()
        plan = []                                               # (variable, file offset, bytes, mask, origin)
        for iv, d in enumerate(self.dss):
            plan += [(iv,) + c for c in d.chunk_plan(starts, stops)]
        offs, pos = [], 0
        for _iv, _addr, nbytes, _mask, _org in plan:
            offs.append(pos)
            pos += (nbytes + 15) & ~15
        total = pos + 4096                                      # the decoder may look a little past the last stream
        if self._pinned is None or self._pinned.numel() < total:
            if self._last_ready is not None:
                self._last_ready.synchronize()
            self._pinned = torch.empty(int(total * 1.25) + 4096, dtype=torch.uint8, pin_memory=True)
        if self._last_ready is not None:
            self._last_ready.synchronize()                      # the previous block has left the pinned buffer
        hbuf = self._pinned.numpy()
        fbufs = [numpy.frombuffer(d._f._buf, numpy.uint8) for d in self.dss]

        def copy(lo, hi):
            for k in range(lo, hi):
                iv, addr, nbytes = plan[k][0], plan[k][1], plan[k][2]
                hbuf[offs[k]:offs[k] + nbytes] = fbufs[iv][addr:addr + nbytes]
        if len(plan) >= 2 * self.workers and self.workers > 1:
            from concurrent.futures import ThreadPoolExecutor
            step = -(-len(plan) // self.workers)
            with ThreadPoolExecutor(self.workers) as pool:
                list(pool.map(lambda lo: copy(lo, min(len(plan), lo + step)), range(0, len(plan), step)))
        else:
            copy(0, len(plan))
        # the staged bytes start their way over PCIe right away, on a side stream and into the device buffer the decoder
        # is NOT reading (two device buffers): the copy of block i + 1 hides behind the decode of block i
        slot = self._slot = self._slot ^ 1
        ready = None
        if plan:
            with torch.cuda.device(self.device):
                if self._dev[slot] is None or self._dev[slot].numel() < total:
                    self._dev[slot] = torch.empty(self._pinned.numel(), dtype=torch.uint8, device=self.device)
                if self._copy_stream is None:
                    self._copy_stream = torch.cuda.Stream(device=self.device)
                with torch.cuda.stream(self._copy_stream):
                    self._dev[slot][:total].copy_(self._pinned[:total], non_blocking=True)
                    ready = torch.cuda.Event()
                    ready.record(self._copy_stream)
        self._last_ready = ready
        return dict(plan=plan, offs=offs, total=total, starts=list(starts), stops=list(stops), slot=slot, ready=ready)

    def decode(self, staged, out=None):
        """device half: H2D of the staged bytes, inflate + unshuffle + placement; returns the cuda tensor (with a
        leading axis over the variables when the reader was built from a list)"""
        torch = _torch()
        plan, offs, total = staged['plan'], staged['offs'], staged['total']
        shape = [b - a for a, b in zip(staged['starts'], staged['stops'])]
        nvar = len(self.dss)
        if out is None:
            out = torch.empty([nvar] + shape, dtype=self.tdtype, device=self.device)
        full = out.view([nvar * shape[0]] + shape[1:]) if shape else out          # variables stacked along axis 0
        for iv, d in enumerate(self.dss):
            blk = out[iv] if nvar > 1 or out.dim() == len(shape) + 1 else out
            if d.fill is not None:
                blk.fill_(float(numpy.frombuffer(d.fill, d.dtype, 1)[0]))
            else:
                blk.zero_()
        if plan:
            dev = self._dev[staged['slot']]
            torch.cuda.current_stream(self.device).wait_event(staged['ready'])
            groups = {}
            for k, (iv, _addr, _nbytes, mask, _org) in enumerate(plan):   # a chunk may have skipped filters (its mask bits)
                flags = 0
                for i, (fid, _cd) in enumerate(self.dss[iv]._filters):
                    if not (mask >> i) & 1:
                        flags |= {1: _lib.NFX_H5_DEFLATE, 2: _lib.NFX_H5_SHUFFLE, 3: _lib.NFX_H5_FLETCHER32}[fid]
                groups.setdefault(flags, []).append(k)
            # one launch for all variables when a chunk is one index thick along axis 0 (NetCDF's usual time chunking):
            # the variables are stacked along that axis and no chunk can hang over into its neighbour; else a launch
            # per variable, clipped by its own block
            together = nvar == 1 or self.ds.chunk_dims[0] == 1
            for flags, ks_all in sorted(groups.items()):
                for iv in ([None] if together else range(nvar)):
                    ks = ks_all if together else [k for k in ks_all if plan[k][0] == iv]
                    if not ks:
                        continue
                    start = [[plan[k][4][d] - staged['starts'][d] + (plan[k][0] * shape[0] if d == 0 and together else 0)
                              for d in range(len(shape))] for k in ks]
                    h5DecodeChunks(dev[:total], [offs[k] for k in ks], [plan[k][2] for k in ks], flags,
                                   self.ds.chunk_dims, full if together else out[iv], start, swap_bytes=self.swap)
            self.bytes_compressed += sum(p[2] for p in plan)
        self.bytes_decoded += out.numel() * out.element_size()
        return out if self.many or out.dim() == len(shape) else out[0]

    def read(self, starts, stops, out=None):
        return self.decode(self.stage(starts, stops), out=out)


def probeReadBandwidth(buf, reps=5, groups=None):
    """read-only HBM ceiling (GB/s) of the device of `buf` (a CUDA tensor of >= 9.3 GB whose contents do not matter)
    with the access pattern of the edge-flux kernels -- the denominator bench.py quotes next to the copy peak.
    groups (int32 CUDA tensor, ascending 256-bit vector indices < 30046 of the probe's 362 x 332 plane): walk only
    those, the pattern of the sparse fused pass; the rate then counts the bytes of the listed groups."""
    torch = _torch()
    if not isinstance(buf, torch.Tensor) or not buf.is_cuda or not buf.is_contiguous():
        raise TypeError('buf must be a contiguous CUDA tensor')
    r = ctypes.c_double()
    with torch.cuda.device(buf.device):
        if groups is None:
            _lib.call('nfx_probe_read_bandwidth', _t_ptr(buf), int(buf.numel() * buf.element_size()), int(reps),
                      ctypes.byref(r), _stream_ptr())
        else:
            _require_cuda(groups, torch.int32, 'groups')
            _lib.call('nfx_probe_read_bandwidth_groups', _t_ptr(buf), int(buf.numel() * buf.element_size()),
                      _t_ptr(groups), int(groups.numel()), int(reps), ctypes.byref(r), _stream_ptr())
    return r.value


def edgeFluxAbsMax(eflux):
    """max |edge flux| over everything in eflux (Field.maxAbsFlux, field.py:230-234)"""
    torch = _torch()
    _require_cuda(eflux, torch.float64, 'eflux')
    r = ctypes.c_double()
    with torch.cuda.device(eflux.device):
        _lib.call('nfx_edgeflux_absmax', _t_ptr(eflux), eflux.shape[0], eflux.shape[1] // 2, ctypes.byref(r),
                  _stream_ptr())
    return r.value
