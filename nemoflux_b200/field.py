"""Field -- mirror of nemoflux/field.py with the compute step on the GPU.

Same constructor, attributes and methods as the reference class (field.py:15-234):
``Field(tFile, uFile, vFile, lonLatZPoints, sverdrup=False)``, ``timeIndex``, ``nt nz ny nx``, ``plis``,
``thickness``, ``arcLengths``, ``edgeFluxesUArray / edgeFluxesVArray`` (absolute values, field.py:230-232),
``integratedVelocity`` ((ncell,4), field.py:209-228), ``maxAbsFlux`` (running maximum, field.py:234),
``update()``, ``getFluxText()``, ``getUV()``, ``readField()``.

What differs: ONE locator is built per grid and shared by all transects (the reference builds one per
transect, field.py:44-49); the vertical integration, edge-flux assembly and the transect integrals run in
libnemoflux_gpu.so (K2, K3); ``fluxSeries()`` is new and evaluates every time step and transect in a few
launches (the loop of fluxplot.py:51-59).  ``vectorPoints`` / ``vectorValues`` (the arrow glyphs, field.py:71-95)
come from nemoflux_gpu.VectorInterp.  ``meshFile`` (optional, new -- SURVEY 8f rank 4): a NEMO mesh_mask-style
file whose per-column vertical scale factors ``e3u_0/e3v_0`` (partial bottom cells) replace the 1-D
``deptht_bounds`` thickness of field.py:51 and whose horizontal scale factors ``e2u/e1v`` (metres), when present,
replace the arc lengths of field.py:170-181.
"""
import re

import numpy

from . import geo
from . import ncio
from . import timeobj
from .horizgrid import HorizGrid
from .latlonreader import LatLonReader  # noqa: F401  (re-exported like the reference module)
from . import nemoflux_gpu

EARTH_RADIUS = 6371000.0          # field.py:12


class _TransectView(object):
    """element of Field.plis: getIntegral(data, placement) of one transect of the shared batch (field.py:102)"""

    def __init__(self, pli, index):
        self._pli, self._index = pli, index          # no reference back to the Field: no reference cycle

    def getIntegral(self, data, placement=nemoflux_gpu.CELL_BY_CELL_DATA):
        return float(self._pli.getIntegral(data, placement)[self._index])

    def getWeights(self):
        return self._pli.getWeights(self._index)


class Field(object):

    def __init__(self, tFile, uFile, vFile, lonLatZPoints, sverdrup=False, verbose=True, meshFile=None):
        import torch
        self.sverdrup = sverdrup
        self.tFile = tFile
        with ncio.open_dataset(tFile) as nc:
            bounds_lat = nc['bounds_lat'][:]
            bounds_lon = nc['bounds_lon'][:]
            self.bounds_depth = nc['deptht_bounds'][:]
        self.lonmin, self.lonmax = bounds_lon.min(), bounds_lon.max()
        self.latmin, self.latmax = bounds_lat.min(), bounds_lat.max()
        if verbose:
            print(f'lon-lat box: {self.lonmin}, {self.latmin} -> {self.lonmax}, {self.latmax}')

        self.timeIndex = 0
        self.ncU = ncio.open_dataset(uFile)
        self.ncV = ncio.open_dataset(vFile)
        self.timeObj = timeobj.TimeObj(self.ncU)
        self.nt, self.nz, self.ny, self.nx = self.getSizes()

        # grid + ONE locator + all transects in one batch
        self.device = torch.device('cuda', torch.cuda.current_device())
        self.gr = HorizGrid(bounds_lon=bounds_lon, bounds_lat=bounds_lat)
        self.pli = nemoflux_gpu.PolylineIntegral()
        self.pli.build(self.gr.getMintGrid(), periodX=360.)
        self.lonLatZPoints = [numpy.array(p, numpy.float64).reshape(-1, 3) for p in lonLatZPoints]
        self.pli.computeWeights(self.lonLatZPoints, counterclock=False)
        self.plis = [_TransectView(self.pli, i) for i in range(len(self.lonLatZPoints))]

        self.thickness = numpy.asarray(self.bounds_depth[:, 1] - self.bounds_depth[:, 0], numpy.float64)   # field.py:51

        numCells = self.ny * self.nx
        self.dx = min((self.lonmax - self.lonmin) / float(self.nx), (self.latmax - self.latmin) / float(self.ny))
        self.arcLengths = numpy.zeros((numCells, 4), numpy.float64)
        self.computeArcLengths()
        self.e3u = self.e3v = None              # (nz, ny, nx) in the storage dtype of uo/vo, from meshFile
        self._d_e3u = self._d_e3v = None
        if meshFile:
            self.readMeshFile(meshFile, verbose)
        self._d_thickness = torch.from_numpy(numpy.ascontiguousarray(self.thickness)).to(self.device)
        self._d_arc1 = torch.from_numpy(numpy.ascontiguousarray(self.arcLengths[:, 1])).to(self.device)
        self._d_arc2 = torch.from_numpy(numpy.ascontiguousarray(self.arcLengths[:, 2])).to(self.device)

        self.edgeFluxesUArray = numpy.zeros((numCells,), numpy.float64)
        self.edgeFluxesVArray = numpy.zeros((numCells,), numpy.float64)
        self.integratedVelocity = numpy.zeros((numCells, 4), numpy.float64)
        self.maxAbsFlux = 0.
        self.fluxes = numpy.zeros(len(self.plis))

        # sample points along the target lines where the viewer draws its arrows (field.py:71-87) and the
        # vector interpolator that feeds them (field.py:90-95)
        vectorPoints = []
        self.uVectors = []
        for lonlatpts in self.lonLatZPoints:
            for i in range(len(lonlatpts) - 1):
                begPoint, endPoint = lonlatpts[i], lonlatpts[i + 1]
                u = endPoint - begPoint
                distance = numpy.sqrt(u.dot(u))
                if distance == 0.:
                    continue
                u = u / distance
                nvpts = max(2, int(distance / self.dx))
                vdx = distance / float(nvpts - 1)
                for j in range(nvpts):
                    vectorPoints.append(begPoint + u * j * vdx)
                    self.uVectors.append(u)
        self.vectorPoints = numpy.array(vectorPoints).reshape(-1, 3)
        self.vinterp = nemoflux_gpu.VectorInterp()
        self.vinterp.setGrid(self.gr.getMintGrid())
        self.vinterp.buildLocator(numCellsPerBucket=128, periodX=360.)
        self.vinterp.findPoints(self.vectorPoints, tol2=1.e-12)
        self.vectorValues = numpy.zeros((self.vectorPoints.shape[0], 3))

        self.update()
        if verbose:
            print(f'max vertically integrated edge |flux|: {self.maxAbsFlux}')
        self.buildEdgeUVGrids(bounds_lon, bounds_lat)

    # ---- reference helpers -------------------------------------------------------------------------------
    def getSizes(self):
        nt, nz, ny, nx = 1, 1, 0, 0
        shapeU = self.ncU['uo'].shape
        if len(shapeU) == 4:
            nt, nz, ny, nx = shapeU
        elif len(shapeU) == 3:
            nz, ny, nx = shapeU
        elif len(shapeU) == 2:
            ny, nx = shapeU
        else:
            raise RuntimeError("ERROR: uo's shape does not match (t, z, y, x), (z, y, x) or (y, x)")
        return nt, nz, ny, nx

    def buildEdgeUVGrids(self, bounds_lon, bounds_lat):
        self.lonlat = numpy.zeros((self.ny, self.nx, 4, 3), numpy.float64)
        self.lonlat[..., 0] = bounds_lon
        self.lonlat[..., 1] = bounds_lat

    def computeArcLengths(self):
        self.arcLengths[:] = geo.cellArcLengths(self.gr.getPoints())

    def readMeshFile(self, meshFile, verbose=False):
        """NEMO mesh_mask conventions: e3u_0/e3v_0 (or e3u/e3v) as (1, z, y, x) or (z, y, x) -- time-invariant
        vertical scale factors at the U and V points; e2u/e1v as (1, y, x) or (y, x) in metres -- the lengths of the
        east and north cell edges, i.e. arcLengths[:, 1] and [:, 2] (field.py:195-196) times the earth radius.
        The scale factors are kept in the storage dtype of uo/vo (the kernels stream all four arrays as one type)."""
        import torch
        want = numpy.dtype(self.ncU['uo'].dtype).newbyteorder('=')

        def pick(nc, names, ndim):
            for name in names:
                if name in nc:
                    a = numpy.asarray(nc[name][:], numpy.float64)       # missing values decoded to NaN (count as 0)
                    while a.ndim > ndim:
                        if a.shape[0] != 1:
                            raise RuntimeError(f'ERROR: {name} in {meshFile} has {a.shape[0]} time steps, expected 1')
                        a = a[0]
                    return name, a
            return None, None
        with ncio.open_dataset(meshFile) as nc:
            nu, e3u = pick(nc, ('e3u_0', 'e3u'), 3)
            nv, e3v = pick(nc, ('e3v_0', 'e3v'), 3)
            n2, e2u = pick(nc, ('e2u',), 2)
            n1, e1v = pick(nc, ('e1v',), 2)
        if e3u is None or e3v is None:
            raise RuntimeError(f'ERROR: {meshFile} holds no e3u_0/e3v_0 (or e3u/e3v) variables')
        shape = (self.nz, self.ny, self.nx)
        if e3u.shape != shape or e3v.shape != shape:
            raise RuntimeError(f'ERROR: {nu}/{nv} shapes {e3u.shape}/{e3v.shape} do not match uo {shape}')
        self.e3u, self.e3v = e3u.astype(want), e3v.astype(want)
        self._d_e3u = torch.from_numpy(self.e3u.reshape(1, self.nz, -1)).to(self.device)
        self._d_e3v = torch.from_numpy(self.e3v.reshape(1, self.nz, -1)).to(self.device)
        if e2u is not None and e1v is not None:
            if e2u.shape != shape[1:] or e1v.shape != shape[1:]:
                raise RuntimeError(f'ERROR: e2u/e1v shapes {e2u.shape}/{e1v.shape} do not match the grid {shape[1:]}')
            self.arcLengths[:, 1] = e2u.reshape(-1) / EARTH_RADIUS
            self.arcLengths[:, 2] = e1v.reshape(-1) / EARTH_RADIUS
        if verbose:
            print(f'mesh file: {nu}, {nv}' + (', e2u, e1v' if e2u is not None and e1v is not None else ''))

    def _slab(self, nc, fieldName, t0, n):
        """(n, nz, ny, nx) block of time steps AS STORED: the missing-value marker (_FillValue, 1e20 in NEMO and
        datagen.py:191) is not decoded on the host -- K2 maps it (and NaN) to 0, which is what xarray's decoding
        followed by fillna(0.0) does in the reference (field.py:149-157)"""
        var = nc[fieldName]
        # packed variables (scale_factor / add_offset) or two different missing-value markers: decoded values (NaN for
        # missing data) instead of the raw fast path -- what xarray hands the reference (field.py:149)
        get = (lambda i: var[i]) if self._decoded(var) else var.raw
        try:
            if len(var.shape) == 4:
                a = get(slice(t0, t0 + n))
            elif len(var.shape) == 3:
                a = get(Ellipsis)[None]
            else:
                a = get(Ellipsis)[None, None]
        except Exception:
            raise RuntimeError(f'ERROR: could not read {fieldName} field')
        return numpy.ascontiguousarray(a)

    @staticmethod
    def _decoded(var):
        return var.packed or len(var.fill_values()) > 1

    def _uv_slabs(self, t0, n):
        """u, v blocks and the one missing-value marker K2 is given; if vo uses another marker than uo it is
        rewritten to NaN on the host (NEMO uses 1e20 for both)"""
        u = self._slab(self.ncU, 'uo', t0, n)
        v = self._slab(self.ncV, 'vo', t0, n)
        fu, fv = self._fill(self.ncU, 'uo'), self._fill(self.ncV, 'vo')
        if fv == fv and fv != fu:
            v = numpy.where(v == v.dtype.type(fv), numpy.nan, v)
        return u, v, fu

    def _fill(self, nc, fieldName):
        if self._decoded(nc[fieldName]):
            return float('nan')                    # decoded on the host: missing data are NaN already
        fv = nc[fieldName].fill_value()
        if nc[fieldName].dtype.itemsize == 4 and fv == fv:
            fv = float(numpy.float32(fv))          # compare in the storage precision
        return fv

    def readField(self, nc, fieldName):
        """vertically integrated field of the current time index, (ny, nx) host array (field.py:145-163);
        computed by K2 with unit metric factors"""
        import torch
        a = torch.from_numpy(self._slab(nc, fieldName, self.timeIndex, 1)).to(self.device)
        ones = torch.ones(self.ny * self.nx, dtype=torch.float64, device=self.device)
        if self._d_e3u is not None:
            e3 = self._d_e3u if fieldName == 'uo' else self._d_e3v
            ef = nemoflux_gpu.edgeFluxAssemble(a.reshape(1, self.nz, -1), a.reshape(1, self.nz, -1), None, ones, ones,
                                               fill=self._fill(nc, fieldName), e3u=e3, e3v=e3)
        else:
            ef = nemoflux_gpu.edgeFluxAssemble(a, a, self._d_thickness, ones, ones, fill=self._fill(nc, fieldName))
        return ef[0, :self.ny * self.nx].reshape(self.ny, self.nx).cpu().numpy()

    def getUV(self):
        return self.readField(self.ncU, 'uo'), self.readField(self.ncV, 'vo')

    # ---- the compute step ----------------------------------------------------------------------------------
    def update(self):
        """edge fluxes and transect fluxes of self.timeIndex (field.py:112-120): K2 + K3 on the device"""
        import torch
        uh, vh, fill = self._uv_slabs(self.timeIndex, 1)
        u, v = torch.from_numpy(uh).to(self.device), torch.from_numpy(vh).to(self.device)
        if self._d_e3u is not None:
            eflux = nemoflux_gpu.edgeFluxAssemble(u.reshape(1, self.nz, -1), v.reshape(1, self.nz, -1), None, self._d_arc1,
                                                  self._d_arc2, sverdrup=self.sverdrup, fill=fill, e3u=self._d_e3u,
                                                  e3v=self._d_e3v)
        else:
            eflux = nemoflux_gpu.edgeFluxAssemble(u, v, self._d_thickness, self._d_arc1, self._d_arc2,
                                                  sverdrup=self.sverdrup, fill=fill)
        self.fluxes = self.pli.integrate(eflux).cpu().numpy()[0]
        ncell = self.ny * self.nx
        self.integratedVelocity[:] = nemoflux_gpu.edgeFluxToCellByCell(eflux, self.ny, self.nx)[0].cpu().numpy()
        ef = eflux[0].abs().cpu().numpy()                     # from now on, edge fluxes are abs values (field.py:230)
        self.edgeFluxesUArray[:] = ef[:ncell]
        self.edgeFluxesVArray[:] = ef[ncell:]
        self.maxAbsFlux = max(self.maxAbsFlux, nemoflux_gpu.edgeFluxAbsMax(eflux))
        self.vectorValues[:] = self.vinterp.getFaceVectors(self.integratedVelocity, placement=0)   # field.py:119-120

    def computeIntegratedFlux(self, uVerticallyIntegrated, vVerticallyIntegrated):
        """field.py:183-234 for callers that hold their own vertically integrated (ny, nx) fields"""
        import torch
        u = torch.from_numpy(numpy.ascontiguousarray(uVerticallyIntegrated, numpy.float64).reshape(1, 1, -1)).to(self.device)
        v = torch.from_numpy(numpy.ascontiguousarray(vVerticallyIntegrated, numpy.float64).reshape(1, 1, -1)).to(self.device)
        one = torch.ones(1, dtype=torch.float64, device=self.device)
        eflux = nemoflux_gpu.edgeFluxAssemble(u, v, one, self._d_arc1, self._d_arc2, sverdrup=self.sverdrup)
        ncell = self.ny * self.nx
        self.integratedVelocity[:] = nemoflux_gpu.edgeFluxToCellByCell(eflux, self.ny, self.nx)[0].cpu().numpy()
        ef = eflux[0].abs().cpu().numpy()
        self.edgeFluxesUArray[:] = ef[:ncell]
        self.edgeFluxesVArray[:] = ef[ncell:]
        self.fluxes = self.pli.integrate(eflux).cpu().numpy()[0]
        self.maxAbsFlux = max(self.maxAbsFlux, float(ef.max()))

    def getFluxText(self):
        """title text of the viewer (field.py:98-109): one %4.3g value per transect and the units"""
        txt = ""
        for totalFlux in self.fluxes:
            txt += f"{totalFlux:4.3g}, "
        txt += "(Sv) " if self.sverdrup else "(A m^2/s) "
        return re.sub(r',\s*\(', ' (', txt)

    def _device_readers(self):
        """(reader of uo, reader of vo) when both are chunked NetCDF-4 variables whose filter pipeline the device undoes
        (nfx_h5_decode_chunks): 4-D float32/float64, one missing-value marker, not packed; else None"""
        from . import ncio
        readers = []
        for nc, name in ((self.ncU, 'uo'), (self.ncV, 'vo')):
            var = nc[name]
            data = getattr(var, '_data', None)
            if not isinstance(data, ncio._H5Data) or len(var.shape) != 4 or self._decoded(var):
                return None
            ds = data._ds
            if ds.chunk_dims is None or ds.device_filter_flags() is None or ds.dtype.kind != 'f' or \
                    ds.dtype.itemsize not in (4, 8):
                return None
            readers.append(ds)
        fu, fv = self._fill(self.ncU, 'uo'), self._fill(self.ncV, 'vo')
        if fv == fv and fv != fu:
            return None                                 # two different markers: the host path rewrites one of them
        try:
            return [nemoflux_gpu.H5DeviceReader(readers, self.device)]       # uo and vo in ONE decode launch
        except ValueError:
            if readers[0].dtype.itemsize != readers[1].dtype.itemsize:
                return None
            return [nemoflux_gpu.H5DeviceReader(d, self.device) for d in readers]

    def _flux_series_device_decode(self, readers, chunk_steps, prefetch, fn, steps, aux=None):
        """fn over chunked + deflated uo / vo: the COMPRESSED chunks cross PCIe and are inflated, unshuffled and
        placed on the device (csrc/nfx_inflate.cu), then fn (the series' K2 + K3, or the section) runs on the decoded
        slab.  A reader thread copies the compressed chunks of block i + 1 from the memory-mapped files into pinned
        staging while block i is decoded."""
        import threading
        import torch
        t_lo, t_hi = steps
        nt = t_hi - t_lo
        esize = readers[0].ds.dtype.itemsize
        step_bytes = esize * self.nz * self.ny * self.nx
        # The decoder works on one chunk per warp and 20 warps fit an SM: a block of as many chunks as the device holds
        # at once (2 960 on a B200) is decoded in one wave; smaller blocks take as long, larger ones leave a tail wave.
        # Capped at 3 GB of decoded data per block.
        ds = readers[0].ds
        chunks_per_step = len(readers[0].dss) * len(readers) * max(1, int(numpy.prod(
            [-(-ext // c) for ext, c in zip(ds.shape[1:], ds.chunk_dims[1:])]))) // max(1, ds.chunk_dims[0])
        wave = 20 * torch.cuda.get_device_properties(self.device).multi_processor_count
        n = chunk_steps if chunk_steps > 0 else max(1, min(nt, wave // max(chunks_per_step, 1),
                                                           (3 << 30) // max(2 * step_bytes, 1)))
        if chunk_steps <= 0:                            # blocks of equal size: a short last block costs a full chunk latency
            nblk = -(-nt // n)
            n = -(-nt // nblk)
        blocks = [(t0, min(n, t_hi - t0)) for t0 in range(t_lo, t_hi, n)]
        fill = self._fill(self.ncU, 'uo')
        staged = {}

        def stage(i):
            t0, m = blocks[i]
            staged[i] = tuple(r.stage([t0, 0, 0, 0], [t0 + m, self.nz, self.ny, self.nx]) for r in readers)
            if aux is not None:
                staged[('aux', i)] = aux(t0, m, numpy.dtype(str(readers[0].tdtype).replace('torch.', '')))

        # stage() ends by sending its bytes to one of the reader's two device buffers; the reader thread prepares block
        # i + 1 (file -> pinned -> device) while block i is inflated and integrated
        stage(0)
        for i, (t0, m) in enumerate(blocks):
            st = staged.pop(i)
            th = None
            if i + 1 < len(blocks) and prefetch:
                th = threading.Thread(target=stage, args=(i + 1,))
                th.start()
            if len(readers) == 1:
                ud, vd = readers[0].decode(st[0])
            else:
                ud, vd = readers[0].decode(st[0]), readers[1].decode(st[1])
            if i + 1 < len(blocks) and not prefetch:
                stage(i + 1)
            more = {} if aux is None else dict(aux=staged.pop(('aux', i)))
            fn(t0, m, ud, vd, self._d_thickness, self._d_arc1, self._d_arc2, sverdrup=self.sverdrup, fill=fill,
               e3u=self._d_e3u, e3v=self._d_e3v, **more)
            if th is not None:
                th.join()
        self.last_ingest = dict(path='device decode', bytes_compressed=sum(r.bytes_compressed for r in readers),
                                bytes_decoded=sum(r.bytes_decoded for r in readers))

    def _series_shape(self, layers):
        return (self.nt, len(self.plis)) if layers is None else (self.nt, len(layers) - 1, len(self.plis))

    def levelsForDepths(self, depths):
        """depths in metres, ascending -> level boundaries for fluxSeries(layers=), see levelsForDepths below"""
        return levelsForDepths(self.bounds_depth, depths)

    def layerInterfaces(self):
        return layerInterfaces(self.bounds_depth)

    def fluxSeries(self, chunk_steps=0, prefetch=True, device_decode=None, layers=None):
        """(nt, M) flux of every transect at every time step -- the loop of fluxplot.py:51-59 in a few launches.
        layers (level boundaries, see levelsForDepths): (nt, nlayers, M), the flux of every layer of model levels.

        The time axis is streamed from the files in chunks: a reader thread fills one of two PINNED host buffers
        (file read, numpy releases the GIL) while the previous chunk goes through the host-buffer entry point of
        the C ABI (double-buffered H2D, K2, K3) -- file I/O, PCIe and the kernels overlap (SURVEY 8f rank 1).
        NetCDF classic files are big-endian: the bytes are copied as stored and swapped on the device
        (NFX_BIG_ENDIAN), so the host does no conversion pass.
        Chunked + deflated NetCDF-4 variables (device_decode=None: whenever possible, True: required, False: host zlib)
        travel COMPRESSED and are inflated / unshuffled on the device, see _flux_series_device_decode."""
        out = numpy.zeros(self._series_shape(layers))

        def fn(t0, m, *args, **kw):
            out[t0:t0 + m] = _host(self.pli.fluxSeries(*args, layers=layers, **kw))
        self._over_chunks(fn, chunk_steps, prefetch, device_decode)
        return out

    def fluxSection(self, layers=None, chunk_steps=0, prefetch=True, device_decode=None, windows=None):
        """(nt, nlayers, nsub) transport section: the flux across every cell crossing of every transect per layer of
        model levels (layers: level boundaries, see levelsForDepths; None = one layer per level), see
        PolylineIntegral.fluxSection and getSectionGeometry.  Reads the files as fluxSeries does.

        windows: step boundaries [b0 < ... < bK] (see timeobj.timeWindows) -> (K, nlayers, nsub), the time mean of
        every window, PolylineIntegral.fluxSection(windows=) of the whole record bit for bit.  Only the steps
        [b0, bK) are read; one (K, nlayers, nsub) array of sums is kept, each block of steps read from the files
        continues the windows it shares with the block before, and the sums are divided at the end."""
        lev = list(range(self.nz + 1)) if layers is None else layers
        nsub = self.pli.getNumberOfSubsegments()
        if windows is None:
            out = numpy.zeros((self.nt, len(lev) - 1, nsub))

            def fn(t0, m, *args, **kw):
                out[t0:t0 + m] = _host(self.pli.fluxSection(*args, layers=lev, **kw))
            self._over_chunks(fn, chunk_steps, prefetch, device_decode)
            return out
        b = numpy.asarray(windows).reshape(-1)
        if b.size < 2 or b.dtype.kind not in 'iu' or b[0] < 0 or b[-1] > self.nt or numpy.any(numpy.diff(b) <= 0):
            raise ValueError(f'windows must be strictly ascending step indices in [0, nt = {self.nt}], got {windows!r}')
        b = b.astype(numpy.int64)
        sums = numpy.zeros((b.size - 1, len(lev) - 1, nsub))

        def fn(t0, m, u, v, *args, **kw):
            # the windows [wa, wb) this block touches, their bounds inside the block; window wa continues its sums when
            # it began in an earlier block
            wa = max(int(numpy.searchsorted(b, t0, 'right')) - 1, 0)
            wb = min(int(numpy.searchsorted(b, t0 + m, 'left')), b.size - 1)
            if wa >= wb:
                return
            local = numpy.clip(b[wa:wb + 1] - t0, 0, m)
            if isinstance(u, numpy.ndarray):
                self.pli.sectionWindowSums(u, v, *args, windows=local, layers=lev, sums=sums[wa:wb],
                                           continue_first=b[wa] < t0, **kw)
            else:
                import torch
                part = torch.from_numpy(sums[wa:wb]).to(u.device)
                self.pli.sectionWindowSums(u, v, *args, windows=local, layers=lev, sums=part,
                                           continue_first=b[wa] < t0, **kw)
                sums[wa:wb] = part.cpu().numpy()
        self._over_chunks(fn, chunk_steps, prefetch, device_decode, steps=(int(b[0]), int(b[-1])))
        sums /= numpy.diff(b).astype(numpy.float64)[:, None, None]
        return sums

    def fluxClasses(self, var, bounds, file=None, chunk_steps=0, prefetch=True, device_decode=None):
        """(nt, K, M) class transport: every transect's flux binned by the T-grid variable `var` (thetao, so, sigma0...)
        into the classes [b_j, b_{j+1}) of bounds, see PolylineIntegral.fluxClasses.  var is read from `file` (default:
        the T file), (nt, nz, ny, nx) or time-invariant (nz, ny, nx), with its _FillValue, block by block next to uo/vo
        on the pipeline of fluxSeries, and converted to the storage type of uo/vo."""
        b = numpy.asarray(bounds, numpy.float64).reshape(-1)
        out = numpy.zeros((self.nt, b.size - 1, len(self.plis)))

        def run(t0, m, c, cfill, *args, **kw):
            out[t0:t0 + m] = _host(self.pli.fluxClasses(*args, cfield=c, bounds=b, cfill=cfill, **kw))
        self._over_chunks_with(var, file, run, chunk_steps, prefetch, device_decode)
        return out

    def fluxTracer(self, var, file=None, ref=0.0, layers=None, section=False, chunk_steps=0, prefetch=True,
                   device_decode=None):
        """tracer transport: every transect's flux weighted by the T-grid variable `var` (thetao, so...) at the C-grid
        faces, minus ref, see PolylineIntegral.fluxTracer: (nt, M), or (nt, nlayers, M) with layers (level
        boundaries, see levelsForDepths); section=True: (nt, nlayers, nsub) per crossing, one layer per level by
        default.  var is read as fluxClasses reads its class field: from `file` (default: the T file), with its
        _FillValue, block by block next to uo/vo, converted to the storage type of uo/vo."""
        if section:
            nlev = self.nz if layers is None else len(layers) - 1
            out = numpy.zeros((self.nt, nlev, self.pli.getNumberOfSubsegments()))
        else:
            out = numpy.zeros(self._series_shape(layers))

        def run(t0, m, c, tfill, *args, **kw):
            out[t0:t0 + m] = _host(self.pli.fluxTracer(*args, tracer=c, ref=ref, tfill=tfill, layers=layers,
                                                       section=section, **kw))
        self._over_chunks_with(var, file, run, chunk_steps, prefetch, device_decode)
        return out

    def _over_chunks_with(self, var, file, run, chunk_steps, prefetch, device_decode):
        """run(t0, m, c, cfill, u, v, thickness, arc1, arc2, sverdrup=, fill=, e3u=, e3v=) over the blocks of
        _over_chunks, with c the T-grid variable `var` of `file` (default: the T file) next to uo/vo in their storage
        type and cfill its _FillValue: (nt, nz, ny, nx) read block by block on the reader thread, or (nz, ny, nx) (or
        one step) converted, and uploaded, once"""
        import torch
        nc = ncio.open_dataset(file or self.tFile)
        try:
            cv = nc[var]
            shape = tuple(cv.shape)
            if shape[-3:] != (self.nz, self.ny, self.nx) or len(shape) not in (3, 4) or \
                    (len(shape) == 4 and shape[0] not in (1, self.nt)):
                raise RuntimeError(f'ERROR: {var} has shape {shape}, expected (nt, nz, ny, nx) or (nz, ny, nx) = '
                                   f'({self.nt}, {self.nz}, {self.ny}, {self.nx})')
            steady = len(shape) == 3 or shape[0] == 1
            cfill = self._fill(nc, var)
            fixed = self._slab(nc, var, 0, 1) if steady else None
            once = {}                       # the time-invariant field, converted (and uploaded) once per form

            def read(t0, m, dtype):
                """on the reader thread, next to uo/vo: the block in the storage type and byte order of uo/vo"""
                return numpy.ascontiguousarray(self._slab(nc, var, t0, m).astype(dtype))

            def fn(t0, m, u, v, *args, aux=None, **kw):
                on_host = isinstance(u, numpy.ndarray)
                if steady:
                    key = u.dtype if on_host else (u.device, u.dtype)
                    if key not in once:
                        c = numpy.ascontiguousarray(fixed.astype(u.dtype if on_host else fixed.dtype.newbyteorder('=')))
                        once[key] = c if on_host else torch.from_numpy(c).to(u.device, u.dtype).reshape(1, self.nz, -1)
                    c = once[key]
                else:
                    c = aux if on_host else torch.from_numpy(aux).to(u.device).reshape(m, self.nz, -1)
                run(t0, m, c, cfill, u, v, *args, **kw)
            self._over_chunks(fn, chunk_steps, prefetch, device_decode, aux=None if steady else read)
        finally:
            nc.close()

    def _over_chunks(self, fn, chunk_steps, prefetch, device_decode, steps=None, aux=None):
        """fn(t0, m, u, v, thickness, arc1, arc2, sverdrup=, fill=, e3u=, e3v=) over blocks [t0, t0 + m) of the time
        steps [steps[0], steps[1]) (default: all) read from the files: the pipeline of fluxSeries.  aux(t0, m, dtype)
        (optional) reads one more array per block on the reader thread, dtype the numpy type of the block's uo/vo;
        fn gets it as aux="""
        import threading
        import torch
        steps = (0, self.nt) if steps is None else steps
        if device_decode is not False:
            readers = self._device_readers()
            if readers is not None:
                return self._flux_series_device_decode(readers, chunk_steps, prefetch, fn, steps, aux)
            if device_decode is True:
                raise RuntimeError('ERROR: uo / vo are not chunked HDF5 variables with a [shuffle,] [deflate] pipeline')
        t_lo, t_hi = steps
        dtype = numpy.dtype(self.ncU['uo'].dtype).newbyteorder('=')
        step_bytes = dtype.itemsize * self.nz * self.ny * self.nx
        # ~300 MB per variable and chunk (sweep in profiles/r1_file_e2e_C3.json: 4 f64 / 8 f32 ORCA1 steps): small enough that reading chunk i+1 overlaps the upload of chunk i even
        # for a short series, large enough for full-rate PCIe copies
        n = chunk_steps if chunk_steps > 0 else max(1, min(t_hi - t_lo, (300 << 20) // max(step_bytes, 1)))
        arc1, arc2 = self.arcLengths[:, 1].copy(), self.arcLengths[:, 2].copy()
        tdtype = {4: torch.float32, 8: torch.float64}[dtype.itemsize]
        shape = (n, self.nz, self.ny, self.nx)
        nbuf = 2 if prefetch and t_hi - t_lo > n else 1
        cache = getattr(self, '_pinned', None)      # page-locked allocations are slow (~0.1 s/GB): keep them
        if cache is None or cache[0] != (shape, tdtype) or len(cache[1]) < nbuf:
            cache = ((shape, tdtype), [(torch.empty(shape, dtype=tdtype, pin_memory=True),
                                        torch.empty(shape, dtype=tdtype, pin_memory=True)) for _ in range(nbuf)])
            self._pinned = cache
        bufs = cache[1][:nbuf]
        chunks = [(t0, min(n, t_hi - t0)) for t0 in range(t_lo, t_hi, n)]
        state = {}
        raw_u, raw_v = numpy.dtype(self.ncU['uo'].dtype), numpy.dtype(self.ncV['vo'].dtype)
        as_stored = raw_u == raw_v and not raw_u.isnative       # both files big-endian: no conversion on the host
        views = [tuple(b.numpy().view(raw_u) if as_stored else b.numpy() for b in pair) for pair in bufs]

        fill_u, fill_v = self._fill(self.ncU, 'uo'), self._fill(self.ncV, 'vo')
        four_d = len(self.ncU['uo'].shape) == 4 and len(self.ncV['vo'].shape) == 4 and \
            not self._decoded(self.ncU['uo']) and not self._decoded(self.ncV['vo'])
        from concurrent.futures import ThreadPoolExecutor
        import os as _os
        workers = max(1, min(8, (_os.cpu_count() or 2) // 2))
        if not (self.ncU['uo'].thread_safe and self.ncV['vo'].thread_safe):
            workers = 1     # netCDF4 backend: libnetcdf / HDF5 are not thread-safe, reads are serialised by ncio's lock
        pool = ThreadPoolExecutor(max_workers=workers)

        def read(i, slot):
            """file -> pinned buffer, one task per (variable, time step): byte-order conversion in parallel"""
            t0, m = chunks[i]
            nu, nv = views[slot]
            if aux is not None:
                state[('aux', i)] = aux(t0, m, nu.dtype)
            if four_d and (fill_v != fill_v or fill_v == fill_u):
                # one task per (variable, time step, slab of levels): enough tasks to keep every worker copying
                nsplit = max(1, min(self.nz, -(-2 * workers // (2 * m))))
                zs = [(k * self.nz // nsplit, (k + 1) * self.nz // nsplit) for k in range(nsplit)]
                jobs = [pool.submit(var.read_into, dst[j, z0:z1], (t0 + j, slice(z0, z1)))
                        for var, dst in ((self.ncU['uo'], nu), (self.ncV['vo'], nv)) for j in range(m) for z0, z1 in zs]
                for job in jobs:
                    job.result()
                state[i] = fill_u
            else:
                u, v, fill = self._uv_slabs(t0, m)
                nu[:m] = u                          # numpy converts to the view's byte order
                nv[:m] = v
                state[i] = fill

        read(0, 0)
        for i, (t0, m) in enumerate(chunks):
            slot = i % len(bufs)
            th = None
            if i + 1 < len(chunks) and len(bufs) == 2:
                th = threading.Thread(target=read, args=(i + 1, 1 - slot))
                th.start()
            nu, nv = views[slot]                    # numpy views of the pinned buffers (kept alive by `bufs`)
            more = {} if aux is None else dict(aux=state.pop(('aux', i)))
            fn(t0, m, nu[:m], nv[:m], self.thickness, arc1, arc2, sverdrup=self.sverdrup, fill=state.pop(i),
               e3u=self._d_e3u, e3v=self._d_e3v, **more)
            if th is not None:
                th.join()
            elif i + 1 < len(chunks):
                read(i + 1, slot)
        pool.shutdown()

    def close(self):
        self.ncU.close()
        self.ncV.close()


def _host(x):
    """a result of PolylineIntegral as numpy (CUDA tensors of the device-decode path are copied back)"""
    return x if isinstance(x, numpy.ndarray) else x.cpu().numpy()


def layerInterfaces(bounds_depth):
    """(nz + 1) depths in metres of the level interfaces of deptht_bounds (nz, 2): the top of every level, then the
    bottom of the last"""
    b = numpy.asarray(bounds_depth, numpy.float64)
    return numpy.concatenate([b[:, 0], b[-1:, 1]])


def levelsForDepths(bounds_depth, depths):
    """depths in metres, ascending -> level boundaries: each depth snapped to the nearest interface of
    layerInterfaces(bounds_depth) (ties go to the shallower one).  Raises ValueError when two depths snap to the same
    interface (the layer between them would be empty) or the snapped depths are not ascending."""
    iface = layerInterfaces(bounds_depth)
    d = numpy.asarray(depths, numpy.float64).reshape(-1)
    if d.size < 2 or not numpy.all(numpy.isfinite(d)):
        raise ValueError('depths: at least two finite depths are needed')
    levels = [int(numpy.argmin(numpy.abs(iface - x))) for x in d]
    for i in range(len(levels) - 1):
        if levels[i + 1] == levels[i]:
            raise ValueError(f'depths {d[i]:g} and {d[i + 1]:g} m snap to the same level interface '
                             f'({iface[levels[i]]:g} m): the layer between them would be empty')
        if levels[i + 1] < levels[i]:
            raise ValueError('depths must be ascending')
    return levels


def parseLonLatPoints(text):
    """'(lon0,lat0),(lon1,lat1),...'  ->  [polyline]        (the README.md:32 form, field.py:250)
       '[(..),(..)],[(..),(..)]'      ->  [polyline, ...]   (the fluxviz.py:378 form)
    each polyline an (n,3) array with z = 0"""
    import ast
    val = ast.literal_eval(text.strip())
    if len(val) == 0:
        raise RuntimeError('ERROR: empty list of target points')

    def is_point(p):
        return isinstance(p, (tuple, list)) and len(p) in (2, 3) and all(isinstance(c, (int, float)) for c in p)
    lines = [val] if is_point(val[0]) else list(val)
    out = []
    for ln in lines:
        out.append(numpy.array([(p[0], p[1], 0.0) for p in ln], numpy.float64))
    return out


def main(argv=None):
    import argparse
    ap = argparse.ArgumentParser(description='Compute fluxes')
    ap.add_argument('-t', '--tFile', required=True, help='netcdf file holding the T-grid')
    ap.add_argument('-u', '--uFile', required=True, help='netcdf file holding u data')
    ap.add_argument('-v', '--vFile', required=True, help='netcdf file holding v data')
    ap.add_argument('-l', '--lonLatPoints', default='', help='target points "(lon0, lat0), (lon1, lat1),..."')
    ap.add_argument('-i', '--iFile', default='', help='alternatively read target points from text file')
    ap.add_argument('-s', '--sverdrup', action='store_true')
    ap.add_argument('--meshFile', default='', help='optional mesh_mask file: e3u_0/e3v_0 (and e2u/e1v) scale factors')
    a = ap.parse_args(argv)
    if a.lonLatPoints:
        pts = parseLonLatPoints(a.lonLatPoints)
    elif a.iFile:
        ll = LatLonReader(a.iFile).getLonLats()
        pts = [numpy.array([(p[0], p[1], 0.) for p in ll])]
    else:
        raise RuntimeError('ERROR must provide either iFile or lonLatPoints!')
    print(f'target points:\n {pts}')
    f = Field(a.tFile, a.uFile, a.vFile, pts, a.sverdrup, meshFile=a.meshFile or None)
    print(f'flux = {f.getFluxText()}')
    return f


if __name__ == '__main__':
    main()
