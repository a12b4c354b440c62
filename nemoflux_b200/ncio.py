"""Minimal NetCDF access for the nemoflux file conventions (T.nc / U.nc / V.nc).

The reference reads with xarray (field.py:22-35, horizgrid.py:12-15) and writes with netCDF4
(datagen.py:168-208).  Neither is installed in this image, so this module uses netCDF4 when it is
importable and falls back to ``scipy.io.netcdf_file`` for classic / 64-bit-offset NetCDF-3 files and to the
package's own minimal HDF5 reader (``h5lite``) for NetCDF-4 files in the classic data model -- the format of the
reference's data/sa/T.nc and of real NEMO output.  Missing values (``_FillValue`` / ``missing_value``)
are decoded to NaN like xarray's default ``mask_and_scale`` does, so ``fillna(0)`` semantics
(field.py:157) carry over.
"""
import contextlib
import threading

import numpy

# libnetcdf / HDF5 are not thread-safe and netCDF4-python releases the GIL around nc_get_vara: every read through that
# backend takes this process-wide lock (the memory-mapped scipy and h5lite backends read in parallel without it)
_NETCDF4_LOCK = threading.RLock()


class Variable(object):
    def __init__(self, name, data, dims, attrs, lock=None):
        self.name, self._data, self.dimensions, self.attrs = name, data, tuple(dims), dict(attrs)
        self.shape = tuple(data.shape)
        self.dtype = data.dtype
        self._lock = lock

    @property
    def thread_safe(self):
        """False when reads are serialised by the backend's lock (netCDF4): parallel readers gain nothing"""
        return self._lock is None

    def _guard(self):
        return self._lock if self._lock is not None else contextlib.nullcontext()

    @property
    def packed(self):
        """CF packing (scale_factor / add_offset): the stored values are not the physical ones"""
        return 'scale_factor' in self.attrs or 'add_offset' in self.attrs

    def _require_unpacked(self, what):
        if self.packed:
            raise NotImplementedError(f'{self.name}: {what} hands out the values as stored, but the variable is packed '
                                      f'(scale_factor / add_offset); index the variable for decoded values')

    def __getattr__(self, key):
        try:
            return self.__dict__['attrs'][key]
        except KeyError:
            raise AttributeError(key)

    def __len__(self):
        return self.shape[0] if self.shape else 0

    @staticmethod
    def _native(a):
        """NetCDF-3 data are big-endian on disk: hand out native byte order (torch.from_numpy needs it)"""
        if a.dtype.byteorder not in ('=', '|') and not a.dtype.isnative:
            a = a.astype(a.dtype.newbyteorder('='))
        return a

    def raw(self, idx=Ellipsis):
        """values as stored (native byte order), missing values NOT decoded: pair with fill_value()"""
        self._require_unpacked('raw()')
        with self._guard():
            return self._native(numpy.array(self._data[idx]))

    def read_into(self, dst, idx=Ellipsis):
        """copy the stored values [idx] into dst (same shape), converting the byte order on the way; missing values
        are NOT decoded.  numpy releases the GIL in the copy loop, so several slices can be read in parallel
        (memory-mapped backends; the netCDF4 backend serialises on its lock)."""
        self._require_unpacked('read_into()')
        with self._guard():
            numpy.copyto(dst, self._data[idx], casting='same_kind')

    def fill_values(self):
        """every distinct missing-data marker of the variable (_FillValue and missing_value may both be present)"""
        out = []
        for key in ('_FillValue', 'missing_value'):
            if key in self.attrs:
                for fv in numpy.asarray(self.attrs[key]).reshape(-1):
                    if float(fv) not in out and fv == fv:
                        out.append(float(fv))
        return out

    def fill_value(self):
        """the value that marks missing data (_FillValue / missing_value), NaN when there is none; raises when the two
        attributes name DIFFERENT markers (the raw fast path handles one: read decoded values instead)"""
        fvs = self.fill_values()
        if len(fvs) > 1:
            raise ValueError(f'{self.name}: _FillValue and missing_value differ ({fvs}); index the variable for decoded values')
        return fvs[0] if fvs else float('nan')

    def __getitem__(self, idx):
        """decoded values like xarray's mask_and_scale: missing data (both markers) -> NaN, then scale_factor /
        add_offset (floating point result)"""
        with self._guard():
            a = self._native(numpy.array(self._data[idx]))
        fvs = self.fill_values()
        if self.packed:
            mask = numpy.zeros(a.shape, bool)
            for fv in fvs:
                mask |= a == a.dtype.type(fv)
            scale = numpy.asarray(self.attrs.get('scale_factor', 1.0)).reshape(-1)[0]
            offset = numpy.asarray(self.attrs.get('add_offset', 0.0)).reshape(-1)[0]
            out_t = numpy.result_type(numpy.float32 if a.dtype.itemsize <= 2 else numpy.float64, numpy.asarray(scale).dtype)
            a = a.astype(out_t) * out_t.type(scale) + out_t.type(offset)
            a[mask] = numpy.nan
            return a
        if a.dtype.kind == 'f':
            for fv in fvs:
                a[a == a.dtype.type(fv)] = numpy.nan
        return a


class _H5Data(object):
    """array-like over one h5lite dataset (shape, dtype, indexing): a numpy.memmap of the file for contiguous
    storage -- a time slice of uo/vo touches only its own bytes --, the decoded array (cached) otherwise"""

    def __init__(self, path, h5file, ds):
        self._ds, self._a = ds, None
        self.shape, self.dtype = ds.shape, ds.dtype
        lay = ds._layout
        if lay[0] == 'contiguous' and lay[1] != 0xFFFFFFFFFFFFFFFF and all(n > 0 for n in ds.shape) and ds.shape:
            self._a = numpy.memmap(path, dtype=ds.dtype, mode='r', offset=h5file._base + lay[1], shape=ds.shape)

    def _array(self):
        if self._a is None:
            self._a = self._ds.read()
        return self._a

    def __getitem__(self, idx):
        if self._a is None and self._ds._layout[0] == 'chunked':
            block = self._block(idx)
            if block is not None:
                return block
        return self._array()[idx]

    def _block(self, idx):
        """ints and unit-stride slices on a chunked variable: decode only the chunks under the block"""
        if idx is Ellipsis:
            return None                                         # the whole variable: decode once and keep it
        idx = idx if isinstance(idx, tuple) else (idx,)
        if any(i is Ellipsis for i in idx) or len(idx) > len(self.shape):
            return None
        starts, stops, squeeze = [], [], []
        for d, n in enumerate(self.shape):
            i = idx[d] if d < len(idx) else slice(None)
            if isinstance(i, (int, numpy.integer)):
                i = int(i) + (n if i < 0 else 0)
                if not 0 <= i < n:
                    raise IndexError(f'index {idx[d]} is out of bounds for axis {d} with size {n}')
                starts.append(i)
                stops.append(i + 1)
                squeeze.append(d)
            elif isinstance(i, slice):
                a, b, step = i.indices(n)
                if step != 1:
                    return None
                starts.append(a)
                stops.append(max(a, b))
            else:
                return None
        out = self._ds.read_region(starts, stops)
        return out.reshape([m for d, m in enumerate(out.shape) if d not in squeeze])

    def __len__(self):
        return self.shape[0] if self.shape else 0


class Dataset(object):
    """read-only view: ds['uo'] -> Variable; ds.attrs; ds.close()"""

    def __init__(self, path):
        self.path = path
        self.variables = {}
        self.attrs = {}
        self._h = None
        try:
            import netCDF4
        except ImportError:
            netCDF4 = None
        if netCDF4 is not None:
            h = netCDF4.Dataset(path)
            h.set_auto_maskandscale(False)
            self._h = h
            for name, var in h.variables.items():
                attrs = {k: var.getncattr(k) for k in var.ncattrs()}
                self.variables[name] = Variable(name, var, var.dimensions, attrs, lock=_NETCDF4_LOCK)
            self.attrs = {k: h.getncattr(k) for k in h.ncattrs()}
            return
        with open(path, 'rb') as f:
            magic = f.read(8)
        if magic == b'\x89HDF\r\n\x1a\n':
            self._open_hdf5(path)
            return
        if magic[:3] != b'CDF':
            raise RuntimeError(f'{path}: neither a classic NetCDF-3 nor a NetCDF-4/HDF5 file (magic {magic[:4]!r})')
        from scipy.io import netcdf_file
        h = netcdf_file(path, 'r', mmap=True, maskandscale=False)
        self._h = h
        for name, var in h.variables.items():
            attrs = {k: (v.decode() if isinstance(v, bytes) else v) for k, v in var._attributes.items()}
            self.variables[name] = Variable(name, var.data, var.dimensions, attrs)
        self.attrs = {k: (v.decode() if isinstance(v, bytes) else v) for k, v in h._attributes.items()}

    def _open_hdf5(self, path):
        """NetCDF-4 (HDF5) through h5lite: contiguous variables are memory-mapped in place, chunked ones are decoded
        on first access; dimension names come from the dimension scales (_Netcdf4Dimid / _Netcdf4Coordinates)"""
        from . import h5lite
        h = h5lite.File(path)
        self._h = h
        hidden = ('CLASS', 'NAME', 'DIMENSION_LIST', 'REFERENCE_LIST', '_Netcdf4Dimid', '_Netcdf4Coordinates',
                  '_NCProperties')
        dim_by_id, dim_by_size = {}, {}
        for name, ds in h.datasets.items():
            if ds.attrs.get('CLASS') == 'DIMENSION_SCALE' and len(ds.shape) == 1:
                if '_Netcdf4Dimid' in ds.attrs:
                    dim_by_id[int(ds.attrs['_Netcdf4Dimid'])] = name
                dim_by_size.setdefault(ds.shape[0], name)
        for name, ds in h.datasets.items():
            note = ds.attrs.get('NAME')
            if isinstance(note, str) and note.startswith('This is a netCDF dimension but not a netCDF variable'):
                continue
            coords = ds.attrs.get('_Netcdf4Coordinates')
            if coords is not None and len(numpy.atleast_1d(coords)) == len(ds.shape):
                dims = [dim_by_id.get(int(c), f'dim{i}') for i, c in enumerate(numpy.atleast_1d(coords))]
            elif len(ds.shape) == 1 and ds.attrs.get('CLASS') == 'DIMENSION_SCALE':
                dims = [name]
            else:
                dims = [dim_by_size.get(n, f'dim{i}') for i, n in enumerate(ds.shape)]
            attrs = {k: v for k, v in ds.attrs.items() if k not in hidden}
            self.variables[name] = Variable(name, _H5Data(path, h, ds), dims, attrs)
        self.attrs = {k: v for k, v in h.attrs.items() if k not in hidden}

    def __getitem__(self, name):
        return self.variables[name]

    def __contains__(self, name):
        return name in self.variables

    def items(self):
        return self.variables.items()

    def close(self):
        if self._h is not None:
            for v in self.variables.values():
                v._data = None
            self.variables = {}
            import warnings
            with warnings.catch_warnings():
                warnings.simplefilter('ignore')
                try:
                    self._h.close()
                except Exception:
                    pass
            self._h = None

    def __enter__(self):
        return self

    def __exit__(self, *a):
        self.close()


def open_dataset(path):
    return Dataset(path)


class Writer(object):
    """createDimension / createVariable subset of netCDF4.Dataset(path, 'w') used by datagen.py:168-208"""

    def __init__(self, path, classic=False):
        """classic: NetCDF classic with 64-bit offsets whatever the backend (without netCDF4 it always is)"""
        try:
            import netCDF4
            self._nc4 = netCDF4.Dataset(path, 'w', **({'format': 'NETCDF3_64BIT_OFFSET'} if classic else {}))
            self._h = None
        except ImportError:
            from scipy.io import netcdf_file
            self._nc4 = None
            self._h = netcdf_file(path, 'w', version=2)

    def createDimension(self, name, size):
        (self._nc4 or self._h).createDimension(name, size)

    def createVariable(self, name, dtype, dims, fill_value=None, attrs=None, data=None):
        if self._nc4 is not None:
            v = self._nc4.createVariable(name, dtype, dims, fill_value=fill_value)
        else:
            v = self._h.createVariable(name, numpy.dtype(dtype), dims)
            if fill_value is not None:
                v._FillValue = numpy.array(fill_value, numpy.dtype(dtype))
        for k, val in (attrs or {}).items():
            setattr(v, k, val)
        if data is not None:
            v[:] = data
        return v

    def setAttr(self, name, value):
        setattr(self._nc4 or self._h, name, value)

    def close(self):
        (self._nc4 or self._h).close()
