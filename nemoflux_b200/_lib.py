"""ctypes binding of libnemoflux_gpu.so (the C ABI declared in include/nemoflux_gpu.h).

There is no CPU fallback: if the library is missing or no CUDA device is usable, every compute entry
point raises.  Build the library with ``python -m nemoflux_b200.build`` (nvcc, sm_100a).
"""
import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, 'libnemoflux_gpu.so')

NFX_OK = 0
NFX_CELL_BY_CELL_DATA = 0
NFX_F64, NFX_F32 = 0, 1
NFX_BIG_ENDIAN = 0x100
NFX_H5_DEFLATE, NFX_H5_SHUFFLE, NFX_H5_FLETCHER32 = 1, 2, 4
NFX_ORDER_LIST, NFX_ORDER_MAP = 0, 1
NFX_K2_AUTO, NFX_K2_LDG, NFX_K2_TMA, NFX_K2_LDG128 = 0, 1, 2, 3
NFX_OPT_K2_VARIANT, NFX_OPT_K2_UNROLL, NFX_OPT_K2_BLOCK, NFX_OPT_FAST_SERIES, NFX_OPT_RING_SLOT_MB = 1, 2, 3, 4, 5
NFX_OPT_K2_ALU_MASK = 6
NFX_OPT_FUSED_F32_SHAPE = 7
NFX_OPT_LAST_SERIES_PATH = 8
NFX_OPT_FUSED_ORDER = 9
NFX_OPT_FUSED_F64_CTAS = 10
NFX_OPT_FUSED_K3_LAG = 15
NFX_OPT_RING_MAX_MB = 16
NFX_OPT_SPARSE_COLUMNS = 17
NFX_OPT_LAST_SERIES_SPARSE = 18

c_i64 = ctypes.c_int64
c_int = ctypes.c_int
c_dbl = ctypes.c_double
c_vp = ctypes.c_void_p
P = ctypes.POINTER

# name -> argtypes; every function returns int except nfx_last_error
SIGNATURES = {
    'nfx_version': [],
    'nfx_set_option': [c_int, c_int],
    'nfx_get_option': [c_int, P(c_int)],
    'nfx_launch_count': [P(c_i64)],
    'nfx_debug_check_guards': [P(c_i64), P(c_i64)],
    'nfx_debug_poke_guard': [c_int],
    'nfx_grid_new': [P(c_vp)],
    'nfx_grid_del': [P(c_vp)],
    'nfx_grid_set_points': [P(c_vp), c_i64, c_vp],
    'nfx_grid_get_num_cells': [P(c_vp), P(c_i64)],
    'nfx_grid_set_cgrid_shape': [P(c_vp), c_int, c_int],
    'nfx_grid_arc_lengths': [P(c_vp), c_vp, c_vp],
    'nfx_pli_new': [P(c_vp)],
    'nfx_pli_del': [P(c_vp)],
    'nfx_pli_set_grid': [P(c_vp), c_vp],
    'nfx_pli_build_locator': [P(c_vp), c_int, c_dbl, c_int],
    'nfx_pli_compute_weights': [P(c_vp), c_int, c_vp, c_int],
    'nfx_pli_compute_weights_batch': [P(c_vp), c_int, c_vp, c_vp, c_int],
    'nfx_pli_get_num_transects': [P(c_vp), P(c_int)],
    'nfx_pli_get_num_subsegments': [P(c_vp), P(c_i64)],
    'nfx_pli_get_subsegments': [P(c_vp)] + [c_vp] * 10,
    'nfx_pli_get_map_size': [P(c_vp), P(c_i64)],
    'nfx_pli_get_map': [P(c_vp), c_vp, c_vp, c_vp],
    'nfx_pli_get_integral': [P(c_vp), c_vp, c_int, P(c_dbl)],
    'nfx_pli_get_integrals': [P(c_vp), c_vp, c_int, c_int, c_vp],
    'nfx_pli_get_integrals_device': [P(c_vp), c_vp, c_int, c_int, c_vp, c_vp],
    'nfx_vinterp_new': [P(c_vp)],
    'nfx_vinterp_del': [P(c_vp)],
    'nfx_vinterp_set_grid': [P(c_vp), c_vp],
    'nfx_vinterp_build_locator': [P(c_vp), c_int, c_dbl, c_int],
    'nfx_vinterp_find_points': [P(c_vp), c_i64, c_vp, c_dbl, P(c_i64)],
    'nfx_vinterp_get_cells': [P(c_vp), c_vp, c_vp],
    'nfx_vinterp_get_face_vectors': [P(c_vp), c_vp, c_int, c_vp],
    'nfx_vinterp_get_face_vectors_device': [P(c_vp), c_vp, c_vp, c_vp],
    'nfx_edgeflux_assemble': [c_vp, c_vp, c_int, c_vp, c_vp, c_vp, c_int, c_int, c_i64, c_int, c_dbl, c_vp, c_vp],
    'nfx_edgeflux_assemble_ld': [c_vp, c_vp, c_int, c_vp, c_vp, c_vp, c_int, c_int, c_i64, c_i64, c_int, c_dbl, c_vp,
                                 c_vp],
    'nfx_edgeflux_assemble_e3': [c_vp, c_vp, c_vp, c_vp, c_int, c_int, c_vp, c_vp, c_int, c_int, c_i64, c_i64, c_int,
                                 c_dbl, c_vp, c_vp],
    'nfx_flux_series_e3': [P(c_vp), c_vp, c_vp, c_vp, c_vp, c_int, c_int, c_vp, c_vp, c_int, c_int, c_i64, c_int, c_dbl,
                           c_int, c_vp, c_vp, c_vp],
    'nfx_edgeflux_to_cell_by_cell': [c_vp, c_int, c_int, c_int, c_vp, c_vp],
    'nfx_edgeflux_absmax': [c_vp, c_int, c_i64, P(c_dbl), c_vp],
    'nfx_pli_integrate': [P(c_vp), c_vp, c_int, c_int, c_vp, c_vp],
    'nfx_flux_series': [P(c_vp), c_vp, c_vp, c_int, c_vp, c_vp, c_vp, c_int, c_int, c_int, c_dbl, c_int, c_vp, c_vp,
                        c_vp],
    'nfx_flux_series_ld': [P(c_vp), c_vp, c_vp, c_int, c_vp, c_vp, c_vp, c_int, c_int, c_i64, c_int, c_dbl, c_int, c_vp,
                           c_vp, c_vp],
    'nfx_pli_get_num_panels': [P(c_vp), P(c_int), P(c_i64)],
    'nfx_pli_get_num_panels_dtype': [P(c_vp), c_int, P(c_int), P(c_i64)],
    'nfx_pli_series_status': [P(c_vp), c_vp, P(c_int)],
    'nfx_probe_read_bandwidth': [c_vp, c_i64, c_int, P(c_dbl), c_vp],
    'nfx_probe_read_bandwidth_groups': [c_vp, c_i64, c_vp, c_i64, c_int, P(c_dbl), c_vp],
    'nfx_pli_get_column_groups': [P(c_vp), c_int, c_int, c_int, c_vp, c_vp, P(c_i64)],
    'nfx_h5_decode_chunks': [c_vp, c_i64, c_i64, c_vp, c_vp, c_int, c_int, c_int, c_vp, c_vp, c_vp, c_int, c_vp, c_vp, c_vp],
    'nfx_flux_series_range': [P(c_vp), c_vp, c_vp, c_int, c_vp, c_vp, c_vp, c_int, c_int, c_i64, c_int, c_dbl, c_int,
                              c_i64, c_i64, c_vp, c_vp],
    'nfx_flux_series_range_e3': [P(c_vp), c_vp, c_vp, c_vp, c_vp, c_int, c_int, c_vp, c_vp, c_int, c_int, c_i64, c_int,
                                 c_dbl, c_int, c_i64, c_i64, c_vp, c_vp],
    'nfx_flux_series_host': [P(c_vp), c_vp, c_vp, c_int, c_vp, c_vp, c_vp, c_int, c_int, c_int, c_dbl, c_int, c_int,
                             c_vp],
    'nfx_flux_series_host_e3': [P(c_vp), c_vp, c_vp, c_vp, c_vp, c_int, c_int, c_int, c_vp, c_vp, c_int, c_int, c_int,
                                c_dbl, c_int, c_int, c_vp],
}

_LIB = None


class NemofluxGpuError(RuntimeError):
    def __init__(self, code, message):
        super().__init__(f'libnemoflux_gpu error {code}: {message}')
        self.code = code


def load():
    """load the shared library (raises if it was not built -- there is no fallback)"""
    global _LIB
    if _LIB is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(f'{LIB_PATH} is missing: build it with `python -m nemoflux_b200.build` '
                               '(nvcc -gencode arch=compute_100a,code=sm_100a); there is no CPU fallback')
        L = ctypes.CDLL(LIB_PATH)
        L.nfx_last_error.restype = ctypes.c_char_p
        L.nfx_last_error.argtypes = []
        for name, args in SIGNATURES.items():
            f = getattr(L, name)
            f.restype = c_int
            f.argtypes = args
        _LIB = L
    return _LIB


def check(ier):
    if ier != NFX_OK:
        raise NemofluxGpuError(ier, load().nfx_last_error().decode('utf-8', 'replace'))


def call(name, *args):
    check(getattr(load(), name)(*args))


def launch_count():
    n = c_i64()
    call('nfx_launch_count', ctypes.byref(n))
    return n.value


def check_guards():
    """NFX_DEBUG_GUARDS=1: number of library-owned device buffers checked; raises NemofluxGpuError when a guard band
    around one of them was overwritten (0 buffers = the guards are off)"""
    n, bad = c_i64(), c_i64()
    call('nfx_debug_check_guards', ctypes.byref(n), ctypes.byref(bad))
    return n.value


def set_option(option, value):
    call('nfx_set_option', option, value)


def get_option(option):
    v = ctypes.c_int()
    call('nfx_get_option', option, ctypes.byref(v))
    return v.value
