"""
ctypes binding of librr_b200.so (the C ABI declared in include/rr_b200.h).

There is no CPU fallback anywhere in this package: if the shared library is missing the
import fails loudly, and every compute entry point fails with ``RuntimeError`` when no CUDA
device is usable.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

_PKG_DIR = os.path.dirname(os.path.abspath(__file__))
# RR_B200_LIB: measurement builds of the same sources (tools/librr_trace.so); never a different implementation
LIB_PATH = os.environ.get('RR_B200_LIB') or os.path.join(_PKG_DIR, 'librr_b200.so')

c_i32p = C.POINTER(C.c_int32)
c_i64p = C.POINTER(C.c_int64)
c_u8p = C.POINTER(C.c_uint8)
c_f64p = C.POINTER(C.c_double)


class PlanOpts(C.Structure):
    _fields_ = [('time_tile', C.c_int32), ('tile_stride', C.c_int32), ('device', C.c_int32),
                ('threads_per_cta', C.c_int32), ('raw_budget_bytes', C.c_int64), ('renumber', C.c_int32),
                ('staging', C.c_int32)]


class PlanInfo(C.Structure):
    _fields_ = [('n', C.c_int64), ('n_edges', C.c_int64), ('n_blocks', C.c_int64), ('n_export', C.c_int64),
                ('n_internal_edges', C.c_int64), ('max_skew', C.c_int32), ('max_indegree', C.c_int32),
                ('max_block_level', C.c_int32), ('n_outlets_lo', C.c_int32), ('n_dep_edges', C.c_int64),
                ('device_bytes', C.c_int64), ('renumbered', C.c_int32), ('reach_depth', C.c_int32),
                ('all_fast', C.c_int32), ('narrow_blocks', C.c_int32), ('n_headwaters', C.c_int64), ('n_work', C.c_int64)]


MAX_STATS = 16   # RR_MAX_STATS


class StatsSpec(C.Structure):
    _fields_ = [('n_stats', C.c_int32), ('kind', C.c_int32 * MAX_STATS), ('q', C.c_int32 * MAX_STATS)]


def _load() -> C.CDLL:
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f'{LIB_PATH} is missing. Build it with `python -c "import __graft_entry__ as g; g.build()"` '
            f'or `make -C {os.path.join(_PKG_DIR, "csrc")}`. river_route_b200 has no CPU fallback.')
    lib = C.CDLL(LIB_PATH)
    vp = C.c_void_p
    i32, i64, f64p = C.c_int32, C.c_int64, c_f64p
    sig = {
        'rr_last_error': (C.c_char_p, []),
        'rr_version': (C.c_int, []),
        'rr_cuda_available': (C.c_int, []),
        'rr_downstream_index': (C.c_int, [i64, c_i64p, c_i64p, c_i32p, c_i64p]),
        'rr_label_basins': (C.c_int, [i64, c_i32p, c_i32p, c_i64p, i32, c_i32p]),
        'rr_plan_create': (C.c_int, [i64, c_i32p, C.POINTER(PlanOpts), C.POINTER(vp)]),
        'rr_plan_destroy': (None, [vp]),
        'rr_plan_get_info': (C.c_int, [vp, C.POINTER(PlanInfo)]),
        'rr_plan_set_coefficients': (C.c_int, [vp, f64p, f64p, f64p, f64p]),
        'rr_route_dev': (C.c_int, [vp, C.c_int, vp, vp, vp, i64, vp, i64, i64, i64, vp]),
        'rr_route_host': (C.c_int, [vp, C.c_int, f64p, f64p, f64p, i64, f64p, i64, i64, i64]),
        'rr_plan_set_output_subset': (C.c_int, [vp, i64, c_i32p]),
        'rr_route_host_ex': (C.c_int, [vp, C.c_int, f64p, f64p, f64p, i64, vp, i64, i64, i64, C.c_int, i64]),
        'rr_route_host_typed': (C.c_int, [vp, C.c_int, f64p, f64p, vp, C.c_int, i64, vp, i64, i64, i64, C.c_int, i64]),
        'rr_transform_create': (C.c_int, [i64, i64, c_i32p, c_i32p, f64p, f64p, i32, C.POINTER(vp)]),
        'rr_transform_set_uh': (C.c_int, [vp, i64, f64p, i64, f64p, i64]),
        'rr_transform_get_uh_state': (C.c_int, [vp, f64p, i64]),
        'rr_transform_destroy': (None, [vp]),
        'rr_runoff_route_host': (C.c_int, [vp, vp, C.c_int, f64p, vp, C.c_int, i64, i64, C.c_int, C.c_int, C.c_int, vp,
                                           i64, i64, C.c_int, i64]),
        'rr_route_ensemble_dev': (C.c_int, [vp, C.c_int, vp, i32, C.POINTER(vp), i64, C.POINTER(vp), i64,
                                            C.POINTER(vp), i64, i64, vp]),
        'rr_plan_tile_rows': (i64, [vp, i64, i64]),
        'rr_route_ensemble_host': (C.c_int, [vp, C.c_int, f64p, i64, i32, C.POINTER(vp), C.c_int, i64, C.POINTER(vp), i64, C.c_int, f64p, i64,
                                             f64p, i64, i64, i64]),
        'rr_ensemble_stats_dev': (C.c_int, [C.POINTER(StatsSpec), i32, vp, i64, i64, i64, i64, vp, C.POINTER(vp), i64,
                                            C.c_int, vp]),
        'rr_route_ensemble_stats_host': (C.c_int, [vp, C.c_int, f64p, i64, i32, C.POINTER(vp), C.c_int, i64,
                                                   C.POINTER(StatsSpec), C.POINTER(vp), i64, C.c_int, f64p, i64, f64p, i64,
                                                   i64, i64]),
        'rr_plan_set_thresholds': (C.c_int, [vp, i32, f64p, i64]),
        'rr_ensemble_stats_dev_ex': (C.c_int, [C.POINTER(StatsSpec), i32, vp, i64, i64, i64, i64, vp, vp, i64, C.POINTER(vp),
                                               i64, C.c_int, vp, vp, i64, i64, vp]),
        'rr_route_ensemble_stats_host_ex': (C.c_int, [vp, C.c_int, f64p, i64, i32, C.POINTER(vp), C.c_int, i64,
                                                      C.POINTER(StatsSpec), C.POINTER(vp), i64, C.c_int, f64p, i64, f64p,
                                                      i64, i64, i64, f64p, c_i32p, i64]),
        'rr_launch_count': (i64, [C.c_int]),
        'rr_timing_enable': (C.c_int, [C.c_int]),
        'rr_timing_read': (C.c_int, [f64p, c_i64p, C.c_int]),
        'rr_uh_convolve_dev': (C.c_int, [i64, i64, i64, vp, i64, vp, i64, vp, i64, vp, i64, vp]),
        'rr_uh_convolve_host': (C.c_int, [i64, i64, i64, f64p, i64, f64p, i64, f64p, i64, f64p, i64]),
        'rr_weights_transform_dev': (C.c_int, [i64, i64, i64, vp, vp, vp, vp, C.c_int, i64, vp, i64, C.c_int, C.c_int,
                                               vp, vp]),
        'rr_weights_transform_host': (C.c_int, [i64, i64, i64, c_i32p, c_i32p, f64p, vp, C.c_int, i64, f64p, i64,
                                                C.c_int, C.c_int, f64p]),
        'rr_plan_read_profile': (C.c_int, [vp, C.POINTER(C.c_uint64)]),
        'rr_host_alloc': (C.c_int, [C.POINTER(vp), i64]),
        'rr_host_free': (C.c_int, [vp]),
        'rr_synth_forest': (C.c_int, [i64, i64, C.c_uint64, C.c_double, i64, C.c_double, c_i32p]),
        'rr_plan_get_arrays': (C.c_int, [vp] + [C.POINTER(c_i32p), C.POINTER(c_i32p), C.POINTER(c_u8p)]
                               + [C.POINTER(c_i32p)] * 7),
        'rr_plan_schedule': (C.c_int, [vp, i64, i32, c_i64p, c_i32p, c_i32p]),
    }
    for name, (res, args) in sig.items():
        fn = getattr(lib, name)  # AttributeError here means the .so does not match include/rr_b200.h
        fn.restype = res
        fn.argtypes = args
    return lib


lib = _load()
EXPORTED_SYMBOLS = (
    'rr_last_error', 'rr_version', 'rr_cuda_available', 'rr_downstream_index', 'rr_label_basins',
    'rr_plan_create', 'rr_plan_destroy', 'rr_plan_get_info', 'rr_plan_set_coefficients', 'rr_route_dev',
    'rr_route_host', 'rr_plan_set_output_subset', 'rr_route_host_ex', 'rr_route_host_typed', 'rr_transform_create', 'rr_transform_set_uh', 'rr_transform_get_uh_state',
    'rr_transform_destroy', 'rr_runoff_route_host', 'rr_route_ensemble_dev', 'rr_route_ensemble_host', 'rr_plan_tile_rows',
    'rr_ensemble_stats_dev', 'rr_route_ensemble_stats_host', 'rr_plan_set_thresholds', 'rr_ensemble_stats_dev_ex',
    'rr_route_ensemble_stats_host_ex', 'rr_launch_count', 'rr_timing_enable', 'rr_timing_read', 'rr_uh_convolve_dev', 'rr_uh_convolve_host',
    'rr_weights_transform_dev', 'rr_weights_transform_host', 'rr_plan_read_profile', 'rr_host_alloc', 'rr_host_free', 'rr_synth_forest',
    'rr_plan_get_arrays', 'rr_plan_schedule',
)


def last_error() -> str:
    return (lib.rr_last_error() or b'').decode('utf-8', 'replace')


def check(rc: int) -> None:
    """Turn a non-zero status of the C ABI into the exception the reference would raise."""
    if rc == 0:
        return
    msg = last_error()
    if rc in (1, 2, 3):  # the reference's topology ValueErrors (Muskingum.py:153-154, tools.py:101-104)
        raise ValueError(msg)
    raise RuntimeError(f'librr_b200: {msg} (status {rc})')


def cuda_available() -> bool:
    return bool(lib.rr_cuda_available())


def as_f64p(a: np.ndarray):
    assert a.dtype == np.float64
    return a.ctypes.data_as(c_f64p)


def as_i32p(a: np.ndarray):
    assert a.dtype == np.int32 and a.flags.c_contiguous
    return a.ctypes.data_as(c_i32p)


def as_i64p(a: np.ndarray):
    assert a.dtype == np.int64 and a.flags.c_contiguous
    return a.ctypes.data_as(c_i64p)


def rows_ld(a: np.ndarray) -> int:
    """Leading dimension (in elements) of a 2-D array whose rows are contiguous."""
    if a.ndim != 2 or (a.shape[1] > 1 and a.strides[1] != a.itemsize):
        raise ValueError('array rows must be contiguous')
    if a.shape[0] > 1:
        if a.strides[0] % a.itemsize or a.strides[0] < a.shape[1] * a.itemsize:
            raise ValueError('unsupported row stride')
        return a.strides[0] // a.itemsize
    return max(a.shape[1], 1)


def pinned_empty(shape, dtype=np.float64) -> np.ndarray:
    """numpy array backed by page-locked host memory (full-rate cudaMemcpyAsync); freed with the array."""
    dtype = np.dtype(dtype)
    count = int(np.prod(shape))
    nbytes = max(count * dtype.itemsize, 1)
    ptr = C.c_void_p()
    check(lib.rr_host_alloc(C.byref(ptr), nbytes))

    class _Owner:
        def __init__(self, p):
            self.p = p

        def __del__(self):
            try:
                lib.rr_host_free(self.p)
            except Exception:
                pass

    buf = (C.c_char * nbytes).from_address(ptr.value)
    buf._owner = _Owner(ptr)  # keeps the allocation alive as long as any view of it
    return np.frombuffer(buf, dtype=dtype, count=count).reshape(shape)
