"""ctypes binding of libskyopt (include/skyopt.h). No CPU fallback.

The structures mirror the C header field by field; numpy structured dtypes of
the same layout are exported so that callers can build whole batches of
queries / slots / tasks as arrays and hand over plain pointers.
"""
import ctypes
import os
import threading
from typing import Optional

import numpy as np

ABI_VERSION = 4
ACC_SET_WORDS = 32
MAX_CLOUDS = 32
NONE16 = 0xFFFF

F_VALID = 0x0001
F_DEFAULT_FAMILY = 0x0002
F_SSD = 0x0004
F_NVME = 0x0008
F_HOST_FAMILY = 0x0010
F_HAS_INSTANCE = 0x0020
F_PREMIUM_DISK = 0x0040

OP_NONE, OP_EQ, OP_GE, OP_RATIO = 0, 1, 2, 3
DISK_NEAR, DISK_GE = 1, 2
Q_ACC, Q_FUZZY, Q_LIST, Q_KEEP_NAN = 1, 2, 4, 8

_LIB_NAME = 'libskyopt.so'


class SkyoptError(RuntimeError):
    """A libskyopt call failed (code, message from skyopt_last_error)."""

    def __init__(self, code: int, message: str):
        super().__init__(f'libskyopt error {code}: {message}')
        self.code = code


class NativeLibraryMissing(ImportError):
    """libskyopt.so is not built; the product path has no CPU fallback."""


QUERY_DTYPE = np.dtype([
    ('cloud', '<i4'), ('qflags', '<u4'), ('flags_require', '<u4'),
    ('group', '<i4'), ('acc_set', '<i4'), ('fuzzy_set', '<i4'),
    ('price_col', '<i4'), ('cpus_op', '<i4'), ('mem_op', '<i4'),
    ('disk_op', '<i4'), ('region_id', '<i4'), ('zone_id', '<i4'),
    ('flags_require2', '<u4'), ('pad_', '<i4'),
    ('cpus', '<f8'), ('mem', '<f8'), ('disk_size', '<f8'),
    ('max_price', '<f8'),
], align=True)

SCAN_RESULT_DTYPE = np.dtype([
    ('any_stage1', '<i4'), ('best_row', '<i4'), ('best_inst', '<i4'),
    ('n_list', '<i4'), ('n_fuzzy', '<i4'), ('pad_', '<i4'),
    ('best_price', '<f8'),
], align=True)

SLOT_DTYPE = np.dtype([
    ('cloud', '<i4'), ('query', '<i4'), ('inst_id', '<i4'),
    ('gate_query', '<i4'), ('acc_set', '<i4'), ('price_col', '<i4'),
    ('region_id', '<i4'), ('zone_id', '<i4'), ('split_by_zone', '<i4'),
    ('us_first', '<i4'), ('cand_acc_key', '<i4'), ('use_spot', '<i4'),
    ('region_set', '<i4'), ('pad_', '<i4'),
    ('hours', '<f8'), ('node_mult', '<f8'), ('time_value', '<f8'),
], align=True)

BLOCKED_DTYPE = np.dtype([
    ('cloud', '<i4'), ('inst_id', '<i4'), ('region_id', '<i4'),
    ('zone_id', '<i4'), ('acc_key', '<i4'), ('use_spot', '<i4'),
], align=True)

TASK_DTYPE = np.dtype([
    ('slot_begin', '<i4'), ('slot_end', '<i4'), ('n_parents', '<i4'),
    ('parent_begin', '<i4'), ('edge_tariff_begin', '<i4'),
    ('src_tariff_begin', '<i4'),
], align=True)

DAG_DTYPE = np.dtype([
    ('task_begin', '<i4'), ('task_end', '<i4'), ('is_chain', '<i4'),
    ('minimize_cost', '<i4'), ('blocked_begin', '<i4'),
    ('blocked_end', '<i4'),
], align=True)

CANDIDATE_DTYPE = np.dtype([
    ('slot', '<i4'), ('inst_id', '<i4'), ('region_id', '<i4'),
    ('zone_id', '<i4'), ('hourly', '<f8'), ('value', '<f8'),
], align=True)

ZONE_DTYPE = np.dtype([
    ('flags_or', '<u4'), ('sig_lo', '<u4'), ('sig_hi', '<u4'), ('groups', '<u4'),
    ('min_key', '<u8', (2,)),
], align=True)
ZONE_ROWS = 128

RESERVATION_DTYPE = np.dtype([
    ('cloud', '<i4'), ('inst_id', '<i4'), ('zone_id', '<i4'),
    ('available', '<i4'),
], align=True)

DAG_RESULT_DTYPE = np.dtype([
    ('status', '<i4'), ('task_fail', '<i4'), ('objective', '<f8'),
], align=True)

_EXPECTED_SIZES = {
    'query': 88, 'scan_result': 32, 'slot': 80, 'blocked': 24, 'task': 24,
    'dag': 24, 'candidate': 32, 'dag_result': 16, 'reservation': 16
}
assert QUERY_DTYPE.itemsize == _EXPECTED_SIZES['query'], QUERY_DTYPE.itemsize
assert SCAN_RESULT_DTYPE.itemsize == _EXPECTED_SIZES['scan_result']
assert SLOT_DTYPE.itemsize == _EXPECTED_SIZES['slot'], SLOT_DTYPE.itemsize
assert BLOCKED_DTYPE.itemsize == _EXPECTED_SIZES['blocked']
assert TASK_DTYPE.itemsize == _EXPECTED_SIZES['task']
assert DAG_DTYPE.itemsize == _EXPECTED_SIZES['dag']
assert CANDIDATE_DTYPE.itemsize == _EXPECTED_SIZES['candidate']
assert DAG_RESULT_DTYPE.itemsize == _EXPECTED_SIZES['dag_result']
assert RESERVATION_DTYPE.itemsize == _EXPECTED_SIZES['reservation']

_p = ctypes.c_void_p


class CatalogDesc(ctypes.Structure):
    _fields_ = [
        ('n_rows', ctypes.c_int64),
        ('price', _p), ('spot_price', _p), ('vcpus', _p), ('mem', _p),
        ('disk_total', _p), ('acc_key', _p), ('region_id', _p),
        ('zone_id', _p), ('flags', _p), ('inst_id', _p),
        ('n_clouds', ctypes.c_int32), ('n_inst', ctypes.c_int32),
        ('n_acc_keys', ctypes.c_int32), ('n_regions', ctypes.c_int32),
        ('cloud_row_offsets', _p), ('cloud_inst_offsets', _p),
        ('cloud_region_offsets', _p), ('cloud_n_zones', _p),
        ('region_is_us', _p), ('inst_row_offsets', _p), ('inst_rows', _p),
        ('acc_row_offsets', _p), ('acc_rows', _p), ('inst_acc_key', _p),
        ('zone_map', _p),
    ]


class Problem(ctypes.Structure):
    _fields_ = [
        ('queries', _p), ('n_queries', ctypes.c_int32),
        ('acc_sets', _p), ('n_acc_sets', ctypes.c_int32),
        ('slots', _p), ('n_slots', ctypes.c_int32),
        ('tasks', _p), ('n_tasks', ctypes.c_int32),
        ('parents', _p), ('n_parents', ctypes.c_int32),
        ('tariffs', _p), ('n_tariffs', ctypes.c_int32),
        ('blocked', _p), ('n_blocked', ctypes.c_int32),
        ('dags', _p), ('n_dags', ctypes.c_int32),
        ('reservations', _p), ('n_reservations', ctypes.c_int32),
    ]


class Solution(ctypes.Structure):
    _fields_ = [
        ('scan', _p), ('slot_count', _p), ('slot_inst', _p), ('chosen', _p),
        ('chosen_index', _p), ('task_n_candidates', _p), ('dag', _p),
        ('candidates', _p), ('cand_cap', ctypes.c_int64),
        ('task_cand_offset', _p),
    ]


class Stats(ctypes.Structure):
    _fields_ = [
        ('scan_ms', ctypes.c_float), ('expand_ms', ctypes.c_float),
        ('solve_ms', ctypes.c_float), ('total_ms', ctypes.c_float),
        ('scan_launches', ctypes.c_int32), ('total_launches', ctypes.c_int32),
        ('scan_rows', ctypes.c_int64), ('scan_passes_rows', ctypes.c_int64),
        ('scan_kernel_ms', ctypes.c_float), ('scan_blocks', ctypes.c_int32),
        ('scan_form', ctypes.c_int32), ('reserved_', ctypes.c_int32),
    ]

    def as_dict(self):
        return {name: getattr(self, name) for name, _ in self._fields_}


EXPORTS = (
    'skyopt_abi_version', 'skyopt_last_error', 'skyopt_device_count',
    'skyopt_catalog_create', 'skyopt_catalog_destroy', 'skyopt_catalog_bytes',
    'skyopt_scan', 'skyopt_optimize', 'skyopt_optimize_timed',
    'skyopt_catalog_set_scan_mode', 'skyopt_price_key',
    'skyopt_solve_tables', 'skyopt_list_offerings',
    'skyopt_session_open', 'skyopt_session_resolve', 'skyopt_session_close',
)

_lib = None
_lib_lock = threading.Lock()


def library_path() -> str:
    # SKYOPT_LIBRARY: another build of the same sources (kernel tuning A/B)
    override = os.environ.get('SKYOPT_LIBRARY')
    if override:
        return os.path.abspath(override)
    return os.path.join(os.path.dirname(os.path.abspath(__file__)), _LIB_NAME)


def load() -> ctypes.CDLL:
    """Loads libskyopt.so (built by `__graft_entry__.build()`); fails loudly."""
    global _lib
    if _lib is not None:
        return _lib
    with _lib_lock:
        if _lib is not None:
            return _lib
        path = library_path()
        if not os.path.exists(path):
            raise NativeLibraryMissing(
                f'{path} not found. Build it with `python -c "import '
                '__graft_entry__ as g; g.build()"` (nvcc, sm_100a). The '
                'optimizer hot path has no CPU fallback.')
        lib = ctypes.CDLL(path)
        lib.skyopt_abi_version.restype = ctypes.c_int
        lib.skyopt_price_key.restype = ctypes.c_uint64
        lib.skyopt_price_key.argtypes = [ctypes.c_double]
        lib.skyopt_last_error.restype = ctypes.c_char_p
        lib.skyopt_device_count.argtypes = [ctypes.POINTER(ctypes.c_int)]
        lib.skyopt_catalog_create.argtypes = [
            ctypes.POINTER(CatalogDesc), ctypes.c_int,
            ctypes.POINTER(ctypes.c_void_p)
        ]
        lib.skyopt_catalog_destroy.argtypes = [ctypes.c_void_p]
        lib.skyopt_catalog_bytes.argtypes = [
            ctypes.c_void_p,
            ctypes.POINTER(ctypes.c_int64),
            ctypes.POINTER(ctypes.c_int64)
        ]
        lib.skyopt_catalog_set_scan_mode.argtypes = [
            ctypes.c_void_p, ctypes.c_int
        ]
        lib.skyopt_solve_tables.argtypes = [
            ctypes.c_void_p, _p, _p, _p, _p, ctypes.c_int, _p, ctypes.c_int, _p,
            ctypes.c_int, _p, ctypes.c_int, _p, _p
        ]
        lib.skyopt_session_open.argtypes = [
            ctypes.c_void_p,
            ctypes.POINTER(Problem),
            ctypes.POINTER(Solution),
            ctypes.POINTER(Stats),
            ctypes.POINTER(ctypes.c_void_p)
        ]
        lib.skyopt_session_resolve.argtypes = [
            ctypes.c_void_p, _p, ctypes.c_int,
            ctypes.POINTER(Solution),
            ctypes.POINTER(Stats)
        ]
        lib.skyopt_session_close.argtypes = [ctypes.c_void_p]
        lib.skyopt_session_close.restype = None
        lib.skyopt_list_offerings.argtypes = [
            ctypes.c_void_p, ctypes.c_int, ctypes.c_int, _p, ctypes.c_int, _p,
            ctypes.c_int, _p
        ]
        lib.skyopt_scan.argtypes = [
            ctypes.c_void_p, _p, ctypes.c_int, _p, ctypes.c_int, _p, _p, _p,
            ctypes.c_int, _p, _p, ctypes.c_int,
            ctypes.POINTER(Stats)
        ]
        lib.skyopt_optimize.argtypes = [
            ctypes.c_void_p,
            ctypes.POINTER(Problem),
            ctypes.POINTER(Solution),
            ctypes.POINTER(Stats)
        ]
        lib.skyopt_optimize_timed.argtypes = [
            ctypes.c_void_p,
            ctypes.POINTER(Problem),
            ctypes.POINTER(Solution), ctypes.c_int, ctypes.c_int, _p, _p,
            ctypes.POINTER(Stats)
        ]
        for name in EXPORTS:
            getattr(lib, name)  # AttributeError if a symbol is missing
        version = lib.skyopt_abi_version()
        if version != ABI_VERSION:
            raise NativeLibraryMissing(
                f'{path} has ABI {version}, expected {ABI_VERSION}; rebuild.')
        _lib = lib
    return _lib


def check(code: int) -> None:
    if code != 0:
        msg = load().skyopt_last_error()
        raise SkyoptError(code, msg.decode('utf-8', 'replace') if msg else '')


def ptr(arr: Optional[np.ndarray]):
    """Pointer to a C-contiguous numpy array (None -> NULL)."""
    if arr is None:
        return None
    assert arr.flags['C_CONTIGUOUS'], 'array must be C-contiguous'
    return ctypes.c_void_p(arr.ctypes.data)


def device_count() -> int:
    n = ctypes.c_int(0)
    code = load().skyopt_device_count(ctypes.byref(n))
    if code != 0:
        return 0
    return n.value
