"""ctypes binding of libmetis_b200.so (C ABI declared in include/metis_b200.h).

The library is built in-tree by ``metis_b200.build.build_library`` (nvcc, sm_100a).
There is no CPU fallback: if the shared object is missing or a call fails, an
exception is raised.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, 'libmetis_b200.so')

METIS_MAX_TYPES = 8
METIS_MAX_STAGES = 128
METIS_MAX_LAYERS = 256
METIS_MAX_PERMUTE_GROUPS = 32
DETAIL_STRIDE = 3 * METIS_MAX_STAGES + 1

FATAL_NAMES = {1: 'KEY_EXEC', 2: 'KEY_MEMORY', 3: 'INDEX', 4: 'HANG', 5: 'SCRATCH', 6: 'ZERODIV'}


class MetisProblem(C.Structure):
    _fields_ = [
        ('num_types', C.c_int32), ('num_tp', C.c_int32), ('num_bs', C.c_int32), ('num_keys', C.c_int32),
        ('lpad', C.c_int32), ('num_layers', C.c_int32), ('norm_len', C.c_int32), ('gbs', C.c_int32),
        ('max_tp', C.c_int32), ('max_bs', C.c_int32), ('num_nodes', C.c_int32),
        ('devices_per_node', C.c_int32), ('total_devices', C.c_int32), ('num_node_sequences', C.c_int32),
        ('uniform_bw', C.c_int32), ('q10_devices', C.c_int32), ('corrected', C.c_int32), ('reserved1', C.c_int32),
        ('sequence_length', C.c_int64), ('hidden_size', C.c_int64), ('vocab_size', C.c_int64),
        ('optimizer_time', C.c_double), ('batch_generator', C.c_double),
        ('input_params', C.c_double), ('transformer_params', C.c_double), ('output_params', C.c_double),
        ('node0_bandwidth', C.c_double), ('node0_memory', C.c_double),
        ('key_index', C.c_void_p), ('layer_compute', C.c_void_p), ('layer_memory', C.c_void_p),
        ('exec_full', C.c_void_p), ('fb_sync', C.c_void_p), ('norm_lc', C.c_void_p),
        ('type_memory', C.c_void_p), ('type_bw_first', C.c_void_p), ('type_bw_min', C.c_void_p),
        ('ns_run_type', C.c_void_p), ('ns_run_end', C.c_void_p), ('ns_q10_end', C.c_void_p),
    ]


class MetisPlanBlock(C.Structure):
    _fields_ = [('first_ordinal', C.c_int64), ('rows_offset', C.c_int64), ('num_rows', C.c_int32),
                ('ns_idx', C.c_int16), ('label_stage', C.c_int16), ('num_stage', C.c_int16),
                ('reserved', C.c_int16 * 3)]


class MetisPlanSpace(C.Structure):
    _fields_ = [('num_plans', C.c_int64), ('rows_bytes', C.c_int64), ('num_blocks', C.c_int32), ('num_div', C.c_int32),
                ('max_stage', C.c_int32), ('reserved', C.c_int32),
                ('blocks', C.c_void_p), ('batches', C.c_void_p), ('rows', C.c_void_p)]


class MetisRecord(C.Structure):
    _fields_ = [('cost', C.c_double), ('ordinal', C.c_uint32), ('step', C.c_uint16),
                ('num_repartition', C.c_uint8), ('num_stage', C.c_uint8)]


class MetisSearchSummary(C.Structure):
    _fields_ = [('num_records', C.c_uint64), ('num_partition_calls', C.c_uint64),
                ('num_balancer_runs', C.c_uint64), ('num_keyerror', C.c_uint64),
                ('fatal_ordinal', C.c_uint64), ('fatal_code', C.c_uint32), ('fatal_aux', C.c_uint32),
                ('best', MetisRecord), ('reserved', C.c_uint64 * 6)]


class MetisShard(C.Structure):
    _fields_ = [('rank', C.c_int32), ('world', C.c_int32), ('tile', C.c_int32), ('reserved', C.c_int32)]


assert C.sizeof(MetisRecord) == 16 and C.sizeof(MetisPlanBlock) == 32

# numpy dtype twins of the C structs
RECORD_DTYPE = [('cost', '<f8'), ('ordinal', '<u4'), ('step', '<u2'), ('num_repartition', 'u1'), ('num_stage', 'u1')]
BLOCK_DTYPE = [('first_ordinal', '<i8'), ('rows_offset', '<i8'), ('num_rows', '<i4'), ('ns_idx', '<i2'),
               ('label_stage', '<i2'), ('num_stage', '<i2'), ('reserved', '<i2', (3,))]

COMP_DTYPE = [('row_offset', '<i8'), ('pool_offset', '<u4'), ('stages', '<u2'), ('num_groups', '<u2'),
              ('first_row', '<u4'), ('num_rows', '<u4')]

SYMBOLS = ['metis_last_error', 'metis_abi_version', 'metis_set_profile_events', 'metis_het_workspace_bytes', 'metis_het_search',
           'metis_het_detail', 'metis_het_trace', 'metis_homo_cost', 'metis_layer_balance', 'metis_enum_device_groups',
           'metis_enum_device_group_tables', 'metis_sort_workspace_bytes', 'metis_sort_records',
           'metis_enum_compositions', 'metis_generate_rows', 'metis_select_workspace_bytes', 'metis_select_records']
SORT_POSITION, SORT_RANKED, SORT_BY_COST_STABLE = 0, 1, 2

_lib = None


class MetisNativeError(RuntimeError):
    pass


def load_library(path: str = LIB_PATH) -> C.CDLL:
    """dlopen the CUDA library; raises if it has not been built (no fallback)."""
    global _lib
    if _lib is not None and path == LIB_PATH:
        return _lib
    if not os.path.exists(path):
        raise MetisNativeError(
            f'{path} is missing: build it with `python -c "import __graft_entry__ as g; g.build()"` '
            f'(nvcc, sm_100a). metis_b200 has no CPU fallback.')
    lib = C.CDLL(path)
    lib.metis_last_error.restype = C.c_char_p
    lib.metis_abi_version.restype = C.c_int
    lib.metis_set_profile_events.restype = None
    lib.metis_set_profile_events.argtypes = [C.c_void_p, C.c_void_p]
    lib.metis_het_workspace_bytes.restype = C.c_int64
    lib.metis_het_workspace_bytes.argtypes = [C.POINTER(MetisProblem), C.c_int64, C.c_int32]
    lib.metis_het_search.restype = C.c_int
    lib.metis_het_search.argtypes = [C.POINTER(MetisProblem), C.POINTER(MetisPlanSpace), C.POINTER(MetisShard),
                                     C.c_void_p, C.c_int64, C.c_void_p, C.c_int32, C.c_void_p, C.c_int64,
                                     C.c_void_p, C.c_void_p]
    lib.metis_het_detail.restype = C.c_int
    lib.metis_het_detail.argtypes = [C.POINTER(MetisProblem), C.POINTER(MetisPlanSpace), C.c_void_p, C.c_int64,
                                     C.c_void_p, C.c_int32, C.c_void_p, C.c_int64, C.c_void_p]
    lib.metis_het_trace.restype = C.c_int
    lib.metis_het_trace.argtypes = [C.POINTER(MetisProblem), C.POINTER(MetisPlanSpace), C.c_void_p, C.c_int64,
                                    C.c_void_p, C.c_int32, C.c_void_p, C.c_int64, C.c_void_p]
    lib.metis_homo_cost.restype = C.c_int
    lib.metis_homo_cost.argtypes = [C.POINTER(MetisProblem), C.c_int32, C.c_void_p, C.c_int64, C.c_void_p,
                                    C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p]
    lib.metis_layer_balance.restype = C.c_int
    lib.metis_layer_balance.argtypes = [C.c_void_p, C.c_void_p, C.c_int64, C.c_int32, C.c_void_p, C.c_int32,
                                        C.c_int32, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p]
    lib.metis_enum_device_groups.restype = C.c_int64
    lib.metis_enum_device_groups.argtypes = [C.c_int32, C.c_int32, C.c_double, C.c_int32, C.c_void_p, C.c_int64]
    lib.metis_enum_device_group_tables.restype = C.c_int64
    lib.metis_enum_device_group_tables.argtypes = [C.c_int32, C.c_int32, C.c_int32, C.c_double, C.c_int32, C.c_void_p,
                                                   C.c_void_p, C.c_int64]
    lib.metis_enum_compositions.restype = C.c_int64
    lib.metis_enum_compositions.argtypes = [C.c_int32, C.c_int32, C.c_int32, C.c_double, C.c_int32, C.c_void_p, C.c_void_p,
                                            C.c_int64, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p]
    lib.metis_generate_rows.restype = C.c_int
    lib.metis_generate_rows.argtypes = [C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p]
    lib.metis_sort_workspace_bytes.restype = C.c_int64
    lib.metis_sort_workspace_bytes.argtypes = [C.c_int64]
    lib.metis_sort_records.restype = C.c_int
    lib.metis_sort_records.argtypes = [C.c_void_p, C.c_int64, C.c_int32, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p]
    lib.metis_select_workspace_bytes.restype = C.c_int64
    lib.metis_select_workspace_bytes.argtypes = [C.c_int64, C.c_int64]
    lib.metis_select_records.restype = C.c_int
    lib.metis_select_records.argtypes = [C.c_void_p, C.c_int64, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p,
                                         C.c_int64, C.c_void_p]
    if lib.metis_abi_version() != 2:
        raise MetisNativeError('libmetis_b200.so ABI version mismatch; rebuild')
    if path == LIB_PATH:
        _lib = lib
    return lib


def check(rc: int, what: str) -> None:
    if rc != 0:
        msg = load_library().metis_last_error().decode(errors='replace')
        raise MetisNativeError(f'{what} failed (code {rc}): {msg}')
