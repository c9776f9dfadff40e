"""ctypes binding of include/arrow_b200.h (the C-ABI drop-in boundary).

This is the Python-side equivalent of the stub a reference maintainer would add (see
INTEGRATION.md): plain pointers and sizes only.  There is NO fallback: if the CUDA
library is missing or no GPU is visible the import / first call raises.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "lib", "libarrow_b200.so")


class B2Array(C.Structure):
    _fields_ = [
        ("validity", C.c_void_p),
        ("data", C.c_void_p),
        ("data2", C.c_void_p),
        ("length", C.c_int64),
        ("offset", C.c_int64),
        ("null_count", C.c_int64),
        ("type", C.c_int32),
        ("byte_width", C.c_int32),
    ]


class B2Scalar(C.Structure):
    _fields_ = [("bits", C.c_uint64), ("type", C.c_int32), ("is_valid", C.c_int32)]


class B2Value(C.Structure):
    _fields_ = [("array", C.POINTER(B2Array)), ("scalar", C.POINTER(B2Scalar))]


class B2CastOptions(C.Structure):
    _fields_ = [
        ("to_type", C.c_int32),
        ("allow_int_overflow", C.c_int32),
        ("allow_float_truncate", C.c_int32),
        ("reserved", C.c_int32),
    ]


class B2HashAggOptions(C.Structure):
    _fields_ = [
        ("skip_nulls", C.c_int32),
        ("min_count", C.c_uint32),
        ("count_mode", C.c_int32),
        ("reserved", C.c_int32),
    ]


class B2ReduceResult(C.Structure):
    _fields_ = [
        ("count", C.c_int64),
        ("null_count", C.c_int64),
        ("sum_bits", C.c_uint64),
        ("min_bits", C.c_uint64),
        ("max_bits", C.c_uint64),
        ("dsum_bits", C.c_uint64),
        ("acc_type", C.c_int32),
        ("value_type", C.c_int32),
    ]


# status codes (arrow::StatusCode values)
OK, OUT_OF_MEMORY, KEY_ERROR, TYPE_ERROR, INVALID, IO_ERROR, CAPACITY_ERROR, INDEX_ERROR = range(8)
NOT_IMPLEMENTED = 10
CUDA_ERROR = 100

# type ids (arrow::Type::type values)
NA, BOOL, UINT8, INT8, UINT16, INT16, UINT32, INT32, UINT64, INT64, HALF_FLOAT, FLOAT, DOUBLE, STRING, BINARY, FIXED_SIZE_BINARY = range(16)
LARGE_STRING, LARGE_BINARY = 34, 35

ARITH_OPS = {
    "add": 0, "subtract": 1, "multiply": 2, "divide": 3,
    "add_checked": 16, "subtract_checked": 17, "multiply_checked": 18, "divide_checked": 19,
}
COMPARE_OPS = {"equal": 0, "not_equal": 1, "greater": 2, "greater_equal": 3, "less": 4, "less_equal": 5}
BOOLEAN_OPS = {"and": 0, "or": 1, "xor": 2, "and_not": 3, "and_kleene": 4, "or_kleene": 5, "and_not_kleene": 6, "invert": 7}
VALIDITY_OPS = {"is_valid": 0, "is_null": 1, "true_unless_null": 2, "is_nan": 3}
COMM_ID_BYTES = 128
HASH_AGG_KINDS = {"hash_sum": 0, "hash_count": 1, "hash_count_all": 2, "hash_mean": 3, "hash_min": 4,
                  "hash_max": 5, "hash_product": 6, "hash_any": 7, "hash_all": 8, "hash_count_distinct": 9}

# every symbol include/arrow_b200.h declares: (name, restype, argtypes)
_P = C.c_void_p
_A = C.POINTER(B2Array)
_V = C.POINTER(B2Value)
_I64P = C.POINTER(C.c_int64)
PROTOTYPES = [
    ("b2_context_create", C.c_int, [C.c_int, C.POINTER(_P)]),
    ("b2_context_destroy", None, [_P]),
    ("b2_context_device", C.c_int, [_P]),
    ("b2_context_stream", _P, [_P]),
    ("b2_context_set_allocator", C.c_int, [_P, _P, _P, _P]),
    ("b2_alloc", C.c_int, [_P, C.c_size_t, C.POINTER(_P)]),
    ("b2_free", C.c_int, [_P, _P]),
    ("b2_pool_stats", C.c_int, [_P, _I64P, _I64P, _I64P]),
    ("b2_pool_trim", C.c_int, [_P]),
    ("b2_sync", C.c_int, [_P, _P]),
    ("b2_memcpy_h2d", C.c_int, [_P, _P, _P, C.c_size_t, _P]),
    ("b2_memcpy_d2h", C.c_int, [_P, _P, _P, C.c_size_t, _P]),
    ("b2_memset", C.c_int, [_P, _P, C.c_int, C.c_size_t, _P]),
    ("b2_event_create", C.c_int, [_P, C.POINTER(_P)]),
    ("b2_event_destroy", C.c_int, [_P]),
    ("b2_event_record", C.c_int, [_P, _P, _P]),
    ("b2_event_synchronize", C.c_int, [_P]),
    ("b2_stream_wait_event", C.c_int, [_P, _P, _P]),
    ("b2_host_alloc", C.c_int, [C.c_size_t, C.POINTER(_P)]),
    ("b2_host_free", C.c_int, [_P]),
    ("b2_last_error", C.c_char_p, []),
    ("b2_version", C.c_char_p, []),
    ("b2_launch_count", C.c_int64, []),
    ("b2_bitmap_count", C.c_int, [_P, _P, C.c_int64, C.c_int64, _I64P, _P]),
    ("b2_bitmap_copy", C.c_int, [_P, _P, C.c_int64, C.c_int64, _P, _P]),
    ("b2_bitmap_and", C.c_int, [_P, _P, C.c_int64, _P, C.c_int64, C.c_int64, _P, _I64P, _P]),
    ("b2_cast_numeric", C.c_int, [_P, _A, C.POINTER(B2CastOptions), _A, _P]),
    ("b2_binary_arith", C.c_int, [_P, C.c_int, _V, _V, _A, _P]),
    ("b2_compare", C.c_int, [_P, C.c_int, _V, _V, _A, _P]),
    ("b2_filter_output_size", C.c_int, [_P, _A, C.c_int, _I64P, _P]),
    ("b2_filter", C.c_int, [_P, _A, _A, C.c_int, _A, _P]),
    ("b2_filter_indices", C.c_int, [_P, _A, C.c_int, _A, _P]),
    ("b2_take", C.c_int, [_P, _A, _A, C.c_int, _A, _P]),
    ("b2_take_cast_arith", C.c_int, [_P, _A, _A, C.c_int32, C.c_int, _V, _A, _P]),
    ("b2_binary_data_size", C.c_int, [_P, _A, _I64P, _P]),
    ("b2_sort_indices", C.c_int, [_P, _A, C.c_int, C.c_int, _A, _P]),
    ("b2_sort_payload", C.c_int, [_P, _A, _A, C.c_int, C.c_int, _A, _P]),
    ("b2_sort_indices_multi", C.c_int, [_P, _A, C.c_int, C.POINTER(C.c_int32), C.c_int, _A, _P]),
    ("b2_hash_join", C.c_int, [_P, _A, _A, C.c_int, C.c_int, _A, _A, _P]),
    ("b2_select_k", C.c_int, [_P, _A, C.c_int64, C.c_int, C.c_int, _A, _P]),
    ("b2_sort_strings_path", C.c_int, [_P, _A, C.POINTER(C.c_int32), _P]),
    ("b2_grouper_create", C.c_int, [_P, C.POINTER(C.c_int32), C.c_int, C.POINTER(_P)]),
    ("b2_grouper_destroy", None, [_P]),
    ("b2_grouper_consume", C.c_int, [_P, _A, _A, _P]),
    ("b2_grouper_lookup", C.c_int, [_P, _A, _A, _P]),
    ("b2_grouper_num_groups", C.c_int, [_P, C.POINTER(C.c_uint32)]),
    ("b2_grouper_uniques", C.c_int, [_P, _A, _P]),
    ("b2_grouper_reset", C.c_int, [_P]),
    ("b2_vector_hash", C.c_int, [_P, _A, C.c_int, _A, _A, _A, _P]),
    ("b2_reduce", C.c_int, [_P, _A, C.POINTER(B2ReduceResult), _P]),
    ("b2_hashagg_create", C.c_int, [_P, C.c_int, C.c_int32, C.POINTER(B2HashAggOptions), C.POINTER(_P)]),
    ("b2_hashagg_destroy", None, [_P]),
    ("b2_hashagg_resize", C.c_int, [_P, C.c_int64, _P]),
    ("b2_hashagg_consume", C.c_int, [_P, _A, _A, _P]),
    ("b2_hashagg_merge", C.c_int, [_P, _P, _A, _P]),
    ("b2_hashagg_finalize", C.c_int, [_P, _A, _P]),
    ("b2_hashagg_out_type", C.c_int32, [_P]),
    ("b2_groupby_sumcount_create", C.c_int, [_P, C.c_int32, C.c_int32, C.c_int64, C.POINTER(_P)]),
    ("b2_groupby_sumcount_destroy", None, [_P]),
    ("b2_groupby_sumcount_consume", C.c_int, [_P, _A, _A, _P]),
    ("b2_groupby_sumcount_finalize", C.c_int, [_P, _A, _A, _A, _P]),
    ("b2_groupby_sumcount_merge", C.c_int, [_P, _A, _A, _A, _P]),
    ("b2_groupby_sumcount_path_counts", C.c_int, [_P, _I64P, _I64P, _I64P, _I64P]),
    ("b2_hash_partition", C.c_int, [_P, _A, C.c_int, _A, _P]),
    ("b2_range_partition", C.c_int, [_P, _A, _A, C.c_int, _A, _P]),
    ("b2_bincount", C.c_int, [_P, _A, C.c_int, _I64P, _P]),
    ("b2_range_split", C.c_int, [_P, _A, _A, C.c_int, C.c_uint64, _A, _A, _I64P, _P]),
    ("b2_boolean", C.c_int, [_P, C.c_int, _V, _V, _A, _P]),
    ("b2_validity", C.c_int, [_P, C.c_int, _A, C.c_int, _A, _P]),
    ("b2_if_else", C.c_int, [_P, _V, _V, _V, _A, _P]),
    ("b2_comm_unique_id", C.c_int, [_P]),
    ("b2_comm_init", C.c_int, [_P, C.c_int, C.c_int, _P, C.POINTER(_P)]),
    ("b2_comm_destroy", None, [_P]),
    ("b2_comm_rank", C.c_int, [_P]),
    ("b2_comm_world", C.c_int, [_P]),
    ("b2_comm_nccl_version", C.c_int, [C.POINTER(C.c_int)]),
    ("b2_comm_group_start", C.c_int, [_P]),
    ("b2_comm_group_end", C.c_int, [_P]),
    ("b2_comm_all_gather", C.c_int, [_P, _P, _P, C.c_int64, _P]),
    ("b2_comm_all_reduce_i64", C.c_int, [_P, _P, _P, C.c_int64, C.c_int, _P]),
    ("b2_comm_all_to_all_v", C.c_int, [_P, _P, _I64P, _I64P, _P, _I64P, _I64P, _P]),
]

_lib = None


class NativeLibraryMissing(ImportError):
    pass


def lib() -> C.CDLL:
    """Load libarrow_b200.so (built in-tree by __graft_entry__.build()).  Fails loudly."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise NativeLibraryMissing(
                f"{LIB_PATH} is missing: run `python -c 'import __graft_entry__ as g; g.build()'` "
                "(arrow_b200 has no CPU fallback)")
        _lib = C.CDLL(LIB_PATH, mode=C.RTLD_GLOBAL)
        for name, restype, argtypes in PROTOTYPES:
            fn = getattr(_lib, name)  # AttributeError if the symbol is not exported
            fn.restype = restype
            fn.argtypes = argtypes
    return _lib


def last_error() -> str:
    return lib().b2_last_error().decode("utf-8", "replace")
