"""ctypes binding of libimm3gpu.so — exactly the symbols declared in include/imm3.h.

There is no Python or CPU implementation behind these names: if the shared library is missing the
import fails loudly (build it with `python -m immutable3_b200._build`, which needs nvcc).
"""
from __future__ import annotations

import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("IMM3_LIB") or os.path.join(HERE, "libimm3gpu.so")  # IMM3_LIB: experiment builds

OK = 0
ERR_NOT_FOUND, ERR_UNSUPPORTED, ERR_BAD_FORMAT, ERR_CUDA, ERR_OOM, ERR_INVALID_ARG, ERR_IO, ERR_STATE, ERR_COMM = range(-1, -10, -1)
COMM_HANDLE_BYTES = 64
COL_INT, COL_TINYINT, COL_STRING, COL_COUNT, COL_DOUBLE, COL_INT64 = 0, 1, 2, 3, 4, 5
AGG_FLAG_GLOBAL = 0x1  # IMM3_AGG_GLOBAL
AGG_FLAG_ENCODED_FILTER = 0x4  # IMM3_AGG_ENCODED_FILTER
DNF_FLAG_ENCODED_FILTER = 0x4  # IMM3_DNF_ENCODED_FILTER
AGG_COUNT, AGG_MIN, AGG_MAX, AGG_SUM, AGG_AVG = 0, 1, 2, 3, 4
CODEC_PFOR_INT, CODEC_DENSE_INT, CODEC_DENSE_TINYINT, CODEC_DENSE_STRING = 0, 1, 2, 3
OP_GT, OP_LT, OP_EQ, OP_MATCH, OP_NOTMATCH, OP_NOOP = 1, 2, 3, 4, 5, 6
OPEN_HOST_ONLY, OPEN_KEEP_HOST, OPEN_NO_TMA, OPEN_FORCE_BLOCKS, OPEN_NO_STATS = 1, 2, 4, 8, 16


class Pred(C.Structure):
    _fields_ = [("col", C.c_char_p), ("op", C.c_int32), ("num", C.c_double),
                ("strs", C.POINTER(C.c_char_p)), ("nstrs", C.c_int32)]


class Agg(C.Structure):
    _fields_ = [("col", C.c_char_p), ("op", C.c_int32)]


class OpenOpts(C.Structure):
    _fields_ = [("device", C.c_int32), ("rank", C.c_int32), ("world", C.c_int32), ("flags", C.c_uint32)]


class TableDesc(C.Structure):
    _fields_ = [("ncols", C.c_int32), ("block_size", C.c_int32), ("nsegments", C.c_int32), ("seg_begin", C.c_int32),
                ("seg_end", C.c_int32), ("nrows", C.c_int64), ("nblocks", C.c_int64), ("resident_bytes", C.c_int64)]


class ColumnDesc(C.Structure):
    _fields_ = [("name", C.c_char * 64), ("column_type", C.c_int32), ("codec", C.c_int32), ("width", C.c_int32),
                ("reserved", C.c_int32), ("encoded_bytes", C.c_int64)]


# name -> (restype, argtypes); kept in one table so tests can check it against include/imm3.h
_P = C.c_void_p
_PP = C.POINTER(C.c_void_p)
_STRS = C.POINTER(C.c_char_p)
SIGNATURES = {
    "imm3_open": (C.c_int, [C.c_char_p, C.POINTER(OpenOpts), _PP]),
    "imm3_close": (C.c_int, [_P]),
    "imm3_table_count": (C.c_int, [_P]),
    "imm3_table_name": (C.c_char_p, [_P, C.c_int]),
    "imm3_table_info": (C.c_int, [_P, C.c_char_p, C.POINTER(TableDesc)]),
    "imm3_column_info": (C.c_int, [_P, C.c_char_p, C.c_int, C.POINTER(ColumnDesc)]),
    "imm3_segment_file_id": (C.c_int, [_P, C.c_char_p, C.c_int, C.POINTER(C.c_int32)]),
    "imm3_reupload": (C.c_int, [_P, C.c_char_p, _STRS, C.c_int, C.POINTER(C.c_int64)]),
    "imm3_set_stream": (C.c_int, [_P, _P]),
    "imm3_sync": (C.c_int, [_P]),
    "imm3_query": (C.c_int, [_P, C.c_char_p, C.POINTER(Pred), C.c_int, _STRS, C.c_int, C.c_int64, _PP]),
    "imm3_query_begin": (C.c_int, [_P, C.c_char_p, C.POINTER(Pred), C.c_int, _STRS, C.c_int, C.c_int64, _PP]),
    "imm3_query_begin_dnf": (C.c_int, [_P, C.c_char_p, C.POINTER(Pred), C.POINTER(C.c_int32), C.c_int, _STRS, C.c_int, C.c_int64, _PP]),
    "imm3_query_begin_dnf_ext": (C.c_int, [_P, C.c_char_p, C.POINTER(Pred), C.POINTER(C.c_int32), C.c_int, _STRS, C.c_int, C.c_int64, C.c_uint32, _PP]),
    "imm3_result_local_count": (C.c_int64, [_P]),
    "imm3_comm_local_handle": (C.c_int, [_P, _P]),
    "imm3_comm_connect": (C.c_int, [_P, _P, C.c_int]),
    "imm3_result_global_offset": (C.c_int64, [_P]),
    "imm3_result_take": (C.c_int64, [_P]),
    "imm3_result_global_count": (C.c_int64, [_P]),
    "imm3_result_rank_counts": (C.c_int, [_P, C.POINTER(C.c_int64), C.c_int]),
    "imm3_result_fetch": (C.c_int, [_P, C.c_int64]),
    "imm3_result_fetch_async": (C.c_int, [_P, C.c_int64]),
    "imm3_result_wait": (C.c_int, [_P]),
    "imm3_query_agg": (C.c_int, [_P, C.c_char_p, C.POINTER(Pred), C.c_int, C.POINTER(Agg), C.c_int, _STRS, C.c_int, _PP]),
    "imm3_query_agg_global": (C.c_int, [_P, C.c_char_p, C.POINTER(Pred), C.c_int, C.POINTER(Agg), C.c_int, _STRS, C.c_int, _PP]),
    "imm3_query_agg_ext": (C.c_int, [_P, C.c_char_p, C.POINTER(Pred), C.c_int, C.POINTER(Agg), C.c_int, _STRS, C.c_int, C.c_uint32, _PP]),
    "imm3_query_sql": (C.c_int, [_P, C.c_char_p, _PP]),
    "imm3_result_nrows": (C.c_int64, [_P]),
    "imm3_result_ncols": (C.c_int, [_P]),
    "imm3_result_col_type": (C.c_int, [_P, C.c_int]),
    "imm3_result_col_width": (C.c_int, [_P, C.c_int]),
    "imm3_result_col_name": (C.c_char_p, [_P, C.c_int]),
    "imm3_result_col_data": (_P, [_P, C.c_int]),
    "imm3_result_col_device": (_P, [_P, C.c_int]),
    "imm3_result_format_row": (C.c_int, [_P, C.c_int64, C.c_char_p, C.c_size_t]),
    "imm3_result_device_ms": (C.c_double, [_P]),
    "imm3_result_kernel_launches": (C.c_int, [_P]),
    "imm3_result_route": (C.c_char_p, [_P]),
    "imm3_result_stage_ms": (C.c_double, [_P, C.c_int]),
    "imm3_result_host_us": (C.c_double, [_P, C.c_int]),
    "imm3_result_algorithmic_bytes": (C.c_int64, [_P]),
    "imm3_result_free": (C.c_int, [_P]),
    "imm3_filter_bitmap": (C.c_int, [_P, C.c_char_p, C.POINTER(Pred), C.c_int, C.POINTER(C.POINTER(C.c_uint32)),
                                     C.POINTER(C.c_int64), C.POINTER(C.c_int64)]),
    "imm3_explain": (C.c_int, [_P, C.c_char_p, C.POINTER(Pred), C.c_int, _STRS, C.c_int, C.c_int64, C.POINTER(C.c_char_p)]),
    "imm3_writer_open": (C.c_int, [C.c_char_p, C.c_char_p, _STRS, C.c_int, C.c_int32, C.c_int32, C.c_int32, C.c_int, _PP]),
    "imm3_writer_append": (C.c_int, [_P, C.POINTER(C.c_void_p), C.c_int64]),
    "imm3_writer_append_csv_line": (C.c_int, [_P, C.c_char_p]),
    "imm3_writer_close": (C.c_int, [_P]),
    "imm3_load_csv": (C.c_int, [C.c_char_p, C.c_char_p, _STRS, C.c_int, C.c_int32, C.c_int32, C.c_char_p]),
    "imm3_pfor_encode": (C.c_int64, [C.POINTER(C.c_int32), C.c_int32, C.POINTER(C.c_uint8), C.c_int64]),
    "imm3_pfor_encode_blocks_gpu": (C.c_int64, [C.c_int, C.POINTER(C.c_int32), C.c_int64, C.c_int32, C.POINTER(C.c_uint8), C.c_int64,
                                    C.POINTER(C.c_int64)]),
    "imm3_synth_write": (C.c_int, [C.c_char_p, C.c_char_p, C.c_int64, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int]),
    "imm3_synth_row": (None, [C.c_int64, C.POINTER(C.c_int32), C.POINTER(C.c_int8), C.c_char_p]),
    "imm3_last_error": (C.c_char_p, []),
    "imm3_abi_version": (C.c_int, []),
}

_lib = None


def lib() -> C.CDLL:
    """Load libimm3gpu.so (once).  Raises if it has not been built — never falls back."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(
                f"{LIB_PATH} is missing: the CUDA extension has not been built "
                "(run `python -m immutable3_b200._build`); immutable3_b200 has no CPU fallback")
        handle = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(handle, name)  # AttributeError if the library does not export a declared symbol
            fn.restype = res
            fn.argtypes = args
        _lib = handle
    return _lib


class Imm3Error(RuntimeError):
    """Non-zero imm3_status; `.status` holds the code, the message comes from imm3_last_error()."""

    def __init__(self, status: int, message: str):
        super().__init__(f"[imm3 status {status}] {message}")
        self.status = status
        self.message = message


def check(status: int) -> int:
    if status < 0:
        raise Imm3Error(status, (lib().imm3_last_error() or b"").decode("utf-8", "replace"))
    return status


def cstr_array(items):
    arr = (C.c_char_p * max(1, len(items)))()
    for i, s in enumerate(items):
        arr[i] = s.encode() if isinstance(s, str) else s
    return arr
