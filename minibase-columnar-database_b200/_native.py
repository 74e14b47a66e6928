"""ctypes binding of libmbcol.so (include/mbcol.h).

This is the Python stand-in for the Panama FFM / JNI stub a Java maintainer would write
(INTEGRATION.md).  There is no CPU fallback: if the shared library is missing the import
fails loudly, and ``mbc_init`` fails when no sm_100 GPU is present.
"""
from __future__ import annotations

import ctypes as C
import os
import re

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("MBC_LIB_PATH") or os.path.join(_HERE, "csrc", "libmbcol.so")   # override: tuning variants only
HEADER_PATH = os.path.join(os.path.dirname(_HERE), "include", "mbcol.h")

# ---- constants (mirrors of the #defines in mbcol.h) ------------------------------------------
MBC_OK = 0
ATTR_STRING, ATTR_INTEGER, ATTR_REAL, ATTR_SYMBOL = 0, 1, 2, 3
OP_EQ, OP_LT, OP_GT, OP_NE, OP_LE, OP_GE, OP_NOT, OP_NOP, OP_RANGE = range(9)
OPERAND_LITERAL, OPERAND_OUTER, OPERAND_INNER = 0, 1, 2
WANT_POSITIONS, WANT_COLUMNS, WANT_TUPLES, WANT_AGG, WANT_BITMAP, WANT_HOST = 1, 2, 4, 8, 16, 32
AGG_COUNT, AGG_SUM, AGG_MIN, AGG_MAX = 0, 1, 2, 3
ERR_ARG, ERR_CUDA, ERR_NODEVICE, ERR_UNSUPPORTED, ERR_FORMAT, ERR_NOINDEX = -1, -2, -3, -4, -5, -6
BITMAP_NONE, BITMAP_DENSE, BITMAP_SPARSE = 0, 1, 2


class mbc_coldesc(C.Structure):
    _fields_ = [("type", C.c_int32), ("width", C.c_int32)]


class mbc_operand(C.Structure):
    _fields_ = [("kind", C.c_int32), ("type", C.c_int32), ("col", C.c_int32), ("lit_i", C.c_int32),
                ("lit_f", C.c_float), ("lit_slen", C.c_int32), ("lit_s", C.POINTER(C.c_uint8))]


class mbc_term(C.Structure):
    _fields_ = [("op", C.c_int32), ("conj_id", C.c_int32), ("lhs", mbc_operand), ("rhs", mbc_operand)]


class mbc_aggspec(C.Structure):
    _fields_ = [("kind", C.c_int32), ("col", C.c_int32)]


class mbc_projspec(C.Structure):
    _fields_ = [("rel", C.c_int32), ("col", C.c_int32)]


class MbcError(RuntimeError):
    """A non-zero status from libmbcol.so (the Java shim would rethrow a ChainException)."""

    def __init__(self, status: int, message: str):
        super().__init__(f"libmbcol status {status}: {message}")
        self.status = status
        self.message = message


_VP = C.c_void_p
_SIGNATURES = {
    "mbc_init": (C.c_int32, [C.c_int32, C.POINTER(_VP)]),
    "mbc_shutdown": (None, [_VP]),
    "mbc_set_stream": (C.c_int32, [_VP, _VP]),
    "mbc_sync": (C.c_int32, [_VP]),
    "mbc_last_error": (C.c_char_p, []),
    "mbc_abi_version": (C.c_int32, []),
    "mbc_host_alloc": (C.c_int32, [C.POINTER(_VP), C.c_int64]),
    "mbc_host_free": (None, [_VP]),
    "mbc_kernel_launches": (C.c_int64, [_VP]),
    "mbc_h2d_bytes": (C.c_int64, [_VP]),
    "mbc_last_kernel_ms": (C.c_float, [_VP]),
    "mbc_table_create": (C.c_int32, [_VP, C.c_int32, C.POINTER(mbc_coldesc), C.c_int64, C.c_int64, C.POINTER(_VP)]),
    "mbc_table_free": (None, [_VP]),
    "mbc_table_nrows": (C.c_int64, [_VP]),
    "mbc_table_ncols": (C.c_int32, [_VP]),
    "mbc_table_coldesc": (C.c_int32, [_VP, C.c_int32, C.POINTER(mbc_coldesc)]),
    "mbc_table_load_column": (C.c_int32, [_VP, C.c_int32, _VP, C.c_int64]),
    "mbc_table_read_column": (C.c_int32, [_VP, C.c_int32, _VP, C.c_int64]),
    "mbc_table_column_device": (C.c_int32, [_VP, C.c_int32, C.POINTER(_VP), C.POINTER(C.c_int32)]),
    "mbc_table_generate": (C.c_int32, [_VP, C.c_int32, C.c_int32, C.c_uint64, C.c_int64]),
    "mbc_table_ingest_dbfile": (C.c_int32, [_VP, _VP, C.c_int64, C.c_char_p, C.POINTER(_VP)]),
    "mbc_table_set_deleted": (C.c_int32, [_VP, _VP, C.c_int64]),
    "mbc_scan": (C.c_int32, [_VP, C.POINTER(mbc_term), C.c_int32, C.POINTER(C.c_int32), C.c_int32, C.c_uint32,
                             C.POINTER(mbc_aggspec), C.c_int32, C.POINTER(_VP)]),
    "mbc_scan_host": (C.c_int32, [_VP, C.c_int32, C.POINTER(mbc_coldesc), C.POINTER(_VP), C.c_int64, C.c_int64,
                                  C.POINTER(mbc_term), C.c_int32, C.POINTER(C.c_int32), C.c_int32, C.c_uint32,
                                  C.POINTER(mbc_aggspec), C.c_int32, C.POINTER(_VP)]),
    "mbc_bitmap_build": (C.c_int32, [_VP, C.c_int32]),
    "mbc_bitmap_exists": (C.c_int32, [_VP, C.c_int32]),
    "mbc_bitmap_values": (C.c_int32, [_VP, C.c_int32, C.POINTER(_VP), C.POINTER(C.c_int64)]),
    "mbc_bitmap_get": (C.c_int32, [_VP, C.c_int32, _VP, _VP, C.c_int64]),
    "mbc_bitmap_layout": (C.c_int32, [_VP, C.c_int32, C.POINTER(C.c_int64)]),
    "mbc_bitmap_scan": (C.c_int32, [_VP, C.POINTER(mbc_term), C.c_int32, C.POINTER(C.c_int32), C.c_int32, C.c_uint32,
                                    C.POINTER(mbc_aggspec), C.c_int32, C.POINTER(_VP)]),
    "mbc_bitmap_join": (C.c_int32, [_VP, _VP, _VP, _VP, C.POINTER(mbc_term), C.c_int32, C.POINTER(mbc_projspec),
                                    C.c_int32, C.c_uint32, C.POINTER(mbc_aggspec), C.c_int32, C.POINTER(_VP)]),
    "mbc_sort": (C.c_int32, [_VP, C.POINTER(C.c_int32), C.c_int32, C.c_int32, C.POINTER(C.c_int32), C.c_int32, C.c_uint32, C.POINTER(_VP)]),
    "mbc_group_aggregate": (C.c_int32, [_VP, C.POINTER(mbc_term), C.c_int32, C.POINTER(C.c_int32), C.c_int32,
                                        C.POINTER(mbc_aggspec), C.c_int32, C.c_uint32, C.POINTER(_VP)]),
    "mbc_topk": (C.c_int32, [_VP, C.POINTER(mbc_term), C.c_int32, C.POINTER(C.c_int32), C.c_int32, C.c_int32, C.c_int64,
                             C.POINTER(C.c_int32), C.c_int32, C.c_uint32, C.POINTER(_VP)]),
    "mbc_result_count": (C.c_int64, [_VP]),
    "mbc_result_kernel_ms": (C.c_float, [_VP]),
    "mbc_result_phase_ms": (C.c_int32, [_VP, C.POINTER(C.c_float)]),
    "mbc_result_positions": (_VP, [_VP]),
    "mbc_result_positions2": (_VP, [_VP]),
    "mbc_result_column": (_VP, [_VP, C.c_int32, C.POINTER(C.c_int32)]),
    "mbc_result_tuples": (_VP, [_VP, C.POINTER(C.c_int32)]),
    "mbc_result_agg": (C.c_int32, [_VP, C.c_int32, C.POINTER(C.c_int64), C.POINTER(C.c_double), C.POINTER(C.c_int32)]),
    "mbc_result_group_agg": (C.c_int32, [_VP, C.c_int32, C.POINTER(_VP), C.POINTER(_VP)]),
    "mbc_result_bitmap": (_VP, [_VP, C.POINTER(C.c_int64)]),
    "mbc_result_device": (C.c_int32, [_VP, C.POINTER(_VP), C.POINTER(_VP), C.POINTER(_VP), C.POINTER(_VP)]),
    "mbc_result_column_device": (C.c_int32, [_VP, C.c_int32, C.POINTER(_VP), C.POINTER(C.c_int32)]),
    "mbc_result_free": (None, [_VP]),
    "mbc_init_devices": (C.c_int32, [C.c_int32, C.POINTER(C.c_int32), C.POINTER(_VP)]),
    "mbc_shard_create": (C.c_int32, [_VP, C.c_int32, C.c_int32, C.POINTER(_VP)]),
    "mbc_shard_free": (None, [_VP]),
    "mbc_shard_window_create": (C.c_int32, [_VP, C.c_int64, C.c_int32, C.POINTER(C.c_int32), C.POINTER(C.c_uint8)]),
    "mbc_shard_window_open": (C.c_int32, [_VP, C.POINTER(C.c_uint8), C.c_int64, C.c_int32, C.POINTER(C.c_int32)]),
    "mbc_shard_window_attach": (C.c_int32, [_VP, _VP]),
    "mbc_shard_gather": (C.c_int32, [_VP, _VP, C.c_int32]),
    "mbc_shard_fence": (C.c_int32, [_VP]),
    "mbc_shard_push_ms": (C.c_float, [_VP]),
    "mbc_shard_collect": (C.c_int32, [_VP, C.POINTER(C.c_int64), C.POINTER(C.c_int64)]),
    "mbc_shard_agg": (C.c_int32, [_VP, C.c_int32, C.c_int32, C.c_int32, C.POINTER(C.c_int64), C.POINTER(C.c_double), C.POINTER(C.c_int32)]),
    "mbc_shard_window_device": (C.c_int32, [_VP, C.POINTER(_VP), C.c_int32, C.POINTER(_VP)]),
    "mbc_shard_read": (C.c_int32, [_VP, C.c_int32, C.c_int64, C.c_int64, _VP]),
    "mbc_shard_release": (C.c_int32, [_VP]),
}
IPC_HANDLE_BYTES = 64


def header_functions(path: str = HEADER_PATH) -> list[str]:
    """Names of every function include/mbcol.h declares."""
    text = open(path).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(mbc_[a-z0-9_]+)\s*\(", text)))


_lib = None


def lib() -> C.CDLL:
    """Load libmbcol.so (once).  Missing library = hard error, never a fallback."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(make -C minibase-columnar-database_b200/csrc). There is no CPU fallback for this path.")
    handle = C.CDLL(LIB_PATH)
    for name, (restype, argtypes) in _SIGNATURES.items():
        fn = getattr(handle, name)      # AttributeError here = the library does not export the ABI
        fn.restype = restype
        fn.argtypes = argtypes
    _lib = handle
    return handle


def check(status: int) -> None:
    if status != MBC_OK:
        msg = lib().mbc_last_error()
        raise MbcError(status, msg.decode("utf-8", "replace") if msg else "")
