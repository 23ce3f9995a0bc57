"""ctypes binding of libdfdb_b200.so (include/dfdb_b200.h).

This is the Python twin of the `ccall` methods in julia/b200.jl / INTEGRATION.md.  There is
no CPU fallback: if the CUDA library is missing or no B200 is usable, every scan raises.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("DFDB_B200_LIB") or os.path.join(_HERE, "lib", "libdfdb_b200.so")   # override: diagnostics builds only
CSRC = os.path.join(_HERE, "csrc")

DFDB_OK = 0
ERR_IO, ERR_FORMAT, ERR_CORRUPT, ERR_ARGUMENT, ERR_UNSUPPORTED, ERR_KEY, ERR_DIVIDE, ERR_CUDA, ERR_NOMEM, ERR_STATE = range(1, 11)
NEED_EXCHANGE = 11
LOAD_HOST, LOAD_HBM, LOAD_DECODED = 0, 1, 2

KIND_NAMES = {1: "Int8", 2: "Int16", 3: "Int32", 4: "Int64", 5: "Int128", 6: "UInt8", 7: "UInt16", 8: "UInt32", 9: "UInt64",
              10: "UInt128", 11: "Float16", 12: "Float32", 13: "Float64", 14: "Bool", 15: "Char", 16: "String", 17: "Date",
              18: "DateTime", 19: "Time", 20: "Tuple"}


class Agg(C.Structure):
    _fields_ = [("count", C.c_int64), ("nmissing", C.c_int64), ("sum_i64", C.c_int64), ("sum_f64", C.c_double),
                ("sum_f64_lo", C.c_double), ("min_i64", C.c_int64), ("max_i64", C.c_int64), ("min_f64", C.c_double),
                ("max_f64", C.c_double), ("has_nan", C.c_int32), ("value_class", C.c_int32)]


class Zone(C.Structure):
    _fields_ = [("rows", C.c_int64), ("null_count", C.c_int64), ("min_i64", C.c_int64), ("max_i64", C.c_int64), ("min_f64", C.c_double),
                ("max_f64", C.c_double), ("has_value", C.c_int32), ("has_nan", C.c_int32)]


class OutCol(C.Structure):
    _fields_ = [("values", C.c_void_p), ("missing", C.c_void_p), ("str_sizes", C.c_void_p), ("str_chars", C.c_void_p)]


class DfdbError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(msg)
        self.code = code


SYMBOLS = {
    "dfdb_init": (C.c_int32, [C.c_int32]),
    "dfdb_shutdown": (C.c_int32, []),
    "dfdb_last_error": (C.c_char_p, []),
    "dfdb_set_stream": (C.c_int32, [C.c_void_p]),
    "dfdb_synchronize": (C.c_int32, []),
    "dfdb_kernel_launches": (C.c_int64, []),
    "dfdb_numa_node": (C.c_int32, []),
    "dfdb_set_option": (C.c_int32, [C.c_char_p, C.c_int64]),
    "dfdb_profile_enable": (C.c_int32, [C.c_int32]),
    "dfdb_profile_reset": (C.c_int32, []),
    "dfdb_profile_get": (C.c_int32, [C.c_char_p, C.POINTER(C.c_double), C.POINTER(C.c_int64), C.POINTER(C.c_int64)]),
    "dfdb_table_open": (C.c_int32, [C.c_char_p, C.POINTER(C.c_void_p)]),
    "dfdb_table_close": (C.c_int32, [C.c_void_p]),
    "dfdb_table_nrows": (C.c_int64, [C.c_void_p]),
    "dfdb_table_ncols": (C.c_int64, [C.c_void_p]),
    "dfdb_table_block_size": (C.c_int64, [C.c_void_p]),
    "dfdb_table_nblocks": (C.c_int64, [C.c_void_p]),
    "dfdb_table_column": (C.c_int32, [C.c_void_p, C.c_int32, C.POINTER(C.c_int64), C.c_char_p, C.c_int32, C.c_char_p, C.c_int32,
                                      C.POINTER(C.c_int32), C.POINTER(C.c_int32), C.POINTER(C.c_int32)]),
    "dfdb_table_column_stats": (C.c_int32, [C.c_void_p, C.c_int64, C.POINTER(C.c_int64), C.POINTER(C.c_int64)]),
    "dfdb_table_column_stored": (C.c_int32, [C.c_void_p, C.c_int64, C.POINTER(C.c_int64), C.POINTER(C.c_int64)]),
    "dfdb_table_set_shard": (C.c_int32, [C.c_void_p, C.c_int32, C.c_int32]),
    "dfdb_table_shard_range": (C.c_int32, [C.c_void_p, C.POINTER(C.c_int64), C.POINTER(C.c_int64), C.POINTER(C.c_int64), C.POINTER(C.c_int64)]),
    "dfdb_table_load": (C.c_int32, [C.c_void_p, C.POINTER(C.c_int64), C.c_int32, C.c_int32]),
    "dfdb_table_drop_decoded": (C.c_int32, [C.c_void_p]),
    "dfdb_table_build_zonemaps": (C.c_int32, [C.c_void_p, C.POINTER(C.c_int64), C.c_int32]),
    "dfdb_table_zonemap": (C.c_int32, [C.c_void_p, C.c_int64, C.c_int64, C.POINTER(Zone)]),
    "dfdb_scan_pruned": (C.c_int32, [C.c_void_p, C.POINTER(C.c_int64), C.POINTER(C.c_int64)]),
    "dfdb_scan_groupreduce": (C.c_int32, [C.c_void_p, C.POINTER(C.c_int32), C.c_int32, C.POINTER(C.c_int32), C.c_int32, C.POINTER(C.c_int64)]),
    "dfdb_scan_group_results": (C.c_int32, [C.c_void_p, C.c_void_p, C.c_void_p]),
    "dfdb_scan_group_key_bytes": (C.c_int32, [C.c_void_p, C.POINTER(C.c_int64)]),
    "dfdb_scan_group_keys": (C.c_int32, [C.c_void_p, C.POINTER(OutCol), C.c_int32]),
    "dfdb_scan_groupreduce_merge": (C.c_int32, [C.c_void_p, C.POINTER(C.c_int32), C.c_int32, C.c_int32, C.POINTER(OutCol), C.POINTER(C.c_int64),
                                                C.c_void_p, C.POINTER(C.c_int64), C.POINTER(C.c_int64), C.c_int32, C.POINTER(C.c_int64)]),
    "dfdb_scan_groupreduce_all": (C.c_int32, [C.c_void_p, C.POINTER(C.c_int32), C.c_int32, C.POINTER(C.c_int32), C.c_int32, C.POINTER(C.c_int64)]),
    "dfdb_scan_unique": (C.c_int32, [C.c_void_p, C.c_int32, C.POINTER(C.c_int64), C.POINTER(C.c_int64)]),
    "dfdb_scan_unique_values": (C.c_int32, [C.c_void_p, C.POINTER(OutCol)]),
    "dfdb_scan_unique_merge": (C.c_int32, [C.c_void_p, C.POINTER(OutCol), C.POINTER(C.c_int64), C.POINTER(C.c_int64), C.c_int32,
                                           C.POINTER(C.c_int64), C.POINTER(C.c_int64)]),
    "dfdb_scan_unique_all": (C.c_int32, [C.c_void_p, C.c_int32, C.POINTER(C.c_int64), C.POINTER(C.c_int64)]),
    "dfdb_host_alloc": (C.c_int32, [C.c_int64, C.POINTER(C.c_void_p)]),
    "dfdb_host_free": (C.c_int32, [C.c_void_p]),
    "dfdb_scan_prepare": (C.c_int32, [C.c_void_p, C.c_char_p, C.c_int64, C.POINTER(C.c_void_p)]),
    "dfdb_scan_free": (C.c_int32, [C.c_void_p]),
    "dfdb_scan_nproj": (C.c_int32, [C.c_void_p]),
    "dfdb_scan_proj_type": (C.c_int32, [C.c_void_p, C.c_int32, C.POINTER(C.c_int32), C.POINTER(C.c_int32), C.POINTER(C.c_int32)]),
    "dfdb_scan_count": (C.c_int32, [C.c_void_p, C.POINTER(C.c_int64)]),
    "dfdb_scan_aggregate": (C.c_int32, [C.c_void_p, C.c_int32, C.POINTER(Agg)]),
    "dfdb_scan_mask": (C.c_int32, [C.c_void_p, C.c_void_p, C.c_int64]),
    "dfdb_scan_indices": (C.c_int32, [C.c_void_p, C.c_void_p, C.c_int64, C.POINTER(C.c_int64)]),
    "dfdb_scan_materialize_sizes": (C.c_int32, [C.c_void_p, C.POINTER(C.c_int64), C.POINTER(C.c_int64)]),
    "dfdb_scan_materialize": (C.c_int32, [C.c_void_p, C.POINTER(OutCol), C.c_int32]),
    "dfdb_agg_fold": (C.c_int32, [C.POINTER(Agg), C.c_int32, C.POINTER(Agg)]),
    "dfdb_scan_exchange_count": (C.c_int32, [C.c_void_p, C.POINTER(C.c_int64), C.POINTER(C.c_int32)]),
    "dfdb_scan_exchange_offset": (C.c_int32, [C.c_void_p, C.c_int64]),
    "dfdb_scan_aggregate_device": (C.c_int32, [C.c_void_p, C.c_int32, C.c_void_p]),
    "dfdb_comm_unique_id": (C.c_int32, [C.c_void_p]),
    "dfdb_comm_init": (C.c_int32, [C.c_int32, C.c_int32, C.c_void_p]),
    "dfdb_comm_destroy": (C.c_int32, []),
    "dfdb_comm_info": (C.c_int32, [C.POINTER(C.c_int32), C.POINTER(C.c_int32)]),
    "dfdb_scan_aggregate_all": (C.c_int32, [C.c_void_p, C.c_int32, C.POINTER(Agg)]),
    "dfdb_scan_count_all": (C.c_int32, [C.c_void_p, C.POINTER(C.c_int64)]),
    "dfdb_scan_resolve_exchange": (C.c_int32, [C.c_void_p]),
    "dfdb_scan_row_offset_all": (C.c_int32, [C.c_void_p, C.POINTER(C.c_int64), C.POINTER(C.c_int64), C.POINTER(C.c_int64)]),
    "dfdb_write_column_file": (C.c_int32, [C.c_char_p, C.c_int64, C.c_char_p, C.c_int64, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                           C.c_int64, C.POINTER(C.c_int64), C.POINTER(C.c_int64)]),
    "dfdb_write_table_meta": (C.c_int32, [C.c_char_p, C.c_int64, C.c_int32, C.POINTER(C.c_int64), C.POINTER(C.c_char_p), C.POINTER(C.c_char_p)]),
    "dfdb_lz4_compress_blocks": (C.c_int32, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p]),
    "dfdb_lz4_decode_blocks": (C.c_int32, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p]),
    "dfdb_lz4_classify_block": (C.c_int32, [C.c_void_p, C.c_int64, C.c_int64]),
}

_lib = None
_inited_device = None


def build(force: bool = False) -> str:
    """Compile the CUDA library in-tree for sm_100a (nvcc cross-compiles without a GPU)."""
    srcs = [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".cu", ".cpp", ".hpp", ".cuh")) or f == "Makefile"]
    srcs.append(os.path.join(_HERE, "..", "include", "dfdb_b200.h"))
    if force or not os.path.exists(LIB_PATH) or any(os.path.getmtime(s) > os.path.getmtime(LIB_PATH) for s in srcs):
        subprocess.run(["make", "-C", CSRC, "-j4", "-s"], check=True)
    return LIB_PATH


def lib():
    """The loaded C ABI.  Raises if the library has not been built -- never falls back to a CPU path."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise DfdbError(ERR_CUDA, f"{LIB_PATH} is missing: run __graft_entry__.build() (no CPU fallback exists)")
        # dfdb_comm_* bind libnccl.so.2 at run time, and a process holds one libnccl.so.2.  torch links the NCCL it was built
        # with and fails to import next to an older one (such as the system's), so torch -- and its NCCL -- is loaded first.
        import torch  # noqa: F401
        L = C.CDLL(LIB_PATH)
        for name, (res, args) in SYMBOLS.items():
            fn = getattr(L, name)
            fn.restype = res
            fn.argtypes = args
        _lib = L
    return _lib


def check(rc: int):
    if rc != DFDB_OK:
        raise DfdbError(rc, lib().dfdb_last_error().decode("utf-8", "replace"))


def init(device: int | None = None):
    """One process per GPU: LOCAL_RANK (torchrun) selects the device unless given."""
    global _inited_device
    if device is None:
        device = int(os.environ.get("LOCAL_RANK", "0"))
    if _inited_device is None:
        check(lib().dfdb_init(device))
        _inited_device = device
    elif _inited_device != device:
        raise DfdbError(ERR_STATE, f"already initialised on device {_inited_device}")
    return _inited_device


class _PinnedBuffer:
    """A buffer of the library's result arena (dfdb_host_alloc): page-locked host memory that dfdb_scan_materialize
    fills with a direct device-to-host copy.  Goes back to the arena when the last numpy view of it dies."""

    def __init__(self, nbytes: int):
        p = C.c_void_p()
        check(lib().dfdb_host_alloc(nbytes, C.byref(p)))
        self.ptr, self.nbytes = p.value, nbytes
        self.__array_interface__ = {"shape": (nbytes,), "typestr": "|u1", "data": (self.ptr, False), "version": 3}

    def __del__(self):
        try:
            if self.ptr and _lib is not None:
                _lib.dfdb_host_free(C.c_void_p(self.ptr))
        except Exception:
            pass
        self.ptr = None


PINNED_MIN_BYTES = 1 << 20


def result_array(n: int, dtype) -> "np.ndarray":
    """Output vector for materialize: from the pinned result arena when it is large enough to matter."""
    import numpy as np
    dtype = np.dtype(dtype)
    nbytes = max(n, 1) * dtype.itemsize
    if nbytes < PINNED_MIN_BYTES:
        return np.zeros(max(n, 1), dtype=dtype)
    return np.asarray(_PinnedBuffer(nbytes)).view(dtype)
