"""CPU reference for unique(col): the oracle's materialize (its restatement of the reference's block iteration with the
selection stages) followed by Base.unique's first-appearance fold with isequal, in C (tests/native/unique_ref.c).

The shared object is compiled on first use into the system's temporary directory, keyed by the source's hash, so that
neither the tests nor scripts/unique_bench.py write into the source tree."""
import ctypes as C
import hashlib
import os
import subprocess
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
SRC = os.path.join(HERE, "native", "unique_ref.c")
KINDS = {"Float16": 11, "Float32": 12, "Float64": 13}
_LIB = None


def lib():
    global _LIB
    if _LIB is None:
        src = open(SRC, "rb").read()
        so = os.path.join(tempfile.gettempdir(), f"dfdb_unique_ref_{os.getuid()}_{hashlib.sha256(src).hexdigest()[:16]}.so")
        if not os.path.exists(so):
            tmp = f"{so}.{os.getpid()}"
            subprocess.run(["gcc", "-O2", "-std=c11", "-Wall", "-shared", "-fPIC", "-o", tmp, SRC], check=True)
            os.replace(tmp, so)
        L = C.CDLL(so)
        L.uref_fixed.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int64, C.c_void_p]
        L.uref_fixed.restype = C.c_int64
        L.uref_strings.argtypes = [C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p]
        L.uref_strings.restype = C.c_int64
        L.uref_take_strings.argtypes = [C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_int64, C.c_void_p]
        L.uref_take_strings.restype = None
        _LIB = L
    return _LIB


def unique_column(col, typename=None):
    """unique over one column as OracleTable.materialize returns it: ndarray | (values, missing) | FlatStrings.
    Returns the same kind of object holding the distinct values in order of first appearance."""
    from oracle import oracle as O
    L = lib()
    if isinstance(col, O.FlatStrings):
        sizes = np.ascontiguousarray(col.sizes, dtype=np.int32)
        chars = np.frombuffer(col.chars, dtype=np.uint8) if len(col.chars) else np.zeros(1, np.uint8)
        idx = np.zeros(max(len(sizes), 1), dtype=np.int64)
        m = L.uref_strings(sizes.ctypes.data, chars.ctypes.data, len(sizes), idx.ctypes.data)
        assert m >= 0, "out of memory"
        idx = idx[:m]
        keep = sizes[idx]
        out = np.zeros(max(int(np.maximum(keep, 0).sum()), 1), dtype=np.uint8)
        L.uref_take_strings(sizes.ctypes.data, chars.ctypes.data, len(sizes), idx.ctypes.data, m, out.ctypes.data)
        return O.FlatStrings(keep.copy(), out[:int(np.maximum(keep, 0).sum())].tobytes())
    vals, miss = col if isinstance(col, tuple) else (col, None)
    vals = np.ascontiguousarray(vals)
    kind = KINDS.get(typename or vals.dtype.name.capitalize(), 0)
    m8 = np.ascontiguousarray(miss, dtype=np.uint8) if miss is not None else None
    idx = np.zeros(max(len(vals), 1), dtype=np.int64)
    m = L.uref_fixed(vals.ctypes.data, m8.ctypes.data if m8 is not None else None, vals.dtype.itemsize, kind, len(vals), idx.ctypes.data)
    assert m >= 0, "out of memory"
    idx = idx[:m]
    return (vals[idx], np.asarray(miss, dtype=bool)[idx]) if miss is not None else vals[idx]


def unique(ot, plan: bytes, proj_idx: int = 0):
    """unique(col) of projection `proj_idx` of `plan` on the oracle table `ot`."""
    return unique_column(ot.materialize(plan)[proj_idx])
