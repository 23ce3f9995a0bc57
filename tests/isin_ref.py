"""Exact model of Julia's `in.(x, Ref(C))`, written from Base's definitions (not from the library):

- `in(x, itr)` for a vector or tuple is `any(y -> x == y, itr)` under three-valued logic: `true` on the first `y` with
  `x == y`, otherwise `missing` if some comparison was `missing` (x missing and C not empty, or `missing` in C), else `false`.
- `in(x, s::Set)` is `haskey(s.dict, x)`: `isequal(x, y)` for some `y`, a `Bool`.
- `==` between numbers is exact across types (`1 == 1.0 == true`, `0.0 == -0.0`, NaN equals nothing); a String equals only a
  String with the same bytes, never a number.
- `isequal` is `==`, except that NaN is isequal to NaN, `missing` to `missing`, and the sign bits of two numbers must agree
  (`isequal(-0.0, 0.0)` and `isequal(0, -0.0)` are false; an integer's sign bit is its sign).

Values are Python values: None (missing), bool, int, float (Float32 values widened exactly), str.  Python compares int and
float exactly, which is Julia's `==` on numbers.
"""
import math

import numpy as np


def _signbit(v) -> bool:
    return math.copysign(1.0, v) < 0 if isinstance(v, float) else v < 0


def jl_eq(x, y) -> bool:
    """x == y for non-missing x, y"""
    if isinstance(x, str) or isinstance(y, str):
        return isinstance(x, str) and isinstance(y, str) and x == y
    return x == y


def jl_isequal(x, y) -> bool:
    """isequal(x, y) for non-missing x, y"""
    if isinstance(x, str) or isinstance(y, str):
        return jl_eq(x, y)
    xn, yn = isinstance(x, float) and x != x, isinstance(y, float) and y != y
    if xn or yn:
        return xn and yn
    if isinstance(x, float) or isinstance(y, float):
        return _signbit(x) == _signbit(y) and x == y
    return x == y


def isin(x, values, isequal: bool):
    """in(x, Ref(C)): True / False, or None for missing"""
    if isequal:
        if x is None:
            return any(y is None for y in values)
        return any(y is not None and jl_isequal(x, y) for y in values)
    if x is None:
        return None if len(values) else False
    saw_missing = False
    for y in values:
        if y is None:
            saw_missing = True
        elif jl_eq(x, y):
            return True
    return None if saw_missing else False


def isin_column(col, values, isequal: bool):
    """the model over a list of row values, one evaluation per distinct value (keyed by type and bits: 0.0 / -0.0 and NaN
    payloads stay apart)"""
    cache = {}
    out = []
    for x in col:
        key = (type(x), np.float64(x).tobytes()) if isinstance(x, float) else (type(x), x)
        r = cache.get(key, cache)
        if r is cache:
            r = cache[key] = isin(x, values, isequal)
        out.append(r)
    return out


def eltype_nullable(x_nullable: bool, values, isequal: bool) -> bool:
    """whether in.(x, Ref(C)) has eltype Union{Bool, Missing}"""
    return not isequal and (x_nullable or any(v is None for v in values))


def as_list(col):
    """an oracle / library result column as Python values (None = missing)"""
    if hasattr(col, "tolist") and not isinstance(col, (np.ndarray, np.ma.MaskedArray)):
        return col.tolist()                               # strings
    if isinstance(col, tuple):
        vals, miss = col
        return [None if m else v for v, m in zip(np.asarray(vals).tolist(), np.asarray(miss).tolist())]
    if isinstance(col, np.ma.MaskedArray):
        return [None if m else v for v, m in zip(np.ma.getdata(col).tolist(), np.ma.getmaskarray(col).tolist())]
    return np.asarray(col).tolist()
