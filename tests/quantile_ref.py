"""CPU model of median / quantile over a DFColumn: the oracle's materialize of the view (its restatement of the reference's
block iteration with the selection stages), missing values dropped, sorted by an isless key written here in numpy, then
Statistics.jl's formulas (default keywords: alpha = beta = 1), restated.

The key maps every value to a uint64 whose unsigned order is Julia's isless: unsigned and Bool values as they are, signed
values offset by 2^63, floats widened to Float64 (exact) with the sign bit set for positives and every bit flipped for
negatives, so -0.0 sorts before 0.0.  NaN is never sorted here: median returns NaN and quantile refuses it before."""
import math
from fractions import Fraction

import numpy as np


def isless_key(vals: np.ndarray) -> np.ndarray:
    if vals.dtype == np.bool_ or vals.dtype.kind == "u":
        return vals.astype(np.uint64)
    if vals.dtype.kind == "i":
        return vals.astype(np.int64).view(np.uint64) ^ np.uint64(1 << 63)
    u = vals.astype(np.float64).view(np.uint64)
    return np.where(u >> np.uint64(63) != 0, ~u, u | np.uint64(1 << 63))


def split(col):
    """(values, missing mask) of a materialized fixed-width column"""
    if isinstance(col, tuple):
        return col[0], col[1].astype(bool)
    return col, np.zeros(len(col), bool)


def sorted_values(col) -> np.ndarray:
    """the non-missing values of a materialized column in isless order"""
    vals, miss = split(col)
    v = vals[~miss]
    return v[np.argsort(isless_key(v), kind="stable")]


def order_stats(col, ranks) -> np.ndarray:
    s = sorted_values(col)
    return s[np.asarray(ranks, dtype=np.int64) - 1]


def _has_nan(v):
    return v.dtype.kind == "f" and bool(np.isnan(v).any())


def _f64(x):
    return float(int(x)) if x.dtype.kind in "iub" else float(x)


def median(col, skipmissing=False):
    """Statistics.median: ArgumentError (raised as ValueError) without rows, None with a missing value, NaN with a NaN, else
    middle(v[(n+1)÷2]) or middle(v[n÷2], v[n÷2+1]); middle(x) = Float64(x) for integers and Bool, x for floats;
    middle(x, y) = x/2 + y/2 in Float64 for integers and Bool, in the column's type for floats"""
    vals, miss = split(col)
    if len(vals) == 0:
        raise ValueError("empty")
    if miss.any() and not skipmissing:
        return None
    v = vals[~miss]
    if len(v) == 0:
        raise ValueError("empty")
    if _has_nan(v):
        return v.dtype.type(np.nan)
    s = v[np.argsort(isless_key(v), kind="stable")]
    n = len(s)
    if v.dtype.kind == "f":
        return s[(n - 1) // 2] if n % 2 else s[n // 2 - 1] / v.dtype.type(2) + s[n // 2] / v.dtype.type(2)
    return _f64(s[(n - 1) // 2]) if n % 2 else _f64(s[n // 2 - 1]) / 2 + _f64(s[n // 2]) / 2


def _clamp(x, lo, hi):
    # Julia: ifelse(x > hi, hi, ifelse(x < lo, lo, x))
    if x > hi:
        return hi
    return lo if x < lo else x


def _isapprox(a, b):
    """isapprox(a, b) with default tolerances: rtol = sqrt(eps(T)) in T for floats, 0 (so ==) for integers and Bool"""
    if a.dtype.kind != "f":
        return int(a) == int(b)
    if a == b:
        return True
    rtol = np.sqrt(np.finfo(a.dtype).eps).astype(a.dtype)
    return bool(np.isfinite(a) and np.isfinite(b) and abs(a - b) <= rtol * max(abs(a), abs(b)))


def quantile_sorted(s: np.ndarray, p: float) -> float:
    """Statistics._quantile(v, p) on sorted values v (n >= 1), alpha = beta = 1"""
    n = len(s)
    aleph = float(Fraction(n) * Fraction(p) + Fraction(1.0 - p))      # fma(n, p, 1 - p): one rounding
    j = _clamp(math.trunc(aleph), 1, n - 1)
    g = _clamp(aleph - j, 0.0, 1.0)
    a, b = (s[0], s[0]) if n == 1 else (s[j - 1], s[j])
    fin = a.dtype.kind != "f" or bool(np.isfinite(a) and np.isfinite(b))
    if fin and _isapprox(a, b):
        d = (b - a) if a.dtype.kind == "f" else 0      # (a == b for integers: b - a is 0 and cannot overflow)
        return _f64(a) + g * float(d)
    return (1 - g) * _f64(a) + g * _f64(b)


def quantile(col, p, skipmissing=False):
    """Statistics.quantile(col, p): a Float64 per p; ValueError where Statistics throws ArgumentError"""
    ps = [float(x) for x in np.atleast_1d(np.asarray(p, dtype=np.float64))]
    if any(not (0.0 <= x <= 1.0) for x in ps):
        raise ValueError("p out of range")
    vals, miss = split(col)
    v = vals[~miss] if skipmissing else vals
    if len(v) == 0 or (miss.any() and not skipmissing) or _has_nan(v):
        raise ValueError("empty, missing or NaN")
    s = v[np.argsort(isless_key(v), kind="stable")]
    out = [quantile_sorted(s, x) for x in ps]
    return out[0] if np.ndim(p) == 0 else out
