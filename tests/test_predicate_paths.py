"""`column <cmp> constant` predicates against an exact model of Julia's comparisons, on every scan path and under zone maps.

The library implements such a predicate several times: the plan folds mixed-type comparisons into one exact integer or
double comparison (plan.cpp make_term); the fused scan evaluates the terms (scan_kernels.cu term_bits); the TMA scan folds
the conjunction into one closed interval per column (api.cu build_tma_args, scan_tma.cu test_bits); the zone maps decide
that a block holds no selected row (api.cu zone_prune); the expression VM runs whatever is left.  The model below evaluates
every row in plain Python: Python compares int with float exactly and NaN the IEEE way, as Julia does.  numpy is not used to
compare (it rounds Int64 to Float64 first: np.int64(2**53 + 1) == 2.0**53).

Coverage:
- the CPU test runs the whole predicate matrix through the oracle (mask, count, aggregate) against the model;
- the GPU test runs the whole matrix under the default options with zone maps on, and a seeded subset of
  `SUBSET` predicates per table under the default options with zone maps off and under each of no_tma / no_wide / no_fused
  with zone maps on and off;
- two block layouts: 256-row blocks, where every 8-byte column (the nullable ones too) can take the TMA scan, and
  960-row blocks, whose odd number of missing-bit words sends nullable columns to the fused scan.
"""
import ctypes as C
import math
import operator
import random
from contextlib import contextmanager

import numpy as np
import pytest

import dfdb_b200 as D
from dfdb_b200 import JType, R, _capi
from dfdb_b200.api import _bc

CODES = ["==", "!=", "<", "<=", ">", ">="]
OPS = {"==": operator.eq, "!=": operator.ne, "<": operator.lt, "<=": operator.le, ">": operator.gt, ">=": operator.ge}

F32_TENTH = float(np.float32(0.1))
INT_CONSTS = [0, 1, -1, 127, -127, 128, -128, -129, 255, 256, 32767, 32768, 65535, 65536, 2**31 - 1, 2**31, 2**32,
              2**53, -2**53, 2**53 + 1, -(2**53 + 1), 2**63 - 1, -2**63]
FLT_CONSTS = [0.0, -0.0, 0.5, -0.5, 127.5, 255.5, 2.0**53, 2.0**63, 9223372036854774784.0, -2.0**63, 2.0**64, 1e19,
              math.inf, -math.inf, math.nan, 5e-324, -5e-324, 0.1, F32_TENTH, 16777217.0]

# name, type string; every predicate column of every table
COLUMNS = [("i8", "Int8"), ("i16", "Int16"), ("i32", "Int32"), ("i64", "Int64"), ("u8", "UInt8"), ("u16", "UInt16"),
           ("u32", "UInt32"), ("u64", "UInt64"), ("f32", "Float32"), ("f64", "Float64"), ("b", "Bool"),
           ("mi64", "Missing(Int64)"), ("mu8", "Missing(UInt8)"), ("mf32", "Missing(Float32)"), ("mf64", "Missing(Float64)")]
# block rows, full blocks, rows of the ragged last block (an even number of missing-bit words in each 256-row block)
LAYOUTS = {"tma": (256, 16, 200), "odd": (960, 8, 500)}
# what block b of every column holds (index b % len(ROLES))
ROLES = ["single", "nan", "zeros", "eq_nan", "high", "window", "missing", "window_nan"]
SUBSET = 400

_NP = {"Int8": np.int8, "Int16": np.int16, "Int32": np.int32, "Int64": np.int64, "UInt8": np.uint8, "UInt16": np.uint16,
       "UInt32": np.uint32, "UInt64": np.uint64, "Float32": np.float32, "Float64": np.float64, "Bool": np.bool_}
_NAN64 = [0x7FF8000000000000, 0x7FF0000000000001, 0xFFF8000000000000, 0x7FFFFFFFFFFFFFFF, 0x7FF4000000000123]
_NAN32 = [0x7FC00000, 0x7F800001, 0xFFC00000, 0x7FFFFFFF, 0x7FA00123]


def _base(ts):
    return ts[8:-1] if ts.startswith("Missing(") else ts


def _int_range(base):
    info = np.iinfo(_NP[base])
    return int(info.min), int(info.max)


def _int_pool(base):
    lo, hi = _int_range(base)
    cand = {lo, lo + 1, hi - 1, hi, 0, 1, -1, 2, 5, 6}
    for c in INT_CONSTS:
        cand |= {c - 1, c, c + 1}
    return sorted(v for v in cand if lo <= v <= hi)


def _flt_pool(base):
    vals = [-math.inf, -1.7976931348623157e308, -1e19, -2.0**63, -2.0**53, -255.5, -1.0, -0.5, -5e-324, 0.0, 5e-324,
            F32_TENTH, 0.1, 0.5, 1.0, 127.5, 255.5, 16777216.0, 16777217.0, 2.0**53 - 1, 2.0**53, 2.0**53 + 2,
            9223372036854774784.0, 2.0**63, 1e19, 2.0**64, 1.7976931348623157e308, math.inf]
    if base == "Float32":
        with np.errstate(over="ignore"):               # (beyond Float32's range: the infinities)
            vals = [float(np.float32(v)) for v in vals] + [float(np.float32(1e-45)), float(np.float32(-1e-45))]
    return sorted(set(vals))


def _column_block(base, role, rows, rnd):
    """Python values (NaN as a (bits,) tuple) for one block of a column."""
    if base == "Bool":
        if role in ("single", "zeros"):
            return [False] * rows
        if role in ("nan", "high"):
            return [True] * rows
        return [rnd.random() < 0.5 for _ in range(rows)]
    if base.startswith("Float"):
        nans = _NAN32 if base == "Float32" else _NAN64
        pool = _flt_pool(base)
        if role == "single":
            return [0.5] * rows
        if role == "nan":
            return [(nans[rnd.randrange(len(nans))],) for _ in range(rows)]
        if role == "zeros":
            return [rnd.choice((0.0, -0.0)) for _ in range(rows)]
        if role == "eq_nan":
            out = [0.5] * rows
            out[rnd.randrange(rows)] = (nans[0],)
            return out
        if role == "high":
            big = [v for v in pool if abs(v) >= 2.0**53]
            return [rnd.choice(big) for _ in range(rows)]
        s = rnd.randrange(len(pool) - 3)
        win = pool[s:s + 4]
        out = []
        for _ in range(rows):
            if rnd.random() < 0.5 or not all(map(math.isfinite, (win[0], win[3]))):
                out.append(rnd.choice(win))
            else:
                out.append(float(np.float32(rnd.uniform(win[0], win[3]))) if base == "Float32" else rnd.uniform(win[0], win[3]))
        if role == "window_nan":
            out[rnd.randrange(rows)] = (nans[rnd.randrange(len(nans))],)
        return out
    lo, hi = _int_range(base)
    pool = _int_pool(base)
    if role == "single":
        v = pool[rnd.randrange(len(pool))]
        return [v] * rows
    if role == "nan":                                   # the type's extremes
        return [rnd.choice((lo, lo + 1, hi - 1, hi)) for _ in range(rows)]
    if role == "zeros":
        return [rnd.choice([v for v in (-1, 0, 1) if lo <= v <= hi]) for _ in range(rows)]
    if role == "high":                                  # UInt64: every value above 2^63
        a = max(lo, (hi + 1) // 2)
        return [rnd.randint(a, hi) if rnd.random() < 0.7 else rnd.choice((a, hi)) for _ in range(rows)]
    s = rnd.randrange(len(pool) - 3)
    win = pool[s:s + 4]
    return [rnd.choice(win) if rnd.random() < 0.5 else rnd.randint(win[0], win[3]) for _ in range(rows)]


def _to_numpy(base, vals):
    if base.startswith("Float"):
        bits = np.uint32 if base == "Float32" else np.uint64
        ftype = _NP[base]
        raw = np.array([v[0] if isinstance(v, tuple) else np.array(v, dtype=ftype).view(bits).item() for v in vals],
                       dtype=bits)
        return raw.view(ftype)
    return np.array(vals, dtype=_NP[base])


class Table:
    """One table on disk + the Python values the model reads (None = missing)."""

    def __init__(self, oracle, path, layout, seed):
        bs, nfull, last = LAYOUTS[layout]
        self.path, self.block_size = path, bs
        self.blocks = [(b * bs, b * bs + bs) for b in range(nfull)] + [(nfull * bs, nfull * bs + last)]
        self.nrows = nfull * bs + last
        rnd = random.Random(seed)
        cols, self.values, self.numpy = [], {}, {}
        for name, ts in COLUMNS:
            base = _base(ts)
            vals, miss = [], []
            for b, (lo, hi) in enumerate(self.blocks):
                role = ROLES[b % len(ROLES)]
                vals += _column_block(base, role, hi - lo, rnd)
                if ts.startswith("Missing("):
                    miss += [role == "missing" or (role.startswith("window") and rnd.random() < 0.25) for _ in range(hi - lo)]
            arr = _to_numpy(base, vals)
            if ts.startswith("Missing("):
                m = np.array(miss, dtype=bool)
                cols.append((name, ts, (arr, m)))
                self.numpy[name] = (arr, m)
            else:
                m = np.zeros(self.nrows, dtype=bool)
                cols.append((name, ts, arr))
                self.numpy[name] = (arr, None)
            py = arr.tolist() if not base.startswith("Float") else [float(x) for x in arr]
            if base == "Bool":
                py = [int(x) for x in py]
            self.values[name] = [None if mm else v for v, mm in zip(py, m.tolist())]
        # value columns of the aggregates: Int64 with the type's extremes, Float64 with signed zeros, NaN and infinities
        vi, vf = [], []
        for b, (lo, hi) in enumerate(self.blocks):
            role = ROLES[b % len(ROLES)]
            n = hi - lo
            vi += [rnd.randint(-10**6, 10**6) for _ in range(n)]
            if role == "nan":
                vi[lo] = -2**63
                vi[lo + 1] = 2**63 - 1
            blk = [rnd.gauss(0.0, 1000.0) for _ in range(n)]
            if role == "zeros":
                blk = [rnd.choice((0.0, -0.0)) for _ in range(n)]
            elif role == "nan":
                blk[rnd.randrange(n)] = math.nan
            elif role == "high":
                blk[rnd.randrange(n)] = math.inf
            elif role == "eq_nan":
                blk[rnd.randrange(n)] = -math.inf
            vf += blk
        cols += [("vi", "Int64", np.array(vi, dtype=np.int64)), ("vf", "Float64", np.array(vf, dtype=np.float64))]
        self.vi, self.vf = vi, vf
        oracle.write_table(path, cols, block_size=bs)


# ---- the model --------------------------------------------------------------------------------------------------------

def model_term(vals, code, c, const_first):
    """[bool per row] of coalesce(x <code> c, false) (or of c <code> x)."""
    f = OPS[code]
    cache = {}
    out = []
    for v in vals:
        if v is None:
            out.append(False)
            continue
        key = (v, math.copysign(1.0, v)) if isinstance(v, float) else v
        r = cache.get(key) if not (isinstance(v, float) and v != v) else None
        if r is None:
            r = bool(f(c, v) if const_first else f(v, c))
            if not (isinstance(v, float) and v != v):
                cache[key] = r
        out.append(r)
    return out


class Pred:
    """A conjunction of (column, code, constant, constant_first) terms."""

    def __init__(self, terms):
        self.terms = terms

    def __repr__(self):
        return " & ".join((f"{c!r} {code} {col}" if cf else f"{col} {code} {c!r}") for col, code, c, cf in self.terms)

    def expr(self, t):
        out = None
        for col, code, c, cf in self.terms:
            x = getattr(t, col)
            e = _bc(code, c, x) if cf else _bc(code, x, c)
            if x.eltype().nullable:
                e = D.coalesce(e, False)
            out = e if out is None else out & e
        return out

    def mask(self, tb):
        m = np.ones(tb.nrows, dtype=bool)
        for col, code, c, cf in self.terms:
            m &= np.array(model_term(tb.values[col], code, c, cf), dtype=bool)
        return m


def model_agg(tb, mask):
    """(count, int sum wrapped to Int64, int min, int max, float values) of the selected rows of vi and vf."""
    idx = np.nonzero(mask)[0].tolist()
    vi = [tb.vi[i] for i in idx]
    vf = [tb.vf[i] for i in idx]
    s = sum(vi) & (2**64 - 1)
    s = s - 2**64 if s >= 2**63 else s
    return len(idx), s, (min(vi) if vi else None), (max(vi) if vi else None), vf


def julia_sum(vf):
    """Base.sum of Float64 values: NaN with any NaN or with both infinities, else the infinity, else the exact sum."""
    if any(x != x for x in vf) or (math.inf in vf and -math.inf in vf):
        return math.nan
    if math.inf in vf or -math.inf in vf:
        return math.inf if math.inf in vf else -math.inf
    return math.fsum(vf)


def julia_min_max(vf):
    """min / max of non-NaN values with -0.0 ordered before 0.0 (Julia's min / max); None when there is none."""
    xs = [x for x in vf if x == x]
    if not xs:
        return None, None
    key = lambda x: (x, math.copysign(1.0, x))  # noqa: E731
    return min(xs, key=key), max(xs, key=key)


def same_float(a, b):
    return (a != a and b != b) or (a == b and math.copysign(1.0, a) == math.copysign(1.0, b))


def check_agg(got_i, got_f, tb, mask, what):
    n, si, mn, mx, vf = model_agg(tb, mask)
    assert got_i.count == n and got_i.nmissing == 0, (what, got_i.count, n)
    if n:
        assert (got_i.sum_i64, got_i.min_i64, got_i.max_i64) == (si, mn, mx), what
    assert got_f.count == n and got_f.nmissing == 0, (what, got_f.count, n)
    has_nan = any(x != x for x in vf)
    assert bool(got_f.has_nan) == has_nan, what
    exp = julia_sum(vf)
    got = D.agg_sum(got_f, JType("Float64"))
    if math.isfinite(exp):
        tol = 1e-12 * math.fsum(abs(x) for x in vf)
        assert abs(got - exp) <= tol, (what, got, exp)
    else:
        assert same_float(got, exp), (what, got, exp)
    if n and not has_nan:
        lo, hi = julia_min_max(vf)
        assert same_float(got_f.min_f64, lo) and same_float(got_f.max_f64, hi), (what, got_f.min_f64, got_f.max_f64, lo, hi)


# ---- the predicate matrix ---------------------------------------------------------------------------------------------

def _own_extremes(tb, col):
    xs = [v for v in tb.values[col] if v is not None and v == v]
    out = []
    for v in (min(xs), max(xs)):
        if isinstance(v, int) and not -2**63 <= v < 2**63:
            v = float(v)                  # (a UInt64 above 2^63 has no Int64 constant; its double is the nearest one)
        out.append(v)
    return out


def matrix(tb):
    preds = []
    for col, _ in COLUMNS:
        for c in INT_CONSTS + FLT_CONSTS + _own_extremes(tb, col):
            for code in CODES:
                for cf in (False, True):
                    preds.append(Pred([(col, code, c, cf)]))
    nan, inf = math.nan, math.inf
    for x in ("f64", "mf64", "f32"):
        preds += [Pred(t) for t in (
            [(x, ">=", 0.5, False), (x, "<=", 255.5, False)],             # non-empty interval
            [(x, ">", 1.0, False), (x, "<", 0.5, False)],                # empty
            [(x, ">=", 0.5, False), (x, "<=", 0.5, False)],              # one point
            [(x, ">=", -0.0, False), (x, "<=", 0.0, False)],             # the signed zeros
            [(x, ">", -0.0, False)], [(x, "<", 0.0, False)],
            [(x, "==", 0.5, False), (x, "!=", 0.5, False)],
            [(x, "==", 0.0, False), (x, "!=", -0.0, False)],
            [(x, "!=", 0.5, False), (x, "!=", -0.0, False)],             # two != (the TMA scan takes them)
            [(x, "!=", 0.5, False), (x, "!=", 1.0, False), (x, "!=", 0.0, False)],   # three: it refuses
            [(x, "!=", nan, False), (x, "!=", 0.5, False)],
            [(x, "!=", nan, False)],
            [(x, "!=", 0.5, False), (x, "<", inf, False)],
            [(x, "!=", 0.5, False), (x, ">", -1.0, False), (x, "<=", 2.0**63, False)],
            [(x, "<", -inf, False)], [(x, ">", inf, False)], [(x, "<=", inf, False)], [(x, ">=", -inf, False)],
            [(x, "!=", 0.5, False), (x, "<", 1.0, True)],
            [(x, "<", 2**53 + 1, False), (x, ">", -(2**53 + 1), False)],
        )]
    for x, big in (("i64", 2**63 - 1), ("mi64", 2**63 - 1), ("u64", 2**63 - 1)):
        preds += [Pred(t) for t in (
            [(x, ">=", 0, False), (x, "<=", 65536, False)],
            [(x, ">", 5, False), (x, "<", 5, False)],
            [(x, ">=", 6, False), (x, "<=", 6, False)],
            [(x, "==", 1, False), (x, "!=", 1, False)],
            [(x, "!=", 0, False), (x, "!=", 1, False)],
            [(x, "!=", 0, False), (x, "!=", 1, False), (x, "!=", -1, False)],
            [(x, ">", -2**63, False), (x, "<", big, False)],
            [(x, ">=", 0.5, False), (x, "<", 1e19, False)],
            [(x, ">", -0.5, False), (x, "!=", 2.0**63, False)],
        )]
    preds += [
        Pred([("i64", ">", 0, False), ("u64", "<", 2**63 - 1, False), ("f64", "!=", 0.5, False)]),
        Pred([("i64", ">", -2**63, False), ("u64", ">=", 0, False), ("f64", "!=", nan, False),
              ("mf64", ">=", -inf, False)]),                                                     # 4 columns
        Pred([("i64", ">", -2**63, False), ("u64", ">=", 0, False), ("f64", "!=", nan, False),
              ("mf64", ">=", -inf, False), ("mi64", ">", -2**63, False)]),                       # 5 columns
        Pred([("i64", ">=", -1, False), ("u64", "<=", 2.0**64, False), ("f64", "<", 1e19, False),
              ("mi64", "!=", 0, False)]),
        Pred([("i8", ">", -128, False), ("u16", "<", 65535, False), ("f32", "!=", 0.5, False), ("b", "==", 1, False),
              ("mu8", "<=", 200.5, False)]),
        Pred([("mf32", ">=", F32_TENTH, False), ("mu8", "!=", 255, False), ("i32", ">", -2**31, False)]),
    ]
    return preds


@contextmanager
def option(name, value=1):
    L = _capi.lib()
    if name is None:
        yield
        return
    _capi.check(L.dfdb_set_option(name, value))
    try:
        yield
    finally:
        _capi.check(L.dfdb_set_option(name, 0))


# ---- CPU: the model against the oracle ---------------------------------------------------------------------------------

@pytest.fixture(scope="module")
def cpu_tables(tmp_path_factory, oracle):
    out = {}
    for i, layout in enumerate(LAYOUTS):
        p = str(tmp_path_factory.mktemp("pred_" + layout) / "t")
        out[layout] = Table(oracle, p, layout, 0xC0DE + i)
    return out


@pytest.mark.parametrize("layout", list(LAYOUTS))
def test_the_model_and_the_oracle_agree_on_every_predicate(cpu_tables, oracle, layout):
    tb = cpu_tables[layout]
    t = D.open_table(tb.path)                     # plans only: no device is touched
    ot = oracle.OracleTable(tb.path)
    try:
        for p in matrix(tb):
            exp = p.mask(tb)
            v = t[p.expr(t), ["vi", "vf"]]
            pb = D.plan_bytes(v)
            assert np.array_equal(ot.mask(pb), exp), p
            assert ot.count(pb) == int(exp.sum()), p
            n, si, mn, mx, vf = model_agg(tb, exp)
            ai, af = ot.aggregate(pb, 0), ot.aggregate(pb, 1)
            assert ai.count == af.count == n, p
            if n:
                assert (ai.sum_i64, ai.min_i64, ai.max_i64) == (si, mn, mx), p
            assert bool(af.has_nan) == any(x != x for x in vf), p
    finally:
        ot.close()
        t.close()


def test_the_model_compares_exactly():
    """The edges the model exists for: exact int / float comparison, NaN, signed zeros."""
    assert model_term([2**53 + 1, 2**53], "==", 2.0**53, False) == [False, True]
    assert model_term([2**63 - 1], "<", 2.0**63, False) == [True]
    assert model_term([math.nan, 0.5, None], "!=", 0.5, False) == [True, False, False]
    assert model_term([math.nan, -0.0], "<", 0.0, False) == [False, False]
    assert model_term([-0.0], "==", 0.0, True) == [True]
    assert model_term([3], "<", 2, True) == [True]             # 2 < 3
    assert julia_sum([1.0, math.inf]) == math.inf and math.isnan(julia_sum([math.inf, -math.inf, 1.0]))
    assert julia_min_max([0.0, -0.0, math.nan]) == (-0.0, 0.0) and math.copysign(1, julia_min_max([0.0, -0.0])[0]) < 0


# ---- GPU: every path gives the model's answer --------------------------------------------------------------------------

@pytest.fixture(scope="module")
def gpu_tables(tmp_path_factory, oracle):
    _capi.init(0)
    out = {}
    for i, layout in enumerate(LAYOUTS):
        p = str(tmp_path_factory.mktemp("gpred_" + layout) / "t")
        tb = Table(oracle, p, layout, 0xC0DE + i)
        t = D.open_table(p)
        t.build_zonemaps()
        t.close()
        out[layout] = tb
    return out


def _run(t, p):
    v = t[p.expr(t), ["vi", "vf"]]
    return D.selection_mask(v), D.nrow(v), D.aggregate(v.vi), D.aggregate(v.vf)


def _zone(on):
    return option(b"no_zonemap", 0 if on else 1)


@pytest.mark.gpu
@pytest.mark.parametrize("layout", list(LAYOUTS))
def test_every_scan_path_gives_the_model_answer(gpu_tables, layout):
    tb = gpu_tables[layout]
    preds = matrix(tb)
    exp = [p.mask(tb) for p in preds]
    subset = sorted(random.Random(0x5EED).sample(range(len(preds)), SUBSET))
    failures = []                                          # (every divergence of a run is reported, up to 40)
    for opt in (None, b"no_tma", b"no_wide", b"no_fused"):
        with option(opt):
            t = D.open_table(tb.path)
            try:
                got = {}
                for zone_on in (True, False):
                    which = range(len(preds)) if (opt is None and zone_on) else subset
                    with _zone(zone_on):
                        for k in which:
                            got[(k, zone_on)] = r = _run(t, preds[k])
                            what = (layout, opt, zone_on, preds[k])
                            try:
                                assert np.array_equal(r[0], exp[k]), (what, np.nonzero(r[0] != exp[k])[0][:8])
                                assert r[1] == int(exp[k].sum()), (what, r[1], int(exp[k].sum()))
                                check_agg(r[2], r[3], tb, exp[k], what)
                            except AssertionError as e:
                                failures.append(str(e).split("\n")[0][:300])
                            assert len(failures) < 40, failures
                for k in subset:                          # zone maps change which blocks are read, never a bit of the result
                    on, off = got[(k, True)], got[(k, False)]
                    if not (on[1] == off[1] and bytes(on[2]) == bytes(off[2]) and bytes(on[3]) == bytes(off[3])):
                        failures.append(f"zone maps changed the result: {(opt, preds[k])}")
            finally:
                t.close()
    assert not failures, (len(failures), failures)


# ---- zone maps ---------------------------------------------------------------------------------------------------------

@pytest.mark.gpu
@pytest.mark.parametrize("layout", list(LAYOUTS))
def test_zone_map_statistics_match_the_data(gpu_tables, layout):
    tb = gpu_tables[layout]
    t = D.open_table(tb.path)
    try:
        for name, ts in COLUMNS:
            base = _base(ts)
            arr, miss = tb.numpy[name]
            for b, (lo, hi) in enumerate(tb.blocks):
                z = t.zonemap(name, b)
                assert z is not None, (name, b)
                vals = arr[lo:hi]
                m = miss[lo:hi] if miss is not None else np.zeros(hi - lo, dtype=bool)
                assert (z.rows, z.null_count) == (hi - lo, int(m.sum())), (name, b)
                live = vals[~m]
                if base.startswith("Float"):
                    nan = np.isnan(live)
                    assert bool(z.has_nan) == bool(nan.any()), (name, b)
                    live = live[~nan]
                    assert bool(z.has_value) == (live.size > 0), (name, b)
                    if live.size:
                        assert (z.min_f64, z.max_f64) == (float(live.min()), float(live.max())), (name, b)
                else:
                    assert not z.has_nan and bool(z.has_value) == (live.size > 0), (name, b)
                    if live.size:
                        mask64 = (1 << 64) - 1 if base in ("UInt64",) else None
                        zmin, zmax = (z.min_i64 & mask64, z.max_i64 & mask64) if mask64 else (z.min_i64, z.max_i64)
                        assert (zmin, zmax) == (int(live.min()), int(live.max())), (name, b)
    finally:
        t.close()


def _decoded_bytes(fn):
    L = _capi.lib()
    L.dfdb_profile_reset()
    L.dfdb_profile_enable(1)
    try:
        out = fn()
    finally:
        L.dfdb_profile_enable(0)
    ms, n, b = C.c_double(), C.c_int64(), C.c_int64()
    L.dfdb_profile_get(b"decode", C.byref(ms), C.byref(n), C.byref(b))
    return out, b.value


@pytest.mark.gpu
@pytest.mark.parametrize("layout", list(LAYOUTS))
def test_zone_maps_prune_exactly_where_it_is_safe(gpu_tables, layout):
    """Each predicate is decided by a block's min / max / NaN flag, so the pruned blocks are exactly those without a
    selected row: `!=` on a block of one value (pruned) and on one value plus NaN (not), `< 0.0` on a block of signed zeros
    (pruned), `u > 5` on a UInt64 block above 2^63 (not)."""
    tb = gpu_tables[layout]
    t = D.open_table(tb.path)
    try:
        cases = [  # predicate, block roles without a selected row, block roles with one
            (Pred([("f64", "!=", 0.5, False)]), ["single"], ["eq_nan"]),
            (Pred([("mf64", "!=", 0.5, False)]), ["single", "missing"], ["eq_nan"]),
            (Pred([("f64", "<", 0.0, False)]), ["zeros", "nan"], []),
            (Pred([("u64", ">", 5, False)]), [], ["high"]),
        ]
        for p, empty_roles, live_roles in cases:
            exp = p.mask(tb)
            live = [bool(exp[lo:hi].any()) for lo, hi in tb.blocks]
            dead = live.count(False)
            for b, role in enumerate(ROLES[b % len(ROLES)] for b in range(len(tb.blocks))):
                assert (role not in empty_roles or not live[b]) and (role not in live_roles or live[b]), (p, b, role)

            def run():
                v = t[p.expr(t), ["vf"]]
                return D.materialize(v)["vf"], D.pruned_blocks(v)
            with _zone(True):
                (col, (pruned, nb)), on_bytes = _decoded_bytes(run)
            with _zone(False):
                (col0, _), off_bytes = _decoded_bytes(run)
            assert nb == len(tb.blocks)
            assert pruned == dead, (p, pruned, dead)
            assert np.array_equal(col.view(np.uint64), col0.view(np.uint64)) and len(col) == int(exp.sum()), p
            assert (on_bytes < off_bytes) == (dead > 0), (p, on_bytes, off_bytes)
    finally:
        t.close()


# ---- multi-stage plans: pruning must not reach across a range stage ---------------------------------------------------

@pytest.fixture(scope="module")
def sorted_table(tmp_path_factory, oracle):
    _capi.init(0)
    p = str(tmp_path_factory.mktemp("stages") / "t")
    nrows = 12 * 4096 + 777
    rng = np.random.default_rng(0x57A6)
    oracle.write_table(p, [("q", "Int64", np.arange(1, nrows + 1, dtype=np.int64)),
                           ("a", "Int64", rng.integers(1, 101, nrows).astype(np.int64))], block_size=4096)
    t = D.open_table(p)
    t.build_zonemaps()
    t.close()
    return p, nrows


def _stage_plans(t, nrows):
    cut = 3 * 4096
    return {
        "pred_range_pred": t[t.a > 50, :][R(1, 3000), :][t.q > cut, ["q", "a"]],
        "pred_index_pred": t[t.a > 50, :][[1, 2, 5, 100, 2999, 3000], :][t.q > cut, ["q", "a"]],
        "range_pred_range_pred": t[R(100, nrows - 100), :][t.a > 50, :][R(1, 3000), :][t.q > cut, ["q", "a"]],
        "pruning_pred_then_range": t[t.q > cut, :][R(1, 3000), :][t.a > 50, ["q", "a"]],
    }


@pytest.mark.gpu
def test_zone_maps_do_not_prune_blocks_an_earlier_range_stage_counts(sorted_table, oracle):
    """A range / index-vector stage ranks the survivors of the stages before it.  A later predicate whose constants rule a
    block out must not empty that block for those earlier stages: here the first 3000 rows with a > 50 all lie below
    q = 3 * 4096, so q > 3 * 4096 keeps none of them."""
    p, nrows = sorted_table
    ot = oracle.OracleTable(p)
    try:
        t = D.open_table(p)
        exp = {k: ot.materialize(D.plan_bytes(v)) for k, v in _stage_plans(t, nrows).items()}
        masks = {k: ot.mask(D.plan_bytes(v)) for k, v in _stage_plans(t, nrows).items()}
        assert len(exp["pred_range_pred"][0]) == len(exp["pred_index_pred"][0]) == 0
        assert len(exp["range_pred_range_pred"][0]) == 0 and len(exp["pruning_pred_then_range"][0]) > 1000
        t.close()
        for zone_on in (True, False):
            with _zone(zone_on):
                t = D.open_table(p)
                for k, v in _stage_plans(t, nrows).items():
                    fr = D.materialize(v)
                    assert np.array_equal(fr["q"], exp[k][0]) and np.array_equal(fr["a"], exp[k][1]), (k, zone_on, fr.nrow(), len(exp[k][0]))
                    assert D.nrow(v) == len(exp[k][0]), (k, zone_on)
                    assert np.array_equal(D.selection_mask(v), masks[k]), (k, zone_on)
                t.close()
                for world in (2, 3):
                    shards = [D.open_table(p, rank=r, world=world) for r in range(world)]
                    try:
                        for k in exp:
                            views = [_stage_plans(ts, nrows)[k] for ts in shards]
                            D.resolve_sharded_selection(views)
                            got = np.concatenate([np.asarray(D.materialize(v)["q"]) for v in views])
                            assert np.array_equal(got, exp[k][0]), (k, zone_on, world, len(got), len(exp[k][0]))
                            assert sum(D.nrow(v) for v in views) == len(exp[k][0]), (k, zone_on, world)
                    finally:
                        for ts in shards:
                            ts.close()
    finally:
        ot.close()
