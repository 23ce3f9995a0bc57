"""median / quantile over a DFColumn -- exact order statistics by radix select on the device (dfdb_scan_order_*).

CPU: the model (tests/quantile_ref.py) against Python's sorted and numpy's quantile, and the Julia shim's bindings.  GPU: the
library's order statistics, medians and quantiles against the model, bit for bit, on one GPU and across shards."""
import ctypes as C
import math

import numpy as np
import pytest

import dfdb_b200 as D
import quantile_ref as Q
from dfdb_b200 import R, _capi
from test_julia_binding import header_prototypes, jl_ok, shim_ccalls

NROWS, BLOCK = 3001, 1000
TYPES = ["Int8", "Int16", "Int32", "Int64", "UInt8", "UInt16", "UInt32", "UInt64", "Float32", "Float64", "Bool"]
REFUSED = ["String", "Float16", "Char", "Date", "DateTime", "Time"]


def _pool(base):
    """values clustered on the edges of the order: type extremes, +-0.0, +-Inf, subnormals, neighbours in the lowest bit"""
    if base.startswith("Float"):
        dt = np.dtype(base.lower())
        fi = np.finfo(dt)
        one = dt.type(1)
        return np.array([0.0, -0.0, -0.0, 0.0, np.inf, -np.inf, fi.max, -fi.max, fi.smallest_subnormal, -fi.smallest_subnormal,
                         fi.tiny, one, np.nextafter(one, dt.type(2)), np.nextafter(one, dt.type(0)), -one, 2.5, 2.5, 2.5], dtype=dt)
    if base == "Bool":
        return np.array([False, True], dtype=np.bool_)
    dt = np.dtype(base.lower())
    ii = np.iinfo(dt)
    vals = [ii.min, ii.max, 0, 1, 2, 3, 3, 3, ii.max - 1, ii.min + 1]
    if dt.kind == "i":
        vals += [-1, -2, -3]
    if dt == np.uint64:
        vals += [2**63, 2**63 + 1, 2**63 - 1]
    return np.array(vals, dtype=dt)


def _col(ts, rng):
    base = ts[8:-1] if ts.startswith("Missing(") else ts
    pool = _pool(base)
    v = pool[rng.integers(0, len(pool), NROWS)]
    return (v, rng.random(NROWS) < 0.2) if base != ts else v


def _refused_col(ts, rng):
    if ts == "String":
        return ["a", "b", "c"] * (NROWS // 3) + ["d"] * (NROWS % 3)
    dt = {"Float16": np.float16, "Char": np.uint32}.get(ts, np.int64)
    return (rng.integers(1, 90, NROWS)).astype(dt)


@pytest.fixture(scope="module")
def typed(tmp_path_factory, oracle):
    p = str(tmp_path_factory.mktemp("quant") / "t")
    rng = np.random.default_rng(20261021)
    names = TYPES + [f"Missing({b})" for b in TYPES]
    cols = [("k", "Int64", np.arange(1, NROWS + 1, dtype=np.int64) % 10)]
    cols += [(f"c{i}", ts, _col(ts, rng)) for i, ts in enumerate(names)]
    cols += [("eq", "Int64", np.full(NROWS, -7, np.int64)), ("eqf", "Float64", np.full(NROWS, 2.5))]
    cols += [(f"x{i}", ts, _refused_col(ts, rng)) for i, ts in enumerate(REFUSED)]
    nan = np.where(rng.random(NROWS) < 0.01, np.nan, rng.random(NROWS))
    cols += [("nan", "Float64", nan), ("nan32", "Float32", nan.astype(np.float32))]
    oracle.write_table(p, cols, block_size=BLOCK)
    ot = oracle.OracleTable(p)
    types = {f"c{i}": ts for i, ts in enumerate(names)}
    types.update(eq="Int64", eqf="Float64")
    yield p, types, ot
    ot.close()


def _selections(t, name):
    return {
        "none": t[:, [name]],
        "predicate": t[t.k > 3, [name]],
        "range_after_predicate": t[t.k > 3, :][R(5, 2, 1500), [name]],
        "index_vector": t[[1, 2, 7, 999, 1000, 1001, 2500, 3001], [name]],
        "single_row": t[[1717], [name]],
        "two_rows": t[[5, 2999], [name]],
        "empty": t[t.k > 100, [name]],
    }


def _bits(x):
    """bit pattern of a result (None stays None): Float32 results as Float32, every other number as Float64"""
    if x is None:
        return None
    if isinstance(x, np.floating) and x.dtype == np.float32:
        return ("f32", np.float32(x).tobytes())
    return ("f64", np.float64(x).tobytes())


# ---- CPU: the model -----------------------------------------------------------------------------------------------------

def _py_isless_key(x):
    """isless as a Python sort key: numbers by value, -0.0 before 0.0"""
    if isinstance(x, float):
        return (x, math.copysign(1.0, x))
    return (x, 0)


def test_model_order_is_isless():
    rng = np.random.default_rng(7)
    for base in TYPES:
        pool = _pool(base)
        for _ in range(20):
            v = pool[rng.integers(0, len(pool), rng.integers(1, 40))]
            got = Q.sorted_values(v)
            want = sorted(v.tolist(), key=_py_isless_key)
            assert [_py_isless_key(x) for x in got.tolist()] == [_py_isless_key(x) for x in want], base
    big = np.array([2**64 - 1, 2**63, 5, 2**63 - 1, 2**63 + 7], dtype=np.uint64)
    assert Q.sorted_values(big).tolist() == sorted(big.tolist())
    z = np.array([0.0, -0.0, 0.0, -0.0, 5e-324, -5e-324], dtype=np.float64)
    got = Q.sorted_values(z)
    assert [math.copysign(1.0, x) for x in got.tolist()] == [-1.0, -1.0, -1.0, 1.0, 1.0, 1.0]
    assert got[0] == -5e-324 and got[-1] == 5e-324


def test_model_quantile_matches_numpy_linear():
    rng = np.random.default_rng(8)
    for n in (1, 2, 3, 10, 101, 1000):
        v = rng.standard_normal(n)
        ps = np.concatenate([[0.0, 1.0, 0.5], rng.random(20)])
        got = Q.quantile(v, ps)
        want = np.quantile(v, ps, method="linear")
        for g, w in zip(got, want):
            assert abs(g - w) <= 4 * np.spacing(np.abs(v).max()), (n, g, w)       # a few ulps of the data's scale
    assert Q.median(np.array([1, 2, 3, 4], np.int64)) == 2.5
    assert Q.median((np.array([1.0, 9.0]), np.array([False, True]))) is None
    assert Q.median((np.array([1.0, 9.0]), np.array([False, True])), skipmissing=True) == 1.0


def test_julia_shim_binds_the_order_entry_points():
    protos = header_prototypes()
    calls = {c[0]: c for c in shim_ccalls()}
    for name in ("dfdb_scan_order_prepare", "dfdb_scan_order_prepare_all", "dfdb_scan_order_round", "dfdb_scan_order_values",
                 "dfdb_scan_order_stats_all"):
        assert name in protos and name in calls, name
        _, ret, argl, nvals = calls[name]
        cret, cargs = protos[name]
        assert len(argl) == len(cargs) == nvals and jl_ok(ret, cret, is_return=True), name
        assert all(jl_ok(j, c) for j, c in zip(argl, cargs)), name
    src = open(Q.__file__.replace("tests/quantile_ref.py", "julia/b200.jl")).read()
    for hook in ("Statistics.median(c::DFColumn)", "Statistics.median(c::Base.SkipMissing{<:DFColumn})",
                 "Statistics.quantile(c::DFColumn, p;", "Statistics.quantile(c::Base.SkipMissing{<:DFColumn}, p;"):
        assert hook in src, hook


# ---- GPU -------------------------------------------------------------------------------------------------------------------

@pytest.fixture(scope="module")
def gpu():
    _capi.init(0)
    yield


def _rank_sets(n, rng):
    if n == 0:
        return []
    sets = [[1], [n]]
    if n <= 64:
        sets.append(list(range(1, n + 1)))
    sets.append(rng.integers(1, n + 1, 200).tolist())
    return sets


def _check_column(col, ref, what, rng):
    vals, miss = Q.split(ref)
    n = int((~miss).sum())
    for ranks in _rank_sets(n, rng):
        got = D.order_stats(col, ranks)
        assert got.tobytes() == Q.order_stats(ref, ranks).tobytes(), (what, ranks[:5])
    if len(vals) == 0:
        with pytest.raises(D.ArgumentError):
            D.median(col)
        with pytest.raises(D.ArgumentError):
            D.quantile(col, 0.5)
        return
    ps = [0.0, 0.01, 0.1, 0.25, 0.5, 0.75, 0.9, 0.99, 1.0, 1 / 3]
    for skip in (False, True):
        for lib_fn, model_fn in ((lambda: D.median(col, skipmissing=skip), lambda: Q.median(ref, skipmissing=skip)),
                                 (lambda: D.quantile(col, ps, skipmissing=skip), lambda: Q.quantile(ref, ps, skipmissing=skip))):
            try:
                want = model_fn()
            except ValueError:                  # where Statistics throws ArgumentError
                with pytest.raises(D.ArgumentError):
                    lib_fn()
                continue
            got = lib_fn()
            if isinstance(want, list):
                assert [_bits(x) for x in got] == [_bits(x) for x in want], (what, skip)
            else:
                assert _bits(got) == _bits(want), (what, skip)


@pytest.mark.gpu
def test_every_type_and_selection_matches_the_model(gpu, typed):
    path, types, ot = typed
    t = D.open_table(path)
    rng = np.random.default_rng(99)
    for name, ts in types.items():
        for sel, v in _selections(t, name).items():
            ref = ot.materialize(D.plan_bytes(v))[0]
            _check_column(getattr(v, name), ref, (ts, name, sel), rng)
    t.close()


@pytest.mark.gpu
def test_ties_and_zero_signs_straddling_ranks(gpu, tmp_path, oracle):
    """ranks that fall between -0.0 and 0.0, between equal neighbours and between keys one bit apart"""
    p = str(tmp_path / "z")
    n = 4000
    z = np.where(np.arange(n) % 2 == 0, -0.0, 0.0)
    lowbit = np.array([1.0, np.nextafter(1.0, 2.0)])[np.arange(n) % 2]
    ints = (np.arange(n) % 2 + (1 << 40)).astype(np.int64)
    oracle.write_table(p, [("z", "Float64", z), ("z32", "Float32", z.astype(np.float32)), ("lb", "Float64", lowbit), ("i", "Int64", ints)],
                       block_size=1024)
    t, ot = D.open_table(p), oracle.OracleTable(p)
    for name in ("z", "z32", "lb", "i"):
        col = getattr(t, name)
        ref = ot.materialize(D.plan_bytes(col))[0]
        ranks = [1, n // 2, n // 2 + 1, n, 1999, 2001]
        assert D.order_stats(col, ranks).tobytes() == Q.order_stats(ref, ranks).tobytes(), name
        assert _bits(D.median(col)) == _bits(Q.median(ref)), name
    t.close()
    ot.close()


@pytest.mark.gpu
@pytest.mark.parametrize("spec", ["r:Int64:iseq", "a:Int64:iuniform:1:100", "b:Float64:funiform"])
def test_multi_block_tables_with_and_without_zone_maps(gpu, tmp_path, oracle, spec):
    p = str(tmp_path / "g")
    nrows = 1_500_000
    oracle.gen_table(p, spec + ";q:Int64:iseq", nrows, 65536, 0xDFDB0201, 4)
    name = spec.split(":")[0]
    t, ot = D.open_table(p), oracle.OracleTable(p)
    t.build_zonemaps()
    t.close()
    t = D.open_table(p)
    rng = np.random.default_rng(5)
    views = {"all": t[:, [name]], "pred": t[t.q > 700_000, [name]], "range_after_pred": t[t.q > 1000, :][R(10, 3, 900_000), [name]]}
    L = _capi.lib()
    for key, v in views.items():
        col = getattr(v, name)
        ref = ot.materialize(D.plan_bytes(v))[0]
        ranks = rng.integers(1, len(ref) + 1, 200).tolist() + [1, len(ref)]
        want = Q.order_stats(ref, ranks).tobytes()
        results = []
        for off in (0, 1):
            _capi.check(L.dfdb_set_option(b"no_zonemap", off))
            try:
                results.append((D.order_stats(col, ranks).tobytes(), _bits(D.median(col)),
                                [_bits(x) for x in D.quantile(col, [0.01, 0.25, 0.5, 0.99])]))
            finally:
                _capi.check(L.dfdb_set_option(b"no_zonemap", 0))
        assert results[0] == results[1], key
        assert results[0][0] == want, key
        assert results[0][1] == _bits(Q.median(ref)), key
        assert results[0][2] == [_bits(x) for x in Q.quantile(ref, [0.01, 0.25, 0.5, 0.99])], key
    t.close()
    ot.close()


@pytest.mark.gpu
def test_sharded_order_stats_equal_the_unsharded_result(gpu, tmp_path, oracle):
    p = str(tmp_path / "m")
    nrows = 4 * 65536 + 777
    oracle.gen_table(p, "a:Int64:iuniform:1:5000;f:Missing(Float64):funiform:m=0.1;u:Missing(Float64):fgrid:0:0.5:40:m=0.1;r:Int64:iseq", nrows, 65536, 0xDFDB0202, 4)
    t = D.open_table(p)
    rng = np.random.default_rng(11)

    def views(tb):
        return {
            "all": lambda name: getattr(tb[:, [name]], name),
            "pred": lambda name: getattr(tb[tb.a > 2500, [name]], name),
            "one_shard": lambda name: getattr(tb[tb.r > nrows - 500, [name]], name),
            "range_after_pred": lambda name: getattr(tb[tb.a > 100, :][R(3, 5, 200000), [name]], name),
        }
    for world in (2, 3):
        shards = [D.open_table(p, rank=r, world=world) for r in range(world)]
        for key in ("all", "pred", "one_shard", "range_after_pred"):
            for name in ("a", "f", "u"):
                whole = views(t)[key](name)
                agg = D.aggregate(whole)
                n = agg.count - agg.nmissing
                ranks = rng.integers(1, n + 1, 200).tolist() + [1, n]
                cols = [views(ts)[key](name) for ts in shards]
                got = D.order_stats_sharded(cols, ranks)
                assert got.tobytes() == D.order_stats(whole, ranks).tobytes(), (world, key, name)
        for ts in shards:
            ts.close()
    t.close()


@pytest.mark.gpu
def test_one_rank_communicator(gpu, typed):
    path, types, ot = typed
    t = D.open_table(path)
    L = _capi.lib()
    ident = (C.c_uint8 * 128)()
    _capi.check(L.dfdb_comm_unique_id(ident))
    _capi.check(L.dfdb_comm_init(0, 1, ident))
    try:
        for ts in ("Missing(Float64)", "Int32", "UInt64", "Missing(Bool)"):
            name = [k for k, v in types.items() if v == ts][0]
            for v in (t[:, [name]], t[t.k > 3, :][R(5, 2, 1500), [name]]):
                col = getattr(v, name)
                h = D.api._scan_handle(v)
                local, whole = _capi.Agg(), _capi.Agg()
                _capi.check(L.dfdb_scan_order_prepare(h, 0, C.byref(local)))
                everywhere = D.aggregate_all(col)
                _capi.check(L.dfdb_scan_order_prepare_all(h, 0, C.byref(whole)))
                assert bytes(whole) == bytes(everywhere), ts
                n = local.count - local.nmissing
                ranks = [1, n, (n + 1) // 2]
                got = D.order_stats(col, ranks)
                assert got.tobytes() == D.order_stats_sharded([col], ranks).tobytes(), ts
                assert got.tobytes() == Q.order_stats(ot.materialize(D.plan_bytes(v))[0], ranks).tobytes(), ts
    finally:
        _capi.check(L.dfdb_comm_destroy())
    t.close()


@pytest.mark.gpu
def test_nan_missing_and_argument_errors(gpu, typed):
    path, types, ot = typed
    t = D.open_table(path)
    for name in ("nan", "nan32"):
        col = getattr(t, name)
        m = D.median(col)
        assert np.isnan(m) and isinstance(m, np.float32) == (name == "nan32")
        with pytest.raises(D.ArgumentError):
            D.quantile(col, 0.5)
        with pytest.raises(D.ArgumentError):
            D.order_stats(col, [1])
        # a selection without the NaN rows is fine
        v = t[[2, 3], [name]]
        ref = ot.materialize(D.plan_bytes(v))[0]
        if not np.isnan(ref).any():
            assert _bits(D.median(getattr(v, name))) == _bits(Q.median(ref))
    name = [k for k, v in types.items() if v == "Missing(Int64)"][0]
    col = getattr(t, name)
    ref = ot.materialize(D.plan_bytes(col))[0]
    assert D.median(col) is None
    assert _bits(D.median(col, skipmissing=True)) == _bits(Q.median(ref, skipmissing=True))
    with pytest.raises(D.ArgumentError):
        D.quantile(col, 0.5)
    n = int((~ref[1]).sum())
    for bad in ([0], [n + 1], [-3]):
        with pytest.raises(D.ArgumentError):
            D.order_stats(col, bad)
    for bad in (-0.1, 1.5, float("nan"), [0.5, 2.0]):
        with pytest.raises(D.ArgumentError):
            D.quantile(getattr(t, "c3"), bad)
    with pytest.raises(D.ArgumentError):
        D.median(getattr(t[t.k > 100, ["c3"]], "c3"))
    with pytest.raises(D.ArgumentError):
        D.quantile(getattr(t[t.k > 100, ["c3"]], "c3"), 0.5)
    for i in range(len(REFUSED)):
        with pytest.raises(D.ArgumentError):
            D.median(getattr(t, f"x{i}"))
    with pytest.raises(D.ArgumentError):
        D.median(t.k % 7)
    t.close()


@pytest.mark.gpu
def test_calls_out_of_order_are_state_errors(gpu, typed):
    path, types, _ = typed
    t = D.open_table(path)
    L = _capi.lib()
    v = t[:, ["c3"]]
    h = D.api._scan_handle(v)
    counts = np.zeros(_capi.ORDER_MAX_COUNTS, np.int64)
    cp = counts.ctypes.data_as(C.POINTER(C.c_int64))
    nl = C.c_int64()
    whole = _capi.Agg()
    ranks = (C.c_int64 * 1)(1)
    out = np.zeros(4, np.int64)
    assert L.dfdb_scan_order_round(h, C.byref(whole), ranks, 1, None, 0, cp, len(counts), C.byref(nl)) == _capi.ERR_STATE   # before prepare
    assert L.dfdb_scan_order_values(h, out.ctypes.data) == _capi.ERR_STATE
    _capi.check(L.dfdb_scan_order_prepare(h, 0, C.byref(whole)))
    assert L.dfdb_scan_order_round(h, C.byref(whole), ranks, 1, cp, 4, cp, len(counts), C.byref(nl)) == _capi.ERR_STATE    # counts, no round
    assert L.dfdb_scan_order_values(h, out.ctypes.data) == _capi.ERR_STATE
    _capi.check(L.dfdb_scan_order_round(h, C.byref(whole), ranks, 1, None, 0, cp, len(counts), C.byref(nl)))
    assert nl.value > 0
    assert L.dfdb_scan_order_values(h, out.ctypes.data) == _capi.ERR_STATE                                                    # round in flight
    assert L.dfdb_scan_order_round(h, C.byref(whole), ranks, 1, None, 0, cp, 16, C.byref(nl)) == _capi.ERR_ARGUMENT          # cap too small
    t.close()


@pytest.mark.gpu
def test_materialize_on_the_same_handle_is_unchanged(gpu, typed):
    """prepare and the rounds between dfdb_scan_materialize_sizes and dfdb_scan_materialize on one handle leave the
    selection mask and block bases the fill reuses intact"""
    path, types, ot = typed
    t = D.open_table(path)
    L = _capi.lib()
    for ts in ("Missing(Int16)", "Float64"):
        name = [k for k, v in types.items() if v == ts][0]
        v = t[t.k > 3, [name, "k"]]
        h = D.api._scan_handle(v)
        n, sb = C.c_int64(), (C.c_int64 * 2)()
        _capi.check(L.dfdb_scan_materialize_sizes(h, C.byref(n), sb))
        whole = _capi.Agg()
        _capi.check(L.dfdb_scan_order_prepare(h, 0, C.byref(whole)))
        ranks = np.array([1, 2, 3], np.int64)
        vals = np.zeros(3, np.int16 if ts == "Missing(Int16)" else np.float64)
        _capi.check(L.dfdb_scan_order_stats_all(h, ranks.ctypes.data_as(C.POINTER(C.c_int64)), 3, vals.ctypes.data))
        ref_col = ot.materialize(D.plan_bytes(getattr(v, name)))[0]
        assert vals.tobytes() == Q.order_stats(ref_col, [1, 2, 3]).tobytes(), ts
        rows = n.value
        outs = (_capi.OutCol * 2)()
        mv, mm = np.zeros(rows, vals.dtype), np.zeros(rows, np.uint8)
        outs[0].values = mv.ctypes.data
        if ts.startswith("Missing("):
            outs[0].missing = mm.ctypes.data
        k = np.zeros(rows, np.int64)
        outs[1].values = k.ctypes.data
        _capi.check(L.dfdb_scan_materialize(h, outs, 2))
        ref = ot.materialize(D.plan_bytes(v))
        assert np.array_equal(k, ref[1]), ts
        if ts == "Float64":
            assert mv.tobytes() == ref[0].tobytes(), ts
        else:
            m = ref[0][1]
            assert np.array_equal(mm.astype(bool), m) and np.array_equal(mv[~m], ref[0][0][~m]), ts
    t.close()
