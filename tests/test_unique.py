"""unique(col) -- Base.unique over iterate(::DFColumn): distinct values of the selected rows in order of first appearance, isequal.

CPU: the C reference (tests/unique_ref.py over the oracle's materialize) against a plain Python fold, and the Julia shim's
bindings.  GPU: dfdb_scan_unique / _merge / _all against the reference, value bits and order exactly."""
import ctypes as C

import numpy as np
import pytest

import dfdb_b200 as D
import unique_ref
from dfdb_b200 import R, _capi
from test_julia_binding import header_prototypes, jl_ok, shim_ccalls

NROWS, BLOCK = 3001, 1000          # the block size does not divide the row count

F64_POOL = [0.0, -0.0, 1.5, -2.25, float("inf"), 0x7ff8000000000001, 0xfff8000000000000, 0x7ff0000000000123]
F32_POOL = [0.0, -0.0, 1.5, -2.25, float("inf"), 0x7fc00001, 0xffc00000, 0x7f800123]
F16_POOL = [0.0, -0.0, 1.5, -2.25, float("inf"), 0x7e01, 0xfe00, 0x7c01]
STR_POOL = ["sony", "", "apple", "ü-ß", "x" * 40, "dell"]
BASE_TYPES = ["Int8", "Int16", "Int32", "Int64", "UInt8", "UInt16", "UInt32", "UInt64", "Float16", "Float32", "Float64", "Bool", "Char",
              "Date", "DateTime", "Time", "String"]
TYPES = BASE_TYPES + [f"Missing({b})" for b in BASE_TYPES]


def _col(name, rng):
    """values of a column of type `name` with few distinct values, NaNs of several payloads, -0.0, missing and "" """
    base = name[8:-1] if name.startswith("Missing(") else name
    n = NROWS
    if base == "String":
        vals = [STR_POOL[i] for i in rng.integers(0, len(STR_POOL), n)]
        if base != name:
            vals = [None if m else v for v, m in zip(vals, rng.random(n) < 0.2)]
        return vals
    if base.startswith("Float"):
        pool = {"Float64": (F64_POOL, np.float64, np.uint64), "Float32": (F32_POOL, np.float32, np.uint32), "Float16": (F16_POOL, np.float16, np.uint16)}[base]
        bits = np.array([int(p) if isinstance(p, int) else int(np.array(p, dtype=pool[1]).view(pool[2])) for p in pool[0]], dtype=pool[2])
        v = bits[rng.integers(0, len(bits), n)].view(pool[1])
    elif base == "Bool":
        v = rng.integers(0, 2, n).astype(np.bool_)
    elif base == "Char":
        v = np.array([65, 66, 0x1F600, 97, 0x00E9], dtype=np.uint32)[rng.integers(0, 5, n)]
    else:
        dt = {"Date": np.int64, "DateTime": np.int64, "Time": np.int64}.get(base) or np.dtype(base.lower())
        v = (rng.integers(0, 12, n) * 3 - (0 if base.startswith("UInt") else 15)).astype(dt)
    return (v, rng.random(n) < 0.2) if base != name else v


@pytest.fixture(scope="module")
def typed(tmp_path_factory, oracle):
    p = str(tmp_path_factory.mktemp("uniq") / "t")
    rng = np.random.default_rng(20261020)
    cols = [("k", "Int64", np.arange(1, NROWS + 1, dtype=np.int64) % 10)]
    cols += [(f"c{i}", ts, _col(ts, rng)) for i, ts in enumerate(TYPES)]
    oracle.write_table(p, cols, block_size=BLOCK)
    ot = oracle.OracleTable(p)
    yield p, {f"c{i}": ts for i, ts in enumerate(TYPES)}, ot
    ot.close()


def _selections(t, name):
    return {
        "none": t[:, [name]],
        "predicate": t[t.k > 3, [name]],
        "range_after_predicate": t[t.k > 3, :][R(5, 2, 1500), [name]],
        "index_vector": t[[1, 2, 7, 999, 1000, 1001, 2500, 3001], [name]],
        "empty": t[t.k > 100, [name]],
    }


# ---- CPU: the reference against a plain Python fold ----------------------------------------------------------------

def _fold(col, base):
    """Base.unique as a dict fold: the key is isequal's -- missing, one NaN, raw bits otherwise (so -0.0 != 0.0)"""
    from oracle import oracle as O
    if isinstance(col, O.FlatStrings):
        return list(dict.fromkeys(col.tolist()))
    vals, miss = col if isinstance(col, tuple) else (col, np.zeros(len(col), bool))
    seen = {}
    for v, m in zip(vals, miss):
        if m:
            key = None
        elif base.startswith("Float") and np.isnan(v):
            key = "NaN"
        else:
            key = v.tobytes()
        seen.setdefault(key, None if m else v.tobytes())
    return list(seen.values())


def _as_list(col):
    from oracle import oracle as O
    if isinstance(col, O.FlatStrings):
        return col.tolist()
    vals, miss = col if isinstance(col, tuple) else (col, np.zeros(len(col), bool))
    return [None if m else v.tobytes() for v, m in zip(vals, miss)]


def test_reference_unique_matches_a_python_fold(typed):
    path, types, ot = typed
    t = D.open_table(path)                       # host-only: plans, no scan
    for name, ts in types.items():
        base = ts[8:-1] if ts.startswith("Missing(") else ts
        for sel, v in _selections(t, name).items():
            col = ot.materialize(D.plan_bytes(v))[0]
            got = unique_ref.unique_column(col, base)
            assert _as_list(got) == _fold(col, base), (ts, sel)
            if sel == "none" and base.startswith("Float"):
                # every NaN payload is one value (the first one's bits), -0.0 and 0.0 are two
                fl = [x for x in _as_list(got) if x is not None]
                dt = {"Float16": np.float16, "Float32": np.float32, "Float64": np.float64}[base]
                arr = np.frombuffer(b"".join(fl), dtype=dt)
                assert np.isnan(arr).sum() == 1 and (arr == 0).sum() == 2, ts
    t.close()


def test_reference_keeps_empty_string_apart_from_missing(tmp_path, oracle):
    p = str(tmp_path / "s")
    oracle.write_table(p, [("s", "Missing(String)", ["", None, "", "a", None, "a", "b"])], block_size=3)
    ot = oracle.OracleTable(p)
    t = D.open_table(p)
    assert unique_ref.unique(ot, D.plan_bytes(t.s)).tolist() == ["", None, "a", "b"]
    t.close()
    ot.close()


def test_julia_shim_binds_the_unique_entry_points():
    protos = header_prototypes()
    calls = {c[0]: c for c in shim_ccalls()}
    for name in ("dfdb_scan_unique", "dfdb_scan_unique_values", "dfdb_scan_unique_merge", "dfdb_scan_unique_all"):
        assert name in protos and name in calls, name
        _, ret, argl, nvals = calls[name]
        cret, cargs = protos[name]
        assert len(argl) == len(cargs) == nvals and jl_ok(ret, cret, is_return=True), name
        assert all(jl_ok(j, c) for j, c in zip(argl, cargs)), name
    assert "Base.unique(c::DFColumn)" in open(unique_ref.os.path.join(unique_ref.HERE, "..", "julia", "b200.jl")).read()


# ---- GPU ---------------------------------------------------------------------------------------------------------------

def _same(got, ref, what):
    """device result == reference result: values (bits), missing and order"""
    from oracle import oracle as O
    if isinstance(ref, O.FlatStrings):
        assert isinstance(got, D.FlatStringsVector), what
        assert np.array_equal(got.sizes, ref.sizes), what
        assert bytes(got.data) == ref.chars, what
        return
    vals, miss = ref if isinstance(ref, tuple) else (ref, None)
    gv = np.ma.getdata(got)
    assert len(gv) == len(vals), (what, len(gv), len(vals))
    if miss is None:
        assert not isinstance(got, np.ma.MaskedArray), what
        assert gv.tobytes() == np.ascontiguousarray(vals).tobytes(), what
    else:
        gm = np.ma.getmaskarray(got)
        assert np.array_equal(gm, miss), what
        assert gv[~gm].tobytes() == np.ascontiguousarray(vals)[~miss].tobytes(), what


@pytest.fixture(scope="module")
def gpu():
    _capi.init(0)
    yield


@pytest.mark.gpu
def test_unique_every_type_and_selection(gpu, typed):
    path, types, ot = typed
    t = D.open_table(path)
    for name, ts in types.items():
        base = ts[8:-1] if ts.startswith("Missing(") else ts
        for sel, v in _selections(t, name).items():
            col = getattr(v, name)
            ref = unique_ref.unique_column(ot.materialize(D.plan_bytes(v))[0], base)
            _same(D.unique(col), ref, (ts, sel))
    t.close()


@pytest.mark.gpu
@pytest.mark.parametrize("spec,nrows", [("a:Int64:iseq", 1_500_000), ("s:String:decimal", 700_000), ("s:String:brands", 400_000),
                                        ("a:Int64:iuniform:1:100", 400_000)])
def test_unique_cardinality(gpu, tmp_path, oracle, spec, nrows):
    """few distinct values, and every row distinct: 1.5M keys start the group table at 2^16 slots and grow it three times"""
    p = str(tmp_path / "c")
    oracle.gen_table(p, spec, nrows, 65536, 0xDFDB0103, 4)
    t, ot = D.open_table(p), oracle.OracleTable(p)
    name = spec.split(":")[0]
    col = getattr(t, name)
    ref = unique_ref.unique(ot, D.plan_bytes(col))
    _same(D.unique(col), ref, spec)
    if spec.endswith("iseq"):
        assert len(ref) == nrows
    t.close()
    ot.close()


@pytest.mark.gpu
def test_unique_merge_over_shards_equals_unsharded(gpu, tmp_path, oracle):
    p = str(tmp_path / "m")
    nrows = 4 * 65536 + 777
    oracle.gen_table(p, "a:Int64:iuniform:1:5000;s:Missing(String):decimal:m=0.05;f:Missing(Float64):fgrid:0:0.5:40:m=0.1;r:Int64:iseq",
                     nrows, 65536, 0xDFDB0104, 4)
    t = D.open_table(p)

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
            for name in ("a", "s", "f"):
                whole = D.unique(views(t)[key](name))
                cols = [views(ts)[key](name) for ts in shards]
                D.resolve_sharded_selection([c.view for c in cols])
                parts = [D.unique(c) for c in cols]
                merged = D.unique_merge(views(t)[key](name), parts)
                if isinstance(whole, D.FlatStringsVector):
                    assert merged == whole, (world, key, name)
                else:
                    assert np.ma.getdata(merged).tobytes() == np.ma.getdata(whole).tobytes(), (world, key, name)
                    assert np.array_equal(np.ma.getmaskarray(merged), np.ma.getmaskarray(whole)), (world, key, name)
        for ts in shards:
            ts.close()
    t.close()


@pytest.mark.gpu
def test_unique_all_over_a_one_rank_communicator_is_the_local_result(gpu, typed):
    path, types, ot = typed
    t = D.open_table(path)
    L = _capi.lib()
    ident = (C.c_uint8 * 128)()
    _capi.check(L.dfdb_comm_unique_id(ident))
    _capi.check(L.dfdb_comm_init(0, 1, ident))
    try:
        for ts in ("Missing(String)", "String", "Missing(Float64)", "Float16", "Int32", "Missing(Char)"):
            name = [k for k, v in types.items() if v == ts][0]
            for v in (t[:, [name]], t[t.k > 3, :][R(5, 2, 1500), [name]], t[t.k > 100, [name]]):
                col = getattr(v, name)
                local, everywhere = D.unique(col), D.unique_all(col)
                if isinstance(local, D.FlatStringsVector):
                    assert everywhere == local, ts
                else:
                    assert np.ma.getdata(everywhere).tobytes() == np.ma.getdata(local).tobytes(), ts
                    assert np.array_equal(np.ma.getmaskarray(everywhere), np.ma.getmaskarray(local)), ts
    finally:
        _capi.check(L.dfdb_comm_destroy())
    t.close()


@pytest.mark.gpu
def test_materialize_on_the_same_handle_is_unchanged(gpu, typed):
    """dfdb_scan_unique between dfdb_scan_materialize_sizes and dfdb_scan_materialize on one handle: the fill reuses the
    selection mask and block bases of the sizes pass (it does not rerun the selection), so unique must leave them intact"""
    path, types, ot = typed
    t = D.open_table(path)
    L = _capi.lib()
    for ts in ("Missing(String)", "Missing(Int16)", "Float16"):
        name = [k for k, v in types.items() if v == ts][0]
        v = t[t.k > 3, [name, "k"]]
        h = D.api._scan_handle(v)
        n, sb = C.c_int64(), (C.c_int64 * 2)()
        _capi.check(L.dfdb_scan_materialize_sizes(h, C.byref(n), sb))
        nu, nb = C.c_int64(), C.c_int64()
        _capi.check(L.dfdb_scan_unique(h, 0, C.byref(nu), C.byref(nb)))           # unique on projection 0 of the same handle
        ref_u = unique_ref.unique(ot, D.plan_bytes(getattr(v, name)))
        assert nu.value == len(ref_u[0] if isinstance(ref_u, tuple) else ref_u)
        rows = n.value
        outs = (_capi.OutCol * 2)()
        if ts == "Missing(String)":
            sizes, chars = np.zeros(rows, np.int32), np.zeros(max(sb[0], 1), np.uint8)
            outs[0].str_sizes, outs[0].str_chars = sizes.ctypes.data, chars.ctypes.data
        else:
            dt = np.float16 if ts == "Float16" else np.int16
            vals, miss = np.zeros(rows, dt), np.zeros(rows, np.uint8)
            outs[0].values = vals.ctypes.data
            if ts.startswith("Missing("):
                outs[0].missing = miss.ctypes.data
        k = np.zeros(rows, np.int64)
        outs[1].values = k.ctypes.data
        _capi.check(L.dfdb_scan_materialize(h, outs, 2))
        ref = ot.materialize(D.plan_bytes(v))
        assert np.array_equal(k, ref[1]), ts
        if ts == "Missing(String)":
            assert D.FlatStringsVector(sizes, chars[:sb[0]]).tolist() == ref[0].tolist(), ts
        elif ts == "Float16":
            assert vals.tobytes() == ref[0].tobytes(), ts
        else:
            m = ref[0][1]
            assert np.array_equal(miss.astype(bool), m) and np.array_equal(vals[~m], ref[0][0][~m]), ts
    t.close()


@pytest.mark.gpu
def test_unique_merge_of_row_range_parts_on_a_fresh_handle(gpu, typed):
    """every column type: the local results of disjoint row ranges (NaNs of other payloads, -0.0, repeats across parts),
    merged on a handle that has run no scan (a table opened anew), equal the unique of the whole column"""
    path, types, ot = typed
    t = D.open_table(path)
    for name, ts in types.items():
        base = ts[8:-1] if ts.startswith("Missing(") else ts
        for bounds in ([(1, 1500), (1501, 3001)], [(1, 999), (1000, 1000), (1001, 2222), (2223, 3001)]):
            parts = [D.unique(getattr(t[R(lo, hi), [name]], name)) for lo, hi in bounds]
            fresh = D.open_table(path)
            merged = D.unique_merge(getattr(fresh[:, [name]], name), parts)
            fresh.close()
            ref = unique_ref.unique_column(ot.materialize(D.plan_bytes(t[:, [name]]))[0], base)
            _same(merged, ref, (ts, len(bounds)))
    t.close()


@pytest.mark.gpu
def test_unique_of_a_computed_column_is_an_argument_error(gpu, typed):
    path, _, _ = typed
    t = D.open_table(path)
    with pytest.raises(D.ArgumentError):
        D.unique(t.k % 7)
    t.close()

