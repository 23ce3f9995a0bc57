"""groupreduce over every shard: key values from the library, per-shard groups merged and folded on the device.

Expectations: a Python dict fold over the columns the ORACLE materializes for the same plan, in first-appearance order with
isequal keys (missing is one value, all NaNs are one value carrying the first NaN's bits, -0.0 and 0.0 differ, strings by
bytes and "" is not missing); counts, integer sums (wrapping), minima and maxima exact, Float64 sums against math.fsum within
1e-12.  CPU: the fold against a hand-computed answer, and the Julia shim's bindings.  GPU: dfdb_scan_groupreduce /
_group_keys / _groupreduce_merge / _groupreduce_all."""
import ctypes as C
import math
import struct

import numpy as np
import pytest

import dfdb_b200 as D
from dfdb_b200 import R, _capi
from test_julia_binding import header_prototypes, jl_ok, shim_ccalls

BLOCK = 2048
NROWS = 10 * BLOCK - 300                      # ten blocks, the last one short: shards at world 2 and 3 cut through the groups
BRANDS = ["apple", "samsung", "huawai", "", "dell", "xbox", "sony", "intel"]
F_POOL = [0.0, -0.0, 1.5, -2.25, 0x7ff8000000000001, 0xfff8000000000000, 0x7ff0000000000123]


def _bits(x):
    return struct.unpack("<Q", struct.pack("<d", x))[0]


def _key(x):
    """isequal's image of one key value"""
    if isinstance(x, float):
        return "NaN" if x != x else ("f", _bits(x))
    return x


def _as_lists(cols):
    out = []
    for c in cols:
        if isinstance(c, tuple):
            out.append([None if m else v for v, m in zip(c[0].tolist(), c[1].tolist())])
        else:
            out.append(c.tolist())
    return out


def dict_fold(cols, nkeys, rows):
    """The groups of columns `cols` (keys first, oracle layout) over the selected table rows `rows` (1-based), in order of
    first appearance: a list of (first key values, first row, [values of each value column])."""
    lists = _as_lists(cols)
    groups, order = {}, []
    for i in range(len(rows)):
        tup = tuple(lists[k][i] for k in range(nkeys))
        key = tuple(_key(x) for x in tup)
        if key not in groups:
            groups[key] = (tup, int(rows[i]), [[] for _ in lists[nkeys:]])
            order.append(key)
        for j, col in enumerate(lists[nkeys:]):
            groups[key][2][j].append(col[i])
    return [groups[k] for k in order]


def _wrap(x, ts):
    if ts.startswith("UInt"):
        return x % (1 << 64)
    if ts.startswith("Int"):
        return (x + (1 << 63)) % (1 << 64) - (1 << 63)
    return x


def expect(ot, view, by, cols):
    v = view[:, by + list(cols.values())]
    plan = D.plan_bytes(v)
    rows = np.flatnonzero(ot.mask(plan)) + 1
    return dict_fold(ot.materialize(plan), len(by), rows)


def check(got, exp, by, cols, types, what):
    """a groupreduce-shaped result dict against the dict fold"""
    keys = list(zip(*[got[k] for k in by])) if exp else []
    bits = lambda tup: tuple(("f", _bits(x)) if isinstance(x, float) else x for x in tup)       # (a NaN key carries the first NaN's bits)
    assert [bits(k) for k in keys] == [bits(e[0]) for e in exp], (what, keys[:4], [e[0] for e in exp[:4]])
    assert got["first_row"] == [e[1] for e in exp], what
    if not cols:
        assert got["ngroups"] == len(exp), what
    for j, (name, src) in enumerate(cols.items()):
        rec, ts = got[name], types[src].replace("Missing(", "").rstrip(")")
        for gi, e in enumerate(exp):
            xs = e[2][j]
            present = [x for x in xs if x is not None]
            assert rec["count"][gi] == len(xs) and rec["nmissing"][gi] == len(xs) - len(present), (what, name, e[0])
            if not present:
                assert rec["min"][gi] is None, (what, name)
                continue
            if ts == "Float64":
                s = math.fsum(present)
                if s != s:
                    assert rec["sum"][gi] != rec["sum"][gi] and rec["min"][gi] != rec["min"][gi] and rec["max"][gi] != rec["max"][gi], (what, name)
                    continue
                assert abs(rec["sum"][gi] - s) <= 1e-12 * max(abs(s), 1e-300), (what, name, e[0])
            else:
                assert rec["sum"][gi] == _wrap(sum(int(x) for x in present), ts), (what, name, e[0])
            assert rec["min"][gi] == min(present) and rec["max"][gi] == max(present), (what, name, e[0])


def same(a, b, by, cols, what):
    """two groupreduce-shaped results: keys (bits), first rows, counts, integer sums, minima and maxima equal; Float64 sums
    within 1e-12 relative (the local pass adds a group's Float64 values in arrival order, so two runs of it may differ in the
    last bits)"""
    canon = lambda xs: [("f", _bits(x)) if isinstance(x, float) else x for x in xs]
    for k in by:
        assert canon(a[k]) == canon(b[k]), (what, k)
    assert a["first_row"] == b["first_row"], what
    for name in cols:
        for f in ("count", "nmissing", "min", "max"):
            assert canon(a[name][f]) == canon(b[name][f]), (what, name, f)
        for x, y in zip(a[name]["sum"], b[name]["sum"]):
            if isinstance(x, float):
                assert (x != x and y != y) or abs(x - y) <= 1e-12 * max(abs(y), 1e-300), (what, name)
            else:
                assert canon([x]) == canon([y]), (what, name)


@pytest.fixture(scope="module")
def small(tmp_path_factory, oracle):
    rng = np.random.default_rng(20261020)
    n = NROWS
    fbits = np.array([p if isinstance(p, int) else _bits(p) for p in F_POOL], dtype=np.uint64)
    s = [BRANDS[i] for i in rng.integers(0, len(BRANDS), n)]
    for i in range(n - 700, n, 7):
        s[i] = "only-in-the-last-block"                          # a key that occurs on one shard only
    price = rng.random(n) * 100
    price[rng.random(n) < 0.002] = np.nan
    cols = [
        ("s", "String", s),
        ("ms", "Missing(String)", [None if m else ("" if e else BRANDS[i]) for i, m, e in
                                   zip(rng.integers(0, len(BRANDS), n), rng.random(n) < 0.15, rng.random(n) < 0.1)]),
        ("f", "Float64", fbits[rng.integers(0, len(fbits), n)].view(np.float64)),
        ("mk", "Missing(Int64)", (rng.integers(-3, 4, n).astype(np.int64), rng.random(n) < 0.2)),
        ("k", "Int64", rng.integers(0, 300, n).astype(np.int64)),
        ("qty", "Missing(Int64)", (rng.integers(-(1 << 62), 1 << 62, n).astype(np.int64), rng.random(n) < 0.15)),
        ("price", "Float64", price),
        ("u", "UInt64", rng.integers(0, 1 << 63, n, dtype=np.uint64) * np.uint64(2) + np.uint64(1)),
        ("b", "Bool", rng.random(n) < 0.3),
        ("a", "Int64", rng.integers(1, 101, n).astype(np.int64)),
        ("r", "Int64", np.arange(1, n + 1, dtype=np.int64)),
    ]
    p = str(tmp_path_factory.mktemp("grp") / "t")
    oracle.write_table(p, cols, block_size=BLOCK)
    ot = oracle.OracleTable(p)
    yield p, {c[0]: c[1] for c in cols}, ot
    ot.close()


@pytest.fixture(scope="module")
def big(tmp_path_factory, oracle):
    p = str(tmp_path_factory.mktemp("grpbig") / "t")
    nrows = 4 * 65536 + 777
    oracle.gen_table(p, "k:Int64:iuniform:1:50000;b:Float64:funiform;r:Int64:iseq", nrows, 65536, 0xDFDB0107, 4)
    ot = oracle.OracleTable(p)
    yield p, {"k": "Int64", "b": "Float64", "r": "Int64"}, ot, nrows
    ot.close()


def cases(t):
    """(name, view, by, value columns): every key type of the issue, every value type, nvals = 0, a shard without selected
    rows, a selection empty everywhere, a range stage behind a predicate"""
    return [
        ("string_key", t[t.a > 20, :], ["s"], {"p": "price", "q": "qty"}),
        ("missing_string_key", t[:, :], ["ms"], {"u": "u", "b": "b"}),
        ("float_key", t[:, :], ["f"], {"q": "qty", "p": "price"}),
        ("missing_int_key", t[:, :], ["mk"], {"p": "price", "u": "u", "b": "b", "q": "qty"}),
        ("two_keys", t[t.a <= 60, :], ["s", "k"], {"q": "qty"}),
        ("distinct_tuples", t[:, :], ["ms", "mk"], {}),
        ("last_shard_only", t[t.r > NROWS - 500, :], ["s"], {"p": "price"}),
        ("empty", t[t.a > 1000, :], ["s"], {"p": "price"}),
        ("range_after_predicate", t[t.a > 30, :][R(5, 3, 12000), :], ["s", "mk"], {"q": "qty", "p": "price"}),
    ]


# ---- CPU ---------------------------------------------------------------------------------------------------------------

def test_dict_fold_matches_a_hand_computed_fold(tmp_path, oracle):
    p = str(tmp_path / "h")
    nan1, nan2 = struct.unpack("<d", struct.pack("<Q", 0x7ff8000000000001))[0], struct.unpack("<d", struct.pack("<Q", 0xfff8000000000000))[0]
    oracle.write_table(p, [("s", "Missing(String)", ["", None, "", "a", None, "a", "b"]),
                           ("f", "Float64", np.array([0.0, -0.0, nan1, 0.0, nan2, -0.0, 1.0])),
                           ("x", "Missing(Int64)", (np.array([1, 2, 3, 4, 5, 6, 7], dtype=np.int64), np.array([0, 0, 1, 0, 0, 0, 0], bool)))],
                       block_size=3)
    ot = oracle.OracleTable(p)
    t = D.open_table(p)                          # host-only: plans, no scan
    by_s = expect(ot, t[:, :], ["s"], {"x": "x"})
    assert [(e[0], e[1], e[2]) for e in by_s] == [(("",), 1, [[1, None]]), ((None,), 2, [[2, 5]]), (("a",), 4, [[4, 6]]), (("b",), 7, [[7]])]
    by_f = expect(ot, t[:, :], ["f"], {"x": "x"})
    assert [(_bits(e[0][0]), e[1], e[2]) for e in by_f] == [(0, 1, [[1, 4]]), (1 << 63, 2, [[2, 6]]), (0x7ff8000000000001, 3, [[None, 5]]),
                                                           (_bits(1.0), 7, [[7]])]
    pairs = expect(ot, t[R(2, 6), :], ["s", "f"], {})
    assert [(e[0][0], _key(e[0][1]), e[1]) for e in pairs] == [(None, ("f", 1 << 63), 2), ("", "NaN", 3), ("a", ("f", 0), 4), (None, "NaN", 5),
                                                              ("a", ("f", 1 << 63), 6)]
    t.close()
    ot.close()


def test_julia_shim_binds_the_group_entry_points():
    protos = header_prototypes()
    calls = {c[0]: c for c in shim_ccalls()}
    for name in ("dfdb_scan_groupreduce", "dfdb_scan_group_results", "dfdb_scan_group_key_bytes", "dfdb_scan_group_keys",
                 "dfdb_scan_groupreduce_merge", "dfdb_scan_groupreduce_all"):
        assert name in protos and name in calls, name
        _, ret, argl, nvals = calls[name]
        cret, cargs = protos[name]
        assert len(argl) == len(cargs) == nvals and jl_ok(ret, cret, is_return=True), name
        assert all(jl_ok(j, c) for j, c in zip(argl, cargs)), name
    src = open(__import__("os").path.join(__import__("os").path.dirname(__file__), "..", "julia", "b200.jl")).read()
    assert "groupreduce_local!" in src and "groupreduce_merge!" in src and "keys = group_keys(" in src


# ---- GPU ---------------------------------------------------------------------------------------------------------------

@pytest.fixture(scope="module")
def gpu():
    _capi.init(0)
    yield


def _handle(view, by, cols):
    return D.api._scan_handle(view[:, by + list(cols.values())])


@pytest.mark.gpu
def test_keys_come_from_the_library(gpu, small):
    """after groupreduce on the unsharded table, dfdb_scan_group_keys equals materialize at first_rows bit for bit, and
    groupreduce_all without a communicator is groupreduce (Float64 sums: to rounding, see `same`)"""
    path, types, ot = small
    t = D.open_table(path)
    L = _capi.lib()
    with pytest.raises(D.DfdbError):
        _capi.check(L.dfdb_scan_group_key_bytes(D.api._scan_handle(t[:, ["s", "k"]]), (C.c_int64 * 2)()))     # no group-by yet
    for name, view, by, cols in cases(t):
        got = D.groupreduce(view, by, **cols)
        h = _handle(view, by, cols)
        n = len(got["first_row"])
        keys = D.api._group_keys(h, n, len(by))
        if n:
            ref = D.materialize(D.DFView(t)[got["first_row"], by])
            for k, col in enumerate(keys):
                r = ref.columns[k]
                if isinstance(r, D.FlatStringsVector):
                    assert np.array_equal(col.sizes, r.sizes) and bytes(col.data) == bytes(r.data), (name, k)
                else:
                    assert np.ma.getdata(col).tobytes() == np.ma.getdata(r).tobytes(), (name, k)
                    assert np.array_equal(np.ma.getmaskarray(col), np.ma.getmaskarray(r)), (name, k)
        else:
            assert all(len(c) == 0 for c in keys), name
        check(got, expect(ot, view, by, cols), by, cols, types, name)
        same(D.groupreduce_all(view, by, **cols), got, by, cols, name)
    t.close()


def _shard_parts(path, world, view_of, by, cols):
    shards = [D.open_table(path, rank=r, world=world) for r in range(world)]
    views = [view_of(s)[:, by + list(cols.values())] for s in shards]
    D.resolve_sharded_selection(views)
    parts = [D.groupreduce_local(v, by, **cols) for v in views]
    for s in shards:
        s.close()
    return parts


@pytest.mark.gpu
def test_shards_merge_to_the_unsharded_result(gpu, small):
    path, types, ot = small
    t = D.open_table(path)
    for world in (2, 3):
        for i, (name, view, by, cols) in enumerate(cases(t)):
            parts = _shard_parts(path, world, lambda s: cases(s)[i][1], by, cols)
            whole = D.groupreduce(view, by, **cols)
            merged = D.groupreduce_merge(view, by, parts, **cols)             # (replaces the handle's result: read below)
            same(merged, whole, by, cols, (world, name))
            check(merged, expect(ot, view, by, cols), by, cols, types, (world, name))
            # the fold is dfdb_agg_fold over the key's per-part aggregates in rank order, bit for bit
            nv = len(cols)
            if not nv:
                continue
            h = _handle(view, by, cols)
            first, aggs = D.api._group_results(h, len(merged["first_row"]), nv)
            norm = lambda tup: tuple(_key(x) for x in tup)                 # (each part's NaN key carries its own first NaN's bits)
            index = [{norm(k): g for g, k in enumerate(zip(*[D.Frame(by, p["keys"]).to_dict()[b] for b in by]))} for p in parts]
            for g, key in enumerate(zip(*[merged[b] for b in by])):
                for j in range(nv):
                    per = [p["aggs"][ix[norm(key)] * nv + j] for p, ix in zip(parts, index) if norm(key) in ix]
                    assert bytes(aggs[g * nv + j]) == bytes(D.fold(per)), (world, name, key, j)
    t.close()


@pytest.mark.gpu
def test_high_cardinality_shards_merge(gpu, big):
    """about 50000 groups, and a key where every row is its own group.  The unsharded side is groupreduce_all without a
    communicator, whose keys come from the library like the merge's"""
    path, types, ot, nrows = big
    t = D.open_table(path)
    for by, cols in ((["k"], {"s": "b", "n": "r"}), (["r"], {"s": "b"})):
        whole = D.groupreduce_all(t[:, :], by, **cols)
        if by == ["r"]:
            assert len(whole["first_row"]) == nrows
        for world in (2, 3):
            parts = _shard_parts(path, world, lambda s: s[:, :], by, cols)
            same(D.groupreduce_merge(t[:, :], by, parts, **cols), whole, by, cols, (world, by))
        check(whole, expect(ot, t[:, :], by, cols), by, cols, types, by)
    t.close()


@pytest.mark.gpu
def test_row_range_parts_merge_on_a_fresh_handle(gpu, small):
    """parts made of disjoint row ranges, merged on a handle that has never run a scan, equal the whole-column result"""
    path, types, ot = small
    t = D.open_table(path)
    for by, cols in ((["s"], {"p": "price"}), (["ms"], {"q": "qty"}), (["f"], {"u": "u"}), (["mk"], {"b": "b"}), (["s", "k"], {"p": "price", "q": "qty"}),
                     (["ms", "f"], {})):
        whole = D.groupreduce(t[:, :], by, **cols)
        for bounds in ([(1, 9000), (9001, NROWS)], [(1, 2047), (2048, 2048), (2049, 11111), (11112, NROWS)]):
            parts = [D.groupreduce_local(t[R(lo, hi), :], by, **cols) for lo, hi in bounds]
            fresh = D.open_table(path)
            merged = D.groupreduce_merge(fresh[:, :], by, parts, **cols)
            fresh.close()
            same(merged, whole, by, cols, (by, len(bounds)))
    t.close()


@pytest.mark.gpu
def test_one_rank_communicator(gpu, small):
    path, types, ot = small
    t = D.open_table(path)
    L = _capi.lib()
    ident = (C.c_uint8 * 128)()
    _capi.check(L.dfdb_comm_unique_id(ident))
    _capi.check(L.dfdb_comm_init(0, 1, ident))
    try:
        for name, view, by, cols in cases(t):
            everywhere = D.groupreduce_all(view, by, **cols)
            local = D.groupreduce(view, by, **cols)
            same(everywhere, local, by, cols, name)
        with pytest.raises(D.ArgumentError):
            D.groupreduce_all(t[:, :], ["k"], x="s")              # a String value column fails the local pass on the rank
        same(D.groupreduce_all(t[:, :], ["k"], q="qty"), D.groupreduce(t[:, :], ["k"], q="qty"), ["k"], {"q": "qty"}, "after a failure")
    finally:
        _capi.check(L.dfdb_comm_destroy())
    t.close()


@pytest.mark.gpu
def test_materialize_on_the_same_handle_is_unchanged(gpu, small):
    """a group-by call between dfdb_scan_materialize_sizes and dfdb_scan_materialize on one handle leaves the selection mask and
    block bases that the fill reuses intact"""
    path, types, ot = small
    t = D.open_table(path)
    L = _capi.lib()
    v = t[t.a > 20, ["ms", "k", "price"]]
    h = D.api._scan_handle(v)
    n, sb = C.c_int64(), (C.c_int64 * 3)()
    _capi.check(L.dfdb_scan_materialize_sizes(h, C.byref(n), sb))
    ng = C.c_int64()
    _capi.check(L.dfdb_scan_groupreduce(h, (C.c_int32 * 2)(0, 1), 2, (C.c_int32 * 1)(2), 1, C.byref(ng)))
    assert ng.value == len(expect(ot, v, ["ms", "k"], {"p": "price"}))
    rows = n.value
    sizes, chars = np.zeros(rows, np.int32), np.zeros(max(sb[0], 1), np.uint8)
    k, price = np.zeros(rows, np.int64), np.zeros(rows, np.float64)
    outs = (_capi.OutCol * 3)()
    outs[0].str_sizes, outs[0].str_chars = sizes.ctypes.data, chars.ctypes.data
    outs[1].values, outs[2].values = k.ctypes.data, price.ctypes.data
    _capi.check(L.dfdb_scan_materialize(h, outs, 3))
    ref = ot.materialize(D.plan_bytes(v))
    assert D.FlatStringsVector(sizes, chars[:sb[0]]).tolist() == ref[0].tolist()
    assert np.array_equal(k, ref[1]) and price.tobytes() == ref[2].tobytes()
    t.close()
