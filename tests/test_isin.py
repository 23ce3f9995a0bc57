"""in.(x, Ref(C)) with collections of any size and element type, under `==` (vectors, tuples) and isequal (Set).

The reference is the exact model of tests/isin_ref.py over the oracle's materialize of the left operand (the oracle itself is
the fixed yardstick of the older plans and is not extended).  CPU: the model against Julia's documented answers, the result
eltypes of the Python mirror, the plan bytes of both opcodes, and the refusals of dfdb_scan_prepare.  GPU: every position a
predicate can take (selection stage, projected Bool column, inside ~ / & / coalesce, behind a range stage), both probe paths
of the selection stage, zone maps on and off, shards, and a semi-join, exactly."""
import ctypes as C
import struct

import numpy as np
import pytest

import dfdb_b200 as D
import isin_ref as M
from dfdb_b200 import R, _capi
from dfdb_b200 import plan as P

NROWS, BLOCK = 3001, 512

INT_POOL = [0, 1, -1, 3, 5, 99, 1000, 7, -128, 127]
F_POOL = [0.0, -0.0, 0.1, 1.0, 2.5, 3.0, float("inf"), 9007199254740992.0]
NAN_BITS = [0x7ff8000000000000, 0x7ff8000000000001, 0xfff8000000000123]
STR_POOL = ["", "so", "sony", "lg", "ü-ß", "x" * 40, "apple"]
BASE_TYPES = ["Int8", "Int16", "Int32", "Int64", "UInt8", "UInt16", "UInt32", "UInt64", "Float32", "Float64", "Bool", "String"]
TYPES = BASE_TYPES + [f"Missing({b})" for b in BASE_TYPES]


def _nan(bits):
    return struct.unpack("<d", struct.pack("<Q", bits))[0]


COLLECTIONS = {
    "empty": [],
    "one": [3],
    "duplicates": [3, 3, 5, 3, 5],
    "ints64": list(range(-10, 118, 2)),                 # 64 values: the old limit
    "ints65": list(range(-10, 120, 2)),                 # 65 values
    "ints1000": list(range(-500, 500)),
    "mixed": [1, 2.5, "sony", True, 99.0],
    "mixed_missing": [1, 2.5, "lg", None, False],
    "missing_only": [None],
    "zeros_nans": [0.0, _nan(NAN_BITS[1]), _nan(NAN_BITS[2])],
    "neg_zero": [-0.0],
    "awkward": [2 ** 53 + 1, 2.0 ** 53 - 1, 2 ** 64 - 1, -1, 0.1, float(np.float32(0.1)), 2 ** 63, 127.0, 1.5],
    "strings": ["", "so", "ü-ß", "x" * 40, "x" * 39, "sonyy"],
}


def _typed_column(ts, rng):
    base = ts[8:-1] if ts.startswith("Missing(") else ts
    n = NROWS
    if base == "String":
        vals = [STR_POOL[i] for i in rng.integers(0, len(STR_POOL), n)]
        return [None if m else v for v, m in zip(vals, rng.random(n) < 0.2)] if base != ts else vals
    if base.startswith("Float"):
        dt, bt = (np.float64, np.uint64) if base == "Float64" else (np.float32, np.uint32)
        pool = np.array(F_POOL, dtype=dt).view(bt).tolist()
        pool += [b if base == "Float64" else (b >> 32) | 1 for b in NAN_BITS]      # NaNs of several payloads
        v = np.array(pool, dtype=bt)[rng.integers(0, len(pool), n)].view(dt)
    elif base == "Bool":
        v = rng.integers(0, 2, n).astype(np.bool_)
    else:
        dt = np.dtype(base.lower())
        pool = [x for x in INT_POOL if np.iinfo(dt).min <= x <= np.iinfo(dt).max] + [int(np.iinfo(dt).max)]
        v = np.array(pool, dtype=dt)[rng.integers(0, len(pool), n)]
    return (v, rng.random(n) < 0.2) if base != ts else v


def _columns():
    rng = np.random.default_rng(20261022)
    cols = [("k", "Int64", np.arange(1, NROWS + 1, dtype=np.int64))]
    cols += [(f"c{i}", ts, _typed_column(ts, rng)) for i, ts in enumerate(TYPES)]
    cols += [("d", "Date", np.arange(NROWS, dtype=np.int64) + 730000)]
    return cols


@pytest.fixture(scope="module")
def typed(tmp_path_factory, oracle):
    p = str(tmp_path_factory.mktemp("isin") / "t")
    cols = _columns()
    oracle.write_table(p, cols, block_size=BLOCK)
    ot = oracle.OracleTable(p)
    yield p, {f"c{i}": ts for i, ts in enumerate(TYPES)}, ot
    ot.close()


def _variants(values):
    """the collection as a vector (`==`) and as a Set (isequal)"""
    return [(list(values), False), (set(values), True)]


def _model(ot, t, name, c, isequal):
    col = M.as_list(ot.materialize(D.plan_bytes(getattr(t, name)))[0])
    return M.isin_column(col, P.InSet(c).values, isequal)


# ---- CPU --------------------------------------------------------------------------------------------------------------

def test_model_gives_julias_answers():
    nan, nan2 = _nan(NAN_BITS[0]), _nan(NAN_BITS[2])
    vec = [  # (x, C, in(x, C)) from Julia's `in(x, ::Vector)`
        (1, [1.0], True), (True, [1], True), (0.0, [-0.0], True), (-0.0, [0], True), (nan, [nan], False),
        (2 ** 53 + 1, [9.007199254740992e15], False), (float(np.float32(0.1)), [0.1], False), (2 ** 64 - 1, [-1], False),
        (1, [1.5], False), ("1", [1], False), ("", [""], True), (None, [1], None), (None, [], False), (2, [1, None], None),
        (1, [1, None], True), (None, [None], None), ("a", ["b", None], None),
    ]
    for x, c, want in vec:
        assert M.isin(x, c, False) is want, (x, c)
    st = [  # in(x, ::Set): isequal
        (nan, [nan2], True), (0.0, [-0.0], False), (0, [-0.0], False), (-0.0, [-0.0], True), (1, [1.0], True), (True, [1.0], True),
        (None, [None], True), (None, [1], False), (2, [None], False), ("a", ["a"], True), ("1", [1], False),
    ]
    for x, c, want in st:
        assert M.isin(x, c, True) is want, (x, c)


def test_mirror_eltypes(typed):
    path, types, _ = typed
    t = D.open_table(path)
    for name, ts in types.items():
        for cname, values in COLLECTIONS.items():
            for c, isequal in _variants(values):
                e = D.isin(getattr(t, name), c)
                nullable = M.eltype_nullable(ts.startswith("Missing("), P.InSet(c).values, isequal)
                assert e.eltype() == D.JType("Bool", nullable), (ts, cname, isequal)
    assert D.isin(t.k % 7, [1, None]).eltype() == D.JType("Bool", True)
    t.close()


def test_plan_bytes_of_both_opcodes():
    col = P.ColRef("a", P.JType("Int64"), 7)
    # all-Int64 vectors keep the IN opcode, byte for byte
    e = P.BlockBroadcasting("in", (col, P.InSet([3, 5, 99, 1000])))
    assert P.encode_expr(e) == struct.pack("<IBqBI4q", 2, P.OP_COL, 7, P.OP_IN, 4, 3, 5, 99, 1000)
    assert P.InSet(np.array([1, 2], dtype=np.int64)).legacy
    # everything else is INSET: semantics, count, tagged elements
    s = P.InSet([1, 2 ** 63, 2.5, np.float32(0.1), "ü", True, None])
    assert not s.legacy and not s.isequal
    want = struct.pack("<BBI", P.OP_INSET, 0, 7) + struct.pack("<Bq", 1, 1) + struct.pack("<BQ", 2, 2 ** 63) + \
        struct.pack("<Bd", 3, 2.5) + struct.pack("<Bd", 3, float(np.float32(0.1))) + struct.pack("<BI", 4, 2) + "ü".encode() + \
        struct.pack("<BB", 5, 1) + struct.pack("<B", 6)
    assert s.wire == want
    assert P.InSet({3}).wire == struct.pack("<BBIBq", P.OP_INSET, 1, 1, 1, 3)
    assert P.InSet(np.ma.MaskedArray([1, 2], mask=[False, True])).values == (1, None)
    assert P.InSet(D.FlatStringsVector(np.array([2, -1], np.int32), b"ab")).values == ("ab", None)
    assert P.InSet([1.9]).values == (1.9,)                              # no truncation
    with pytest.raises(P.ArgumentError):
        P.InSet([2 ** 64])
    with pytest.raises(P.ArgumentError):
        P.InSet([object()])


def _prepare(t, expr_body: bytes):
    plan = struct.pack("<IIIB", P.MAGIC, 0, 1, P.PJ_EXPR) + expr_body
    h = C.c_void_p()
    rc = _capi.lib().dfdb_scan_prepare(t._h, plan, len(plan), C.byref(h))
    if rc == 0:
        _capi.lib().dfdb_scan_free(h)
    return rc


def test_prepare_refuses_bad_collections_and_operands(typed, tmp_path, oracle):
    path, types, _ = typed
    t = D.open_table(path)
    head = struct.pack("<IBq", 2, P.OP_COL, t.k.view.projection.cols[0][1].col_id)
    good = head + struct.pack("<BBIBq", P.OP_INSET, 0, 1, 1, 3)
    assert _prepare(t, good) == 0
    for bad in (good[:-3], head + struct.pack("<BBIB", P.OP_INSET, 0, 1, 9), head + struct.pack("<BBI", P.OP_INSET, 2, 0),
                head + struct.pack("<BBIBI", P.OP_INSET, 0, 1, 4, 10) + b"abc", head + struct.pack("<BBI", P.OP_INSET, 0, 5)):
        assert _prepare(t, bad) == _capi.ERR_ARGUMENT, bad
    # Date through the INSET form is refused; through IN it stays accepted
    did = t.d.view.projection.cols[0][1].col_id
    dhead = struct.pack("<IBq", 2, P.OP_COL, did)
    assert _prepare(t, dhead + struct.pack("<BBIBq", P.OP_INSET, 0, 1, 1, 3)) == _capi.ERR_UNSUPPORTED
    assert _prepare(t, dhead + struct.pack("<BIq", P.OP_IN, 1, 730001)) == 0
    with pytest.raises(P.ArgumentError):
        D.isin(t.d, [1.5])
    t.close()
    p = str(tmp_path / "odd")
    oracle.write_table(p, [("ch", "Char", np.array([65, 66], np.uint32)), ("h", "Float16", np.array([1, 2], np.float16))])
    t = D.open_table(p)
    for name in ("ch", "h"):
        ref = getattr(t, name).view.projection.cols[0][1]
        body = struct.pack("<IBq", 2, P.OP_COL, ref.col_id) + struct.pack("<BBIBq", P.OP_INSET, 1, 1, 1, 65)
        assert _prepare(t, body) == _capi.ERR_UNSUPPORTED, name
        with pytest.raises(P.ArgumentError):
            D.isin(getattr(t, name), {65})
    t.close()


# ---- GPU --------------------------------------------------------------------------------------------------------------

@pytest.fixture(scope="module")
def gpu():
    _capi.init(0)
    yield


def _option(name, value):
    _capi.check(_capi.lib().dfdb_set_option(name, value))


def _sel_rows(model, k):
    return [kk for kk, r in zip(k, model) if r is True]


def _check_selection(t, ot, sel, want_k, what):
    """selection stage `sel` (a Bool DFColumn) over the table: nrow, materialize, sum and minimum of k"""
    v = t[sel, ["k"]]
    assert D.nrow(v) == len(want_k), what
    got = D.materialize(v)["k"].tolist()
    assert got == want_k, what
    assert D.sum(v.k) == sum(want_k), what
    if want_k:
        assert D.minimum(v.k) == min(want_k), what


@pytest.mark.gpu
def test_every_type_collection_and_position(gpu, typed):
    path, types, ot = typed
    t = D.open_table(path)
    k = list(range(1, NROWS + 1))
    for name, ts in types.items():
        x = getattr(t, name)
        for cname, values in COLLECTIONS.items():
            for c, isequal in _variants(values):
                what = (ts, cname, isequal)
                model = _model(ot, t, name, c, isequal)
                e = D.isin(x, c)
                # projected Bool column, missings included
                got = M.as_list(D.materialize(t[:, {"r": e}])["r"])
                assert got == model, what
                nullable = e.eltype().nullable
                # coalesce(in, false), ~, & another term, behind a range stage; each on both selection paths
                cz = D.coalesce(e, False)
                cases = [(cz, _sel_rows(model, k)),
                         (~cz, [kk for kk, r in zip(k, model) if r is not True]),
                         (cz & (t.k > 1500), [kk for kk, r in zip(k, model) if r is True and kk > 1500])]
                if not nullable:
                    cases.append((e, _sel_rows(model, k)))
                for fused in (0, 1):
                    _option(b"no_fused", fused)
                    try:
                        for sel, want in cases:
                            _check_selection(t, ot, sel, want, what + (fused,))
                        ranged = t[R(5, 3, NROWS), :][cz, ["k"]]
                        want = [kk for kk, r in zip(k, model) if kk >= 5 and (kk - 5) % 3 == 0 and r is True]
                        assert D.materialize(ranged)["k"].tolist() == want, what + (fused, "range")
                    finally:
                        _option(b"no_fused", 0)
    t.close()


def _big_table(tmp_path, nrows=400_000, block=65536):
    p = str(tmp_path / "big")
    rng = np.random.default_rng(7)
    ids = rng.integers(1, 2 * nrows, nrows).astype(np.int64)
    strs = ["k%d" % v for v in ids[:nrows] % 200_000]
    D.create_table(p, [("k", "Int64", np.arange(1, nrows + 1, dtype=np.int64)), ("id", "Int64", ids),
                       ("f", "Float64", ids.astype(np.float64) / 2), ("s", "String", strs)], block_size=block).close()
    return p, ids, strs


@pytest.mark.gpu
@pytest.mark.parametrize("size", [1, 64, 65, 1000, 4096, 4097, 100_000, 1_000_000])
def test_set_sizes_on_both_probe_paths(gpu, tmp_path, oracle, size):
    """the selection stage stages tables of up to INSET_SMEM_SLOTS slots (4096 keys) in shared memory and probes larger ones
    in global memory; the VM probes the same tables.  About half the rows hit."""
    nrows = 400_000
    p, ids, strs = _big_table(tmp_path, nrows)
    t, ot = D.open_table(p), oracle.OracleTable(p)
    # exactly `size` distinct keys: ids of a sample of the rows, the rest values no row holds
    rng = np.random.default_rng(size)
    keys = np.unique(ids[rng.integers(0, nrows, max(1, min(size, nrows) // 2))])
    keys = np.concatenate([keys, -np.arange(1, size - len(keys) + 1, dtype=np.int64)])
    assert len(np.unique(keys)) == size
    hit = np.isin(ids, keys)
    for c in (keys, set(keys.tolist())):
        for fused in (0, 1):
            _option(b"no_fused", fused)
            try:
                v = t[D.isin(t.id, c), ["k"]]
                assert D.nrow(v) == int(hit.sum()), (size, fused)
                assert np.array_equal(D.materialize(v)["k"], np.nonzero(hit)[0] + 1), (size, fused)
            finally:
                _option(b"no_fused", 0)
        assert D.nrow(t[D.isin(t.id + 0, c), ["k"]]) == int(hit.sum())
        fl = t[D.isin(t.f, keys.astype(np.float64) / 2), ["k"]]
        assert D.nrow(fl) == int(hit.sum())
    if size <= 100_000:
        skeys = ["k%d" % v for v in np.unique(keys % 200_000)]
        ss = set(skeys)
        want = [i + 1 for i, s in enumerate(strs) if s in ss]
        v = t[D.isin(t.s, skeys), ["k"]]
        assert D.materialize(v)["k"].tolist() == want
    t.close()
    ot.close()


@pytest.mark.gpu
def test_cached_set_zone_maps_and_shards(gpu, tmp_path, oracle):
    p, ids, strs = _big_table(tmp_path, 300_000, 16384)
    t, ot = D.open_table(p), oracle.OracleTable(p)
    t.build_zonemaps(["k", "id", "f"])
    cases = {   # name -> (column, collection, whether the zone maps must rule out blocks)
        "disjoint_sorted": ("k", [10 ** 9, 10 ** 9 + 7], True),
        "two_blocks": ("k", {3, 200_000}, True),
        "float": ("f", [0.5, 1.0, 1.5, float("nan")], False),
        "set_nan": ("f", {float("nan"), 2.0}, False),
        "ids": ("id", list(range(1, 5000)), False),
        "strings": ("s", ["k1", "k2", "k19"], False),
    }
    for name, (cn, c, prune) in cases.items():
        def mk(tb):
            return D.isin(getattr(tb, cn), c)
        col = M.as_list(ot.materialize(D.plan_bytes(getattr(t, cn)))[0])
        model = M.isin_column(col, P.InSet(c).values, isinstance(c, set))
        ref = np.array([i + 1 for i, r in enumerate(model) if r is True], dtype=np.int64)
        v = t[mk(t), ["k"]]
        # on a handle, then again on the same handle (the set table is kept), then on a fresh table
        for _ in range(2):
            assert np.array_equal(D.materialize(v)["k"], ref), name
        if prune:
            assert D.pruned_blocks(v)[0] > 0, name
        fresh = D.open_table(p)
        assert np.array_equal(D.materialize(fresh[mk(fresh), ["k"]])["k"], ref), name
        fresh.close()
        _option(b"no_zonemap", 1)
        try:
            off = D.materialize(t[mk(t), ["k"]])["k"]
        finally:
            _option(b"no_zonemap", 0)
        assert np.array_equal(off, ref), name
        for world in (2, 3):
            shards = [D.open_table(p, rank=r, world=world) for r in range(world)]
            parts = [D.materialize(s[mk(s), ["k"]])["k"] for s in shards]
            assert np.array_equal(np.concatenate(parts), ref), (name, world)
            assert sum(D.nrow(s[mk(s), ["k"]]) for s in shards) == len(ref), (name, world)
            for s in shards:
                s.close()
    t.close()
    ot.close()


@pytest.mark.gpu
def test_semi_join_through_unique(gpu, tmp_path):
    p = str(tmp_path / "sj")
    rng = np.random.default_rng(11)
    n = 200_000
    user = rng.integers(0, 50_000, n).astype(np.int64)
    country = ["fr" if u % 7 == 0 else "de" for u in user]
    names = ["u%d" % u for u in user]
    score = rng.random(n)
    t = D.create_table(p, [("user", "Int64", user), ("name", "String", names), ("country", "String", country), ("score", "Float64", score)],
                       block_size=32768)
    for key in ("user", "name"):
        keys = D.unique(getattr(t[(t.country == "fr") & (t.score > 0.5), [key]], key))
        vals = M.as_list(keys)
        want_set = set(vals)
        col = user.tolist() if key == "user" else names
        want = [i + 1 for i, x in enumerate(col) if x in want_set]
        got = D.selection_indices(t[D.isin(getattr(t, key), keys), [key]]).tolist()
        assert got == want, key
        model = M.isin_column(col, P.InSet(keys).values, False)
        assert [i + 1 for i, r in enumerate(model) if r] == want, key
    t.close()
