"""CPU: plan algebra (mirror of the reference's SelectionQueue / Projection / BlockBroadcasting), plan wire
format, C-ABI surface, table indexing by the product's host code (no compute calls)."""
import ctypes as C
import os
import re
import struct
import subprocess
import sys

import numpy as np
import pytest

import dfdb_b200 as D
import fixtures
from dfdb_b200 import R, _capi
from dfdb_b200.plan import BlockBroadcasting as BB, ColRef, JType, Projection, SelectionQueue, add, encode_plan

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_selection_queue_algebra():
    """test/selection.jl:5-37"""
    sel = SelectionQueue()
    assert sel.isempty()
    a = ColRef("a", JType("Int64"), 1)
    test_b = BB("==", (a, 1))
    assert add(sel, slice(None)).isempty()
    sel2 = add(sel, R(5, 20))
    assert len(sel2) == 1
    sel2 = add(sel2, R(1, 5))
    assert len(sel2) == 1 and sel2.queue[0] == R(5, 9)
    sel2 = add(sel2, test_b)
    assert len(sel2) == 2
    sel3 = add(add(sel, test_b), test_b)
    assert len(sel3) == 1 and sel3.queue[0].f == "&"
    assert len(add(sel3, R(1, 3))) == 2
    with pytest.raises(D.ArgumentError):
        add(sel3, BB("*", (a, 3)))
    # reindexing of ranges and index vectors (selection.jl:40)
    assert add(add(sel, R(1, 10, 1000)), R(1, 10)).queue[0] == R(1, 10, 91)
    assert add(add(sel, [5, 9, 2]), R(2, 3)).queue[0] == (9, 2)
    assert add(add(sel, R(10, 20)), [1, 3]).queue[0] == (10, 12)


def test_projection_algebra():
    """test/projection.jl:10-55"""
    a = ColRef("a", JType("Int64"), 1)
    p = Projection([("a", a), ("b", BB("*", (a, 2)))])
    assert p.keys() == ("a", "b")
    with pytest.raises(D.ArgumentError):
        p.add([("a", a)])
    p2 = Projection([("a", a)]).add([("c", ColRef("a", JType("Float64"), 1)), ("e", ColRef("e", JType("Float64"), 5))])
    assert p2.keys() == ("a", "c", "e")
    assert p2[2].keys() == ("c",) and p2[R(1, 2)].keys() == ("a", "c") and p2[[1, 3]].keys() == ("a", "e")
    assert p2[["a", "e"]].keys() == ("a", "e")
    assert p.required_columns() == ("a",)
    assert Projection().isempty()


def test_broadcast_typing():
    """test/broadcast.jl:12-36 result types; arrays rejected :73-81"""
    a, c, s = ColRef("a", JType("Int64"), 1), ColRef("c", JType("Float64"), 3), ColRef("s", JType("String"), 2)
    m = ColRef("m", JType("Int64", True), 4)
    assert BB("*", (a, 2)).eltype() == JType("Int64")
    assert BB("+", (a, c)).eltype() == JType("Float64")
    assert BB("+", (a, BB("+", (a, c)))).eltype() == JType("Float64")
    assert BB("/", (a, 50)).eltype() == JType("Float64")
    assert BB(">", (m, 5)).eltype() == JType("Bool", True)
    assert BB("coalesce", (BB(">", (m, 5)), False)).eltype() == JType("Bool")
    assert BB("startswith", (s, "x")).eltype() == JType("Bool")
    assert BB("<", (s, 3)).eltype() is None
    from dfdb_b200.plan import required_columns
    assert required_columns(BB("+", (a, BB("+", (a, c))))) == ("a", "c")
    with pytest.raises(D.ArgumentError):
        BB("in", (a, [1, 11, 21]))


def test_plan_wire_format():
    a = ColRef("a", JType("Int64"), 7)
    q = add(add(SelectionQueue(), R(5, 2, 20)), BB(">", (a, 50)))
    plan = encode_plan(q, Projection([("a", a), ("x", BB("*", (a, 2.5)))]))
    assert plan[:4] == b"DFP1" and struct.unpack_from("<I", plan, 4)[0] == 2
    assert struct.unpack_from("<Bqqq", plan, 8) == (1, 5, 2, 19)
    assert plan[33] == 3 and struct.unpack_from("<I", plan, 34)[0] == 3


def test_header_declares_exactly_the_exported_symbols():
    hdr = open(os.path.join(ROOT, "include", "dfdb_b200.h")).read()
    declared = set(re.findall(r"DFDB_API\s+[\w\s\*]+?\b(dfdb_\w+)\s*\(", hdr))
    assert declared == set(_capi.SYMBOLS), declared ^ set(_capi.SYMBOLS)
    _capi.build()
    lib = C.CDLL(_capi.LIB_PATH)
    for name in declared:
        assert hasattr(lib, name), name


def test_product_fails_loudly_without_a_gpu(tmp_path, oracle):
    import torch
    if torch.cuda.is_available():
        pytest.skip("needs a box without a GPU")
    p = str(tmp_path / "t")
    fixtures.make_selection_fixture(oracle, p, 50)
    t = D.open_table(p)                     # host-only: parses headers, indexes blocks
    assert t.total_rows() == 100 and t.nblocks() == 2 and t.names() == ["a", "b"]
    with pytest.raises(D.DfdbError) as e:
        D.nrow(t[t.a > 5, :])
    assert e.value.code == _capi.ERR_CUDA


def test_torch_imports_after_the_library_binds_nccl():
    """dfdb_comm_unique_id binds libnccl.so.2 (no GPU needed for the id); torch must still import afterwards in that process,
    which it cannot once an NCCL older than its own is loaded."""
    code = ("import ctypes as C\n"
            "from dfdb_b200 import _capi\n"
            "L = _capi.lib()\n"
            "_capi.check(L.dfdb_comm_unique_id((C.c_uint8 * 128)()))\n"
            "import torch\n")
    r = subprocess.run([sys.executable, "-c", code], cwd=ROOT, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-2000:]


def test_table_index_and_open_errors(tmp_path, oracle):
    p = str(tmp_path / "t")
    data = fixtures.make_reference_fixture(oracle, p, sz=1000, block_size=100)
    t = D.open_table(p)
    assert (t.total_rows(), t.nblocks(), t.block_size) == (1000, 10, 100)
    assert [(m.id, m.name, m.typestring) for m in t.meta] == [(1, "a", "Int64"), (2, "b", "String"), (3, "c", "Int64")]
    assert oracle.OracleTable(p).columns() == [(1, "a", "Int64"), (2, "b", "String"), (3, "c", "Int64")]
    L = _capi.lib()
    comp, unc = C.c_int64(), C.c_int64()
    _capi.check(L.dfdb_table_column_stats(t._h, 1, C.byref(comp), C.byref(unc)))
    assert unc.value == 8000
    _capi.check(L.dfdb_table_set_shard(t._h, 1, 3))
    lo, hi, rlo, rhi = C.c_int64(), C.c_int64(), C.c_int64(), C.c_int64()
    _capi.check(L.dfdb_table_shard_range(t._h, C.byref(lo), C.byref(hi), C.byref(rlo), C.byref(rhi)))
    assert (lo.value, hi.value, rlo.value, rhi.value) == (3, 6, 300, 600)
    with pytest.raises(KeyError):
        t.getmeta("nope")
    # header mismatch: block size in the column file differs from meta (filesystem.jl:47-54)
    f = os.path.join(p, "1.bin")
    raw = bytearray(open(f, "rb").read())
    raw[0:8] = struct.pack("<q", 64)
    open(f, "wb").write(raw)
    with pytest.raises(RuntimeError):
        D.open_table(p)
    # plan validation happens on the host: unknown column, non-Bool predicate, empty range
    p2 = str(tmp_path / "t2")
    fixtures.make_selection_fixture(oracle, p2, 50)
    t2 = D.open_table(p2)
    h = C.c_void_p()
    for plan, code in [(encode_plan(SelectionQueue((BB(">", (ColRef("zz", JType("Int64"), 99), 1)),)), Projection()), _capi.ERR_KEY),
                       (encode_plan(SelectionQueue((R(1, 0),)), Projection()), _capi.ERR_ARGUMENT),
                       (b"XXXX" + bytes(8), _capi.ERR_ARGUMENT)]:
        assert L.dfdb_scan_prepare(t2._h, plan, len(plan), C.byref(h)) == code


def test_agg_fold_is_a_fixed_order_host_fold():
    parts = []
    for cnt, s, mn, mx in [(3, 1.5, 0.25, 0.75), (0, 0.0, 0.0, 0.0), (2, 1e-17, -0.0, 0.5)]:
        a = _capi.Agg()
        a.count, a.sum_f64, a.min_f64, a.max_f64, a.value_class = cnt, s, mn, mx, (3 if cnt else 0)
        parts.append(a)
    f = D.fold(parts)
    assert f.count == 5 and f.min_f64 == 0.0 and np.signbit(f.min_f64) and f.max_f64 == 0.75
    assert f.sum_f64 + f.sum_f64_lo == 1.5 + 1e-17 or abs((f.sum_f64 + f.sum_f64_lo) - 1.5) < 1e-15


def test_flat_strings_vector_views():
    """FlatStringsVector (src/FlatStringsVectors.jl:5-9,61-70,83-85): sizes + flat chars, offsets = exclusive scan of max(size, 0)
    built on first use; the char buffer may be bytes or a zero-copy view of a result array."""
    import numpy as np
    sizes = np.array([4, -1, 0, 5, 3], dtype=np.int32)
    chars = b"sonyapplexyz"
    a = D.FlatStringsVector(sizes, chars)
    b = D.FlatStringsVector(sizes, np.frombuffer(chars, dtype=np.uint8))
    assert a._offsets is None and len(a) == 5
    assert a.tolist() == ["sony", None, "", "apple", "xyz"] == b.tolist()
    assert a.offsets.tolist() == [0, 4, 4, 4, 9]
    assert a == b and a == ["sony", None, "", "apple", "xyz"] and a[3] == "apple" and a[1] is None
    assert a[np.array([True, False, False, True, False])] == ["sony", "apple"]
    assert len(b.data) == len(chars) and bytes(b.data) == chars
    empty = D.FlatStringsVector(np.zeros(0, dtype=np.int32), np.zeros(0, dtype=np.uint8))
    assert len(empty) == 0 and empty.tolist() == []


def test_result_array_small_results_stay_in_ordinary_memory():
    """results below _capi.PINNED_MIN_BYTES do not touch the (GPU-side) result arena"""
    import numpy as np
    from dfdb_b200 import _capi
    a = _capi.result_array(10, np.int64)
    assert a.dtype == np.int64 and a.shape == (10,) and not a.any()
    assert _capi.result_array(0, np.uint8).shape == (1,)


def test_bench_plan_constants_match_the_plan_encoder(tmp_path, oracle):
    """bench.py's reference arm must not import the product, so it carries the benchmark query as constant plan bytes: they
    are the encoder's output for `t[(t.a .> 25) .& (t.a .<= 75), [:b]]` / `t[t.a .> 50, [:b]]` and the committed golden plan."""
    import json
    import bench
    import dfdb_b200 as D
    p = str(tmp_path / "t")
    oracle.gen_table(p, bench.SPEC, 1000, 256, 1, 1)
    t = D.open_table(p)
    assert D.plan_bytes(t[(t.a > 25) & (t.a <= 75), ["b"]].b) == bench.BENCH_PLAN
    assert D.plan_bytes(t[t.a > 50, ["b"]].b) == bench.C1_PLAN
    golden = json.load(open(os.path.join(os.path.dirname(__file__), "golden", "queries.json")))
    assert bytes.fromhex(next(q["plan"] for q in golden if q["name"] == "range_predicate_aggregate")) == bench.BENCH_PLAN
    t.close()


def test_zone_map_sidecar_is_optional_and_validated(tmp_path, oracle):
    """<id>.zmap (block index + zone maps) is only trusted while it matches the column file; any mismatch falls back to the
    header walk of the reference (skip_block, BlockStreams.jl:74-78).  Host side only: the sidecars here are hand-made."""
    import struct as st
    p = str(tmp_path / "t")
    oracle.gen_table(p, "q:Int64:iseq;b:Float64:funiform", 5 * 256 + 10, 256, 3, 1)
    t = D.open_table(p)
    L = _capi.lib()
    qid = t.getmeta("q").id
    nb = t.nblocks()
    assert nb == 6 and t.zonemap("q", 0) is None
    t.close()
    # write a sidecar by hand from the header walk of the oracle-side format description
    binp = os.path.join(p, f"{qid}.bin")
    raw = open(binp, "rb").read()
    pos = 8 + 4 + len("Int64")
    entries = []
    blk = 0
    while pos < len(raw):
        rows, origin, comp = st.unpack_from("<iqq", raw, pos)
        lo = blk * 256 + 1
        entries.append(st.pack("<qiiqqqQQ", pos + 20, rows, 1, origin, comp, 0, lo, lo + rows - 1))
        pos += 20 + comp
        blk += 1
    stt = os.stat(binp)
    head = b"DFDBZM01" + st.pack("<qqqqqiiii", 256, len(entries), qid, stt.st_size, stt.st_mtime_ns, 4, 0, 8, 1)
    zm = os.path.join(p, f"{qid}.zmap")
    open(zm, "wb").write(head + b"".join(entries))
    t = D.open_table(p)
    z = t.zonemap("q", 2)
    assert z is not None and (z.rows, z.min_i64, z.max_i64, z.has_value) == (256, 513, 768, 1)
    assert t.total_rows() == 5 * 256 + 10 and t.nblocks() == 6
    t.close()
    # wrong size recorded, truncated file, wrong magic, an index that does not tile the file: all ignored
    for bad in (head[:40] + st.pack("<q", stt.st_size + 1) + head[48:] + b"".join(entries),
                head + b"".join(entries)[:-8],
                b"DFDBZM99" + head[8:] + b"".join(entries),
                head + b"".join(entries[:2] + [st.pack("<qiiqqqQQ", 5, 256, 1, 2048, 10, 0, 1, 2)] + entries[3:])):
        open(zm, "wb").write(bad)
        t = D.open_table(p)
        assert t.zonemap("q", 0) is None and t.total_rows() == 5 * 256 + 10
        t.close()


def test_k1_flavour_is_chosen_from_the_token_stream():
    """dfdb_table_load picks a K1 decoder per column from a token sample of its blocks (api.cu: sample_flavour; no device needed):
    word-regular bodies -> verified word runs (2), match-only byte streams -> byte decoder (4), long sequences -> window decoder (3),
    everything else -> walker / consumer (1).  Bodies are the kinds of src/io/blocks.jl:2-33, compressed by the oracle's codec."""
    import numpy as np
    from dfdb_b200 import _capi
    from oracle import oracle as O
    O.build()
    L = _capi.lib()
    rng = np.random.default_rng(5)
    N = 65536
    brands = ["apple", "samsung", "huawai", "microsoft", "dell", "xbox", "sony", "intel"]
    bodies = {
        "rand100": (rng.integers(1, 101, N).astype(np.int64).tobytes(), 2),
        "sorted": (np.arange(1, N + 1, dtype=np.int64).tobytes(), 2),
        "brands": (O.block_body("String", [brands[i] for i in rng.integers(0, 8, N)], 0, N), 4),
        "missing_float": (O.block_body("Missing(Float64)", (rng.random(N), rng.random(N) < 0.1), 0, N), 3),
        "decimals": (O.block_body("String", [str(int(v)) for v in rng.integers(-2**31, 2**31, N)], 0, N), 1),
        "price_grid": ((1 + 0.1 * rng.integers(0, 19991, N)).astype(np.float64).tobytes(), 1),
        "tiny": (b"abc" * 10, -1),
    }
    for name, (body, want) in bodies.items():
        comp = O.compress_block(body)
        buf = np.frombuffer(comp, dtype=np.uint8)
        got = L.dfdb_lz4_classify_block(buf.ctypes.data, len(comp), len(body))
        assert got == want, (name, got, want)
