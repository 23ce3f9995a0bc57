#!/usr/bin/env python
"""make_golden.py -- writes the committed golden fixtures under tests/golden/.

The reference is Julia and cannot run in this image, and it ships no golden byte vectors of its own (its tests build
tables at run time and compare with an in-memory DataFrame, SURVEY.md section 4).  So the fixtures are made from the two
things that ARE fixed by the reference: its on-disk format (src/io/table_io.jl:9-19, filesystem.jl:14-23,
BlockStreams.jl:50-53, blocks.jl:2-33) and its codec, liblz4 (`LZ4_compress_fast`, acceleration 2, BlockStreams.jl:39-48),
which is present here as the system library (1.9.4).  Expected results are computed from the raw column data with plain
numpy / Python in this script -- never by the oracle and never by the CUDA path, which are the two things the fixtures
are there to check.

  tables/<name>/{meta.bin,<id>.bin}   tables in the reference's format, blocks compressed by the system liblz4
  tables.json                         per table: raw column data (lists; None = missing) and block size
  queries.json                        per query: table, the plan bytes (hex) the host-side plan algebra emits for it, and
                                      the expected count / selected 1-based row ids / materialized columns / aggregates
  lz4_vectors.json                    compressed blocks produced by the system liblz4 (base64) + sha256 of the body
  lz4_upstream.json                   what the system liblz4 makes of the inputs of tests/test_oracle_lz4.py (sha256 of its
                                      compressed streams; its LZ4_decompress_safe verdict on the damaged streams)

Run from the repo root:  python tests/golden/make_golden.py     (needs the system liblz4, liblz4.so.1)
"""
import base64
import ctypes as C
import hashlib
import json
import math
import os
import shutil
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import dfdb_b200 as D  # noqa: E402
from dfdb_b200 import R  # noqa: E402
from oracle import oracle as O  # noqa: E402

BRANDS = ["apple", "samsung", "huawai", "microsoft", "dell", "xbox", "sony", "intel"]   # docs/src/index.md:58


def opt(values, missing):
    return [None if m else v for v, m in zip(values, missing)]


def build_tables():
    rng = np.random.default_rng(0xDFDB)
    n = 2000
    a = rng.integers(1, 101, n).astype(np.int64)
    b = rng.random(n)
    s = [BRANDS[i] for i in rng.integers(0, 8, n)]
    ma_v, ma_m = rng.integers(1, 101, n).astype(np.int64), rng.random(n) < 0.1
    mb_v, mb_m = rng.random(n), rng.random(n) < 0.1
    sm_m = rng.random(n) < 0.1
    sm = [None if m else BRANDS[i] for m, i in zip(sm_m, rng.integers(0, 8, n))]
    sz = 1000
    tables = {
        # test/view.jl:8-15
        "view": dict(block_size=100, cols=[("a", "Int64", np.arange(1, sz + 1, dtype=np.int64)),
                                           ("b", "String", [str(i) for i in range(1, sz + 1)]),
                                           ("c", "Int64", np.arange(1, sz + 1, dtype=np.int64))]),
        # test/missings.jl:4
        "missings": dict(block_size=4, cols=[("x", "Missing(Int64)", (np.array([1, 0, 2, 3, 0, 5, 6, 0, 10, 11, 0], dtype=np.int64),
                                                                      np.array([0, 1, 0, 0, 1, 0, 0, 1, 0, 0, 1], dtype=bool)))]),
        # the shape of BASELINE.json's configs at toy size: ragged last block (2000 = 7 * 256 + 208)
        "mixed": dict(block_size=256, cols=[("a", "Int64", a), ("b", "Float64", b), ("s", "String", s),
                                            ("ma", "Missing(Int64)", (ma_v, ma_m)), ("mb", "Missing(Float64)", (mb_v, mb_m)),
                                            ("sm", "Missing(String)", sm)]),
    }
    return tables


def raw(col):
    name, ts, data = col
    if ts.startswith("Missing(") and "String" not in ts:
        return opt(data[0].tolist(), data[1].tolist())
    return data.tolist() if isinstance(data, np.ndarray) else list(data)


def sys_compress(lib, body, accel):
    cap = lib.LZ4_compressBound(len(body))
    buf = C.create_string_buffer(cap)
    n = lib.LZ4_compress_fast(body, buf, len(body), cap, accel)
    return buf.raw[:n]


def upstream_codec(lib):
    """lz4_upstream.json: upstream's compressed streams of test_oracle_lz4's bodies at accelerations 1 / 2 / 8, and upstream's
    LZ4_decompress_safe on its damaged streams (sha256 of the output when it accepts one, null when it refuses)."""
    import test_oracle_lz4 as T

    def sha(b):
        return hashlib.sha256(b).hexdigest()

    comp = {}
    for name, body in T._bodies(O).items():
        streams = {str(a): sys_compress(lib, body, a) for a in (1, 2, 8)}
        comp[name] = {"body_sha256": sha(body), "accel": {a: {"size": len(c), "sha256": sha(c)} for a, c in streams.items()}}
    body, good, streams = T.corrupt_streams(O)
    verdicts = []
    for bad in streams:
        out = C.create_string_buffer(len(body))
        verdicts.append(sha(out.raw) if lib.LZ4_decompress_safe(bad, out, len(bad), len(body)) == len(body) else None)
    return {"compress": comp, "corrupt": {"good_sha256": sha(good), "verdicts": verdicts}}


def main():
    if O.system_liblz4() is None:
        raise SystemExit("the system liblz4 is required: the fixtures must carry the reference codec's own streams")
    shutil.rmtree(os.path.join(HERE, "tables"), ignore_errors=True)
    tables = build_tables()
    tj = {}
    for name, t in tables.items():
        path = os.path.join(HERE, "tables", name)
        os.makedirs(os.path.dirname(path), exist_ok=True)
        O.write_table(path, t["cols"], block_size=t["block_size"], prefer_system_lz4=True)
        tj[name] = {"block_size": t["block_size"], "columns": {c[0]: {"type": c[1], "data": raw(c)} for c in t["cols"]}}
    json.dump(tj, open(os.path.join(HERE, "tables.json"), "w"))

    mixed = {k: v["data"] for k, v in tj["mixed"]["columns"].items()}
    view = {k: v["data"] for k, v in tj["view"]["columns"].items()}
    n = len(mixed["a"])
    queries = []

    def add(name, table, v, rows0, cols, agg=None):
        """rows0: expected selected 0-based rows; cols: {name: list}; plan bytes from the host-side plan algebra"""
        q = {"name": name, "table": table, "plan": D.plan_bytes(v).hex(), "count": len(rows0), "rows": [int(r) + 1 for r in rows0],
             "columns": cols}
        if agg is not None:
            q["aggregate"] = agg
        queries.append(q)

    t = D.open_table(os.path.join(HERE, "tables", "mixed"))
    tv = D.open_table(os.path.join(HERE, "tables", "view"))
    tm = D.open_table(os.path.join(HERE, "tables", "missings"))
    # configs[0]/[1]: range predicate + aggregate of b
    sel = [i for i in range(n) if 25 < mixed["a"][i] <= 75]
    bs = [mixed["b"][i] for i in sel]
    add("range_predicate_aggregate", "mixed", t[(t.a > 25) & (t.a <= 75), ["b"]], sel, {"b": bs},
        {"count": len(bs), "sum": math.fsum(bs), "min": min(bs), "max": max(bs)})
    sel = [i for i in range(n) if mixed["a"][i] > 50]
    add("docs_example", "mixed", t[t.a > 50, ["b"]], sel, {"b": [mixed["b"][i] for i in sel]},
        {"count": len(sel), "sum": math.fsum(mixed["b"][i] for i in sel)})
    # reductions over computed columns (test/columnbroadcast.jl:28-33,55-60): sum / extrema of a broadcast expression
    sel = [i for i in range(n) if mixed["a"][i] > 50]
    vals = [mixed["a"][i] * 2 + 1 for i in sel]
    add("computed_int_aggregate", "mixed", t[t.a > 50, ["a"]], sel, {"a": [mixed["a"][i] for i in sel]},
        {"expr": "a*2+1", "count": len(vals), "sum_i": sum(vals), "min_i": min(vals), "max_i": max(vals)})
    fvals = [mixed["a"][i] * mixed["b"][i] for i in sel]
    add("computed_float_aggregate", "mixed", t[t.a > 50, ["b"]], sel, {"b": [mixed["b"][i] for i in sel]},
        {"expr": "a*b", "count": len(fvals), "sum": math.fsum(fvals), "min": min(fvals), "max": max(fvals)})
    # configs[2]: string equality / prefix + projection
    sel = [i for i in range(n) if mixed["s"][i] == "sony"]
    add("string_equality", "mixed", t[t.s == "sony", ["s", "a"]], sel, {"s": [mixed["s"][i] for i in sel], "a": [mixed["a"][i] for i in sel]})
    sel = [i for i in range(n) if mixed["s"][i].startswith("s")]
    add("string_prefix", "mixed", t[D.startswith(t.s, "s"), ["s"]], sel, {"s": [mixed["s"][i] for i in sel]})
    # configs[3]: predicate over missing-bearing columns, four projected columns
    sel = [i for i in range(n) if mixed["ma"][i] is not None and mixed["ma"][i] > 50 and mixed["mb"][i] is not None and mixed["mb"][i] < 0.5]
    add("missing_predicate", "mixed", t[D.coalesce(t.ma > 50, False) & D.coalesce(t.mb < 0.5, False), ["ma", "mb", "sm", "b"]], sel,
        {k: [mixed[k][i] for i in sel] for k in ("ma", "mb", "sm", "b")})
    sel = [i for i in range(n) if mixed["sm"][i] is None]
    add("ismissing_strings", "mixed", t[D.ismissing(t.sm), ["a", "sm"]], sel, {"a": [mixed["a"][i] for i in sel], "sm": [None] * len(sel)})
    # selection.jl:94-111: range stages rank the survivors of the earlier stages, offsets run across blocks
    s1 = list(range(100, 1900))
    s2 = [i for i in s1 if mixed["a"][i] > 50]
    s3 = s2[9:300:3]
    add("range_after_predicate", "mixed", t[R(101, 1900), :][t.a > 50, :][R(10, 3, 300), ["a", "s"]], s3,
        {"a": [mixed["a"][i] for i in s3], "s": [mixed["s"][i] for i in s3]})
    # test/view.jl:19-50
    sel = [i for i in range(1000) if view["a"][i] % 50 == 0 and view["c"][i] < 930]
    v = D.selection(D.selection(D.DFView(tv), tv.a % 50 == 0), tv.c < 930)
    add("view_jl_mod50", "view", v, sel, {k: [view[k][i] for i in sel] for k in ("a", "b", "c")})
    # test/missings.jl
    x = tj["missings"]["columns"]["x"]["data"]
    add("missings_full", "missings", D.DFView(tm), list(range(len(x))), {"x": x})
    sel = [i for i in range(len(x)) if x[i] is not None and x[i] > 2]
    add("missings_gt2", "missings", tm[D.coalesce(tm.x > 2, False), ["x"]], sel, {"x": [x[i] for i in sel]})
    json.dump(queries, open(os.path.join(HERE, "queries.json"), "w"))

    # codec vectors: the system liblz4's own compressed streams
    rng = np.random.default_rng(5)
    bodies = {
        "int64_rand100": rng.integers(1, 101, 2048).astype(np.int64).tobytes(),
        "int64_seq": np.arange(1, 2049, dtype=np.int64).tobytes(),
        "float64_grid": (1 + 0.1 * rng.integers(0, 19991, 2048)).astype(np.float64).tobytes(),
        "float64_uniform": rng.random(512).tobytes(),
        "missing_float64": O.block_body("Missing(Float64)", (rng.random(2048), rng.random(2048) < 0.1), 0, 2048),
        "strings_brands": O.block_body("String", [BRANDS[i] for i in rng.integers(0, 8, 2048)], 0, 2048),
        "zeros": bytes(5000),
        "short": b"abc",
        "empty_literal": b"",
    }
    lib = O.system_liblz4()
    vec = []
    for k, body in bodies.items():
        for accel in (1, 2):
            comp = sys_compress(lib, body, accel) if body else b"\x00"
            vec.append({"name": k, "accel": accel, "origin": len(body), "sha256": hashlib.sha256(body).hexdigest(),
                        "compressed": base64.b64encode(comp).decode()})
    json.dump(vec, open(os.path.join(HERE, "lz4_vectors.json"), "w"))
    json.dump(upstream_codec(lib), open(os.path.join(HERE, "lz4_upstream.json"), "w"), indent=0)
    print("wrote", len(tables), "tables,", len(queries), "queries,", len(vec), "codec vectors, upstream codec expectations")


if __name__ == "__main__":
    main()
