"""Predicate bits from the spec decoder: an aggregate whose predicate tests one column has that column's decoder write the
selection bits, and the TMA scan then stages only the aggregated column (api.cu run_aggregate, lz4_decode_spec.cu
flush_bits, scan_tma.cu's mask-in form).

- CPU: the lane-exact model of the decoder with the kernel's chunk rule (tests/models/spec_bits_model.py) writes the bits on real
  streams of every word-regular body kind, odd block lengths and blocks too short for the fast path; they must equal numpy's
  predicate over the decoded values.
- GPU: `aggregate` and `count` are bit for bit the same with the bits on and off (option pred_bits: 1 = always, 2 = never),
  under every forced decoder flavour, with zone maps on and off, on shards, in every residency mode, with float predicates
  (NaN, -0.0, `!=`), and a corrupt block still fails.
"""
import ctypes as C
import math
import os
from contextlib import contextmanager

import numpy as np
import pytest

from models.spec_bits_model import decode_block_spec_bits

BLOCK = 4096
ROWS = 5 * BLOCK + 1237          # an odd last block


@pytest.fixture(scope="module")
def O():
    from oracle import oracle
    oracle.build()
    return oracle


def _mask_words(sel):
    return np.packbits(np.concatenate([sel, np.zeros(-len(sel) % 32, bool)]), bitorder="little").view("<u4").tolist()


def test_spec_model_writes_the_predicate_bits(O):
    rng = np.random.default_rng(5)
    n = 16384
    bodies = {
        "rand100": rng.integers(1, 101, n),
        "rand1000": rng.integers(1, 1001, n),
        "sorted": np.arange(1, n + 1),           # runs of (2, 6) sequences (token 0x22)
        "rand4": rng.integers(1, 5, n),
        "odd": rng.integers(1, 101, 12345),      # a last mask word of 25 rows
        "short": rng.integers(1, 101, 37),       # shorter than the fast path's stream margin
        "tiny": rng.integers(1, 101, 3),
    }
    tests = {"rand100": (25, 75), "rand1000": (100, 900), "sorted": (1000, 9000), "rand4": (1, 2), "odd": (25, 75),
             "short": (25, 75), "tiny": (0, 100)}
    shapes = {}
    for name, vals in bodies.items():
        vals = vals.astype(np.int64)
        body = vals.tobytes()
        lo, hi = tests[name]
        exp = _mask_words((vals > lo) & (vals <= hi))
        for comp in (O.compress_block(body), O.lz4_compress(body, 1)):
            got, st, bits = decode_block_spec_bits(comp, len(body), lambda v: lo < (v - (1 << 64) if v >> 63 else v) <= hi)
            assert got == body, name
            assert bits == exp, name
            for k, v in st.items():
                shapes[k] = shapes.get(k, 0) + v
    assert all(shapes.get(k, 0) > 0 for k in ("fb", "fb1", "fb1b", "nfb", "one")), shapes


# ---- GPU: bits on and off give the same bits ------------------------------------------------------------------------------

@contextmanager
def option(name, value=1):
    from dfdb_b200 import _capi
    L = _capi.lib()
    _capi.check(L.dfdb_set_option(name.encode(), value))
    try:
        yield
    finally:
        _capi.check(L.dfdb_set_option(name.encode(), 0))


def _fields(a):
    from dfdb_b200 import _capi
    return tuple(np.float64(getattr(a, f)).tobytes() if t is C.c_double else getattr(a, f) for f, t in _capi.Agg._fields_)


@pytest.fixture(scope="module")
def table(tmp_path_factory, O):
    rng = np.random.default_rng(0xB175)
    p = str(tmp_path_factory.mktemp("predbits") / "t")
    a = rng.integers(1, 101, ROWS).astype(np.int64)
    s = np.arange(ROWS, dtype=np.int64)
    fvals = np.array([-0.0, 0.0, 1.5, math.nan, 2.5, -3.0, math.inf, 7.25])
    f = fvals[rng.integers(0, len(fvals), ROWS)]
    b = rng.random(ROWS) * 100 - 50
    b[rng.integers(0, ROWS, 50)] = -0.0
    vi = rng.integers(-2**62, 2**62, ROWS).astype(np.int64)
    O.write_table(p, [("a", "Int64", a), ("s", "Int64", s), ("f", "Float64", f), ("b", "Float64", b), ("vi", "Int64", vi)],
                  block_size=BLOCK)
    return p


def _queries(t):
    return [
        ((t.a > 25) & (t.a <= 75), "b"),
        (t.a != 50, "vi"),
        ((t.s >= 3000) & (t.s < 17000), "b"),     # zone maps rule out whole blocks
        (t.f > -0.0, "b"),
        (t.f != 1.5, "vi"),                         # NaN passes
        ((t.f >= -0.0) & (t.f != 2.5), "b"),
        (t.f != math.nan, "b"),
    ]


def _run(path, mode, rank=0, world=1):
    import dfdb_b200 as D
    t = D.open_table(path, mode=mode, rank=rank, world=world)
    try:
        out = []
        for pred, col in _queries(t):
            v = t[pred, :]
            out.append((_fields(D.aggregate(getattr(v, col))), D.count(v.a)))
        return out
    finally:
        t.close()


def _both(path, mode=1, rank=0, world=1):
    with option("pred_bits", 1):                 # (these tables are far below the size at which the bits pay)
        on = _run(path, mode, rank, world)
    with option("pred_bits", 2):
        off = _run(path, mode, rank, world)
    assert on == off


@pytest.mark.gpu
@pytest.mark.parametrize("flavour", [0, 2, 3, 4, 5, 6])
@pytest.mark.parametrize("zonemap", [True, False])
def test_bits_match_the_scan_under_every_flavour(table, flavour, zonemap):
    with option("lz4_flavour", flavour), option("no_zonemap", 0 if zonemap else 1):
        _both(table)


@pytest.mark.gpu
@pytest.mark.parametrize("world", [2, 3])
def test_bits_match_the_scan_on_shards(table, world):
    for rank in range(world):
        _both(table, rank=rank, world=world)


@pytest.mark.gpu
@pytest.mark.parametrize("mode", [0, 1, 2])
def test_bits_match_the_scan_in_every_residency_mode(table, mode):
    _both(table, mode=mode)


@pytest.mark.gpu
def test_bits_match_the_oracle(table, O):
    import dfdb_b200 as D
    t = D.open_table(table)
    ot = O.OracleTable(table)
    try:
        for pred, col in _queries(t):
            v = t[pred, [col]]
            ref = ot.aggregate(D.plan_bytes(v), 0)
            got = D.aggregate(getattr(t[pred, :], col))
            assert got.count == ref.count
    finally:
        ot.close()
        t.close()


@pytest.mark.gpu
def test_corrupt_block_still_fails(tmp_path, O):
    import dfdb_b200 as D
    p = str(tmp_path / "c")
    O.gen_table(p, "a:Int64:iuniform:1:100;b:Float64:funiform", 200000, 65536, 5, 2)
    f = os.path.join(p, "1.bin")
    raw = bytearray(open(f, "rb").read())
    raw[len(raw) // 2] ^= 0xFF
    raw[len(raw) // 2 + 1] ^= 0xFF
    open(f, "wb").write(raw)
    ot = O.OracleTable(p)

    def run():
        t = D.open_table(p)
        try:
            v = t[(t.a > 25) & (t.a <= 75), :]
            return _fields(D.aggregate(v.b))
        except (AssertionError, D.DfdbError) as e:   # (the API raises DFDB_ERR_CORRUPT as an AssertionError, like the reference)
            return ("error", str(e))
        finally:
            t.close()

    t0 = D.open_table(p)
    try:
        ref = ot.count(D.plan_bytes(t0[t0.a > 50, :]))
    except O.OracleError:
        ref = None
    finally:
        t0.close()
        ot.close()
    with option("pred_bits", 1):
        on = run()
    with option("pred_bits", 2):
        off = run()
    assert on == off
    if ref is None:
        assert on[0] == "error" and "decompression error" in on[1], on
