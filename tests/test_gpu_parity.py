"""GPU parity tests: the CUDA library, called through its C ABI, against the CPU oracle and the reference's
known-answer cases.  Bar: bit-exact masks, row indices, counts, integer aggregates, strings and missings;
Float64 sums within 1e-12 relative of the oracle's compensated (Kahan/Neumaier) sum."""
import ctypes as C
import os

import numpy as np
import pytest

import cases
import dfdb_b200 as D
import fixtures
from dfdb_b200 import R, _capi
from engines import GpuEngine, OracleEngine

pytestmark = pytest.mark.gpu

FSUM_RTOL = 1e-12


@pytest.fixture(scope="module", autouse=True)
def _init():
    _capi.init(0)
    yield


# ---- K1 codec hook -------------------------------------------------------------------------------------

def _bodies(oracle):
    rng = np.random.default_rng(7)
    N = 65536
    brands = ["apple", "samsung", "huawai", "microsoft", "dell", "xbox", "sony", "intel"]
    out = {
        "rand100": rng.integers(1, 101, N).astype(np.int64).tobytes(),
        "rand1000": rng.integers(1, 1001, N).astype(np.int64).tobytes(),
        "iseq": np.arange(1, N + 1, dtype=np.int64).tobytes(),
        "price": (1 + 0.1 * rng.integers(0, 19991, N)).astype(np.float64).tobytes(),
        "f01": rng.random(N).tobytes(),
        "zeros": bytes(100000),
        "short3": b"abc",
        "len13": b"0123456789abc",
        "len1": b"x",
        "rle_then_random": bytes(5000) + rng.integers(0, 256, 7001).astype(np.uint8).tobytes() + b"ab" * 3000,
        "brands": oracle.block_body("String", [brands[i] for i in rng.integers(0, 8, N)], 0, N),
        "missing_int": oracle.block_body("Missing(Int64)", (rng.integers(1, 101, N).astype(np.int64), rng.random(N) < 0.1), 0, N),
        # literal-heavy: nearly every token carries a literal-length extension
        "missing_float": oracle.block_body("Missing(Float64)", (rng.random(N), rng.random(N) < 0.1), 0, N),
        "decimals": oracle.block_body("String", [str(int(v)) for v in rng.integers(-2**31, 2**31, N)], 0, N),
        # long matches (match-length extensions) between long literal runs
        "repeats": b"".join(rng.integers(0, 256, 700).astype(np.uint8).tobytes() * 3 for _ in range(40)),
        "small_ints": rng.integers(0, 4, 30011).astype(np.uint8).tobytes(),
        "period3": (b"abc" * 20000)[:50001],
        "odd_sizes": rng.integers(0, 2, 777).astype(np.uint8).tobytes(),
    }
    return out


def _gpu_decode(blocks, origins):
    L = _capi.lib()
    n = len(blocks)
    comp = b"".join(blocks)
    coff = np.cumsum([0] + [len(b) for b in blocks[:-1]]).astype(np.int64)
    clen = np.array([len(b) for b in blocks], dtype=np.int64)
    ooff = np.cumsum([0] + list(origins[:-1])).astype(np.int64)
    orig = np.array(origins, dtype=np.int64)
    out = np.zeros(max(int(orig.sum()), 1), dtype=np.uint8)
    status = np.zeros(n, dtype=np.int32)
    cbuf = np.frombuffer(comp, dtype=np.uint8)
    _capi.check(L.dfdb_lz4_decode_blocks(cbuf.ctypes.data, coff.ctypes.data, clen.ctypes.data, out.ctypes.data, ooff.ctypes.data,
                                         orig.ctypes.data, n, status.ctypes.data))
    return [bytes(out[o:o + s]) for o, s in zip(ooff, orig)], status


def _set_variant(variant):
    """K1 variants: the warp-per-block decoder with verified runs, the lane-per-block decoder, the walker / consumer decoder and the sequential decoder."""
    L = _capi.lib()
    L.dfdb_set_option(b"lz4_simple", 0)
    L.dfdb_set_option(b"lz4_flavour", 0)
    L.dfdb_set_option(b"lane_hot", -1)
    if variant == "v3":
        _capi.check(L.dfdb_set_option(b"lz4_flavour", 2))
    elif variant == "lane":
        _capi.check(L.dfdb_set_option(b"lz4_flavour", 3))
    elif variant == "long":           # warp per block, one sequence at a time, headers parsed out of a shared-memory window of the stream
        _capi.check(L.dfdb_set_option(b"lz4_flavour", 5))
    elif variant == "bytes":          # warp per block, bare-match byte streams: verified positions, byte copies by pointer jumping
        _capi.check(L.dfdb_set_option(b"lz4_flavour", 6))
    elif variant == "spec":           # warp per block, plain token runs verified in parallel
        _capi.check(L.dfdb_set_option(b"lz4_flavour", 4))
    elif variant == "lane_hot":       # the lane-per-block decoder on the hot-step schedule of word-regular columns
        _capi.check(L.dfdb_set_option(b"lz4_flavour", 3))
        _capi.check(L.dfdb_set_option(b"lane_hot", 1))
    elif variant is not None:
        _capi.check(L.dfdb_set_option(variant.encode(), 1))


@pytest.mark.parametrize("variant", ["spec", "long", "bytes", "lane", "lane_hot", "v3", "lz4_simple"], ids=["verified_runs", "long_sequences", "byte_streams", "lane_per_block", "lane_hot_steps", "walker_consumer", "sequential"])
def test_lz4_decode_matches_reference_codec(oracle, variant):
    """read_block BlockStreams.jl:101-119: decoded bytes are determined by the LZ4 block format."""
    bodies = _bodies(oracle)
    names = list(bodies)
    blocks = [oracle.compress_block(bodies[k]) for k in names] + [oracle.lz4_compress(bodies[k], 1) for k in names]
    origins = [len(bodies[k]) for k in names] * 2
    _set_variant(variant)
    try:
        got, status = _gpu_decode(blocks, origins)
    finally:
        _set_variant(None)
    for i, k in enumerate(names + names):
        assert status[i] == 0, (k, status[i])
        assert got[i] == bodies[k], f"decoded bytes differ for {k} (first diff at {next(j for j in range(len(got[i])) if got[i][j] != bodies[k][j])})"


@pytest.mark.parametrize("variant", ["spec", "long", "bytes", "lane", "lane_hot", "v3"], ids=["verified_runs", "long_sequences", "byte_streams", "lane_per_block", "lane_hot_steps", "walker_consumer"])
def test_lz4_decode_many_small_blocks(oracle, variant):
    """More blocks than the persistent decoder has slots (148 SMs x 87), ragged sizes, every body kind: slots are
    reused, rings wrap, windows re-base after long literal / match runs."""
    rng = np.random.default_rng(11)
    kinds = list(_bodies(oracle).values())
    pool = []
    for body in kinds:
        for _ in range(6):
            n = int(rng.integers(1, min(len(body), 6000) + 1))
            s0 = int(rng.integers(0, len(body) - n + 1))
            pool.append(body[s0:s0 + n])
    pool.append(b"")
    comp = [oracle.compress_block(b) if b else b"\x00" for b in pool]
    idx = rng.integers(0, len(pool), 14000)
    blocks = [comp[i] for i in idx]
    origins = [len(pool[i]) for i in idx]
    _set_variant(variant)
    try:
        got, status = _gpu_decode(blocks, origins)
    finally:
        _set_variant(None)
    bad = [k for k in range(len(idx)) if status[k] != 0 or got[k] != pool[idx[k]]]
    assert not bad, f"{len(bad)} of {len(idx)} blocks differ, first: block {bad[0]} (pool {idx[bad[0]]}, origin {origins[bad[0]]}, status {status[bad[0]]})"


@pytest.mark.parametrize("variant", ["spec", "long", "bytes", "lane", "lane_hot", "v3"], ids=["verified_runs", "long_sequences", "byte_streams", "lane_per_block", "lane_hot_steps", "walker_consumer"])
def test_lz4_decode_rejects_corrupt_blocks(oracle, variant):
    """@assert size == sizes.origin "decompression error" (BlockStreams.jl:112)"""
    body = np.random.default_rng(3).integers(1, 101, 4096).astype(np.int64).tobytes()
    good = oracle.compress_block(body)
    bad_trunc = good[: len(good) // 2]
    bad_origin = good
    bad_offset = bytes([0x00, 0xFF, 0xFF]) + good          # match with offset 65535 before any output
    _set_variant(variant)
    try:
        got, status = _gpu_decode([good, bad_trunc, bad_origin, bad_offset], [len(body), len(body), len(body) - 8, len(body)])
    finally:
        _set_variant(None)
    assert status[0] == 0 and got[0] == body
    assert status[1] != 0 and status[2] != 0 and status[3] != 0
    for blk, org in [(bad_trunc, len(body)), (bad_origin, len(body) - 8), (bad_offset, len(body))]:
        with pytest.raises(oracle.OracleError):
            oracle.lz4_decompress(blk, org)


@pytest.mark.parametrize("variant", ["spec", "long", "bytes", "lane", "lane_hot", "v3"], ids=["verified_runs", "long_sequences", "byte_streams", "lane_per_block", "lane_hot_steps", "walker_consumer"])
def test_lz4_decode_fuzzed_streams(oracle, variant):
    """LZ4_decompress_safe contract on damaged streams (@assert size == sizes.origin, BlockStreams.jl:110-112): no crash, no
    out-of-bounds write, a stream is refused exactly when the CPU codec refuses it, and an accepted one decodes to the same
    bytes."""
    rng = np.random.default_rng(23)
    brands = ["apple", "samsung", "huawai", "microsoft", "dell", "xbox", "sony", "intel"]
    bodies = [rng.integers(1, 101, 4096).astype(np.int64).tobytes(),
              oracle.block_body("String", [brands[i] for i in rng.integers(0, 8, 4096)], 0, 4096),
              oracle.block_body("Missing(Float64)", (rng.random(4096), rng.random(4096) < 0.1), 0, 4096)]
    blocks, origins, expect = [], [], []
    for body in bodies:
        good = oracle.compress_block(body)
        for _ in range(100):
            bad = bytearray(good)
            for _ in range(int(rng.integers(1, 4))):
                bad[int(rng.integers(0, len(bad)))] = int(rng.integers(0, 256))
            if rng.random() < 0.2:
                bad = bad[: int(rng.integers(1, len(bad)))]
            bad = bytes(bad)
            try:
                ref = oracle.lz4_decompress(bad, len(body))
            except oracle.OracleError:
                ref = None
            blocks.append(bad)
            origins.append(len(body))
            expect.append(ref)
    _set_variant(variant)
    try:
        got, status = _gpu_decode(blocks, origins)
    finally:
        _set_variant(None)
    for k, ref in enumerate(expect):
        if ref is not None:
            assert status[k] == 0 and got[k] == ref, f"stream {k}: the CPU codec accepts it, GPU status {status[k]}"
        else:
            # liblz4's end-of-block rules are enforced on the device (the lane-per-block decoder gives the verdict for every
            # flavour): identical accept / reject
            assert status[k] != 0, f"stream {k}: the CPU codec rejects it, the GPU decoder accepted it"


# ---- reference known-answer cases through the C ABI -----------------------------------------------------------

@pytest.fixture(scope="module")
def ref_table(tmp_path_factory, oracle):
    p = str(tmp_path_factory.mktemp("ref") / "test_data")
    data = fixtures.make_reference_fixture(oracle, p)
    t = D.open_table(p)
    yield GpuEngine(), t, data
    t.close()


@pytest.mark.parametrize("case", [cases.case_view_full, cases.case_view_predicates, cases.case_view_projections,
                                  cases.case_range_indexing, cases.case_range_composition, cases.case_column_broadcast,
                                  cases.case_columns, cases.case_aggregates], ids=lambda f: f.__name__)
def test_reference_fixture_cases(ref_table, case):
    case(*ref_table)


@pytest.mark.parametrize("block_size", [100, 50, 7])
def test_selection_stages(tmp_path, oracle, block_size):
    p = str(tmp_path / "sel")
    data = fixtures.make_selection_fixture(oracle, p, block_size)
    cases.case_selection_stages(GpuEngine(), D.open_table(p), data)


def test_broadcast_eval(tmp_path, oracle):
    p = str(tmp_path / "bc")
    data = fixtures.make_broadcast_fixture(oracle, p)
    cases.case_broadcast_eval(GpuEngine(), D.open_table(p), data)


@pytest.mark.parametrize("block_size", [4, 64, 3])
def test_missings(tmp_path, oracle, block_size):
    p = str(tmp_path / "ms")
    fixtures.make_missing_fixture(oracle, p, block_size)
    cases.case_missings(GpuEngine(), D.open_table(p), None)


@pytest.mark.parametrize("block_size", [4, 64])
def test_flat_strings(tmp_path, oracle, block_size):
    p = str(tmp_path / "st")
    fixtures.make_strings_fixture(oracle, p, block_size)
    cases.case_flat_strings(GpuEngine(), D.open_table(p), None)


# ---- seeded synthetic tables: GPU vs oracle on the same files ---------------------------------------------------

SPEC = ("a:Int64:iuniform:1:100;b:Float64:funiform;s:String:brands;"
        "ma:Missing(Int64):iuniform:1:100:m=0.1;mb:Missing(Float64):funiform:m=0.1;ms:Missing(String):decimal:m=0.05;"
        "p:Float64:fgrid:1:0.1:2000;q:Int64:iseq")


@pytest.fixture(scope="module")
def synth(tmp_path_factory, oracle):
    p = str(tmp_path_factory.mktemp("synth") / "t")
    nrows = 5 * 65536 + 12345
    oracle.gen_table(p, SPEC, nrows, 65536, 0xDFDB0002, 4)
    t = D.open_table(p)
    ot = oracle.OracleTable(p)
    yield t, ot, nrows
    t.close()
    ot.close()


def _plans(t):
    return {
        "c1_gt50": t[t.a > 50, ["b"]],
        "c2_range_pred": t[(t.a > 25) & (t.a <= 75), ["b", "a"]],
        "float_const_on_int": t[(t.a > 25.5) & (t.a <= 75.0), ["a"]],
        "float_pred": t[(t.b < 0.25) | (t.b >= 0.9), ["b"]],
        "str_eq": t[t.s == "sony", ["s"]],
        "str_prefix": t[D.startswith(t.s, "s"), ["s", "a"]],
        "c4_missing_and": t[D.coalesce(t.ma > 50, False) & D.coalesce(t.mb < 0.5, False), ["ma", "mb", "a", "b"]],
        "missing_str": t[D.coalesce(D.startswith(t.ms, "-1"), False), ["ms", "ma"]],
        "ismissing": t[D.ismissing(t.ms) | D.ismissing(t.mb), ["ms", "mb"]],
        "arith": t[(t.a * 2 + t.q) % 7 == 0, ["q"]],
        "mixed_cmp": t[(t.p > t.a) & (t.q % 1000 < 10), ["p", "q"]],
        "isin": t[D.isin(t.a, [3, 5, 99, 1000]), ["a"]],
        "range_first": t[R(70000, 3, 250000), ["q", "s"]],
        "range_pred_range": t[R(1000, 300000), :][t.a > 90, :][R(5, 7, 20000), ["q", "a"]],
        "indexvec": t[[1, 65536, 65537, 131072, 340000, 17], ["q"]],
        "pred_then_index": t[t.a == 7, :][[1, 2, 3, 500, 501, 3000], ["q", "a"]],
        "computed_cols": t[t.a < 3, {"x": t.a * 2 + 1, "y": t.b / 2, "z": t.a > 1, "w": t.ma + 1}],
        "empty": t[t.a > 1000, ["a", "s"]],
    }


def _same_cols(got, exp):
    assert len(got) == len(exp)
    for g, e in zip(got, exp):
        if isinstance(g, D.FlatStringsVector):
            assert np.array_equal(g.sizes, e.sizes) and g.data == e.chars
        elif isinstance(g, np.ma.MaskedArray):
            ev, em = e
            assert np.array_equal(np.ma.getmaskarray(g), em)
            assert np.array_equal(g.data[~em], ev[~em])
        else:
            assert g.dtype == e.dtype and np.array_equal(g, e), (g[:5], e[:5])


def test_synthetic_plans_match_oracle(synth):
    t, ot, nrows = synth
    for name, v in _plans(t).items():
        pb = D.plan_bytes(v)
        exp_mask = ot.mask(pb)
        assert np.array_equal(D.selection_mask(v), exp_mask), name
        assert D.nrow(v) == ot.count(pb) == int(exp_mask.sum()), name
        assert np.array_equal(D.selection_indices(v), np.nonzero(exp_mask)[0] + 1), name
        _same_cols(D.materialize(v).columns, ot.materialize(pb))


def _check_agg(got, ref, what):
    assert got.count == ref.count and got.nmissing == ref.nmissing, what
    if ref.count - ref.nmissing == 0:
        return
    if ref.kind in (12, 13):
        gsum = got.sum_f64 + got.sum_f64_lo
        assert abs(gsum - ref.sum_kahan) <= FSUM_RTOL * abs(ref.sum_kahan), (what, gsum, ref.sum_kahan)
        assert got.min_f64 == ref.min_f64 and got.max_f64 == ref.max_f64, what
    else:
        assert got.sum_i64 == ref.sum_i64 and got.min_i64 == ref.min_i64 and got.max_i64 == ref.max_i64, what


def test_synthetic_aggregates_match_oracle(synth):
    t, ot, nrows = synth
    views = {
        "all_b": t[:, :], "c1": t[t.a > 50, :], "c2": t[(t.a > 25) & (t.a <= 75), :],
        "missing": t[D.coalesce(t.ma > 50, False) & D.coalesce(t.mb < 0.5, False), :],
        "str": t[t.s == "dell", :], "ranges": t[R(1000, 300000), :][t.a > 90, :][R(5, 7, 20000), :],
        "none": t[t.a > 1000, :],
    }
    for name, v in views.items():
        for col in ["a", "b", "ma", "mb", "p", "q"]:
            c = getattr(v, col)
            _check_agg(D.aggregate(c), ot.aggregate(D.plan_bytes(c), 0), (name, col))
    v = views["c2"]
    assert D.sum(v.a) == int(ot.aggregate(D.plan_bytes(v.a), 0).sum_i64)
    assert D.minimum(v.b) == ot.aggregate(D.plan_bytes(v.b), 0).min_f64
    assert D.sum(views["missing"].ma) is not None and D.sum(t[:, :].ma) is None      # missing + x == missing
    with pytest.raises(D.ArgumentError):
        D.minimum(views["none"].a)                                                    # empty collection
    assert D.sum(views["none"].b) == 0.0
    assert D.sum(D.ismissing(t.ms)) == int(ot.mask(D.plan_bytes(t[D.ismissing(t.ms), :])).sum())


def test_aggregates_over_computed_columns(synth, tmp_path, oracle):
    """sum / minimum / maximum / count of a broadcast column (test/columnbroadcast.jl:28-33,55-60: `sum(t.a .* t.c)`,
    reductions over `v.price .* 2`): the Base folds run over the VM values of the selected rows."""
    t, ot, nrows = synth
    v = t[(t.a > 25) & (t.a <= 75), :]
    vm = t[D.coalesce(t.ma > 50, False), :]
    cols = {
        "int_arith": v.a * 2 + v.q,
        "flt_arith": v.b * 2.5 - 1.0,
        "mixed": v.a * v.b,
        "bool": v.b < 0.5,
        "missing_int": t.ma + t.a,                                                  # missing where ma is
        "missing_flt": vm.mb * 2.0,
        "all_rows": t.a % 7,
        "none": t[t.a > 1000, :].a * 3,
    }
    for name, c in cols.items():
        got, ref = D.aggregate(c), ot.aggregate(D.plan_bytes(c), 0)
        _check_agg(got, ref, name)
        again = D.aggregate(c)
        assert (got.sum_f64, got.sum_f64_lo, got.sum_i64) == (again.sum_f64, again.sum_f64_lo, again.sum_i64), name
    assert D.sum(cols["int_arith"]) == int(ot.aggregate(D.plan_bytes(cols["int_arith"]), 0).sum_i64)
    assert D.maximum(cols["flt_arith"]) == ot.aggregate(D.plan_bytes(cols["flt_arith"]), 0).max_f64
    assert D.sum(cols["missing_int"]) is None                                         # missing + x == missing
    # DivideError raised by the expression surfaces from the reduction as well (broadcast.jl:96-133 evaluates it per row)
    p = str(tmp_path / "div")
    oracle.write_table(p, [("x", "Int64", np.arange(-3, 4, dtype=np.int64))], block_size=4)
    td = D.open_table(p)
    with pytest.raises(ZeroDivisionError):
        D.sum(10 % td.x)                                                           # rem(10, 0)
    td.close()


def test_residency_modes_and_kernel_variants_agree(synth, oracle):
    t, ot, nrows = synth
    v = t[(t.a > 25) & (t.a <= 75), ["b"]]
    ref = ot.aggregate(D.plan_bytes(v.b), 0)
    L = _capi.lib()
    base = D.aggregate(v.b)
    for mode in (D.LOAD_HOST, D.LOAD_DECODED, D.LOAD_HBM):
        t2 = D.open_table(t.path, mode=mode)
        v2 = t2[(t2.a > 25) & (t2.a <= 75), ["b"]]
        for _ in range(2):
            r = D.aggregate(v2.b)
            _check_agg(r, ref, mode)
            # fixed combination order: identical bits run to run and across residency modes
            assert (r.sum_f64, r.sum_f64_lo, r.count) == (base.sum_f64, base.sum_f64_lo, base.count)
        t2.close()
    for opt in (b"no_tma", b"no_wide", b"no_fused", b"lz4_simple", b"no_alias"):
        L.dfdb_set_option(opt, 1)
        try:
            t2 = D.open_table(t.path)
            v2 = t2[(t2.a > 25) & (t2.a <= 75), ["b"]]
            r1, r2 = D.aggregate(v2.b), D.aggregate(v2.b)
            # uniform Float64 is incompressible: every block of b is a stored block, referenced in place unless no_alias
            nst, byt = C.c_int64(), C.c_int64()
            _capi.check(L.dfdb_table_column_stored(t2._h, t2.getmeta("b").id, C.byref(nst), C.byref(byt)))
            assert nst.value == (0 if opt == b"no_alias" else t2.nblocks()), (opt, nst.value)
            _check_agg(r1, ref, opt)
            assert (r1.sum_f64, r1.sum_f64_lo) == (r2.sum_f64, r2.sum_f64_lo)
            for col in ("a", "ma", "mb", "q"):
                c2 = getattr(t2[D.coalesce(t2.ma > 50, False) & (t2.b < 0.5), :], col)
                _check_agg(D.aggregate(c2), ot.aggregate(D.plan_bytes(c2), 0), (opt, col))
            assert np.array_equal(D.selection_mask(v2), D.selection_mask(v))
            t2.close()
        finally:
            L.dfdb_set_option(opt, 0)


def test_decode_scan_overlap_matches_the_plain_path(tmp_path, oracle):
    """A shard with more blocks than the decoder keeps in flight (148 SMs x 60) decodes in rounds, and the scan of the
    earlier rounds runs beside the decode of the last one (api.cu ensure_decoded / run_aggregate).  Same partials, same
    fixed combination order: the result must be bit-identical to the one-kernel-after-the-other path."""
    p = str(tmp_path / "many_blocks")
    nrows, bs = 1_400_000, 128                                   # 10 938 blocks per column
    oracle.gen_table(p, "a:Int64:iuniform:1:100;b:Float64:funiform;c:Int64:iseq", nrows, bs, 0xDFDB0099, 4)
    ot = oracle.OracleTable(p)
    L = _capi.lib()
    results = {}
    for no_overlap in (0, 1):
        _capi.check(L.dfdb_set_option(b"no_overlap", no_overlap))
        try:
            t = D.open_table(p)
            for name, mk in {"b": lambda t: t[(t.a > 25) & (t.a <= 75), ["b"]].b, "c": lambda t: t[t.a > 50, ["c"]].c,
                             "count": lambda t: t[t.c > 700_000, ["a"]].a}.items():
                col = mk(t)
                r1, r2 = D.aggregate(col), D.aggregate(col)
                _check_agg(r1, ot.aggregate(D.plan_bytes(col), 0), (no_overlap, name))
                assert (r1.sum_f64, r1.sum_f64_lo, r1.sum_i64, r1.count) == (r2.sum_f64, r2.sum_f64_lo, r2.sum_i64, r2.count)
                results[(no_overlap, name)] = (r1.sum_f64, r1.sum_f64_lo, r1.sum_i64, r1.count, r1.min_f64, r1.max_f64, r1.min_i64, r1.max_i64)
            t.close()
        finally:
            L.dfdb_set_option(b"no_overlap", 0)
    for name in ("b", "c", "count"):
        assert results[(0, name)] == results[(1, name)], name
    ot.close()


@pytest.mark.parametrize("bs", [128, 65536])
def test_filter_aggregate_over_word_regular_columns_matches_the_oracle(tmp_path, oracle, bs):
    """Filter + aggregate whose predicate column still has to be decoded and is word-regular (the spec decoder, then the
    scan; api.cu run_aggregate).  Every result matches the oracle and is reproducible bit for bit; the decoded column it
    leaves behind serves the next query like any other decode."""
    p = str(tmp_path / "spec_filter")
    nrows = 1_000_003 if bs == 128 else 3_000_017                  # (a partial last block)
    oracle.gen_table(p, "a:Int64:iuniform:1:100;b:Float64:funiform;c:Int64:iseq;d:Int64:iuniform:-5:5", nrows, bs, 0xDFDB0F5E, 4)
    ot = oracle.OracleTable(p)
    L = _capi.lib()
    queries = {
        "sum b": lambda t: t[(t.a > 25) & (t.a <= 75), ["b"]].b,
        "sum c": lambda t: t[t.a > 50, ["c"]].c,
        "sum d": lambda t: t[(t.a != 7) & (t.a != 93), ["d"]].d,
        "point": lambda t: t[t.a == 13, ["c"]].c,
        "none": lambda t: t[t.a > 1000, ["b"]].b,
        "all": lambda t: t[t.a >= 1, ["b"]].b,
    }
    def key(r):
        return (r.sum_f64, r.sum_f64_lo, r.sum_i64, r.count, r.min_f64, r.max_f64, r.min_i64, r.max_i64)
    for name, mk in queries.items():
        runs = []
        for run in range(2):
            if bs == 128:
                _capi.check(L.dfdb_set_option(b"lz4_flavour", 4))   # (blocks this small give the token sample at load no verdict)
            try:
                t = D.open_table(p)
                col = mk(t)
                r = D.aggregate(col)
                _check_agg(r, ot.aggregate(D.plan_bytes(col), 0), (name, run))
                # the predicate column decoded on the way is complete: the same query again runs the scan over it
                _check_agg(D.aggregate(col), ot.aggregate(D.plan_bytes(col), 0), (name, run, "again"))
                assert D.nrow(t[t.a > 25, ["b"]]) == ot.count(D.plan_bytes(t[t.a > 25, ["b"]]))
                runs.append(key(r))
                t.close()
            finally:
                L.dfdb_set_option(b"lz4_flavour", 0)
        assert runs[0] == runs[1], name                           # reproducible bit for bit
    # count without a projection column, fresh table
    t = D.open_table(p)
    v = t[(t.a > 25) & (t.a <= 75), ["b"]]
    assert D.nrow(v) == ot.count(D.plan_bytes(v))
    t.close()
    ot.close()


def test_leading_range_stage_prunes_the_decode(synth):
    """skip_block / skipblocks (blocksiterator.jl:69-78, selection.jl:177-184): blocks that a leading range stage rules out
    are not decompressed -- and the result is the same as when they are."""
    t, ot, nrows = synth
    L = _capi.lib()

    def decoded_bytes(view, fn):
        L.dfdb_profile_reset()
        L.dfdb_profile_enable(1)
        out = fn(view)
        L.dfdb_profile_enable(0)
        ms, n, b = C.c_double(), C.c_int64(), C.c_int64()
        L.dfdb_profile_get(b"decode", C.byref(ms), C.byref(n), C.byref(b))
        return out, b.value

    cols = ["a", "s", "ma"]
    full = t[t.a > 50, cols]
    _, full_bytes = decoded_bytes(full, D.materialize)
    for lo, hi in [(70_000, 140_000), (1, 10), (nrows - 5, nrows), (65_536, 65_537)]:
        v = t[R(lo, hi), :][t.a > 50, cols]
        fr, part_bytes = decoded_bytes(v, D.materialize)
        exp = ot.materialize(D.plan_bytes(v))
        got = fr.to_dict()
        assert got["a"] == exp[0].tolist() and got["s"] == exp[1].tolist(), (lo, hi)
        assert got["ma"] == [None if m else x for x, m in zip(exp[2][0].tolist(), exp[2][1].tolist())], (lo, hi)
        nblk = (hi - 1) // 65536 - (lo - 1) // 65536 + 1
        assert 0 < part_bytes <= full_bytes * (nblk + 0.5) / 6, (lo, hi, part_bytes, full_bytes)
        assert D.nrow(v) == len(exp[0])
        c = v.ma
        _check_agg(D.aggregate(c), ot.aggregate(D.plan_bytes(c), 0), (lo, hi))
    # an index vector and a single row are windows too
    v = t[[5, 70_000, 70_001], cols]
    assert D.materialize(v).to_dict()["a"] == ot.materialize(D.plan_bytes(v))[0].tolist()
    # and a scan over everything afterwards still sees every block
    fr, again_bytes = decoded_bytes(full, D.materialize)
    assert again_bytes == full_bytes and fr.to_dict()["a"] == ot.materialize(D.plan_bytes(full))[0].tolist()


def test_projection_blocks_without_selected_rows_are_not_decoded(synth):
    """skip_cols (blocksiterator.jl:84-95,112-115): `isempty(range) ? skip_cols(proj_cols) : read_cols(proj_cols)` -- the
    projection columns of a block are only decompressed when the block holds a selected row."""
    t, ot, nrows = synth
    L = _capi.lib()

    def run(view):
        L.dfdb_profile_reset()
        L.dfdb_profile_enable(1)
        fr = D.materialize(view)
        L.dfdb_profile_enable(0)
        ms, n, b = C.c_double(), C.c_int64(), C.c_int64()
        L.dfdb_profile_get(b"decode", C.byref(ms), C.byref(n), C.byref(b))
        return fr.to_dict(), b.value

    cols = ["a", "s", "ma", "ms"]
    everything, all_bytes = run(t[t.q > 0, cols])
    for pred in (t.q == 70_000, (t.q == 5) | (t.q == nrows), t.q > nrows - 3):
        v = t[pred, cols]
        got, some_bytes = run(v)
        exp = ot.materialize(D.plan_bytes(v))
        assert got["a"] == exp[0].tolist() and got["s"] == exp[1].tolist()
        assert got["ma"] == [None if m else x for x, m in zip(exp[2][0].tolist(), exp[2][1].tolist())]
        assert got["ms"] == exp[3].tolist()
        assert len(got["a"]) > 0 and some_bytes < 0.6 * all_bytes, (some_bytes, all_bytes)
    # twice in a row (the column state a filtered decode leaves behind must not leak into the next scan)
    again, again_bytes = run(t[t.q > 0, cols])
    assert again == everything and again_bytes == all_bytes


def test_result_arena(synth):
    """dfdb_host_alloc / dfdb_host_free: page-locked result buffers, reused after they are freed; materialize fills both
    arena buffers (direct copy) and ordinary memory (bounce buffers) with the same bytes."""
    t, ot, nrows = synth
    L = _capi.lib()
    p1, p2 = C.c_void_p(), C.c_void_p()
    _capi.check(L.dfdb_host_alloc(3 << 20, C.byref(p1)))
    assert p1.value and p1.value % 4096 == 0
    (C.c_uint8 * (3 << 20)).from_address(p1.value)[(3 << 20) - 1] = 7          # writable to the last byte
    _capi.check(L.dfdb_host_free(p1))
    seen = set()
    for _ in range(64):                                                          # freed buffers are handed out again
        _capi.check(L.dfdb_host_alloc(3 << 20, C.byref(p2)))
        seen.add(p2.value)
        _capi.check(L.dfdb_host_free(p2))
    assert len(seen) < 64
    assert L.dfdb_host_free(C.c_void_p(12345)) != 0                              # not an arena buffer
    v = t[t.a > 50, ["a", "b", "s", "ma"]]
    old = _capi.PINNED_MIN_BYTES
    try:
        _capi.PINNED_MIN_BYTES = 1                                               # every result vector from the arena
        pinned = D.materialize(v).to_dict()
        _capi.PINNED_MIN_BYTES = 1 << 62                                         # none
        pageable = D.materialize(v).to_dict()
    finally:
        _capi.PINNED_MIN_BYTES = old
    assert pinned == pageable
    exp = ot.materialize(D.plan_bytes(v))
    assert pinned["a"] == exp[0].tolist() and pinned["s"] == exp[2].tolist()


def test_sharded_scan_folds_to_the_unsharded_result(synth):
    t, ot, nrows = synth
    v = t[(t.a > 25) & (t.a <= 75), ["b", "s"]]
    whole = D.aggregate(v.b)
    exp_rows = D.materialize(v)
    for world in (2, 3):
        parts, counts, frames = [], [], []
        for rank in range(world):
            ts = D.open_table(t.path, rank=rank, world=world)
            vs = ts[(ts.a > 25) & (ts.a <= 75), ["b", "s"]]
            parts.append(D.aggregate(vs.b))
            counts.append(D.nrow(vs))
            frames.append(D.materialize(vs))
            ts.close()
        f = D.fold(parts)
        assert f.count == whole.count == sum(counts)
        assert abs((f.sum_f64 + f.sum_f64_lo) - (whole.sum_f64 + whole.sum_f64_lo)) <= 1e-13 * abs(whole.sum_f64)
        assert f.min_f64 == whole.min_f64 and f.max_f64 == whole.max_f64
        assert np.array_equal(np.concatenate([fr["b"] for fr in frames]), exp_rows["b"])
        assert sum((fr["s"].tolist() for fr in frames), []) == exp_rows["s"].tolist()


def test_sharded_range_stage_after_predicate(synth):
    """selection.jl:94-111: a range / index-vector stage behind a predicate ranks rows among ALL survivors, so every
    shard needs the survivor counts of the lower-ranked shards (dfdb_scan_exchange_count / _offset)."""
    t, ot, nrows = synth

    def plans(tb):
        return {
            "pred_range": tb[tb.a > 90, :][R(5, 7, 20000), ["q", "a"]],
            "pred_index": tb[tb.a == 7, :][[1, 2, 3, 500, 501, 3000], ["q"]],
            "range_pred_range_pred_range": tb[R(1000, 300000), :][tb.a > 50, :][R(3, 2, 90000), :][tb.b < 0.5, :][R(10, 3, 5000), ["q", "b"]],
        }

    whole = {k: D.materialize(v) for k, v in plans(t).items()}
    for k, v in plans(t).items():   # the unsharded results are the oracle's
        _same_cols([whole[k][n] for n in whole[k].names], ot.materialize(D.plan_bytes(v)))
    for world in (2, 3):
        shards = [D.open_table(t.path, rank=r, world=world) for r in range(world)]
        for k in whole:
            views = [plans(ts)[k] for ts in shards]
            with pytest.raises(D.DfdbError) as ei:      # not resolved yet: the scan says what it needs
                D.nrow(views[-1])
            assert ei.value.code == _capi.NEED_EXCHANGE
            D.resolve_sharded_selection(views)
            frames = [D.materialize(v) for v in views]
            assert sum(D.nrow(v) for v in views) == whole[k].nrow(), (k, world)
            for name in whole[k].names:
                got = np.concatenate([np.asarray(fr[name]) for fr in frames])
                assert np.array_equal(got, np.asarray(whole[k][name])), (k, world, name)
        for ts in shards:
            ts.close()


def test_corrupt_block_is_reported(tmp_path, oracle):
    p = str(tmp_path / "c")
    oracle.gen_table(p, "a:Int64:iuniform:1:100", 200000, 65536, 5, 2)
    f = os.path.join(p, "1.bin")
    raw = bytearray(open(f, "rb").read())
    raw[len(raw) // 2] ^= 0xFF
    raw[len(raw) // 2 + 1] ^= 0xFF
    open(f, "wb").write(raw)
    t = D.open_table(p)
    ot = oracle.OracleTable(p)
    v = t[t.a > 50, :]
    try:
        ref = ot.count(D.plan_bytes(v))
    except oracle.OracleError:
        ref = None
    if ref is None:
        with pytest.raises((AssertionError, D.DfdbError)):
            D.nrow(v)
    else:   # the flipped bytes happened to decode to a valid stream of the same size: results must still agree
        assert D.nrow(v) == ref


def test_size_independent_properties_at_scale(tmp_path, oracle):
    """BASELINE config shapes at a size the test box generates in seconds: partition and complement laws."""
    p = str(tmp_path / "big")
    n = 20_000_000
    oracle.gen_table(p, "a:Int64:iuniform:1:100;b:Float64:funiform", n, 65536, 0xDFDB0002, os.cpu_count() or 4)
    t = D.open_table(p)
    pred = (t.a > 25) & (t.a <= 75)
    sel, rest = D.aggregate(t[pred, :].b), D.aggregate(t[~pred, :].b)
    allb = D.aggregate(t.b)
    assert sel.count + rest.count == allb.count == n
    s1 = (sel.sum_f64 + sel.sum_f64_lo) + (rest.sum_f64 + rest.sum_f64_lo)
    assert abs(s1 - (allb.sum_f64 + allb.sum_f64_lo)) <= 1e-12 * allb.sum_f64
    assert min(sel.min_f64, rest.min_f64) == allb.min_f64 and max(sel.max_f64, rest.max_f64) == allb.max_f64
    ia = D.aggregate(t.a)
    assert 1 <= ia.min_i64 and ia.max_i64 <= 100 and abs(ia.sum_i64 / n - 50.5) < 0.05
    # sampled oracle check on a prefix: range stage first, then the predicate
    v = t[R(1, 1_000_000), :][pred, :]
    ot = oracle.OracleTable(p)
    ref = ot.aggregate(D.plan_bytes(v.b), 0)
    _check_agg(D.aggregate(v.b), ref, "prefix")
    t.close()


# ---- block index + zone maps (SURVEY.md 8f) ------------------------------------------------------------------------

def test_zone_maps_prune_blocks_without_changing_results(tmp_path, oracle):
    """Optional sidecar <id>.zmap (per block min / max / null count, built on the device): a predicate made of
    `column <cmp> constant` terms skips every block its constants rule out -- never copied, never decoded -- and every result
    stays what the reference computes (oracle on the same files, and the same scan with the zone maps switched off).  The
    column files are untouched, so the reference still opens the table."""
    p = str(tmp_path / "z")
    nrows = 40 * 4096 + 777
    rng = np.random.default_rng(0xF3)
    brands = ["apple", "samsung", "huawai", "microsoft", "dell", "xbox", "sony", "intel"]
    oracle.write_table(p, [
        ("q", "Int64", np.arange(1, nrows + 1, dtype=np.int64)),
        ("a", "Int64", rng.integers(1, 101, nrows).astype(np.int64)),
        ("b", "Float64", rng.random(nrows)),
        ("mf", "Missing(Float64)", (rng.random(nrows), rng.random(nrows) < 0.3)),
        ("p", "Float64", 1 + 0.1 * rng.integers(0, 19991, nrows)),
        ("s", "String", [brands[i] for i in rng.integers(0, 8, nrows)]),
        ("u", "UInt8", rng.integers(0, 201, nrows).astype(np.uint8)),
    ], block_size=4096)
    before = {f: open(os.path.join(p, f), "rb").read() for f in os.listdir(p)}
    t = D.open_table(p)
    ot = oracle.OracleTable(p)
    L = _capi.lib()
    assert t.zonemap("q", 0) is None
    t.build_zonemaps()
    for f, data in before.items():
        assert open(os.path.join(p, f), "rb").read() == data, f"{f} changed"          # the reference's files are untouched
    assert sorted(set(os.listdir(p)) - set(before)) == sorted(f"{t.getmeta(n).id}.zmap" for n in ("q", "a", "b", "mf", "p", "u"))
    # the statistics themselves, against the raw data
    qv = ot.materialize(D.plan_bytes(t[:, ["q", "mf", "u"]]))
    for blk in (0, 7, 40):
        lo, hi = blk * 4096, min(nrows, (blk + 1) * 4096)
        z = t.zonemap("q", blk)
        assert (z.rows, z.null_count, z.min_i64, z.max_i64, z.has_value) == (hi - lo, 0, int(qv[0][lo:hi].min()), int(qv[0][lo:hi].max()), 1)
        z = t.zonemap("mf", blk)
        vals, miss = qv[1][0][lo:hi], qv[1][1][lo:hi]
        assert z.null_count == int(miss.sum()) and z.min_f64 == float(vals[~miss].min()) and z.max_f64 == float(vals[~miss].max())
        z = t.zonemap("u", blk)
        assert (z.min_i64, z.max_i64) == (int(qv[2][lo:hi].min()), int(qv[2][lo:hi].max()))
    t.close()

    t = D.open_table(p)                       # a fresh open finds the sidecars (and takes its block index from them)
    assert t.zonemap("q", 3) is not None

    def decoded_bytes(fn):
        L.dfdb_profile_reset()
        L.dfdb_profile_enable(1)
        out = fn()
        L.dfdb_profile_enable(0)
        ms, n, b = C.c_double(), C.c_int64(), C.c_int64()
        L.dfdb_profile_get(b"decode", C.byref(ms), C.byref(n), C.byref(b))
        return out, b.value

    lo, hi = nrows // 2, nrows // 2 + nrows // 100          # a 1 % range of the sorted column
    views = {
        "range_on_sorted": lambda: t[(t.q > lo) & (t.q <= hi), ["q", "a", "s"]],
        "eq_on_sorted": lambda: t[t.q == 12345, ["b", "s"]],
        "none": lambda: t[t.q > nrows + 5, ["a"]],
        "unsorted_is_not_pruned": lambda: t[(t.a > 25) & (t.a <= 75), ["b"]],
        "float_and_missing": lambda: t[D.coalesce(t.mf < 0.001, False) & (t.q <= 9000), ["mf", "q"]],
        "two_stages": lambda: t[t.a > 50, :][t.q < 5000, ["q", "a"]],
        "range_after_pruned_predicate": lambda: t[t.q > nrows - 9000, :][R(10, 3, 200), ["q"]],
        "uint8": lambda: t[(t.u >= 250) | (t.u < 1), ["u", "q"]],
        "ne_all_equal": lambda: t[t.p != 3.5, ["p"]],
    }
    for name, mk in views.items():
        _capi.check(L.dfdb_set_option(b"no_zonemap", 0))
        (fr, n, agg), with_bytes = decoded_bytes(lambda: (D.materialize(mk()), D.nrow(mk()), D.aggregate(mk()[:, list(mk().names())[0]])))
        pruned, nb = D.pruned_blocks(mk())
        _capi.check(L.dfdb_set_option(b"no_zonemap", 1))
        try:
            (fr0, n0, agg0), without_bytes = decoded_bytes(lambda: (D.materialize(mk()), D.nrow(mk()), D.aggregate(mk()[:, list(mk().names())[0]])))
        finally:
            _capi.check(L.dfdb_set_option(b"no_zonemap", 0))
        exp = ot.materialize(D.plan_bytes(mk()))
        assert fr.to_dict() == fr0.to_dict() and n == n0 == fr.nrow(), name
        assert bytes(agg) == bytes(agg0), name
        first = exp[0][0] if isinstance(exp[0], tuple) else exp[0]
        assert fr.nrow() == len(first), name
        if name in ("range_on_sorted", "eq_on_sorted", "none", "two_stages", "range_after_pruned_predicate", "float_and_missing"):
            assert pruned >= nb // 2 and with_bytes < 0.5 * without_bytes, (name, pruned, nb, with_bytes, without_bytes)
        if name == "unsorted_is_not_pruned":
            assert pruned == 0 and with_bytes == without_bytes
    # a stale sidecar (the column file changed) is ignored, not trusted
    qbin = os.path.join(p, f"{t.getmeta('q').id}.bin")
    t.close()
    os.utime(qbin, ns=(1, 1))
    t = D.open_table(p)
    assert t.zonemap("q", 0) is None and t.zonemap("a", 0) is not None
    assert D.nrow(t[(t.q > lo) & (t.q <= hi), ["q"]]) == hi - lo
    t.close()
    ot.close()


# ---- write path: GPU LZ4 compressor + column files (SURVEY.md 8f rank 2) ---------------------------------------------------

def _gpu_compress(bodies):
    L = _capi.lib()
    n = len(bodies)
    src = b"".join(bodies)
    boff = np.cumsum([0] + [len(b) for b in bodies[:-1]]).astype(np.int64)
    blen = np.array([len(b) for b in bodies], dtype=np.int64)
    bound = [len(b) + len(b) // 255 + 16 for b in bodies]
    ooff = np.cumsum([0] + bound[:-1]).astype(np.int64)
    out = np.zeros(max(sum(bound), 1), dtype=np.uint8)
    clen = np.zeros(n, dtype=np.int64)
    sbuf = np.frombuffer(src, dtype=np.uint8) if src else np.zeros(1, dtype=np.uint8)
    _capi.check(L.dfdb_lz4_compress_blocks(sbuf.ctypes.data, boff.ctypes.data, blen.ctypes.data, n, out.ctypes.data, ooff.ctypes.data, clen.ctypes.data))
    return [bytes(out[o:o + c]) for o, c in zip(ooff, clen)]


def test_gpu_compressor_emits_blocks_every_lz4_decoder_accepts(oracle):
    """commit_block_write! (BlockStreams.jl:36-60): the device compressor's blocks decode to the same body with the oracle codec,
    with the system liblz4 (the reference's own codec) and with every GPU decoder; the ratio stays close to
    LZ4_compress_fast(acceleration 2) on the four columns whose ratios the reference's docs print (docs/src/index.md:52-63)."""
    bodies = _bodies(oracle)
    names = list(bodies)
    extra = {"empty": b"", "twelve": bytes(range(12)), "thirteen": bytes(13), "big_incompressible": np.random.default_rng(5).integers(0, 256, 700001).astype(np.uint8).tobytes()}
    names += list(extra)
    bodies.update(extra)
    comp = _gpu_compress([bodies[k] for k in names])
    sysl = oracle.system_liblz4()
    for k, c in zip(names, comp):
        body = bodies[k]
        assert 1 <= len(c) <= len(body) + len(body) // 255 + 16, k
        if body:
            assert oracle.lz4_decompress(c, len(body)) == body, f"oracle codec rejects / differs on {k}"
        if sysl is not None and body:
            dst = C.create_string_buffer(len(body))
            assert sysl.LZ4_decompress_safe(c, dst, len(c), len(body)) == len(body) and dst.raw == body, f"liblz4 rejects / differs on {k}"
    for variant in ("lane", "v3"):
        _set_variant(variant)
        try:
            got, status = _gpu_decode([c for k, c in zip(names, comp) if bodies[k]], [len(bodies[k]) for k in names if bodies[k]])
        finally:
            _set_variant(None)
        assert list(status) == [0] * len(got) and got == [bodies[k] for k in names if bodies[k]], variant
    # ratios: the docs' four columns (Int64 rand 1..100 -> 2.55/2.69, brand strings 2.85, Float64 grid 1.93, Int64 sequence 2.0)
    for k in ("rand100", "brands", "price", "iseq"):
        ref = len(oracle.compress_block(bodies[k]))
        mine = len(comp[names.index(k)])
        assert mine <= 1.05 * ref, f"{k}: {mine} bytes against liblz4's {ref}"


def test_device_write_path_produces_tables_the_reference_reader_opens(tmp_path, oracle):
    """create_table / add_column! (creators.jl:81-89, table.jl:96-124, columns.jl:65-84): column files written by the device
    write path are read back by the oracle (the restated reference reader) and by the GPU reader with identical contents, for
    every body kind of src/io/blocks.jl -- bits, Union{T,Missing}, String, Union{String,Missing} -- ragged last block included."""
    rng = np.random.default_rng(99)
    n = 7 * 1000 + 123
    brands = ["apple", "samsung", "huawai", "microsoft", "dell", "xbox", "sony", "intel", ""]
    data = {
        "a": rng.integers(1, 101, n).astype(np.int64),
        "f": rng.random(n),
        "i8": rng.integers(-100, 100, n).astype(np.int8),
        "ma": np.ma.masked_array(rng.integers(1, 101, n).astype(np.int64), rng.random(n) < 0.2),
        "mf": np.ma.masked_array(rng.random(n).astype(np.float32), rng.random(n) < 0.5),
        "s": [brands[i] for i in rng.integers(0, 9, n)],
        "ms": [None if rng.random() < 0.1 else brands[i] for i in rng.integers(0, 9, n)],
    }
    p = str(tmp_path / "w")
    t = D.create_table(p, data, block_size=1000)
    assert [m.typestring for m in t.meta] == ["Int64", "Float64", "Int8", "Missing(Int64)", "Missing(Float32)", "String", "Missing(String)"]
    assert t.total_rows() == n and t.nblocks() == 8
    ot = oracle.OracleTable(p)
    exp = ot.materialize(D.plan_bytes(t[:, :]))
    got = D.materialize(t[:, :])
    for name, e, g in zip(data, exp, [got[k] for k in got.names]):
        src = data[name]
        if isinstance(src, list):
            assert e.tolist() == src and g.tolist() == src, name
        elif isinstance(src, np.ma.MaskedArray):
            ev, em = e
            assert np.array_equal(em, np.ma.getmaskarray(src)) and np.array_equal(ev[~em], src.data[~em]), name
            assert np.array_equal(np.ma.getmaskarray(g), em) and np.array_equal(g.data[~em], src.data[~em]), name
        else:
            assert np.array_equal(e, src) and np.array_equal(g, src), name
    # add_column! from a computed column of the same table, and from plain data
    t.add_column("a2", t.a * 2)
    t.add_column("tag", ["x%d" % (i % 7) for i in range(n)])
    with pytest.raises(D.ArgumentError):
        t.add_column("a", data["a"])                      # Column :a already exists
    with pytest.raises(D.ArgumentError):
        t.add_column("short", data["a"][:10])             # Column and table have different sizes
    ot2 = oracle.OracleTable(p)
    e2 = ot2.materialize(D.plan_bytes(t[t.a > 50, ["a2", "tag"]]))
    sel = data["a"] > 50
    assert np.array_equal(e2[0], data["a"][sel] * 2) and e2[1].tolist() == [("x%d" % (i % 7)) for i in range(n) if sel[i]]
    g2 = D.materialize(t[t.a > 50, ["a2", "tag"]])
    assert np.array_equal(g2["a2"], e2[0]) and g2["tag"].tolist() == e2[1].tolist()
    with pytest.raises(RuntimeError):
        D.create_table(p, {"x": data["a"]})               # Table ... already exists
    t.close(); ot.close(); ot2.close()


# ---- group-by reduce (SURVEY.md 8f rank 4) --------------------------------------------------------------------------------

def test_groupreduce_matches_a_dictionary_fold_in_first_appearance_order(tmp_path, oracle):
    """groupreduce(view, by; cols...) -- the reference only stubs it (src/tables/aggregate.jl:1-36: a RobinDict from the key tuple
    to a group number in order of first appearance).  Expectations: a plain Python dict fold over the columns the ORACLE
    materializes from the same files; counts, integer sums, minima and maxima exact, Float64 sums within 1e-12."""
    rng = np.random.default_rng(41)
    n = 9 * 2048 + 77
    brands = ["apple", "samsung", "huawai", "microsoft", "dell", "xbox", "sony", "intel"]
    data = [
        ("brand", "String", [brands[i] for i in rng.integers(0, 8, n)]),
        ("mbrand", "Missing(String)", [None if rng.random() < 0.1 else brands[i] for i in rng.integers(0, 8, n)]),
        ("k", "Int64", rng.integers(0, 500, n).astype(np.int64)),
        ("mk", "Missing(Int64)", (rng.integers(0, 5, n).astype(np.int64), rng.random(n) < 0.2)),
        ("fk", "Float64", rng.choice(np.array([0.0, -0.0, 1.5, np.nan, 2.5]), n)),
        ("price", "Float64", rng.random(n) * 100),
        ("qty", "Missing(Int64)", (rng.integers(-50, 50, n).astype(np.int64), rng.random(n) < 0.15)),
        ("a", "Int64", rng.integers(1, 101, n).astype(np.int64)),
    ]
    p = str(tmp_path / "g")
    oracle.write_table(p, data, block_size=2048)
    t = D.open_table(p)
    ot = oracle.OracleTable(p)

    def expect(view, by, vals):
        cols = ot.materialize(D.plan_bytes(view[:, by + vals]))

        def as_list(c):
            if isinstance(c, tuple):
                return [None if m else v for v, m in zip(c[0].tolist(), c[1].tolist())]
            return c.tolist()
        lists = [as_list(c) for c in cols]
        groups, order = {}, []
        for i in range(len(lists[0])):
            key = tuple("NaN" if isinstance(x, float) and x != x else (("-0.0" if str(x) == "-0.0" else x)) for x in (lists[j][i] for j in range(len(by))))
            if key not in groups:
                groups[key] = [[] for _ in vals]
                order.append(key)
            for j in range(len(vals)):
                groups[key][j].append(lists[len(by) + j][i])
        return order, groups

    cases = [
        (t[t.a > 50, :], ["brand"], {"total": "price", "units": "qty"}),
        (t[:, :], ["mbrand", "mk"], {"p": "price"}),
        (t[t.a <= 10, :], ["k"], {"q": "qty", "p": "price", "a": "a"}),
        (t[:, :], ["fk"], {"n": "a"}),
        (t[t.a > 200, :], ["brand"], {"p": "price"}),
    ]
    for view, by, cols in cases:
        got = D.groupreduce(view, by, **cols)
        order, groups = expect(view, by, list(cols.values()))
        gkeys = list(zip(*[got[k] for k in by])) if order else []
        norm = [tuple("NaN" if isinstance(x, float) and x != x else ("-0.0" if str(x) == "-0.0" else x) for x in key) for key in gkeys]
        assert norm == order, (by, norm[:5], order[:5])
        for name, src in cols.items():
            j = list(cols).index(name)
            for gi, key in enumerate(order):
                xs = groups[key][j]
                present = [x for x in xs if x is not None]
                rec = got[name]
                assert rec["count"][gi] == len(xs) and rec["nmissing"][gi] == len(xs) - len(present), (name, key)
                if not present:
                    assert rec["min"][gi] is None
                    continue
                if isinstance(present[0], float):
                    import math
                    assert abs(rec["sum"][gi] - math.fsum(present)) <= 1e-12 * max(abs(math.fsum(present)), 1e-300), (name, key)
                else:
                    assert rec["sum"][gi] == sum(present), (name, key)
                assert rec["min"][gi] == min(present) and rec["max"][gi] == max(present), (name, key)
    # the group table grows when the data has more groups than it first assumed
    big = D.groupreduce(t[:, :], ["price"])
    assert big["ngroups"] == len(set(data[5][2].tolist()))
    with pytest.raises(D.ArgumentError):
        D.groupreduce(t[:, :], ["brand"], s="brand")          # aggregate over a String column
    t.close(); ot.close()


def test_library_communicator_combines_partials_over_nccl(synth):
    """dfdb_comm_init / dfdb_scan_aggregate_all / dfdb_scan_count_all: the combine step inside the library (ncclAllGather of one
    slot per rank on the scan stream + dfdb_agg_fold).  One GPU here, so the communicator has one rank: the NCCL path runs end to
    end and must return exactly the local result; bench.py runs the same entry points at 2 / 4 / 8 ranks."""
    t, ot, nrows = synth
    L = _capi.lib()
    ident = (C.c_uint8 * 128)()
    _capi.check(L.dfdb_comm_unique_id(ident))
    assert any(ident)
    _capi.check(L.dfdb_comm_init(0, 1, ident))
    try:
        r, w = C.c_int32(), C.c_int32()
        _capi.check(L.dfdb_comm_info(C.byref(r), C.byref(w)))
        assert (r.value, w.value) == (0, 1)
        assert L.dfdb_comm_init(0, 1, ident) != 0                       # a communicator already exists
        for v in (t[(t.a > 25) & (t.a <= 75), ["b"]], t[t.a > 50, :][R(10, 7, 5000), ["a"]], t[:, ["b"]]):
            col = v[:, list(v.names())[0]]
            assert bytes(D.aggregate_all(col)) == bytes(D.aggregate(col))
            assert D.nrow_all(v) == D.nrow(v) == ot.count(D.plan_bytes(v))
    finally:
        _capi.check(L.dfdb_comm_destroy())
    _capi.check(L.dfdb_comm_info(C.byref(r), C.byref(w)))
    assert w.value == 0
