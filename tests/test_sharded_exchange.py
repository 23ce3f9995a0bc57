"""The record exchange of the `_all` entry points: one shard / communicator rule for all of them, and each rank's local status
travelling with its record.

One GPU: a communicator that does not serve the table's shard is refused by every `_all` call, and a local failure returns the
local error without spoiling the communicator.  Two GPUs: every `_all` result equals, bit for bit, the host-carried result of
the same two shards computed in one process, and a failure on one rank is an error on both."""
import contextlib
import ctypes as C
import traceback

import pytest

import dfdb_b200 as D
from dfdb_b200 import R, _capi

BLOCK = 4096
NROWS = 6 * BLOCK + 321                      # seven blocks: each shard of two holds several


@pytest.fixture(scope="module")
def table(tmp_path_factory, oracle):
    p = str(tmp_path_factory.mktemp("exch") / "t")
    oracle.gen_table(p, "a:Int64:iuniform:1:50;b:Float64:funiform;r:Int64:iseq", NROWS, BLOCK, 0xDFDB0301, 4)
    return p


@pytest.fixture(scope="module")
def gpu():
    _capi.init(0)
    yield


@contextlib.contextmanager
def one_rank_communicator():
    L = _capi.lib()
    ident = (C.c_uint8 * 128)()
    _capi.check(L.dfdb_comm_unique_id(ident))
    _capi.check(L.dfdb_comm_init(0, 1, ident))
    try:
        yield
    finally:
        _capi.check(L.dfdb_comm_destroy())


def _all_codes(v):
    """the status of every `_all` entry point on the scan of view v (projection 0 is an Int64 column)"""
    L = _capi.lib()
    h = D.api._scan_handle(v)
    agg, n, lo, tot, nb = _capi.Agg(), C.c_int64(), C.c_int64(), C.c_int64(), C.c_int64()
    ranks, vals = (C.c_int64 * 1)(1), (C.c_int64 * 1)()
    return {
        "aggregate_all": L.dfdb_scan_aggregate_all(h, 0, C.byref(agg)),
        "count_all": L.dfdb_scan_count_all(h, C.byref(n)),
        "row_offset_all": L.dfdb_scan_row_offset_all(h, C.byref(n), C.byref(lo), C.byref(tot)),
        "groupreduce_all": L.dfdb_scan_groupreduce_all(h, (C.c_int32 * 1)(0), 1, (C.c_int32 * 1)(1), 1, C.byref(n)),
        "unique_all": L.dfdb_scan_unique_all(h, 0, C.byref(n), C.byref(nb)),
        "order_prepare_all": L.dfdb_scan_order_prepare_all(h, 0, C.byref(agg)),
        "order_stats_all": L.dfdb_scan_order_stats_all(h, ranks, 1, vals),
    }


@pytest.mark.gpu
def test_a_communicator_that_does_not_match_the_shard_is_refused(gpu, table):
    """shard 0 of 2 under a one-rank communicator, with a plan that needs no survivor-count exchange: every `_all` call is
    DFDB_ERR_STATE (none returns shard 0's partial as the whole table's); the same calls on the unsharded table over the same
    communicator then return the local results"""
    L = _capi.lib()
    shard, whole = D.open_table(table, rank=0, world=2), D.open_table(table)
    with one_rank_communicator():
        v = shard[shard.a > 20, ["a", "r"]]
        _capi.check(L.dfdb_scan_order_prepare(D.api._scan_handle(v), 0, C.byref(_capi.Agg())))    # (shard-local: no exchange)
        codes = _all_codes(v)
        assert codes == {name: _capi.ERR_STATE for name in codes}, codes

        w = whole[whole.a > 20, :]
        assert bytes(D.aggregate_all(w.b)) == bytes(D.aggregate(w.b))
        n = D.nrow(w)
        assert D.nrow_all(w) == n
        local, lo, tot = C.c_int64(), C.c_int64(), C.c_int64()
        _capi.check(L.dfdb_scan_row_offset_all(D.api._scan_handle(w), C.byref(local), C.byref(lo), C.byref(tot)))
        assert (local.value, lo.value, tot.value) == (n, 0, n)
        assert D.groupreduce_all(w, ["a"], s="r") == D.groupreduce(w, ["a"], s="r")
        assert D.unique_all(w.a).tobytes() == D.unique(w.a).tobytes()
        h = D.api._scan_handle(w[:, ["b"]])
        mine, everywhere = _capi.Agg(), _capi.Agg()
        _capi.check(L.dfdb_scan_order_prepare(h, 0, C.byref(mine)))
        _capi.check(L.dfdb_scan_order_prepare_all(h, 0, C.byref(everywhere)))
        assert bytes(everywhere) == bytes(mine)
        ranks = [1, n // 2, n]
        assert D.order_stats(w.b, ranks).tobytes() == D.order_stats_sharded([w.b], ranks).tobytes()
    shard.close()
    whole.close()


@pytest.mark.gpu
def test_a_local_failure_returns_the_local_error(gpu, table):
    """over a one-rank communicator, a local pass that fails (a projection index out of range) returns its own error code, and
    the next valid call returns exactly the local result"""
    L = _capi.lib()
    t = D.open_table(table)
    with one_rank_communicator():
        vb, va = t[t.a > 20, ["b"]], t[t.a > 20, ["a"]]
        agg, n, nb = _capi.Agg(), C.c_int64(), C.c_int64()
        assert L.dfdb_scan_aggregate_all(D.api._scan_handle(vb), 3, C.byref(agg)) == _capi.ERR_ARGUMENT
        assert bytes(D.aggregate_all(vb.b)) == bytes(D.aggregate(vb.b))
        assert L.dfdb_scan_unique_all(D.api._scan_handle(va), 3, C.byref(n), C.byref(nb)) == _capi.ERR_ARGUMENT
        assert D.unique_all(va.a).tobytes() == D.unique(va.a).tobytes()
        h = D.api._scan_handle(vb)
        assert L.dfdb_scan_order_prepare_all(h, 3, C.byref(agg)) == _capi.ERR_ARGUMENT
        mine = _capi.Agg()
        _capi.check(L.dfdb_scan_order_prepare_all(h, 0, C.byref(agg)))
        _capi.check(L.dfdb_scan_order_prepare(h, 0, C.byref(mine)))
        assert bytes(agg) == bytes(mine)
    t.close()


# ---- two GPUs ------------------------------------------------------------------------------------------------------------

def _plans(t):
    """the same selections on any table or shard: p is the projection"""
    return {
        "all": lambda p: t[:, p],
        "pred": lambda p: t[t.a > 20, p],
        "range_after_pred": lambda p: t[t.a > 10, :][R(7, 3, 19000), p],      # (ranks survivors of both shards)
    }


def _two_rank_worker(rank, path, store, q):
    """rank `rank` of 2 on device `rank`: the `_all` results against the host-carried merge of both shards, opened in this
    process too; then a failure on rank 1 alone"""
    import torch
    import torch.distributed as dist
    from dfdb_b200 import dist as DD
    bad = []
    try:
        torch.cuda.set_device(rank)
        dist.init_process_group("gloo", init_method=f"file://{store}", rank=rank, world_size=2)
        DD.comm_init_from_torch(rank, 2, device=rank)
        L = _capi.lib()
        mine = D.open_table(path, rank=rank, world=2, device=rank)
        shards = [D.open_table(path, rank=r, world=2, device=rank) for r in range(2)]
        whole = D.open_table(path, device=rank)
        col = slice(None)
        for key in ("all", "pred", "range_after_pred"):
            got = _plans(mine)[key]
            # aggregate: the rank-order fold of the shard aggregates
            parts = [_plans(s)[key](["b"]) for s in shards]
            D.resolve_sharded_selection(parts)
            want = D.fold([D.aggregate(v.b) for v in parts])
            if bytes(D.aggregate_all(got(["b"]).b)) != bytes(want):
                bad.append((key, "aggregate_all"))
            # row offsets and the total
            counts = [D.nrow(v) for v in parts]
            local, lo, tot = C.c_int64(), C.c_int64(), C.c_int64()
            _capi.check(L.dfdb_scan_row_offset_all(D.api._scan_handle(got(["b"])), C.byref(local), C.byref(lo), C.byref(tot)))
            if (local.value, lo.value, tot.value) != (counts[rank], sum(counts[:rank]), sum(counts)):
                bad.append((key, "row_offset_all"))
            # order statistics
            n = want.count - want.nmissing
            ranks = sorted({1, n, (n + 1) // 2, n // 3 + 1})
            if D.order_stats(got(["b"]).b, ranks).tobytes() != D.order_stats_sharded([v.b for v in parts], ranks).tobytes():
                bad.append((key, "order_stats"))
            # unique
            parts = [_plans(s)[key](["a"]) for s in shards]
            D.resolve_sharded_selection(parts)
            merged = D.unique_merge(_plans(whole)[key](["a"]).a, [D.unique(v.a) for v in parts])
            if D.unique_all(got(["a"]).a).tobytes() != merged.tobytes():
                bad.append((key, "unique_all"))
            # group-by (an Int64 value column: its sums do not depend on the order of the local pass)
            parts = [_plans(s)[key](["a", "r"]) for s in shards]
            D.resolve_sharded_selection(parts)
            merged = D.groupreduce_merge(_plans(whole)[key](col), ["a"], [D.groupreduce_local(v, ["a"], s="r") for v in parts], s="r")
            if D.groupreduce_all(got(col), ["a"], s="r") != merged:
                bad.append((key, "groupreduce_all"))
        # rank 1 alone passes a projection index that does not exist
        h = D.api._scan_handle(mine[:, ["a", "b"]])
        agg, n, nb = _capi.Agg(), C.c_int64(), C.c_int64()
        calls = {
            "aggregate_all": lambda p: L.dfdb_scan_aggregate_all(h, p, C.byref(agg)),
            "unique_all": lambda p: L.dfdb_scan_unique_all(h, p, C.byref(n), C.byref(nb)),
            "groupreduce_all": lambda p: L.dfdb_scan_groupreduce_all(h, (C.c_int32 * 1)(p), 1, (C.c_int32 * 1)(1), 1, C.byref(n)),
            "order_prepare_all": lambda p: L.dfdb_scan_order_prepare_all(h, p, C.byref(agg)),
        }
        for name, call in calls.items():
            rc = call(5 if rank == 1 else 0)
            msg = L.dfdb_last_error().decode()
            if rank == 1 and rc != _capi.ERR_ARGUMENT:
                bad.append((name, "rank 1 status", rc, msg))
            if rank == 0 and (rc != _capi.ERR_STATE or "rank 1" not in msg):
                bad.append((name, "rank 0 status", rc, msg))
            rc = call(0)
            if rc != 0:
                bad.append((name, "the next call", rc, L.dfdb_last_error().decode()))
        DD.comm_destroy()
        for t in [mine, whole] + shards:
            t.close()
        dist.destroy_process_group()
    except Exception:
        bad.append(traceback.format_exc())
    q.put((rank, bad))


@pytest.mark.gpu
def test_two_ranks_equal_the_host_carried_merge(table, tmp_path):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip(f"the exchange between ranks needs two GPUs; this machine has {torch.cuda.device_count()}")
    import multiprocessing as mp
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_two_rank_worker, args=(r, table, str(tmp_path / "store"), q)) for r in range(2)]
    for p in procs:
        p.start()
    try:
        res = dict(q.get(timeout=600) for _ in procs)
    finally:
        for p in procs:
            p.join(timeout=60)
            if p.is_alive():
                p.terminate()
                p.join()
    assert res == {0: [], 1: []}, res
