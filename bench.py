#!/usr/bin/env python
"""bench.py -- filtered-scan throughput of the column-scan hot path (BASELINE.json metric).

A step = one pass of the whole path over the table shard: LZ4 decode of every needed column block ->
range predicate `25 < a <= 75` -> sum/min/max/count of `b` -> (N > 1) NCCL all-gather of the per-rank
partials + fixed rank-order fold.  Workload at N = 1 is BASELINE.json configs[1] (1B-row Int64/Float64
table); at N > 1 every rank scans a 1B-row block-range shard of an N*1B-row table (configs[4], weak scaling).

  value      rows/s with the compressed blocks resident in HBM when the timed region starts
  e2e        same metric through the public API with the compressed blocks in pinned HOST memory:
             every step copies them H2D, decodes, scans and reads the aggregate back
  roofline   dominant kernel (K1 LZ4 decode): algorithmic bytes (compressed read + decoded written)
             / CUDA-event time of the launch, against the measured HBM copy peak
  cpu_baseline / --impl reference: the CPU restatement of the reference algorithm (oracle/, a port --
             the reference is Julia and no julia binary exists in this image) on the host cores
"""
import argparse
import ctypes as C
import json
import os
import shutil
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

SPEC = "a:Int64:iuniform:1:100;b:Float64:funiform"
SEED = 0xDFDB0002
BLOCK = 65536


def log(*a):
    print(*a, file=sys.stderr, flush=True)


def mem_available_bytes():
    try:
        for line in open("/proc/meminfo"):
            if line.startswith("MemAvailable:"):
                return int(line.split()[1]) * 1024
    except OSError:
        pass
    return 64 << 30


def table_dir(rows):
    base = "/dev/shm" if os.path.isdir("/dev/shm") and os.access("/dev/shm", os.W_OK) else "/tmp"
    return os.path.join(base, f"dfdb_b200_bench_{rows}_{SEED:x}")


def ensure_table(rows, threads):
    """Synthetic table in the reference's on-disk format (oracle/gen.c); reused when already present."""
    from oracle import oracle as O
    path = table_dir(rows)
    marker = os.path.join(path, ".complete")
    if os.path.exists(marker):
        return path, json.load(open(marker))
    shutil.rmtree(path, ignore_errors=True)
    t0 = time.time()
    unc, comp = O.gen_table(path, SPEC, rows, BLOCK, SEED, threads)
    info = {"rows": rows, "uncompressed": unc, "compressed": comp, "gen_s": round(time.time() - t0, 2)}
    json.dump(info, open(marker, "w"))
    log(f"[bench] generated {rows} rows in {info['gen_s']} s: {unc / 1e9:.2f} GB -> {comp / 1e9:.2f} GB at {path}")
    return path, info


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index = index
        self.lines = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100", "-i", str(self.index)],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append((time.time(), line.strip()))

    def stop(self, t0, t1):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, smax, reasons = [], None, set()
        for ts, line in self.lines:
            f = [x.strip() for x in line.split(",")]
            if len(f) < 9:
                continue
            try:
                smax = float(f[2])
                if t0 - 0.05 <= ts <= t1 + 0.15:
                    sm.append(float(f[1]))
                    for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                        if val.lower().startswith("active"):
                            reasons.add(name)
            except ValueError:
                continue
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": smax, "reasons": sorted(reasons), "samples": len(sm)}


def measured_peak_gbs():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def ncu_traffic(kernel, rows):
    """dram bytes per launch from the committed `ncu --set full` capture, scaled linearly to `rows`."""
    p = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(p):
        try:
            t = json.load(open(p)).get(kernel)
            return int(t["bytes"] * rows / t["rows"]) if t else None
        except Exception:
            return None
    return None


# ---------------------------------------------------------------------------------------------------------
# The benchmark query `t[(t.a .> 25) .& (t.a .<= 75), [:b]]` -> sum / min / max / count of b, as plan bytes (wire format:
# INTEGRATION.md).  A constant, so that the reference arm does not have to import the product package to build it;
# tests/test_host_logic.py checks it against plan_bytes() of the Python mirror and tests/golden/queries.json.
BENCH_PLAN = bytes.fromhex("4446503101000000030700000001010000000000000002190000000000000014010100000000000000024b00000000000000132001000000010200000000000000")
C1_PLAN = bytes.fromhex("444650310100000003030000000101000000000000000232000000000000001401000000010200000000000000")   # t[t.a .> 50, [:b]]


def oracle_scan(ot, plan, nblocks, threads, blk_lo=0):
    """The CPU restatement of the reference's scan over blocks [blk_lo, blk_lo + nblocks) on `threads` host threads."""
    t0 = time.time()
    parts = ot.aggregate_mt(plan, 0, nblocks, threads, blk_lo)
    return parts, time.time() - t0


def run_reference(args):
    """The reference's CPU implementation of the path, restated in C (oracle/): every host thread, the SAME table and query as
    the GPU arm at N = 1 (at N > 1 rank 0 scans a 1B-row shard-sized table: one GPU's share of the workload).  Nothing of the
    product is imported or loaded here."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    from oracle import oracle as O
    threads = os.cpu_count() or 1
    rows = args.rows if args.ref_sample_rows <= 0 else min(args.rows, args.ref_sample_rows)
    avail = mem_available_bytes()
    if rows * 11.1 * 1.3 > avail * 0.8:
        rows = max(BLOCK, int(avail * 0.8 / (11.1 * 1.3)) // BLOCK * BLOCK)
        log(f"[bench] host RAM {avail / 2**30:.0f} GiB: reference arm reduced to {rows} rows")
    path, info = ensure_table(rows, threads)
    ot = O.OracleTable(path)
    nblocks = (rows + BLOCK - 1) // BLOCK
    times = []
    parts = []
    for i in range(args.warmup + args.steps):
        parts, dt = oracle_scan(ot, BENCH_PLAN, nblocks, threads)
        if i >= args.warmup:
            times.append(dt)
    # single thread on a bounded sample (BASELINE.md quotes single-thread figures for the reference)
    nb1 = min(nblocks, 400)
    _, dt1 = oracle_scan(ot, BENCH_PLAN, nb1, 1)
    ot.close()
    total = sum(times)
    value = rows * len(times) / total
    sample = (f"the whole {rows}-row table ({nblocks} blocks) per step, {threads} threads over block ranges" if args.gpus == 1 else
              f"{rows} rows ({nblocks} blocks) per step = one GPU's shard of the {args.gpus}-GPU workload, {threads} threads over block ranges")
    line = {
        "impl": "reference", "metric": "filtered-scan rows/s (LZ4 block decode + range predicate + sum/min/max/count)", "value": value,
        "unit": "rows/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * total / len(times),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "int64/f64", "data": "synthetic",
        "config": workload_config(args, rows, info),
        "cpu_baseline": {"value": value, "unit": "rows/s", "cores": threads, "kind": "port", "sample": sample},
        "cpu_baseline_1t": {"value": min(rows, nb1 * BLOCK) / dt1, "unit": "rows/s", "cores": 1, "kind": "port",
                            "sample": f"{min(rows, nb1 * BLOCK)} rows ({nb1} blocks) of the same table, one thread"},
        "e2e": {"value": value, "unit": "rows/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "same_config": args.gpus == 1 and rows == args.rows,
        "note": "C restatement of the reference's per-block algorithm (oracle/dfdb_oracle.c); the Julia reference cannot run in this image",
        "selected_rows": sum(p.count for p in parts),
    }
    print(json.dumps(line), flush=True)
    return 0


def dump_outputs(out_dir, agg):
    """What the timed path hands its caller -- every field of the dfdb_agg that aggregate() / aggregate_all() return -- as
    <out_dir>/<field>.npy (float64, one element), so that two builds can be compared output for output on the same seeded table."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    for name, _ in type(agg)._fields_:
        np.save(os.path.join(out_dir, f"{name}.npy"), np.array([getattr(agg, name)], dtype=np.float64))


def workload_config(args, rows_per_gpu, info):
    return {
        "workload": "configs[1]: 1B-row Int64 a / Float64 b table, compressed block decode + range predicate 25 < a <= 75 + sum/min/max/count of b"
        if args.gpus == 1 else "configs[4]: N*1B-row table sharded by block range, scan-filter-aggregate + NCCL partial-aggregate combine",
        "rows_per_gpu": rows_per_gpu, "rows_total": rows_per_gpu * args.gpus if args.gpus > 1 else rows_per_gpu, "block_size": BLOCK,
        "columns": "a::Int64 uniform 1..100 (LZ4 ratio 2.69), b::Float64 uniform [0,1) (ratio 1.00)",
        "compressed_bytes": info.get("compressed"), "uncompressed_bytes": info.get("uncompressed"),
        "parallelism": f"block-range shards x{args.gpus}" if args.gpus > 1 else "single GPU",
        "l2": "inputs (compressed + decoded columns, tens of GB) are far larger than the 126 MB L2; no flush needed",
    }


def agg_variant(name, spec, seed, rows, plan_of, threads, local, steps=5, warmup=3):
    """A filter + aggregate query over a generated table, HBM-resident: ms per step (CUDA events on the scan stream, whole
    query through the public API), checked against the oracle over the WHOLE table."""
    import math
    import torch
    import dfdb_b200 as D
    from oracle import oracle as O
    base = "/dev/shm" if os.path.isdir("/dev/shm") and os.access("/dev/shm", os.W_OK) else "/tmp"
    path = os.path.join(base, f"dfdb_b200_variant_{name}_{rows}_{seed:x}")
    if not os.path.exists(os.path.join(path, ".complete")):
        shutil.rmtree(path, ignore_errors=True)
        O.gen_table(path, spec, rows, BLOCK, seed, threads)
        open(os.path.join(path, ".complete"), "w").write("{}")
    t = D.open_table(path, mode=D.LOAD_HBM, device=local)
    col = plan_of(t)
    stream = torch.cuda.current_stream()
    for _ in range(warmup):
        res = D.aggregate(col)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for _ in range(steps):
        res = D.aggregate(col)
    e1.record(stream)
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / steps
    ot = O.OracleTable(path)
    parts, cpu_s = oracle_scan(ot, D.plan_bytes(col), t.nblocks(), threads)
    ot.close()
    cnt = sum(p.count for p in parts)
    ksum = math.fsum(p.sum_kahan for p in parts)
    gsum = res.sum_f64 + res.sum_f64_lo
    ok = (cnt == res.count and abs(gsum - ksum) <= 1e-12 * max(abs(ksum), 1e-300)
          and min(p.min_f64 for p in parts if p.count) == res.min_f64 and max(p.max_f64 for p in parts if p.count) == res.max_f64)
    t.close()
    shutil.rmtree(path, ignore_errors=True)
    return {"rows": rows, "ms_per_step": ms, "value": rows / (ms / 1e3), "unit": "rows/s", "steps": steps, "columns": spec,
            "verified": {"ok": bool(ok), "kind": "full", "count": cnt, "rel_err": abs(gsum - ksum) / max(abs(ksum), 1e-300)},
            "cpu_port_rows_per_s": rows / cpu_s, "cpu_threads": threads}


def run_variants(args, threads, local):
    """configs[0] (the reference's own 10M-row case), configs[1] with a COMPRESSIBLE b (Float64 grid, LZ4 ratio 1.93: the
    headline table's b is incompressible and read in place), configs[2] (string filter + materialize, 200M rows) and configs[3]
    (missing-bearing multi-column predicate + materialize of 4 columns, 500M rows).  Every result is checked over the whole
    table against the CPU oracle (aggregates: count / min / max exact, sum within 1e-12; materialize: row count + a 64-bit
    content hash of every output column)."""
    import bench_configs
    out = {}
    scale = args.rows / 1_000_000_000
    out["config0_10M_gt50_sum_b"] = agg_variant("c0", "a:Int64:iuniform:1:100;b:Float64:funiform;s:String:brands", 0xDFDB0001,
                                                max(BLOCK, int(10_000_000 * min(1.0, scale * 100))), lambda t: t[t.a > 50, ["b"]].b, threads, local, steps=10)
    out["config1_compressible_b"] = agg_variant("c1fg", "a:Int64:iuniform:1:100;b:Float64:fgrid:1:0.1:2000", 0xDFDB0012, args.rows,
                                                lambda t: t[(t.a > 25) & (t.a <= 75), ["b"]].b, threads, local)
    bench_configs.run_query.quiet = True
    for cfg, key in ((3, "config2_strings_200M"), (4, "config3_missings_500M")):
        rows = max(BLOCK, int(bench_configs.CONFIGS[cfg]["rows"] * scale))
        lines = bench_configs.run_config(cfg, rows=rows, reps=3, check="full", quiet=True)
        out[key] = [{k: ln[k] for k in ("query", "rows", "selected", "ms", "rows_per_s", "out_bytes", "phases_ms", "verified")} for ln in lines]
        shutil.rmtree(bench_configs.table_path(bench_configs.CONFIGS[cfg], rows), ignore_errors=True)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--rows", type=int, default=1_000_000_000, help="rows per GPU")
    ap.add_argument("--ref-sample-rows", type=int, default=0, help="reference arm: scan at most this many rows per step (0 = the whole table)")
    ap.add_argument("--no-variants", action="store_true", help="skip the other BASELINE.json configurations (variants)")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-verify", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the result of the last timed step as DIR/<field>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the GPU path's result; the reference arm has none")
    args.warmup = max(args.warmup, 0)
    if args.impl == "reference":
        return run_reference(args)

    import numpy as np
    import torch
    import torch.distributed as dist
    import dfdb_b200 as D
    from dfdb_b200 import _capi

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        log(f"[bench] WORLD_SIZE={world} differs from --gpus {args.gpus}; using WORLD_SIZE")
        args.gpus = world
    torch.cuda.set_device(local)
    if world > 1:
        # NCCL prints its version banner on stdout at NCCL_DEBUG=VERSION; stdout carries exactly one JSON line
        if os.environ.get("NCCL_DEBUG", "VERSION").upper() == "VERSION":
            os.environ["NCCL_DEBUG"] = "WARN"
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    threads = os.cpu_count() or 1

    # ---- size the table to the host (tmpfs file + pinned staging both live in RAM) ----
    rows = args.rows
    if rank == 0:
        avail = mem_available_bytes()
        need_per_row = 11.1 * 2.3          # compressed bytes/row: tmpfs file + pinned copy + slack
        max_rows_total = int(avail * 0.8 / need_per_row)
        if rows * world > max_rows_total:
            rows = max(BLOCK, (max_rows_total // world) // BLOCK * BLOCK)
            log(f"[bench] host RAM {avail / 2**30:.0f} GiB: rows per GPU reduced to {rows}")
    if world > 1:
        rt = torch.tensor([rows], dtype=torch.int64, device="cuda")
        dist.broadcast(rt, 0)
        rows = int(rt.item())
    info = {}
    if rank == 0:
        path, info = ensure_table(rows * world, threads)
    if world > 1:
        dist.barrier()
    path = table_dir(rows * world)
    if not info:
        info = json.load(open(os.path.join(path, ".complete")))

    _capi.init(local)
    L = _capi.lib()
    stream = torch.cuda.current_stream()
    _capi.check(L.dfdb_set_stream(C.c_void_p(stream.cuda_stream)))

    def open_view(mode):
        t = D.open_table(path, mode=mode, rank=rank, world=world, device=local)
        v = t[(t.a > 25) & (t.a <= 75), ["b"]]
        t.load(["a", "b"])
        return t, v

    if world > 1:
        # the LIBRARY's NCCL communicator (dfdb_comm_init): torch.distributed only carries the 128-byte id to the ranks
        from dfdb_b200.dist import comm_init_from_torch
        comm_init_from_torch(rank, world, device=torch.device("cuda", local))

    def step(v):
        """one pass of the hot path over this rank's shard; at N > 1 the partial aggregates are combined inside the library
        (dfdb_scan_aggregate_all: ncclAllGather of the per-rank partials on the scan stream + fixed rank-order fold)"""
        return D.aggregate(v.b) if world == 1 else D.aggregate_all(v.b)

    def timed(v, steps, warmup, profile=False):
        for _ in range(warmup):
            res = step(v)
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        if profile:
            L.dfdb_profile_reset()
            L.dfdb_profile_enable(1)
        l0 = L.dfdb_kernel_launches()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        w0 = time.time()
        e0.record(stream)
        for _ in range(steps):
            res = step(v)
        e1.record(stream)
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        w1 = time.time()
        if profile:
            L.dfdb_profile_enable(0)
        ms = e0.elapsed_time(e1)
        if world > 1:
            mt = torch.tensor([ms], dtype=torch.float64, device="cuda")
            dist.all_reduce(mt, op=dist.ReduceOp.MAX)
            ms = float(mt.item())
        return res, ms, L.dfdb_kernel_launches() - l0, (w0, w1)

    def phase(name):
        ms, n, b = C.c_double(), C.c_int64(), C.c_int64()
        L.dfdb_profile_get(name.encode(), C.byref(ms), C.byref(n), C.byref(b))
        return ms.value, n.value, b.value

    # ---- HBM-resident: compressed blocks on the device, every step decodes + scans ----
    t, v = open_view(D.LOAD_HBM)
    comp_a, unc_a, comp_b, unc_b = C.c_int64(), C.c_int64(), C.c_int64(), C.c_int64()
    L.dfdb_table_column_stats(t._h, t.getmeta("a").id, C.byref(comp_a), C.byref(unc_a))
    L.dfdb_table_column_stats(t._h, t.getmeta("b").id, C.byref(comp_b), C.byref(unc_b))
    shard_comp, shard_unc = comp_a.value + comp_b.value, unc_a.value + unc_b.value
    lo, hi = t.shard_rows()
    shard_rows = hi - lo
    sampler = ClockSampler(local)
    sampler.start()
    time.sleep(0.3)
    res, ms, launches, (w0, w1) = timed(v, args.steps, args.warmup, profile=True)
    clocks = sampler.stop(w0, w1)
    total_rows = rows * world
    value = total_rows * args.steps / (ms / 1e3)
    dec_ms, dec_n, dec_bytes = phase("decode")
    con_ms, con_n, con_bytes = phase("consume")
    peak, peak_src = measured_peak_gbs()
    dec_launch_ms = dec_ms / max(dec_n, 1)
    achieved = (dec_bytes / max(dec_n, 1)) / (dec_launch_ms / 1e3) / 1e9 if dec_ms > 0 else 0.0
    st_blocks, st_bytes = C.c_int64(), C.c_int64()
    L.dfdb_table_column_stored(t._h, t.getmeta("b").id, C.byref(st_blocks), C.byref(st_bytes))
    # which K1 kernel decoded (the library picks a flavour per column from a token sample at load): the one that decoded the most bytes
    k1 = {}
    for nm, kern in (("k1_v1", "lz4_decode_kernel"), ("k1_v3", "lz4_decode_v3_kernel"), ("k1_long", "lz4_decode_long_kernel"), ("k1_bytes", "lz4_decode_bytes_kernel"),
                     ("k1_lane", "lz4_decode_lane_kernel"), ("k1_spec", "lz4_decode_spec_kernel")):
        k1[kern] = phase(nm)[2]            # algorithmic bytes this kernel decoded
    k1_kernel = max(k1, key=k1.get)
    roofline = {"bound": "hbm", "kernel": k1_kernel, "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                "traffic": (lambda tr: int(tr / max(dec_n / max(args.steps, 1), 1)) if tr else tr)(ncu_traffic(k1_kernel, shard_rows)),
                "peak_source": peak_src, "algorithmic_bytes_per_launch": dec_bytes // max(dec_n, 1), "launches_per_step": dec_n / max(args.steps, 1),
                "avg_launch_ms": dec_launch_ms, "share_of_step": dec_ms / ms if ms else None,
                "note": "algorithmic bytes = compressed read + decoded written of the blocks the kernel decodes (column a); "
                        "achieved = those bytes / the decode phase's device time (CUDA events around the launch; when a decode is split in "
                        "two launches, from the start of the first to the end of the second); "
                        f"column b is {st_blocks.value} stored (incompressible) blocks = {st_bytes.value} bytes that the scan reads in place, no copy"}
    scan_achieved = (con_bytes / max(args.steps, 1)) / ((con_ms / max(args.steps, 1)) / 1e3) / 1e9 if con_ms > 0 else 0.0
    hbm_result = res
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, hbm_result)

    # ---- verification + CPU baseline (rank 0, N = 1): oracle over the same files, every host thread ----
    cpu_baseline = None
    verified = None
    if rank == 0 and not args.no_verify:
        from oracle import oracle as O
        ot = O.OracleTable(path)
        pb = D.plan_bytes(v.b)
        nb_total = t.nblocks()
        assert pb == BENCH_PLAN, "bench.py's constant plan bytes no longer match the plan encoder"
        sample_blocks = nb_total if world == 1 else min(nb_total, (1_000_000_000 + BLOCK - 1) // BLOCK)
        parts, dt = oracle_scan(ot, pb, sample_blocks, threads)
        sample_rows = min(total_rows, sample_blocks * BLOCK)
        cpu_baseline = {"value": sample_rows / dt, "unit": "rows/s", "cores": threads, "kind": "port",
                        "sample": f"{sample_rows} rows ({sample_blocks} blocks) of the same table, one thread per block range, {dt:.2f} s"}
        if world == 1:
            import math
            cnt = sum(p.count for p in parts)
            ksum = math.fsum(p.sum_kahan for p in parts)
            gsum = hbm_result.sum_f64 + hbm_result.sum_f64_lo
            ok = (cnt == hbm_result.count and abs(gsum - ksum) <= 1e-12 * abs(ksum)
                  and min(p.min_f64 for p in parts if p.count) == hbm_result.min_f64
                  and max(p.max_f64 for p in parts if p.count) == hbm_result.max_f64)
            verified = {"ok": bool(ok), "count": cnt, "sum_gpu": gsum, "sum_oracle_kahan": ksum, "rel_err": abs(gsum - ksum) / abs(ksum)}
            if not ok:
                log(f"[bench] PARITY FAILURE: gpu count {hbm_result.count} sum {gsum!r} vs oracle {cnt} {ksum!r}")
        ot.close()
    t.close()

    # ---- scan only: decoded columns cached in HBM (the 16 B/row figure of SURVEY.md 8d) ----
    t, v = open_view(D.LOAD_DECODED)
    step(v)
    _, ms_scan, _, _ = timed(v, args.steps, 1, profile=True)
    con2_ms, con2_n, con2_bytes = phase("consume")
    scan_only = {"rows_per_s": total_rows * args.steps / (ms_scan / 1e3), "kernel": "fused_scan_kernel<agg=f64,wide>",
                 "achieved": (16.0 * shard_rows * args.steps) / (con2_ms / 1e3) / 1e9 if con2_ms > 0 else None, "peak": peak, "unit": "GB/s",
                 "algorithmic_bytes_per_row": 16, "kernel_ms_per_step": con2_ms / max(args.steps, 1), "ms_per_step": ms_scan / args.steps}
    if scan_only["achieved"]:
        scan_only["frac"] = scan_only["achieved"] / peak
    t.close()

    # ---- what the box gives: pinned host -> device with every rank copying at once (the roofline of the transfer-inclusive mode) ----
    def h2d_ceiling():
        nb = 1 << 30
        host = torch.empty(nb, dtype=torch.uint8, pin_memory=True)
        host.fill_(1)
        devb = torch.empty(nb, dtype=torch.uint8, device="cuda")
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(stream)
        for _ in range(4):
            devb.copy_(host, non_blocking=True)
        b.record(stream)
        torch.cuda.synchronize()
        mine = torch.tensor([4 * nb / 1e9 / (a.elapsed_time(b) / 1e3)], dtype=torch.float64, device="cuda")
        rates = [mine]
        if world > 1:
            rates = [torch.zeros_like(mine) for _ in range(world)]
            dist.all_gather(rates, mine)
        del host, devb
        return [round(float(r.item()), 2) for r in rates]

    # ---- end to end: compressed blocks in pinned host memory, H2D inside every step ----
    e2e = None
    if not args.no_e2e:
        ceiling = h2d_ceiling()
        t, v = open_view(D.LOAD_HOST)
        k = max(3, min(args.steps, 5))
        res_e, ms_e, _, _ = timed(v, k, 1, profile=True)
        h2d_ms, _, h2d_bytes = phase("h2d")
        e2e = {"value": total_rows * k / (ms_e / 1e3), "unit": "rows/s", "h2d_bytes_per_step": shard_comp, "d2h_bytes_per_step": C.sizeof(_capi.Agg) + 8,
               "steps": k, "ms_per_step": ms_e / k, "h2d_gbs": (h2d_bytes / 1e9) / (h2d_ms / 1e3) if h2d_ms > 0 else None,
               "same_result": (res_e.count, res_e.sum_f64, res_e.sum_f64_lo) == (hbm_result.count, hbm_result.sum_f64, hbm_result.sum_f64_lo),
               "h2d_ceiling_gbs_per_rank": ceiling, "h2d_ceiling_gbs_aggregate": round(sum(ceiling), 2),
               "h2d_ceiling_note": "pinned host -> device, 1 GiB x 4, every rank copying at once, measured in this run; a step ends when the "
                                   "slowest rank ends, so the roofline of the whole job is world x the slowest rank's ceiling"}
        # roofline of the transfer-inclusive mode: bytes every rank must move / the slowest rank's measured H2D ceiling
        e2e["h2d_frac_of_node_ceiling"] = (shard_comp / 1e9 / (ms_e / k / 1e3)) / min(ceiling) if ms_e > 0 else None
        t.close()

    # ---- the other BASELINE.json configurations and the compressible-b variant of this one (SURVEY.md 8d), N = 1 only ----
    variants = None
    if world == 1 and not args.no_variants:
        try:
            variants = run_variants(args, threads, local)
        except Exception as e:                      # a variant must never take the headline line down with it
            log(f"[bench] variants failed: {e!r}")
            variants = {"error": repr(e)}

    if rank == 0:
        line = {
            "metric": "filtered-scan rows/s (LZ4 block decode + range predicate + sum/min/max/count)", "value": value, "unit": "rows/s",
            "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "int64/f64", "data": "synthetic", "config": workload_config(args, rows, info),
            "decoded_gbs": (shard_unc * world * args.steps / 1e9) / (ms / 1e3),
            "roofline": roofline, "cpu_baseline": cpu_baseline, "e2e": e2e, "gpu_launches": int(launches), "clocks": clocks,
            "scan_only": scan_only, "verified": verified, "variants": variants,
            "collective": ("NCCL, inside the library (dfdb_comm_init / dfdb_scan_aggregate_all: ncclAllGather of one 128-byte slot per rank)"
                           if world > 1 else None),
            "phases_ms_per_step": {"decode": dec_ms / args.steps, "consume": con_ms / args.steps,
                                   "consume_gbs": scan_achieved},
            "result": {"count": hbm_result.count, "sum": hbm_result.sum_f64 + hbm_result.sum_f64_lo, "min": hbm_result.min_f64, "max": hbm_result.max_f64},
        }
        print(json.dumps(line), flush=True)
    if world > 1:
        from dfdb_b200.dist import comm_destroy
        comm_destroy()
        dist.barrier()
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
