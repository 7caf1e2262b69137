#!/usr/bin/env python
"""bench.py — the headline benchmark: rows/s of a time-bucketed SUM group-by over a 1e9-row
synthetic fact table (BASELINE.json, config "1e9 rows, 3 filters + time-bucketizer + SUM group-by
2 dims"), on N B200s of one node.

    python bench.py [--gpus N] [--steps K] [--warmup W]            the B200 engine
    python bench.py --impl reference [--gpus N] ...                the reference's CPU path

A step = one whole query: every archive batch of the table goes through ExecuteBatchPlan (one fused
kernel per batch), then AggStateFinalize; with N > 1 the 8 day-batches are dealt round-robin to the
ranks (strong scaling: the table stays 1e9 rows) and the per-GPU group tables are merged over NCCL.
One JSON line on stdout (rank 0).  Zone maps (BatchPlan.Ranges) are PRODUCED by the engine
(ComputeColumnRanges, once per batch when it becomes device resident, timed separately); the result of
every workload is verified once, outside the timed region, against an independent torch restatement
(tests/independent.py) — `"verified": true`.  At N = 1 the line also carries the other BASELINE
configurations as `workloads` sub-results (same data, same code, fewer steps).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

NUM_BATCHES = 8


def _columns():
    from aresdb_b200 import expr as E, synth
    return tuple(E.Col(i, t, n) for i, (t, n) in enumerate(zip(synth.COLUMN_TYPES, synth.COLUMN_NAMES)))


def _q_cfg3():
    from aresdb_b200 import expr as E, synth
    from aresdb_b200.query import AggQuery, Measure
    TS, CITY, STATUS, FARE = _columns()
    t0 = synth.BASE_TS
    return AggQuery([E.eq(STATUS, E.Lit(1)), E.gt(FARE, E.Lit(5.0)), E.ne(CITY, E.Lit(0)),
                     E.ge(TS, E.Lit(t0 + 1800)), E.lt(TS, E.Lit(t0 + NUM_BATCHES * 86400 - 1800))],
                    [E.floor(TS, E.Lit(3600)), CITY], Measure("sum", FARE))


def _q_cfg3_count():
    from aresdb_b200 import expr as E
    from aresdb_b200.query import AggQuery, Measure
    TS, CITY, STATUS, FARE = _columns()
    return AggQuery([E.eq(STATUS, E.Lit(1)), E.gt(FARE, E.Lit(5.0)), E.ne(CITY, E.Lit(0))],
                    [E.floor(TS, E.Lit(3600)), CITY], Measure("count"))


def _q_cfg2():
    from aresdb_b200 import expr as E
    from aresdb_b200.query import AggQuery, Measure
    TS, CITY, STATUS, FARE = _columns()
    return AggQuery([E.eq(STATUS, E.Lit(1))], [CITY], Measure("sum", FARE))


def _q_cfg4():
    from aresdb_b200 import cabi as A, expr as E
    from aresdb_b200.query import AggQuery, Measure
    TS, CITY, STATUS, FARE = _columns()
    return AggQuery([], [CITY, E.floor(TS, E.Lit(60))], Measure("sum", FARE), reduce_mode=A.ARES_REDUCE_HASH)


def _q_cfg4_hll():
    from aresdb_b200 import expr as E
    from aresdb_b200.query import AggQuery, Measure
    TS, CITY, STATUS, FARE = _columns()
    return AggQuery([E.eq(STATUS, E.Lit(1))], [E.floor(TS, E.Lit(86400)), CITY], Measure("countdistincthll", TS))


# name -> description, query, algorithmic bytes per row (SURVEY.md §8d: value widths of the referenced
# columns + 1 bit per referenced null bitmap), default rows, batches, group-table hint, arithmetic
WORKLOADS = {
    "cfg3": dict(desc="cfg3: 1e9-row fact table as 8 day-batches; filters status==1, fare>5.0, city_id!=0, "
                      "request_at in [t0+1800, t0+8d-1800); dims floor(request_at,3600) x city_id; SUM(fare) in f64",
                 query=_q_cfg3, bytes_per_row=4 + 2 + 1 + 4 + 4 / 8.0, rows=1_000_000_000, batches=8, expected_groups=0,
                 dtype="u32/u16/u8 filters; f32 fares summed into f64 (exactly, as integers on the 2^-S grid the zone map allows)",
                 metric="rows/s, 1e9-row time-bucketed SUM group-by (cfg3)", check="cfg3"),
    "cfg3_count": dict(desc="cfg3 count(*) variant: filters status==1, fare>5.0, city_id!=0; dims floor(request_at,3600) x "
                            "city_id; COUNT in u32", query=_q_cfg3_count, bytes_per_row=4 + 2 + 1 + 4 + 4 / 8.0,
                       rows=1_000_000_000, batches=8, expected_groups=0, dtype="u32 count",
                       metric="rows/s, 1e9-row time-bucketed COUNT group-by (cfg3)", check="cfg3_count"),
    "cfg2": dict(desc="cfg2: 1e8-row fact table, one batch; filter status==1; dim city_id; SUM(fare) in f64",
                 query=_q_cfg2, bytes_per_row=1 + 2 + 4 + 3 / 8.0, rows=100_000_000, batches=1, expected_groups=0,
                 dtype="u8 filter, f32->f64 sum", metric="rows/s, 1e8-row SUM group-by 1 dim (cfg2)", check="cfg2"),
    "cfg4": dict(desc="cfg4: 1e9 rows as 8 day-batches, no filter; dims city_id x floor(request_at,60) (1.16e6 groups); "
                      "SUM(fare) in f64, hash-reduce semantics", query=_q_cfg4, bytes_per_row=4 + 2 + 4 + 3 / 8.0,
                 rows=1_000_000_000, batches=8, expected_groups=1_300_000, dtype="f32->f64 sum, 32-bit hash identity",
                 metric="rows/s, 1e9-row high-cardinality SUM group-by (cfg4)", check="cfg4"),
    "cfg4_hll": dict(desc="cfg4 HLL: 1e9 rows as 8 day-batches; filter status==1; dims floor(request_at,86400) x city_id "
                          "(808 groups); countdistincthll(request_at), p=14 registers",
                     query=_q_cfg4_hll, bytes_per_row=4 + 2 + 1 + 3 / 8.0, rows=1_000_000_000, batches=8,
                     expected_groups=0, dtype="u32 murmur3 -> rho/register max (dense registers per group)",
                     metric="rows/s, 1e9-row HLL distinct-count group-by (cfg4)", check="cfg4_hll"),
}
WORKLOADS["cfg3_zipf"] = dict(WORKLOADS["cfg3"], desc=WORKLOADS["cfg3"]["desc"] + "; city_id ~ Zipf(1.1)", city_dist="zipf",
                              metric="rows/s, 1e9-row time-bucketed SUM group-by (cfg3, Zipf cities)")
WL = WORKLOADS["cfg3"]


def select_workload(name: str):
    global WL
    WL = WORKLOADS[name]


def build_query():
    return WL["query"]()


# ---------------------------------------------------------------------------------------------------
# CPU baseline / reference arm: the reference's own per-node call sequence on host cores
# ---------------------------------------------------------------------------------------------------
def _physical_cores() -> list[int]:
    """One logical CPU per physical core of this process's affinity set (first SMT sibling)."""
    allowed = sorted(os.sched_getaffinity(0))
    seen, out = set(), []
    for c in allowed:
        try:
            sib = Path(f"/sys/devices/system/cpu/cpu{c}/topology/thread_siblings_list").read_text().strip()
        except OSError:
            sib = str(c)
        if sib not in seen:
            seen.add(sib)
            out.append(c)
    return out


def _cpu_worker(args):
    """One worker process = one table shard slice, pinned to one core: runs the reference call sequence over its rows,
    `reps` times, every repetition started together with the other workers (barrier)."""
    kind, slot, cpu, rows, reps, wl_name, barrier, out_q = args
    try:
        os.sched_setaffinity(0, {cpu})
    except OSError:
        pass
    select_workload(wl_name)
    sys.path.insert(0, str(ROOT))
    from aresdb_b200 import cabi, columns, synth
    from aresdb_b200.executor import Batch, LegacyBatchExecutor
    from aresdb_b200.memory import HostSpace
    if kind == "reference":
        lib = cabi.Library(ROOT / "oracle" / "_ref" / "libalgorithm.so", ROOT / "oracle" / "_ref" / "libmem_ref.so",
                           has_plan_api=False, name="ref")
    else:
        lib = cabi.Library(ROOT / "oracle" / "build" / "liboracle.so", None, has_plan_api=False, name="oracle")
    sp = HostSpace()
    hb = synth.generate_batch(slot % WL["batches"], rows, seed=777 + slot, city_dist=WL.get("city_dist", "uniform"))
    cols, keep = [], []
    for dt, v, ok in zip(synth.COLUMN_TYPES, hb.values, hb.valid):
        buf, vp = columns.make_column(sp, dt, v, valid=ok)
        cols.append(vp)
        keep.append(buf)
    q = build_query()
    if wl_name == "cfg4":
        # the HOST HashReduce extracts its result in O(g^2) (std::next over the map per slot,
        # reference query/hash_reduction.cu:143-156): time the same grouping through Sort + Reduce
        q.reduce_mode = cabi.ARES_REDUCE_SORT
    devnull = os.open(os.devnull, os.O_WRONLY)
    saved = os.dup(1)
    os.dup2(devnull, 1)  # the reference's HOST build prints a line per call (utils.cu:41-57)
    times, groups = [], 0
    try:
        for _ in range(reps):
            if barrier is not None:
                barrier.wait()
            t = time.perf_counter()
            ex = LegacyBatchExecutor(lib, sp, q)
            ex.process_batch(Batch(cols, rows), is_last=True)
            groups = ex.result_size
            times.append(time.perf_counter() - t)
    finally:
        os.dup2(saved, 1)
        os.close(devnull)
    out_q.put((slot, times, groups))


def _run_workers(ctx, kind, cpus, rows, reps, wl_name):
    barrier = ctx.Barrier(len(cpus)) if len(cpus) > 1 else None
    out_q = ctx.Queue()
    procs = [ctx.Process(target=_cpu_worker, args=((kind, i, c, rows, reps, wl_name, barrier, out_q),)) for i, c in enumerate(cpus)]
    for p in procs:
        p.start()
    res = [out_q.get(timeout=1800) for _ in procs]
    for p in procs:
        p.join()
    return sorted(res)


def cpu_reference_run(steps: int, warmup: int, rows_per_worker: int, workers: int | None = None, wl_name: str = "cfg3"):
    """Times the reference CPU path.  (i) ONE single-threaded executor on one core (the reference's HOST path is
    single-threaded per batch).  (ii) One executor per PHYSICAL core, each pinned, each over its own slice (the
    reference's unit of parallelism is the table shard / batch); every step starts behind a barrier, a step's time is
    its slowest worker, and the reported value is the MEDIAN over the steps."""
    import multiprocessing as mp
    kind = "reference" if (ROOT / "oracle" / "_ref" / "libalgorithm.so").exists() else "port"
    if kind == "port":
        sys.path.insert(0, str(ROOT / "oracle"))
        import build_oracle
        build_oracle.build()
    cores = _physical_cores()
    workers = max(1, min(workers or len(cores), len(cores), 128))
    cpus = cores[:workers]
    ctx = mp.get_context("spawn")
    t0 = time.perf_counter()
    single = _run_workers(ctx, kind, cpus[:1], rows_per_worker, 1 + max(1, min(steps, 3)), wl_name)
    single_s = float(np.median(single[0][1][1:]))
    res = _run_workers(ctx, kind, cpus, rows_per_worker, steps + warmup, wl_name)
    wall = time.perf_counter() - t0
    per_step = [max(r[1][i] for r in res) for i in range(warmup, warmup + steps)]   # barriered: slowest worker of the step
    ms = float(np.median(per_step)) * 1e3
    sample_rows = rows_per_worker * workers
    return {"value": sample_rows / (ms / 1e3), "ms_per_step": ms, "kind": kind, "cores": workers,
            "host_cores": os.cpu_count() or 1, "physical_cores": len(cores),
            "single_core_rows_per_s": rows_per_worker / single_s,
            "step_ms": [round(x * 1e3, 2) for x in per_step],
            "sample": f"{workers} pinned single-threaded workers (one per physical core) x {rows_per_worker} rows of the "
                      f"{wl_name} query per step, barrier per step, median of {steps} steps (reference HOST path is "
                      "single-threaded per batch)",
            "groups": int(res[0][2]), "wall_s": wall}


# ---------------------------------------------------------------------------------------------------
# clocks
# ---------------------------------------------------------------------------------------------------
class ClockSampler:
    def __init__(self, index: int):
        self.samples, self.proc, self.index = [], None, index

    def start(self):
        q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-lms", "100",
                                          "-i", str(self.index)], stdout=subprocess.PIPE, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.samples.append(line.strip())

    def stop(self):
        if self.proc:
            self.proc.terminate()
        sm, mx, reasons = [], 0, set()
        for s in self.samples:
            f = [x.strip() for x in s.split(",")]
            if len(f) < 8:
                continue
            try:
                sm.append(float(f[1]))
                mx = max(mx, float(f[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx or None, "reasons": sorted(reasons),
                "samples": len(sm)}


# ---------------------------------------------------------------------------------------------------
# the B200 arm
# ---------------------------------------------------------------------------------------------------
class DeviceTable:
    """The synthetic fact table of one rank: its day-batches resident in HBM (+ pinned host mirrors for e2e)."""

    def __init__(self, lib, space, dev, days, rows_per_batch, city_dist, mirror_host, shard=0):
        import torch
        from aresdb_b200 import columns, synth
        from aresdb_b200.executor import compute_zone_map
        self.days, self.rows_per_batch = days, rows_per_batch
        self.bufs, self.cols, self.zone_maps, self.host = [], [], [], []
        self.values_off = None
        zm_ms = []
        for d in days:
            bufs, self.values_off = synth.generate_batch_cuda(d, rows_per_batch, dev, city_dist=city_dist, seed=20260922 + shard)
            cols = [columns.slice_of(b.data_ptr(), dt, rows_per_batch, 0, self.values_off, 2) for b, dt in zip(bufs, synth.COLUMN_TYPES)]
            self.bufs.append(bufs)
            self.cols.append(cols)
            # the engine produces the zone map of the batch (ComputeColumnRanges); timed with CUDA events
            torch.cuda.synchronize()
            s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s.record()
            zm = compute_zone_map(lib, space, cols)
            e.record()
            torch.cuda.synchronize()
            zm_ms.append(s.elapsed_time(e))
            self.zone_maps.append(zm)
            if mirror_host:
                hb = []
                for b in bufs:
                    h = torch.empty(b.numel(), dtype=torch.uint8, pin_memory=True)
                    h.copy_(b)
                    hb.append(h)
                self.host.append(hb)
        torch.cuda.synchronize()
        self.zone_map_ms = float(np.median(zm_ms[1:] or zm_ms)) if zm_ms else None

    def batches(self, zone_maps: bool, rows: int | None = None, count: int | None = None):
        from aresdb_b200 import columns, synth
        from aresdb_b200.executor import Batch
        out = []
        for i in range(len(self.days) if count is None else min(count, len(self.days))):
            if rows is None or rows == self.rows_per_batch:
                cols, n = self.cols[i], self.rows_per_batch
            else:   # a prefix of the batch (cfg2: 1e8 rows of day 0)
                n = rows
                cols = [columns.slice_of(b.data_ptr(), dt, n, 0, self.values_off, 2) for b, dt in zip(self.bufs[i], synth.COLUMN_TYPES)]
            out.append(Batch(cols, n, ranges=self.zone_maps[i] if zone_maps else None))
        return out


def _verify(name, ex_result, table: "DeviceTable", dev, rows, count, is_hll, world, dist):
    """Independent check of one workload's result (outside every timed region).  Returns (ok, info)."""
    sys.path.insert(0, str(ROOT / "tests"))
    import independent as I
    from aresdb_b200 import synth
    t0 = synth.BASE_TS
    check = WORKLOADS[name]["check"]
    exp = I.Expected(check, NUM_BATCHES, dev, t0, t0 + 1800, t0 + NUM_BATCHES * 86400 - 1800)
    for i in range(len(table.days) if count is None else min(count, len(table.days))):
        exp.add_batch(table.bufs[i], table.values_off, rows)
    if world > 1:   # every rank holds its own days: the group space is global, sums of exact values are exact
        dist.all_reduce(exp.vals)
        p = exp.present.to(exp.vals.dtype)
        dist.all_reduce(p)
        exp.present = p != 0
        import torch
        k = torch.tensor([exp.rows_kept], device=dev, dtype=torch.int64)
        dist.all_reduce(k)
        exp.rows_kept = int(k.item())
    try:
        if is_hll:
            info = exp.check_hll(ex_result)
        elif name == "cfg4":
            info = _check_hash_identity(exp, ex_result)
        else:
            info = exp.check(ex_result)
        return True, info
    except AssertionError as e:
        return False, {"error": str(e)[:300]}


def _check_hash_identity(exp, res):
    """cfg4 runs with the reference's 32-bit hash identity: groups whose packed rows collide in murmur3-32 are ONE group
    (query/hash_reduction.cu:216-243); everything else must equal the independent result."""
    import hashes
    import independent as I
    from aresdb_b200 import synth
    rows = res.packed_rows()
    h = hashes.murmur3_32(rows)
    present = exp.present.cpu().numpy()
    vals = exp.vals.cpu().numpy()
    gidx = np.nonzero(present)[0]
    tidx, cidx = gidx // I.CITY_SPACE, gidx % I.CITY_SPACE
    tnull, cnull = tidx == exp.tn - 1, cidx == I.CITY_SPACE - 1
    erow = np.zeros((gidx.size, 8), np.uint8)
    erow[:, 0:4] = np.where(tnull, 0, synth.BASE_TS + tidx * 60).astype("<u4").view(np.uint8).reshape(-1, 4)
    erow[:, 4:6] = np.where(cnull, 0, cidx).astype("<u2").view(np.uint8).reshape(-1, 2)
    erow[:, 6] = ~tnull
    erow[:, 7] = ~cnull
    eh = hashes.murmur3_32(erow)
    order = np.argsort(eh, kind="stable")
    uniq, start = np.unique(eh[order], return_index=True)
    sums = np.add.reduceat(vals[gidx][order], start)
    assert res.groups == uniq.size == len(np.unique(h)), f"{res.groups} groups, expected {uniq.size}"
    pos = np.searchsorted(uniq, h)
    assert (uniq[pos] == h).all() and (res.measures.view(np.uint64) == sums[pos].view(np.uint64)).all(), "sums differ"
    return {"groups": int(res.groups), "rows_kept": exp.rows_kept, "distinct_rows": int(gidx.size),
            "merged_by_murmur3_32": int(gidx.size - uniq.size)}


def gpu_run(args):
    # keep stdout clean for the single JSON line: libraries (NCCL prints its version) write to fd 1
    real_stdout = os.dup(1)
    os.dup2(2, 1)
    import torch
    import torch.distributed as dist
    from aresdb_b200 import cabi as A
    from aresdb_b200 import columns, synth
    from aresdb_b200.executor import Batch
    from aresdb_b200.memory import CudaSpace
    from aresdb_b200.query import QueryResult
    from aresdb_b200.sharding import ShardedFusedQuery

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device(f"cuda:{local}")
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    lib = A.load_engine()
    stream = torch.cuda.current_stream().cuda_stream
    space = CudaSpace(local, stream)
    rows_total = args.rows or WL["rows"]
    num_batches = WL["batches"]
    rows_per_batch = rows_total // num_batches
    my_days = [d for d in range(num_batches) if d % world == rank]
    # one table per rank; at N = 1 the sub-workloads reuse it (cfg2 = the first 1e8 rows of day 0)
    table = DeviceTable(lib, space, dev, my_days, rows_per_batch, WL.get("city_dist", "uniform"), mirror_host=not args.no_e2e)
    zone_map_ms = table.zone_map_ms

    def run_workload(name, steps, warmup, zone_maps, table, with_kernel=True, with_e2e=False, verify=True, rows_scale=1,
                     dump_dir=None):
        """Times one workload on `table`; returns the sub-result dict (device-resident value, kernel-alone roofline,
        optional e2e, verification).  dump_dir: where to write the result of the last timed step (dump_outputs)."""
        wl = WORKLOADS[name]
        q = wl["query"]()
        nb = wl["batches"]
        rows_b = (args.rows or wl["rows"]) // nb
        count = len(table.days) if nb > 1 else 1
        batches = table.batches(zone_maps, rows_b, count)
        rows_all = (args.rows or wl["rows"]) * rows_scale
        ex = ShardedFusedQuery(lib, space, q, expected_groups=wl["expected_groups"])

        def finish():
            if q.is_hll:
                return ex.finalize_hll()
            return ex.finalize()

        def step_device():
            ex.reset()
            for b in batches:
                ex.process_batch(b)
            return finish()

        def timed(fn, steps, warmup):
            import gc
            keep = None
            for _ in range(warmup):
                keep = fn()   # (held like the timed loop holds `last`: result buffers reach their steady state here)
            keep = None
            # everything that takes host time happens BEFORE the barrier, so that the ranks leave it together
            gc.collect()
            gc.disable()   # (a collection inside a 0.5 ms step would be the whole step)
            evs = [torch.cuda.Event(enable_timing=True) for _ in range(steps + 1)]
            launches0 = lib.kernel_launch_count()
            torch.cuda.synchronize()
            if world > 1:
                dist.barrier()
            torch.cuda.synchronize()
            evs[0].record()
            last = None
            for i in range(steps):
                last = fn()
                evs[i + 1].record()
            torch.cuda.synchronize()
            gc.enable()
            if world > 1:
                dist.barrier()
            per = [evs[i].elapsed_time(evs[i + 1]) for i in range(steps)]
            ms = evs[0].elapsed_time(evs[steps]) / steps
            launches = (lib.kernel_launch_count() - launches0) // steps
            if world > 1:
                t = torch.tensor([ms] + per, device=dev)
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
                ms, per = float(t[0].item()), [float(x) for x in t[1:].tolist()]
            return ms, per, launches, last

        if name == args.workload and args.profile_range:  # `ncu --profile-from-start off`: only these steps are captured
            torch.cuda.profiler.start()
        ms, per, launches, last = timed(step_device, steps, warmup)
        if name == args.workload and args.profile_range:
            torch.cuda.synchronize()
            torch.cuda.profiler.stop()
        if dump_dir and rank == 0:
            if q.is_hll:
                dump_outputs(dump_dir, last)
            else:
                g, bufs = last
                dump_outputs(dump_dir, QueryResult(q, bufs.dims.get(np.uint8), bufs.capacity, bufs.measures.get(np.uint8), g))
        out = {"value": rows_all / (ms / 1e3), "unit": "rows/s", "ms_per_step": ms, "p50_query_ms": float(np.median(per)),
               "step_ms": [round(x, 4) for x in per],
               "steps": steps, "gpu_launches": int(launches), "zone_maps": bool(zone_maps)}

        # dominant kernel timed alone (one launch per batch, back to back), L2 cold because a batch >> L2
        if with_kernel and batches:
            ex.reset()
            torch.cuda.synchronize()
            s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            reps = max(2, min(steps, 5))
            l0 = lib.kernel_launch_count()
            s.record()
            for _ in range(reps):
                for b in batches:
                    ex.process_batch(b)
            e.record()
            torch.cuda.synchronize()
            kern_ms = s.elapsed_time(e) / (reps * len(batches))
            algo = wl["bytes_per_row"] * rows_b
            out["roofline"] = {"bound": "hbm", "kernel": "aresFusedJit (NVRTC-specialised fused scan-filter-aggregate)",
                               "achieved": algo / (kern_ms / 1e3) / 1e9, "peak": PEAK, "unit": "GB/s",
                               "frac": algo / (kern_ms / 1e3) / 1e9 / PEAK, "kernel_ms": kern_ms,
                               "launches_per_batch": (lib.kernel_launch_count() - l0) / (reps * len(batches)),
                               "algorithmic_bytes_per_launch": algo, "peak_source": PEAK_SRC}

        # result check, once, outside the timed regions
        if verify:
            if q.is_hll:
                res = last
            else:
                g, bufs = last
                res = QueryResult(q, bufs.dims.get(np.uint8), bufs.capacity, bufs.measures.get(np.uint8), g)
            ok, info = _verify(name, res, table, dev, rows_b, count, q.is_hll, world, dist)
            out["verified"] = bool(ok)
            out["check"] = info
            out["groups"] = int(res.groups)
        else:
            out["groups"] = int(last.groups if q.is_hll else last[0])

        if with_e2e and table.host:
            out["e2e"] = run_e2e(ex, q, table, batches, rows_all, timed, steps)
        ex.close()
        return out

    def run_e2e(ex, q, table, batches, rows_all, timed, steps):
        """The same query from HOST (pinned) columns: every step copies every batch host->device through the boundary's
        own libmem (AsyncCopyHostToDevice on a copy stream created by CreateCudaStream, WaitForCudaStream — the
        reference's transferBatch protocol, memstore/batch.go + cgoutils/memory.go), double-buffered against the
        fused kernels by a copier thread, produces the batch's zone map on the device, and reads the result back."""
        from aresdb_b200.executor import compute_zone_map
        copy_stream = lib.CreateCudaStream(local)

        class CopySpace:   # what compute_zone_map needs of a memory space: the stream and device to run on
            stream, device = copy_stream, local
        staging = [[torch.empty_like(b) for b in table.bufs[0]] for _ in range(2)]
        nb = len(batches)
        rows_b = batches[0].num_rows
        stats = {}

        def step_e2e():
            ex.reset()
            main = torch.cuda.current_stream()
            ready = [threading.Event() for _ in range(nb)]
            zms = [None] * nb
            freed = [None] * nb
            freed_set = [threading.Event() for _ in range(nb)]
            h2d = [0]
            err = []

            def copier():
                try:
                    torch.cuda.set_device(local)
                    for i in range(nb):
                        slot = i & 1
                        if i >= 2:
                            freed_set[i - 2].wait()
                            freed[i - 2].synchronize()   # the kernel that read this staging slot is done
                        for dst, src in zip(staging[slot], table.host[i]):
                            lib.AsyncCopyHostToDevice(dst.data_ptr(), src.data_ptr(), src.numel(), copy_stream, local)
                            h2d[0] += src.numel()
                        if batches[i].ranges is not None:
                            # the zone map of the freshly resident batch, on the COPY stream (it overlaps the fused kernel of
                            # the previous batch on the main stream); ComputeColumnRanges synchronises that stream
                            cols = [columns.slice_of(t.data_ptr(), dt, rows_b, 0, table.values_off, 2)
                                    for t, dt in zip(staging[slot], synth.COLUMN_TYPES)]
                            zms[i] = compute_zone_map(lib, CopySpace, cols)
                        else:
                            lib.WaitForCudaStream(copy_stream, local)
                        ready[i].set()
                except Exception as e:   # noqa: BLE001
                    err.append(e)
                    for r in ready:
                        r.set()

            if nb:
                main.synchronize()      # staging slots of the previous step are free
            th = threading.Thread(target=copier)
            th.start()
            for i in range(nb):
                ready[i].wait()
                if err:
                    raise err[0]
                slot = i & 1
                cols = [columns.slice_of(t.data_ptr(), dt, rows_b, 0, table.values_off, 2) for t, dt in zip(staging[slot], synth.COLUMN_TYPES)]
                ex.process_batch(Batch(cols, rows_b, ranges=zms[i]))
                ev = torch.cuda.Event()
                ev.record(main)
                freed[i] = ev
                freed_set[i].set()
            th.join()
            if q.is_hll:
                r = ex.finalize_hll()
                d2h = int(r.regs.size + r.counts.size * 2 + r.groups * q.row_bytes)
                stats.update(h2d=h2d[0], d2h=d2h)
                return r
            g, out = ex.finalize()
            dims_h = out.dims.handle[: max(out.dims.nbytes, 1)].cpu()
            meas_h = out.measures.handle[: g * q.measure_bytes].cpu()
            stats.update(h2d=h2d[0], d2h=int(dims_h.numel() + meas_h.numel()))
            return g, out

        e_ms, per, _, _ = timed(step_e2e, max(1, steps // 2), 1)
        lib.DestroyCudaStream(copy_stream, local)
        return {"value": rows_all / (e_ms / 1e3), "unit": "rows/s", "ms_per_step": e_ms,
                "h2d_bytes_per_step": int(stats.get("h2d", 0)) * world, "d2h_bytes_per_step": int(stats.get("d2h", 0)),
                "copy_path": "libmem AsyncCopyHostToDevice + WaitForCudaStream (C ABI), zone map computed on the device per batch"}

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    main = run_workload(args.workload, args.steps, args.warmup, not args.no_zone_maps, table, with_e2e=not args.no_e2e,
                        dump_dir=args.dump_outputs)
    clocks = sampler.stop() if rank == 0 else None

    subs = {}
    if world == 1 and not args.no_sub and args.workload == "cfg3" and not args.rows:
        sub_steps, sub_warm = max(3, min(args.steps, 5)), 3
        subs["cfg3_nozm"] = run_workload("cfg3", sub_steps, sub_warm, False, table)
        for name in ("cfg3_count", "cfg2", "cfg4", "cfg4_hll"):
            subs[name] = run_workload(name, sub_steps, sub_warm, True, table)
        if not args.no_zipf:
            del table
            torch.cuda.empty_cache()
            ztable = DeviceTable(lib, space, dev, list(range(NUM_BATCHES)), 125_000_000, "zipf", mirror_host=False)
            subs["cfg3_zipf"] = run_workload("cfg3_zipf", sub_steps, sub_warm, True, ztable)
            del ztable

    # N > 1: the headline keeps the table at 1e9 rows (strong scaling, as the metric is worded); the same query over a
    # table that grows with the ranks — every rank holds a 1e9-row SHARD of all the days (AresDB shards a table by key, so
    # every shard sees every group), 1e9 x N rows in all — is reported beside it
    weak = None
    if world > 1 and not args.no_weak and not args.rows:
        del table
        torch.cuda.empty_cache()
        wtable = DeviceTable(lib, space, dev, list(range(num_batches)), rows_per_batch, WL.get("city_dist", "uniform"),
                             mirror_host=False, shard=rank)
        w = run_workload(args.workload, args.steps, args.warmup, not args.no_zone_maps, wtable, with_kernel=False, rows_scale=world)
        weak = {"scaling": "weak", "rows": rows_total * world, "rows_per_gpu": rows_total, "value": w["value"], "unit": "rows/s",
                "ms_per_step": w["ms_per_step"], "p50_query_ms": w["p50_query_ms"], "verified": w.get("verified"),
                "groups": w.get("groups"), "gpu_launches": w["gpu_launches"]}
        del wtable

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    traffic = None
    try:  # DRAM bytes per launch from the committed ncu capture of this workload's kernel, scaled to this batch size
        for f in ("r02_traffic.json", "r01_traffic.json"):
            if (ROOT / "profiles" / f).exists():
                t = json.loads((ROOT / "profiles" / f).read_text()).get(args.workload)
                if t:
                    traffic = (t["dram_bytes_read"] + t["dram_bytes_write"]) * (rows_total // num_batches) / t["rows_per_launch"]
                    break
    except Exception:
        pass
    cpu = None
    if world == 1 and not args.no_cpu:
        cpu = cpu_reference_run(steps=3, warmup=1, rows_per_worker=args.cpu_rows, wl_name=args.workload)
        cpu = {k: cpu[k] for k in ("value", "kind", "cores", "host_cores", "physical_cores", "single_core_rows_per_s", "step_ms", "sample")}
        cpu["unit"] = "rows/s"
    roof = main.get("roofline") or {}
    roof["traffic"] = traffic
    out = {
        "metric": WL["metric"], "value": main["value"], "unit": "rows/s",
        "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": main["ms_per_step"],
        "p50_query_ms": main["p50_query_ms"], "step_ms": main["step_ms"],
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": WL["dtype"],
        "data": "synthetic", "groups": main["groups"], "verified": main.get("verified"), "check": main.get("check"),
        "config": {"workload": WL["desc"], "rows": rows_total, "batches": num_batches, "rows_per_batch": rows_total // num_batches,
                   "parallelism": f"batches round-robin over {world} GPU(s), NCCL merge of the per-GPU group tables" if world > 1 else "1 GPU",
                   "l2": f"inputs ({WL['bytes_per_row'] * (rows_total // num_batches) / 1e9:.2f} GB per batch) larger than the 126 MB L2; no flush needed",
                   "zone_maps": "off" if args.no_zone_maps else "per-batch column min/max produced by the engine (ComputeColumnRanges, once per "
                                "resident batch) and passed as BatchPlan.Ranges (direct-indexed aggregation where every dimension is bounded)",
                   "zone_map_ms_per_batch": zone_map_ms},
        "gpu_launches": main["gpu_launches"],
        "roofline": roof, "roofline_nozm": (subs.get("cfg3_nozm") or {}).get("roofline"),
        "e2e": main.get("e2e"), "cpu_baseline": cpu, "clocks": clocks, "workloads": subs or None,
        "weak_scaling": weak,
    }
    os.write(real_stdout, (json.dumps(out) + "\n").encode())
    if world > 1:
        dist.destroy_process_group()


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(out_dir, res):
    """Writes the groups of a QueryResult / HLLResult as DIR/<name>.npy, one row per group, ordered by the packed
    dimension row (the order a hash table hands groups out in is not part of the result), so that two builds can be
    compared array for array:
        dim<i>        float64, the i-th dimension's value (NaN for NULL)
        measures      float64 (SUM / COUNT / MIN / MAX / AVG), counts float64 for AVG
        hll_counts    float64, non-zero registers per group;  hll_registers float32 [groups, 16384], rho + 1 per register
    Above DUMP_LIMIT_BYTES in all, a fixed seeded sample of the groups is written and group_index names its rows."""
    from aresdb_b200.query import HLLResult
    hll = isinstance(res, HLLResult)
    qr = res.dims if hll else res
    rows = qr.packed_rows()
    order = np.lexsort(rows.T[::-1]) if rows.shape[1] else np.arange(qr.groups)
    arrays = {}
    for i, col in enumerate(qr.decoded_dims()):
        arrays[f"dim{i}"] = np.array([np.nan if v is None else float(v) for v in col], np.float64)[order]
    if hll:
        dense = res.dense_registers()
        arrays["hll_counts"] = res.counts.astype(np.float64)[order]
        arrays["hll_registers"] = np.stack([dense[qr.rows[g]] for g in order]).astype(np.float32) if qr.groups \
            else np.zeros((0, 1 << 14), np.float32)
    else:
        arrays["measures"] = qr.measures.astype(np.float64)[order]
        if qr.counts is not None:
            arrays["counts"] = qr.counts.astype(np.float64)[order]
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_LIMIT_BYTES:
        keep = int(qr.groups * DUMP_LIMIT_BYTES // (total + 8 * qr.groups))     # 8 bytes more per row: group_index
        idx = np.sort(np.random.default_rng(0).choice(qr.groups, size=keep, replace=False))
        arrays = {k: v[idx] for k, v in arrays.items()}
        arrays["group_index"] = idx.astype(np.float64)
    out = Path(out_dir)
    out.mkdir(parents=True, exist_ok=True)
    for f in out.glob("*.npy"):      # what an earlier dump left (another workload's dims, a sample's group_index)
        if f.stem in ("measures", "counts", "hll_counts", "hll_registers", "group_index") or \
                (f.stem.startswith("dim") and f.stem[3:].isdigit()):
            f.unlink()
    for k, v in arrays.items():
        np.save(out / f"{k}.npy", v)


PEAK, PEAK_SRC = 6650.0, "fallback 6650 GB/s"


def _load_peak():
    global PEAK, PEAK_SRC
    try:
        peaks = json.loads((ROOT / "MEASURED_PEAKS.json").read_text())
        PEAK, PEAK_SRC = float(peaks["hbm_gbs"]), "MEASURED_PEAKS.json hbm_gbs (burst copy bandwidth; the kernel is timed alone)"
    except Exception:
        pass


def reference_run(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    r = cpu_reference_run(args.steps, args.warmup, rows_per_worker=args.cpu_rows, wl_name=args.workload)
    out = {"impl": "reference", "metric": WL["metric"], "value": r["value"],
           "unit": "rows/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": r["ms_per_step"],
           "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": WL["dtype"],
           "data": "synthetic", "config": {"workload": WL["desc"], "rows": r["cores"] * args.cpu_rows,
                                           "note": "bounded sample of the workload; CPU throughput is size-independent"},
           "cpu_baseline": {"value": r["value"], "unit": "rows/s", "kind": r["kind"], "cores": r["cores"],
                            "host_cores": r["host_cores"], "physical_cores": r["physical_cores"],
                            "single_core_rows_per_s": r["single_core_rows_per_s"], "step_ms": r["step_ms"], "sample": r["sample"]},
           "e2e": {"value": r["value"], "unit": "rows/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
           "gpu_launches": 0}
    print(json.dumps(out))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="cfg3", choices=sorted(WORKLOADS),
                    help="cfg3 (default) is the headline; the others are the remaining BASELINE configs")
    ap.add_argument("--rows", type=int, default=0, help="override the workload's table size")
    ap.add_argument("--cpu-rows", type=int, default=4_000_000, help="rows per CPU worker per step (baseline sample)")
    ap.add_argument("--profile-range", action="store_true",
                    help="bracket the device-resident steps (warm-up included) with cudaProfilerStart/Stop for ncu")
    ap.add_argument("--no-zone-maps", action="store_true",
                    help="do not pass the per-batch column min/max (BatchPlan.Ranges): hash-table aggregation only")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-sub", action="store_true", help="N = 1: skip the sub-results of the other BASELINE configs")
    ap.add_argument("--no-weak", action="store_true", help="N > 1: skip the weak-scaling leg (1e9 rows per GPU)")
    ap.add_argument("--no-zipf", action="store_true", help="skip the Zipf-city sub-result (a second 11.5 GB table)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="B200 path: write the result of the last timed step of --workload as DIR/<name>.npy (see dump_outputs)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    select_workload(args.workload)
    _load_peak()
    if args.impl == "reference":
        reference_run(args)
    else:
        gpu_run(args)


if __name__ == "__main__":
    main()
