#!/usr/bin/env python
"""bench.py — rows/s of scan + filter + hash-aggregate on the 100M-row Parca schema (BASELINE.json).

  python bench.py --gpus N --steps K --warmup W [--impl frostgpu|reference] [--dump-outputs DIR]

One process per GPU (torchrun sets RANK / LOCAL_RANK / WORLD_SIZE).  A step is one execution of

    ScanTable(t).Filter(timestamp in the middle 50% of the range)
                .Aggregate([Sum(value), Count(value)], [labels.l00, labels.l01])

over this rank's parts: 100M rows per GPU (weak scaling), 16 dynamic label columns, parts of 4Mi
rows sorted the way compaction leaves them, row groups of 1Mi rows.  N > 1 adds the one exchange
step the path has, inside the library (fgpu_query_execute_collective): every rank's partial table is
stored into every rank's peer-mapped mailbox over NVLink and merged behind a flag wait.

The line also carries `parity` (the timed result compared bit-exact with the oracle on the same rows;
a mismatch fails the run) and `extra` (the other BASELINE.json configurations: cfg 2 latency, cfg 3
without filter and on unsorted parts, the cfg 5 selectivity sweep), each with kernel time, algorithmic
bytes and roofline fraction.

`value`  parts resident in HBM before the timed region (fgpu_query_execute only).
`e2e`    the same query through the public C-ABI from HOST Parquet buffers: every step puts the
         parts (host parse + H2D), executes, reads the result record back and drops the parts.
`--impl reference` times the CPU restatement of the reference path (oracle/, a port: the Go
         engine cannot be built here) on all host cores, on a bounded sample of the same workload.
`--dump-outputs DIR` writes the result record of the last timed step to DIR, one float64 .npy per
         column (see dump_outputs).  The inputs are generated from a fixed seed, so two builds run
         with the same arguments can be compared output for output.
"""
from __future__ import annotations

import argparse
import hashlib
import json
import os
import re
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import bench_data as bd  # noqa: E402
from frostdb_b200 import logicalplan as lp  # noqa: E402

METRIC = "rows/sec scan+filter+hash-agg (100M-row Parca schema)"
N_LABELS = 16
TABLE = "bench"


def env_int(name, default):
    return int(os.environ.get(name, default))


def headline_query_exprs(total_first_row: int, rows: int):
    lo = bd.T0 + total_first_row + rows // 4
    hi = bd.T0 + total_first_row + (3 * rows) // 4
    filt = lp.And(lp.Col("timestamp").GtEq(lp.Literal(lo)), lp.Col("timestamp").Lt(lp.Literal(hi)))
    aggs = [lp.Sum(lp.Col("value")), lp.Count(lp.Col("value"))]
    groups = [lp.Col("labels.l00"), lp.Col("labels.l01")]
    return filt, aggs, groups



def result_rows(batches):
    """Result records -> {key tuple: aggregate tuple} (dictionary key columns decoded; aggregates are the trailing
    columns named func(expr))."""
    import pyarrow as pa
    out = {}
    for b in batches:
        names = b.schema.names
        cols = []
        for i, n in enumerate(names):
            a = b.column(i)
            if pa.types.is_dictionary(a.type):
                a = a.dictionary_decode()
            vals = a.to_pylist()
            cols.append([v.decode() if isinstance(v, (bytes, bytearray)) else v for v in vals])
        nk = sum(1 for n in names if not (n.endswith(")") and "(" in n))
        order = sorted(range(nk), key=lambda i: names[i])  # key columns by name: both engines may order them differently
        for r in range(b.num_rows):
            key = tuple((names[i], cols[i][r]) for i in order)
            out[key] = tuple(cols[i][r] for i in range(nk, len(names)))
    return out


def parity_of(gpu_rows: dict, ref_rows: dict) -> dict:
    """Bit-exact comparison of two results (integer aggregates)."""
    mism = 0
    for k, v in ref_rows.items():
        if gpu_rows.get(k) != v:
            mism += 1
    mism += sum(1 for k in gpu_rows if k not in ref_rows)
    return {"checked": True, "groups": len(ref_rows), "gpu_groups": len(gpu_rows), "mismatches": mism}


DUMP_BYTES = 64 << 20


def dump_outputs(out_dir, rows: dict, key_names, agg_names) -> None:
    """Writes a result ({key tuple: aggregate tuple}, as result_rows returns it) as out_dir/<column>.npy, float64, one file
    per key column (by name, as in the key tuples) and per aggregate.  Rows are in key order (NULL last), so two runs
    compare element for element whatever order the engine returned the groups in.  A string key is written as a 48-bit
    BLAKE2b digest of its UTF-8 bytes (exact in float64), NULL as NaN.  A result of more than DUMP_BYTES keeps a fixed,
    seeded sample of its rows."""
    items = sorted(rows.items(), key=lambda kv: tuple((v is None, v) for _, v in kv[0]))
    cap = DUMP_BYTES // (8 * max(1, len(key_names) + len(agg_names)))
    if len(items) > cap:
        keep = np.sort(np.random.default_rng(0).choice(len(items), cap, replace=False))
        items = [items[i] for i in keep]

    def num(v):
        if v is None:
            return np.nan
        if isinstance(v, str):
            return float(int.from_bytes(hashlib.blake2b(v.encode(), digest_size=6).digest(), "little"))
        return float(v)

    cols = {n: [num(k[j][1]) for k, _ in items] for j, n in enumerate(key_names)}
    cols.update({n: [num(a[j]) for _, a in items] for j, n in enumerate(agg_names)})
    os.makedirs(out_dir, exist_ok=True)
    for n, vals in cols.items():
        np.save(os.path.join(out_dir, re.sub(r"[^0-9A-Za-z.]+", "_", n).strip("_") + ".npy"), np.asarray(vals, dtype=np.float64))


def oracle_rows(bufs, plan_scan, agg_names, threads, sample_rows=0, reps=1):
    """Runs the oracle over the given Parquet buffers; returns (result rows, best seconds, rows scanned)."""
    from oracle import oracle as orc
    table = orc.OracleTable()
    for b in bufs:
        table.add_pinned(b.ctypes.data, b.nbytes, b)
    plan, keep = plan_scan._plan()
    best, scanned, rows = None, 0, {}
    for _ in range(reps):
        t0 = time.perf_counter()
        r = table.execute(plan, threads=threads, max_rows=sample_rows)
        d = time.perf_counter() - t0
        scanned = r.rows_scanned
        if not rows:
            rows = result_rows([r.to_batch(agg_names)])
        r.close()
        best = d if best is None else min(best, d)
    table.close()
    return rows, best, scanned


def load_files(paths):
    return [np.fromfile(p, dtype=np.uint8) for p in paths]


class ClockSampler(threading.Thread):
    """nvidia-smi clocks + throttle reasons during the timed region (B200_PROFILING.md)."""

    def __init__(self, gpu_index: int):
        super().__init__(daemon=True)
        self.gpu_index, self.samples, self.stop_flag, self.proc = gpu_index, [], False, None

    def run(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.gpu_index}", f"--query-gpu={q}", "--format=csv,noheader,nounits",
                                          "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            for line in self.proc.stdout:
                if self.stop_flag:
                    break
                self.samples.append([x.strip() for x in line.split(",")])
        except Exception:
            pass

    def stop(self):
        self.stop_flag = True
        if self.proc:
            try:
                self.proc.terminate()
                self.proc.wait(timeout=5)
            except Exception:
                pass

    def summary(self):
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for s in self.samples:
            try:
                sm.append(float(s[0]))
                mx.append(float(s[1]))
                for n, v in zip(names, s[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(n)
            except Exception:
                continue
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(mx)), "reasons": sorted(reasons), "samples": len(sm)}


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def run_reference(args, rows_per_gpu):
    """CPU restatement of the reference path on all host cores, bounded sample (rank 0 only)."""
    rank = env_int("RANK", 0)
    if rank != 0:
        return
    from frostdb_b200.physicalplan import GPUScan
    from frostdb_b200 import _lib
    from oracle import oracle as orc
    cores = os.cpu_count() or 1
    threads = min(cores, env_int("FROSTGPU_REF_THREADS", cores))
    sample_rows = min(rows_per_gpu, env_int("FROSTGPU_REF_SAMPLE_ROWS", 128 * bd.RG_ROWS))
    paths = bd.generate_parts(rows_per_gpu, N_LABELS)
    need_parts = (sample_rows + bd.PART_ROWS - 1) // bd.PART_ROWS
    bufs = load_files(paths[:need_parts])
    table = orc.OracleTable()
    for b in bufs:
        table.add_pinned(b.ctypes.data, b.nbytes, b)
    filt, aggs, groups = headline_query_exprs(0, rows_per_gpu)
    scan = GPUScan(None, TABLE, filt, _lib.PLAN_AGGREGATE, groups, aggs)
    plan, keep = scan._plan()
    agg_names = [a.Name() for a in aggs]
    times, scanned = [], 0
    for it in range(args.warmup + args.steps):
        t0 = time.perf_counter()
        res = table.execute(plan, threads=threads, max_rows=sample_rows)
        dt = time.perf_counter() - t0
        scanned = res.rows_scanned
        if args.dump_outputs and it == args.warmup + args.steps - 1:
            dump_outputs(args.dump_outputs, result_rows([res.to_batch(agg_names)]), sorted(g.Name() for g in groups), agg_names)
        res.close()
        if it >= args.warmup:
            times.append(dt)
    total = sum(times)
    value = scanned * len(times) / total
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": "rows/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1000.0 * total / len(times), "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "int64", "data": "synthetic",
        "config": workload_config(rows_per_gpu, args.gpus),
        "cpu_baseline": {"value": value, "unit": "rows/s", "cores": threads, "kind": "port",
                         "sample": f"{scanned} rows ({scanned // bd.RG_ROWS} row groups of the same parts) per step, C port of the "
                                   "reference's decode->filter->hash-aggregate chain (oracle/frost_oracle.c), one chain per thread"},
        "e2e": {"value": value, "unit": "rows/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def workload_config(rows_per_gpu, n_gpus):
    return {"workload": f"cfg3+filter: {rows_per_gpu} rows per GPU x {n_gpus} GPU(s), Parca SampleDefinition with {N_LABELS} dynamic "
                        "label columns, Filter(timestamp in the middle 50% of the rank's own time range) + Sum(value),Count(value) GROUP BY labels.l00,labels.l01 "
                        "(<=16705 groups); parts of 4Mi rows sorted in compaction order, 1Mi-row row groups, uncompressed, DataPageV2",
            "rows_per_gpu": rows_per_gpu, "label_columns": N_LABELS, "part_rows": bd.PART_ROWS, "row_group_rows": bd.RG_ROWS,
            "l2": "inputs (>=0.5 GB read per step per GPU) exceed the 126 MB L2; no explicit flush",
            "parallelism": f"parts sharded one range per GPU x{n_gpus}; the partial -> final aggregate step runs inside the library "
                           "(fgpu_query_execute_collective: NVLink stores into peer-mapped mailboxes, flag wait, merge kernel)"}


def run_case(eng, lib, table, rows, kind, filt, groups, aggs, peak, reps=5, env=None, note=None):
    """One query on resident parts: kernel time (CUDA events around the scan launches), Execute wall time, bytes."""
    import ctypes as C
    from frostdb_b200 import _lib
    from frostdb_b200.physicalplan import GPUScan
    env = env or {}
    os.environ.update(env)
    try:
        scan = GPUScan(eng, table, filt, kind, groups, aggs)
        q, keep = scan.prepare()
        ks, ws, st = [], [], None
        for i in range(reps + 1):
            res = C.c_void_p()
            t0 = time.perf_counter()
            _lib.check(lib.fgpu_query_execute(eng.handle, q, eng.table_watermark(table), C.byref(res)))
            w = (time.perf_counter() - t0) * 1e3
            st = eng.stats(res)
            lib.fgpu_result_free(res)
            if i:
                ks.append(st["scan_kernel_ms"])
                ws.append(w)
        lib.fgpu_query_free(q)
    finally:
        for k in env:
            os.environ.pop(k)
    k = float(np.median(ks))
    out = {"rows": int(rows), "kernel_ms": round(k, 4), "exec_ms": round(float(np.median(ws)), 4),
           "algorithmic_bytes": int(st["algorithmic_bytes"]), "GBps": round(st["algorithmic_bytes"] / k / 1e6, 1) if k > 0 else None,
           "frac": round(st["algorithmic_bytes"] / k / 1e6 / peak, 4) if k > 0 else None, "rows_selected": int(st["rows_selected"]),
           "result_rows": int(st["groups"]), "row_groups": int(st["row_groups"]), "row_groups_pruned": int(st["row_groups_pruned"]),
           "row_groups_runs": int(st["row_groups_runs"]), "row_groups_tiles": int(st["row_groups_tiles"])}
    if note:
        out["note"] = note
    return out


def extra_configs(eng, lib, rows_per_gpu, peak):
    """The other BASELINE.json configurations, measured on one GPU next to the headline (N == 1 only)."""
    from frostdb_b200 import _lib
    AGG, FILT = _lib.PLAN_AGGREGATE, _lib.PLAN_FILTER
    ts, val = lp.Col("timestamp"), lp.Col("value")
    K01 = [lp.Col("labels.l00"), lp.Col("labels.l01")]
    SC = [lp.Sum(val), lp.Count(val)]
    out = {}
    # cfg 3 as BASELINE.json states it: no filter, Sum + Count by two dictionary keys, all 100M rows
    out["cfg3_sorted_nofilter"] = run_case(eng, lib, TABLE, rows_per_gpu, AGG, None, K01, SC, peak)
    # cfg 5: filter-only compaction (timestamp, value of the passing rows) and filter + Sum, int64 and dictionary predicates
    sweep = {}
    for sel in (0.001, 0.01, 0.1, 0.5, 0.9):
        f = ts.Lt(lp.Literal(bd.T0 + int(sel * rows_per_gpu)))
        sweep[f"rows_ts_lt_{sel}"] = run_case(eng, lib, TABLE, rows_per_gpu, FILT, f, [ts, val], [], peak, reps=2)
        sweep[f"sum_ts_lt_{sel}"] = run_case(eng, lib, TABLE, rows_per_gpu, AGG, f, [], [lp.Sum(val)], peak, reps=3)
    for sel in (0.001, 0.1, 0.5):  # spread over every row group: no pruning possible
        f = val.Lt(lp.Literal(int(sel * 1000)))
        sweep[f"rows_value_lt_{int(sel * 1000)}"] = run_case(eng, lib, TABLE, rows_per_gpu, FILT, f, [ts, val], [], peak, reps=2)
    fd = lp.Col("labels.l02").Eq(lp.Literal("v000003"))
    sweep["rows_l02_eq"] = run_case(eng, lib, TABLE, rows_per_gpu, FILT, fd, [ts, val], [], peak, reps=2)
    sweep["sum_l02_eq"] = run_case(eng, lib, TABLE, rows_per_gpu, AGG, fd, [], [lp.Sum(val)], peak, reps=3)
    out["cfg5_selectivity_sweep_sorted_100M"] = sweep
    out["cfg3_sorted_sum_by_l02_short_runs"] = run_case(eng, lib, TABLE, rows_per_gpu, AGG, None, [lp.Col("labels.l02")], [lp.Sum(val)], peak)
    # cfg 3 on UNSORTED parts (arrival order, table.go:1410-1426): bit-packed keys, the tile-aggregate kernel
    n_un = min(rows_per_gpu, env_int("FROSTGPU_BENCH_UNSORTED_ROWS", 32 * 1024 * 1024))
    paths = bd.generate_parts(n_un, N_LABELS, sort=False)
    for pth in paths:
        eng.put_parquet("bench_unsorted", np.fromfile(pth, dtype=np.uint8))
    lo, hi = bd.T0 + n_un // 4, bd.T0 + (3 * n_un) // 4
    f50 = lp.And(ts.GtEq(lp.Literal(lo)), ts.Lt(lp.Literal(hi)))
    out["cfg3_unsorted_nofilter"] = run_case(eng, lib, "bench_unsorted", n_un, AGG, None, K01, SC, peak)
    out["cfg3_unsorted_filter50"] = run_case(eng, lib, "bench_unsorted", n_un, AGG, f50, K01, SC, peak)
    out["cfg3_unsorted_general_kernel"] = run_case(eng, lib, "bench_unsorted", n_un, AGG, None, K01, SC, peak, reps=2, env={"FROSTGPU_NO_TILE": "1"},
                                                  note="the same query with the tile-aggregate kernel switched off (k_scan)")
    eng.drop_table("bench_unsorted")
    # cfg 2: 1M rows, 4 label columns, Filter(timestamp range 50%) + Sum(value) GROUP BY labels.l00 (C = 64): latency
    n2 = 1_000_000
    for pth in bd.generate_parts(n2, 4, part_rows=n2, rg_rows=bd.RG_ROWS):
        eng.put_parquet("bench_cfg2", np.fromfile(pth, dtype=np.uint8))
    f2 = lp.And(ts.Gt(lp.Literal(bd.T0 + n2 // 4)), ts.Lt(lp.Literal(bd.T0 + (3 * n2) // 4)))
    out["cfg2_1M_rows_latency"] = run_case(eng, lib, "bench_cfg2", n2, AGG, f2, [lp.Col("labels.l00")], [lp.Sum(val)], peak, reps=20,
                                           note="launch / latency bound: exec_ms is the number")
    eng.drop_table("bench_cfg2")
    # cfg 4's key space on one GPU: C0 = C1 = 1024 (~1M groups, ~4 rows per group and 4 Mi-row part), Sum + Count by two
    # keys.  Runs this short are bit-packed: the tile-aggregate kernel with its table in global memory (L2).  (The full
    # config — 1 B rows, 64 label columns over 8 GPUs — is not run here.)
    n4 = min(rows_per_gpu, env_int("FROSTGPU_BENCH_CFG4_ROWS", 32 * 1024 * 1024))
    for pth in bd.generate_parts(n4, N_LABELS, c0=1024, c1=1024):
        eng.put_parquet("bench_cfg4", np.fromfile(pth, dtype=np.uint8))
    out["cfg4_keyspace_1M_groups"] = run_case(eng, lib, "bench_cfg4", n4, AGG, None, K01, SC, peak, reps=3,
                                              note="1025 x 1025 dense slots (25 MB table in L2), result of ~1M rows: exec_ms includes its export")
    eng.drop_table("bench_cfg4")
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="frostgpu", choices=["frostgpu", "reference"])
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the result of the last timed step to DIR/<column>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3)
    rows_per_gpu = env_int("FROSTGPU_BENCH_ROWS", 100_000_000)
    if args.impl == "reference":
        run_reference(args, rows_per_gpu)
        return

    import torch
    import torch.distributed as dist
    from frostdb_b200 import _lib
    from frostdb_b200.physicalplan import GPUScan
    from frostdb_b200.store import GPUEngine
    import ctypes as C

    rank, world, local = env_int("RANK", 0), env_int("WORLD_SIZE", 1), env_int("LOCAL_RANK", 0)
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the frostgpu arm has no CPU fallback")
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    lib = _lib.load()

    first_row = rank * rows_per_gpu
    t_gen = time.perf_counter()
    paths = bd.generate_parts(rows_per_gpu, N_LABELS, first_row=first_row)
    bufs = load_files(paths)
    t_gen = time.perf_counter() - t_gen
    file_bytes = sum(b.nbytes for b in bufs)

    eng = GPUEngine(local)
    # cross-rank dictionary ids: union of every rank's dictionary entries, in rank order, preloaded
    # before the parts are put (one-time, at upload)
    key_cols = ["labels.l00", "labels.l01"]
    unions = {}
    if world > 1:
        for col in key_cols:
            seen, mine = set(), []
            for b in bufs:
                for v in _lib.parquet_dict_values(b, col):
                    if v not in seen:
                        seen.add(v)
                        mine.append(v)
            allv = [None] * world
            dist.all_gather_object(allv, mine)
            seen, union = set(), []
            for vs in allv:
                for v in vs:
                    if v not in seen:
                        seen.add(v)
                        union.append(v)
            unions[col] = union
            eng.dict_preload(TABLE, col, union)

        def exchange(handle):  # the mailbox handles travel once, at setup
            allh = [None] * world
            dist.all_gather_object(allh, handle)
            return allh
        eng.comm_open(rank, world, exchange, slot_bytes=8 << 20)
    t_up = time.perf_counter()
    for b in bufs:
        eng.put_parquet(TABLE, b)
    t_up = time.perf_counter() - t_up

    filt, aggs, groups = headline_query_exprs(first_row, rows_per_gpu)
    agg_names = [a.Name() for a in aggs]
    scan = GPUScan(eng, TABLE, filt, _lib.PLAN_AGGREGATE, groups, aggs)
    q, keep = scan.prepare()
    tx = eng.table_watermark(TABLE)
    execute = lib.fgpu_query_execute_collective if world > 1 else lib.fgpu_query_execute

    def step(q_=None, tx_=None):
        """ONE C call per step: scan (+ at N > 1 the exchange and the merge, inside the library) -> result record."""
        res = C.c_void_p()
        _lib.check(execute(eng.handle, q if q_ is None else q_, tx if tx_ is None else tx_, C.byref(res)))
        st = eng.stats(res)
        batches = list(eng.drain(res))
        lib.fgpu_result_free(res)
        return st, batches

    def sync_all():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    for _ in range(args.warmup):
        st, batches = step()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
        time.sleep(0.3)
    sync_all()
    t0 = time.perf_counter()
    scan_ms, launches, alg_bytes = [], 0, 0
    for _ in range(args.steps):
        st, batches = step()
        scan_ms.append(st["scan_kernel_ms"])
        launches += st["kernel_launches"]
        alg_bytes = st["algorithmic_bytes"]
    sync_all()
    dt = time.perf_counter() - t0
    if rank == 0:
        time.sleep(0.2)
        sampler.stop()
    tmax = torch.tensor([dt], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
    dt = float(tmax.item())
    total_rows = rows_per_gpu * world
    value = total_rows * args.steps / dt
    gpu_rows = result_rows(batches)  # the last timed step's record (at N > 1: the merged result, on every rank)
    if rank == 0 and args.dump_outputs:
        dump_outputs(args.dump_outputs, gpu_rows, sorted(g.Name() for g in groups), agg_names)

    # ---- e2e: host Parquet buffers -> result record, every step --------------------------------------
    # The parts sit in page-locked host memory (where the Go side would have written them); a step
    # registers them (footer + page-header parse), executes the query — which builds and uploads only
    # the projected columns, PLAIN pages DMA'd straight from the host buffers — reads the result
    # record back and drops the parts again.
    e2e = None
    if not os.environ.get("FROSTGPU_SKIP_E2E"):
        from frostdb_b200.store import PinnedBuffer
        e2e_steps = max(1, min(args.steps, env_int("FROSTGPU_E2E_STEPS", 3)))
        E2E = "bench_e2e"
        pinned = []
        for b in bufs:
            pb = PinnedBuffer(b.nbytes)
            pb.array[:] = b
            pinned.append(pb)
        scan_e = GPUScan(eng, E2E, filt, _lib.PLAN_AGGREGATE, groups, aggs)
        h2d = {"bytes": 0}

        def e2e_step():
            for col, union in unions.items():  # (multi-rank) same dictionary ids on every rank
                eng.dict_preload(E2E, col, union)
            for pb in pinned:
                eng.put_parquet(E2E, pb.array, borrow=True)
            qe, keep_e = scan_e.prepare()  # the shim prepares per Execute; equal plans share their compiled state
            st_e, batches_e = step(qe, eng.table_watermark(E2E))
            lib.fgpu_query_free(qe)
            h2d["bytes"] = st_e["h2d_bytes"]
            d2h = sum(x.nbytes for x in batches_e)
            eng.drop_table(E2E)
            return d2h

        e2e_step()  # warm
        sync_all()
        t0 = time.perf_counter()
        d2h = 0
        for _ in range(e2e_steps):
            d2h = e2e_step()
        sync_all()
        de = time.perf_counter() - t0
        tde = torch.tensor([de], dtype=torch.float64, device="cuda")
        tb = torch.tensor([float(h2d["bytes"])], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(tde, op=dist.ReduceOp.MAX)
            dist.all_reduce(tb, op=dist.ReduceOp.SUM)
        de, h2d["bytes"] = float(tde.item()), int(tb.item())
        e2e = {"value": rows_per_gpu * world * e2e_steps / de, "unit": "rows/s", "h2d_bytes_per_step": int(h2d["bytes"]),
               "d2h_bytes_per_step": int(d2h), "steps": e2e_steps, "ms_per_step": 1000.0 * de / e2e_steps,
               "note": "every step: fgpu_part_put_parquet(BORROW_PINNED) of all parts from page-locked host memory (footer/page "
                       "parse), fgpu_query_prepare + execute (builds + uploads the projected columns, then the scan), result record read "
                       "back, fgpu_table_drop"}
        for pb in pinned:
            pb.close()

    # ---- parity of the timed result + CPU baseline -------------------------------------------------------
    # Every rank runs the oracle (test infrastructure, oracle/) over ITS OWN 100M rows with the same plan; the
    # per-rank oracle results are added up (Sum and Count are additive) and compared bit for bit with the record the
    # last timed step returned.  At N == 1 the same oracle runs are the cpu_baseline (best of 3).
    cpu, parity = None, {"checked": False}
    if not os.environ.get("FROSTGPU_SKIP_CPU"):
        cores = os.cpu_count() or 1
        threads = max(1, cores // world)
        ref_rows, best, scanned = oracle_rows(bufs, scan, agg_names, threads, sample_rows=0, reps=3 if world == 1 else 1)
        if world > 1:
            allr = [None] * world
            dist.all_gather_object(allr, ref_rows)
            merged = {}
            for rr in allr:
                for k_, v_ in rr.items():
                    merged[k_] = tuple(a + b_ for a, b_ in zip(merged[k_], v_)) if k_ in merged else v_
            ref_rows = merged
        parity = parity_of(gpu_rows, ref_rows)
        parity["rows"] = int(total_rows)
        parity["how"] = ("oracle (oracle/frost_oracle.c) over the same %d rows per rank, per-rank results added; compared bit-exact with the "
                         "record of the last timed step" % rows_per_gpu)
        if world == 1:
            cpu = {"value": scanned / best, "unit": "rows/s", "cores": threads, "kind": "port",
                   "sample": f"{scanned} rows of the same parts, best of 3, C port of the reference chain (oracle/frost_oracle.c)"}

    extra = None
    if rank == 0 and world == 1 and not os.environ.get("FROSTGPU_SKIP_EXTRA"):
        extra = extra_configs(eng, lib, rows_per_gpu, measured_peak()[0])

    rc = 0
    if rank == 0:
        peak, peak_src = measured_peak()
        avg_scan_ms = float(np.mean(scan_ms))
        achieved = alg_bytes / (avg_scan_ms * 1e-3) / 1e9 if avg_scan_ms > 0 else 0.0
        # DRAM traffic of the dominant kernel: from the committed ncu --set full capture of this same
        # workload (profiles/*_traffic.json), only when the launch processes the same bytes
        traffic, traffic_src = None, None
        for name in ("r2_traffic.json", "r1_traffic.json"):
            try:
                with open(os.path.join(ROOT, "profiles", name)) as f:
                    tr = json.load(f)
                if tr["workload_rows_per_gpu"] == rows_per_gpu and abs(tr["algorithmic_bytes"] - alg_bytes) <= 0.01 * alg_bytes:
                    traffic = int(tr["dram_bytes_read"] + tr["dram_bytes_write"])
                    traffic_src = f"profiles/{name} (ncu --set full capture of this workload's scan launch; not re-measured in this run)"
                    break
            except (OSError, KeyError, ValueError):
                pass
        line = {
            "metric": METRIC, "value": value, "unit": "rows/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": 1000.0 * dt / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "int64", "data": "synthetic", "config": workload_config(rows_per_gpu, world),
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": traffic, "traffic_source": traffic_src,
                         "kernel": "fgpu::k_runs_tma (sorted-run scan, TMA-staged tiles); unsorted / short-run / nullable keys: fgpu::k_tile_agg, see extra",
                         "kernel_ms": avg_scan_ms, "algorithmic_bytes": int(alg_bytes), "peak_source": peak_src},
            "cpu_baseline": cpu, "e2e": e2e, "gpu_launches": int(launches), "clocks": sampler.summary(),
            "parity": parity, "groups": int(st["groups"]), "rows_selected_per_gpu": int(st["rows_selected"]),
            "rows_touched_per_gpu": int(st["rows_touched"]),
            "row_groups": {"scanned": int(st["row_groups"]), "pruned": int(st["row_groups_pruned"])},
            "setup": {"generate_s": round(t_gen, 2), "upload_s": round(t_up, 2), "parquet_bytes_per_gpu": int(file_bytes)},
            "extra": extra,
        }
        print(json.dumps(line), flush=True)
        if parity.get("checked") and parity["mismatches"]:
            print(f"bench.py: PARITY FAILURE: {parity['mismatches']} of {parity['groups']} groups differ from the oracle", file=sys.stderr)
            rc = 3
    lib.fgpu_query_free(q)
    if world > 1:
        sync_all()
        eng.comm_close()
    eng.close()
    if world > 1:
        dist.destroy_process_group()
    if rc:
        sys.exit(rc)


if __name__ == "__main__":
    main()
