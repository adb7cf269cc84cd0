#!/usr/bin/env python
"""bench.py — scanned rows/s of the per-segment filter + group-by hot path (BASELINE.json metric).

Workload at N=1 (BASELINE.json configs[1]): 8 segments x 12.5 M rows = 100 M rows of the 20-column synthetic table
(only the 8 columns the query touches are materialised), inverted index on c1 disabled so both predicates scan:

    SELECT d0,d1,d2, SUM(m0), COUNT(*), MIN(m1), MAX(m2) FROM t
    WHERE c1 IN (16 values) AND c2 < k(50 %) GROUP BY d0,d1,d2            -- 4 096 groups, ~0.8 % selectivity

A step = one pass of the whole query over all segments of this rank through the C ABI (host planning layer ->
pb_query_execute, merged result table back in pinned host memory).  `value` = rows / wall time of K steps with the
segments already resident in HBM; `e2e` = the same call sequence starting from page-locked HOST buffers inside the timed
region (pb_segment_stage + execute + result read-back; headline policy PB_Q_GATHER_IN_PLACE = copy the predicate columns,
gather the group-by / aggregation columns of the matching rows over PCIe; the copy-every-touched-column policy is
measured alongside as e2e.legs.stage_all).  N > 1 (one process per GPU under torchrun): the per-rank tables are merged
INSIDE libpinot_b200.so (pb_comm_init + PB_Q_ALL_RANKS: one ncclAllGather of the table block + a merge kernel on the call's
stream) and every rank gets the merged table.  Two curves are measured in every run: weak (every GPU owns its own 8 x
12.5 M rows) and strong (the same 100 M-row table, 64 segments, 64 / N per GPU); `scaling` / `value` are the headline's
(--scaling, default weak), the other curve is reported under its own key.  Before anything is timed the (merged) device
result is compared with the oracle's over all ranks' segments (`parity_checked`).

`--impl reference` times the CPU restatement of the reference path (oracle/, the one place this file may run it
besides the cpu_baseline legs and the parity check) on ALL host cores, one segment per core.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "scanned rows/sec for filter+groupby(3 dims,4 aggs) @1/2/4/8 B200; %HBM BW"


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--segments", type=int, default=8)
    ap.add_argument("--docs-per-segment", type=int, default=12_500_000)
    ap.add_argument("--in-values", type=int, default=16)
    ap.add_argument("--flags", type=int, default=0, help="extra PB_Q_* flags (A/B: 4 = generic predicate path, 8 = no TMA)")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--e2e-policy", choices=("in_place", "stage_all"), default="in_place",
                    help="cold-segment staging policy of the e2e leg (stage_all is always measured and reported alongside)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--scaling", choices=("weak", "strong"), default="weak",
                    help="which curve is the headline (value / ms_per_step); the other one is measured too and reported alongside")
    ap.add_argument("--strong-segments", type=int, default=64, help="segments of the fixed 100 M-row table of the strong-scaling curve")
    ap.add_argument("--no-variants", action="store_true", help="skip the 25 %% selectivity variant and the second scaling curve")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the result table of the last timed headline step as DIR/<name>.npy (float64), so that two builds "
                         "can be compared output for output on the same seeded table")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs applies to --impl b200")
    return args


def measured_peak_gbs():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """SM clock + throttle reasons sampled DURING the timed region (NVML in a thread; same fields as the
    nvidia-smi line of B200_PROFILING.md, without forking a process inside the timed region)."""

    def __init__(self, gpu_index: int, period_s: float = 0.001):
        self.gpu, self.period = gpu_index, period_s
        self.sm, self.reasons, self.smmax = [], set(), None
        self._stop = threading.Event()
        self.t = None
        self.err = None

    def mark(self):
        """samples taken before this call (warm-up) are dropped"""
        self.sm = []
        self.reasons = set()

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            idx = self.gpu
            if vis:
                try:
                    idx = int(vis.split(",")[self.gpu])
                except Exception:
                    idx = self.gpu
            self.h = pynvml.nvmlDeviceGetHandleByIndex(idx)
            self.smmax = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
        except Exception as e:   # pragma: no cover
            self.err = repr(e)
            return
        self.t = threading.Thread(target=self._run, daemon=True)
        self.t.start()

    def _run(self):
        nv = self.nv
        bits = {"hw_slowdown": getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8),
                "hw_thermal_slowdown": getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40),
                "sw_thermal_slowdown": getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20),
                "sw_power_cap": getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4)}
        while not self._stop.is_set():
            try:
                self.sm.append(float(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)))
                try:
                    r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for k, b in bits.items():
                    if r & b:
                        self.reasons.add(k)
            except Exception as e:   # pragma: no cover
                self.err = repr(e)
                break
            self._stop.wait(self.period)

    def stop(self):
        self._stop.set()
        if self.t:
            self.t.join(timeout=1)
        out = {"sm_mhz": float(np.median(self.sm)) if self.sm else None, "sm_max_mhz": self.smmax,
               "reasons": sorted(self.reasons), "samples": len(self.sm)}
        if self.err:
            out["error"] = self.err
        return out


def build_table(args, rank):
    from pinot_b200 import datagen
    segs = datagen.make_table(args.segments, args.docs_per_segment, columns=datagen.CONFIG2_COLUMNS,
                              first_index=rank * args.segments)
    return segs


def algorithmic_bytes(segs, q, part="all"):
    """BASELINE.md §3: sum over segments of numDocs x sum over touched columns of storedBits / 8 (full-scan convention).
    part = "filter": only the predicate columns (what pb_filter_kernel streams); "agg": the group-by/metric columns."""
    _, preds = q.filter_postfix()
    fcols = {p.column for p in preds}
    acols = set(q.group_by) | {a.column for a in q.aggregations if a.column}
    touched = fcols | acols if part == "all" else (fcols if part == "filter" else acols - fcols)
    total = 0.0
    for s in segs:
        bits = 0
        for c in touched:
            col = s.columns[c]
            bits += col.bits_per_element if col.has_dictionary else 8 * col.dict_entry_bytes
        total += s.num_docs * bits / 8.0
    return total


_oracle_prepared = {}


def oracle_query_all_threads(segs, q, threads):
    """One CombineOperator-style pass on the CPU: the segments on `threads` pooled native worker threads (pthreads inside
    liboracle.so, the segments and the query marshalled once), every worker folding its segments' results into an IndexedTable
    of its own, tables merged at the end -- GroupByCombineOperator without the interpreter anywhere in the timed loop."""
    from oracle import oracle
    key = (id(segs[0]), len(segs), id(q))
    prep = _oracle_prepared.get(key)
    if prep is None:
        prep = _oracle_prepared[key] = oracle.PreparedBatch(segs, q)
    merged = oracle.execute_combined(prep, threads)      # segments AND merge on native worker threads
    if merged is not None:
        return merged
    res = oracle.execute_batch(prep, threads)
    return oracle.combine_numeric(res)


def run_reference(args, rank, world):
    """The reference's own CPU path (restated in C: oracle/) on ALL the host cores the box has: the same 100 M rows and the
    same query, cut into one segment per core (at most 128; Pinot parallelises a query over segments,
    BaseCombineOperator.java:97-142, so the segment count is what bounds its parallelism), one thread per segment, then the
    cross-segment merge.  Each step is one full pass over the table."""
    if rank != 0:
        return
    from oracle import oracle
    from pinot_b200 import datagen
    from pinot_b200.query import parse_sql
    oracle.build()
    cores = os.cpu_count() or 1
    total_rows = args.segments * args.docs_per_segment
    n_segs = max(args.segments, min(cores, 128))
    docs = total_rows // n_segs
    segs = [datagen.make_segment_synth(200_000 + i, docs, columns=datagen.CONFIG2_COLUMNS) for i in range(n_segs)]
    q = parse_sql(datagen.config2_sql(segs, args.in_values))
    threads = min(len(segs), cores)
    rows = sum(s.num_docs for s in segs)
    for _ in range(args.warmup):
        oracle_query_all_threads(segs, q, threads)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        oracle_query_all_threads(segs, q, threads)
    dt = time.perf_counter() - t0
    value = rows * args.steps / dt
    cfg = workload_config(args, segs)
    cfg["workload"] = (f"BASELINE.json configs[1]: the {rows}-row table as {n_segs} segments x {docs} rows (one per host core), "
                       f"WHERE c1 IN({args.in_values}) AND c2<k GROUP BY d0,d1,d2 SUM/COUNT/MIN/MAX, skipIndexes c1=inverted")
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": "rows/s", "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1000 * dt / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": cfg,
            "cpu_baseline": {"value": value, "unit": "rows/s", "cores": threads, "kind": "port",
                             "sample": f"full {rows}-row query per step as {n_segs} segments, one thread per segment ({threads} threads of {cores} cores), {args.steps} steps"},
            "e2e": {"value": value, "unit": "rows/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    _emit(line)


def workload_config(args, segs, w=None):
    return {"workload": f"BASELINE.json configs[1]: {len(segs)} segments x {segs[0].num_docs} rows{' per GPU' if args.gpus > 1 else ''}, "
                        f"WHERE c1 IN({args.in_values}) AND c2<k GROUP BY d0,d1,d2 SUM/COUNT/MIN/MAX, skipIndexes c1=inverted",
            "segments_per_gpu": len(segs), "rows_per_gpu": sum(s.num_docs for s in segs),
            "columns_materialised": "8 touched of the 20-column table", "l2_policy": "inputs (>1 GB/GPU) larger than the 126 MB L2",
            "parallelism": (f"segments sharded over {args.gpus} GPUs, one process per GPU; per-rank group tables merged inside libpinot_b200.so "
                            f"(PB_Q_ALL_RANKS: one ncclAllGather of the table block + pb_merge_blocks_kernel on the call's stream)") if args.gpus > 1 else "1 GPU"}


def _teardown(native, dist):
    """Communicator and process-group teardown after the line is out.  Every rank has finished its work by now; a teardown that
    cannot complete (a peer that died, a collective library waiting for a resource) must not keep the job alive: a watchdog
    ends the process 20 s later whatever happens."""
    import threading
    threading.Thread(target=lambda: (time.sleep(20), os._exit(0)), daemon=True).start()
    native.comm_destroy()
    dist.destroy_process_group()


_JSON_OUT = None


def _claim_stdout():
    """The contract is ONE JSON line on stdout.  Libraries loaded later write banners to file descriptor 1 from C (NCCL prints
    its version there): keep a private duplicate of the real stdout for the JSON line and point fd 1 at stderr for everyone else."""
    global _JSON_OUT
    if _JSON_OUT is None:
        sys.stdout.flush()
        _JSON_OUT = os.fdopen(os.dup(1), "w")
        os.dup2(2, 1)


def _emit(line: dict):
    out = _JSON_OUT or sys.stdout
    out.write(json.dumps(line) + "\n")
    out.flush()


class Workload:
    """One rank's share of a table + the query over it, staged and ready to step."""

    def __init__(self, args, rank, world, scaling, dist=None):
        from pinot_b200 import datagen, native
        from pinot_b200.query import parse_sql
        self.scaling, self.rank, self.world = scaling, rank, world
        if scaling == "weak":        # every GPU owns 8 x 12.5 M rows (BASELINE.json configs[1] per GPU)
            self.segs = datagen.make_table(args.segments, args.docs_per_segment, columns=datagen.CONFIG2_COLUMNS,
                                           first_index=rank * args.segments)
            self.table_rows = args.segments * args.docs_per_segment * world
        else:                        # the SAME 100 M-row table at every N: 64 x 1 562 500 rows, 64 / N segments per GPU
            n_total, docs = args.strong_segments, args.segments * args.docs_per_segment // args.strong_segments
            from pinot_b200.distributed import shard_segments
            mine = shard_segments(n_total, rank, world)
            self.segs = [datagen.make_segment_synth(100_000 + i, docs, columns=datagen.CONFIG2_COLUMNS) for i in mine]
            self.table_rows = n_total * docs
        self.sql = datagen.config2_sql(self.segs, args.in_values)
        self.q = parse_sql(self.sql)
        self.rows_rank = sum(s.num_docs for s in self.segs)
        self.flags = native.PB_Q_COMBINE | args.flags | (native.PB_Q_ALL_RANKS if world > 1 else 0)
        # page-lock the host copies of the touched columns (what a server does once for its mmap'd segments)
        for s in self.segs:
            for c in s.columns.values():
                native.host_register(c.forward_index)
        self.staged = [native.StagedSegment(s) for s in self.segs]
        self.group = native.SegmentGroup(self.staged)
        if world > 1:
            # the ranks agree on the global dictionaries of the group-by columns once (dense tables must line up)
            from pinot_b200.distributed import TorchExchange, agree_global_dictionaries, dictionary_columns
            cols = dictionary_columns(self.q, self.segs[0])
            agree_global_dictionaries(self.group, cols, [int(self.segs[0].columns[c].data_type) for c in cols], TorchExchange(dist))
        self.prepared = native.prepare(self.q)

    def with_query(self, sql):
        """the same staged segments under another query (e.g. the 25 % selectivity variant)"""
        import copy
        from pinot_b200 import native
        from pinot_b200.query import parse_sql
        w = copy.copy(self)
        w.sql, w.q = sql, parse_sql(sql)
        w.prepared = native.prepare(w.q)
        return w

    def step(self, group=None, extra_flags=0):
        """one pass of the hot path over this rank's segments THROUGH THE C ABI: plan + kernels + (N > 1) the NCCL merge
        of the per-rank tables inside libpinot_b200.so + result hand-back.  Every rank gets the merged table."""
        from pinot_b200 import native
        return native.execute(group or self.group, self.q, self.flags | extra_flags, self.prepared)

    def release(self):
        from pinot_b200 import native
        self.group.release()
        for st in self.staged:
            st.release()
        for s in self.segs:
            for c in s.columns.values():
                try:
                    native.host_unregister(c.forward_index)
                except Exception:
                    pass


def _merge_oracle_tables(tables, q):
    """key -> row dicts of several ranks (oracle.combine output) -> one table: SUM/COUNT add, MIN/MAX fold, AVG pairs add"""
    from pinot_b200.query import AggOp
    out = {}
    for t in tables:
        for k, row in t.items():
            if k not in out:
                out[k] = list(row)
                continue
            cur = out[k]
            for a, agg in enumerate(q.aggregations):
                if agg.op in (AggOp.COUNT, AggOp.SUM):
                    cur[a] = cur[a] + row[a]
                elif agg.op == AggOp.MIN:
                    cur[a] = min(cur[a], row[a])
                elif agg.op == AggOp.MAX:
                    cur[a] = max(cur[a], row[a])
                elif agg.op == AggOp.AVG:
                    cur[a] = (cur[a][0] + row[a][0], cur[a][1] + row[a][1])
                else:
                    raise ValueError("parity check: unsupported aggregation")
    return out


def parity_check(w, dist, threads):
    """BEFORE anything is timed: the (merged) device result of the bench query must equal the oracle's over ALL ranks'
    segments -- every group, every aggregate, bit for bit (sums of this workload are integers < 2^53), plus the statistics.
    Every rank runs the oracle on its own segments (the checker, not the product path); the per-rank oracle tables are
    exchanged and merged on the host.  Raises on the first difference."""
    from concurrent.futures import ThreadPoolExecutor
    from oracle import oracle
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from tests.parity import assert_rows_equal, combined_rows
    oracle.build()
    with ThreadPoolExecutor(max_workers=threads) as ex:
        orc = list(ex.map(lambda s: oracle.execute(s, w.q), w.segs))
    mine = combined_rows(oracle.combine(orc), w.q)
    docs = sum(o.stats["num_docs_scanned"] for o in orc)
    if w.world > 1:
        gathered = [None] * w.world
        dist.all_gather_object(gathered, (mine, docs))
        exp = _merge_oracle_tables([g[0] for g in gathered], w.q)
        docs = sum(g[1] for g in gathered)
    else:
        exp = mine
    r = w.step()
    t = r.tables[0]
    assert_rows_equal(t.rows(), exp, w.q, exact_float=True, what=f"bench parity ({w.scaling}, rank {w.rank} of {w.world})")
    assert t.stats["num_docs_scanned"] == docs, (t.stats, docs)
    assert t.stats["num_total_docs"] == w.table_rows, (t.stats, w.table_rows)
    n = t.num_groups
    r.free()
    return {"groups": int(n), "docs_matched": int(docs), "ranks_checked": w.world}


def result_arrays(table, q):
    """The merged result table a caller of the hot path receives, copied out of the result's pinned memory as float64 arrays:
    `keys` [groups, group-by columns], one array per aggregation named after it (COUNT from the long slot, SUM / MIN / MAX
    from the double slot) and `stats` (docs scanned, entries scanned in / post filter, total docs).  A GROUP BY without
    ORDER BY returns its groups in no defined order, so the rows are put in key order.  The bench query has at most
    8 x 16 x 32 groups: well under a megabyte in all."""
    from pinot_b200.query import AggOp
    keys = np.stack([np.asarray(v, dtype=np.float64) for v in table.key_values], axis=1)
    order = np.lexsort(keys.T[::-1])
    out = {"keys": keys[order]}
    for a, agg in enumerate(q.aggregations):
        src = table.longs if agg.op == AggOp.COUNT else table.doubles
        out[f"{agg.op.name.lower()}_{agg.column or 'star'}"] = np.asarray(src[a], dtype=np.float64)[order]
    out["stats"] = np.array([table.stats[k] for k in ("num_docs_scanned", "num_entries_scanned_in_filter",
                                                      "num_entries_scanned_post_filter", "num_total_docs")], dtype=np.float64)
    return out


def run_timed(w, steps, warmup, torch, dist, sampler=None):
    """W warm-up steps, then exactly K timed steps bracketed by barrier + synchronize; returns the timing record (max over
    ranks) and the per-kernel CUDA-event times measured by the library on the call's stream."""
    import gc
    world = w.world

    def barrier():
        if world > 1:
            dist.barrier()

    gc.collect()
    gc.disable()          # no cyclic-GC pauses inside the timed region (re-enabled right after)
    for _ in range(max(warmup, 3)):
        w.step().free()
    rec = {k: [] for k in ("scan", "filt", "agg", "comm", "wall", "device", "host_us")}
    launches = 0
    barrier()
    torch.cuda.synchronize()
    if sampler:
        sampler.mark()
    t0 = time.perf_counter()
    last = None
    for _ in range(steps):
        ts = time.perf_counter()
        if last is not None:
            last.free()            # the operator frees a result before it runs the next query (same as the warm-up)
        r = w.step()
        rec["wall"].append(1000 * (time.perf_counter() - ts))
        rec["scan"].append(r.scan_ms())
        f_, a_ = r.phase_ms()      # CUDA events on the call's stream (a cached plan samples them on every 8th replay and repeats the sample in between)
        rec["filt"].append(f_)
        rec["agg"].append(a_)
        rec["comm"].append(r.comm_ms())
        launches += lib_launches(r)
        rec["device"].append(getattr(r, "device_ms", 0.0))
        rec["host_us"].append(r.host_timing_us())
        last = r
    torch.cuda.synchronize()
    barrier()
    elapsed = time.perf_counter() - t0
    gc.enable()
    in_region = len(sampler.sm) if sampler else 0
    if world > 1:
        t = torch.tensor([elapsed, float(np.mean(rec["scan"])), float(np.mean(rec["comm"]))], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        elapsed, scan_max, comm_max = (float(x) for x in t.tolist())
    else:
        scan_max, comm_max = float(np.mean(rec["scan"])), 0.0
    out = {"elapsed": elapsed, "ms_per_step": 1000 * elapsed / steps, "value": w.rows_rank * world * steps / elapsed,
           "scan_ms": scan_max, "comm_ms": comm_max, "filter_ms": float(np.mean(rec["filt"])), "agg_ms": float(np.mean(rec["agg"])),
           "device_ms": float(np.mean(rec["device"])) if rec["device"] else None, "launches": launches,
           "host_us": [round(float(x), 1) for x in np.mean(np.array(rec["host_us"]), axis=0)],
           "step_wall": rec["wall"], "in_region_samples": in_region, "last": last}
    return out


def main():
    args = parse_args()
    _claim_stdout()
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return 0

    import torch
    import torch.distributed as dist
    from pinot_b200 import datagen, native

    os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")   # keep NCCL's banner off stdout (one JSON line only)
    torch.cuda.set_device(local_rank)
    native.init(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
        # the data-path communicator lives INSIDE libpinot_b200.so (pb_comm_init); torch.distributed only carries the
        # rendezvous (NCCL id, dictionary agreement), the barriers and the max-over-ranks of the timings
        from pinot_b200.distributed import TorchExchange, init_comm
        init_comm(TorchExchange(dist))
    oracle_threads = max(1, min(args.segments, os.cpu_count() or 1))

    head_scaling = args.scaling
    w = Workload(args, rank, world, head_scaling, dist)
    segs, q = w.segs, w.q
    parity = {head_scaling: parity_check(w, dist, oracle_threads)}

    # ---- headline: W warm-up + exactly K timed steps ----
    sampler = ClockSampler(local_rank)
    sampler.start()
    T = run_timed(w, args.steps, args.warmup, torch, dist, sampler)
    elapsed, last = T["elapsed"], T["last"]
    outputs = result_arrays(last.tables[0], q) if args.dump_outputs else None
    # A K-step region of this workload lasts only a few ms, shorter than a handful of NVML reads: keep the SAME steps
    # running (untimed, same count on every rank) right after it so the clock median is taken under the identical load.
    n_extra = 0 if elapsed >= 0.25 else min(5000, int(0.25 / max(elapsed / max(args.steps, 1), 1e-5)))
    for _ in range(n_extra):
        last.free()
        last = w.step()
    torch.cuda.synchronize()
    clocks = sampler.stop()
    clocks["samples_in_timed_region"] = T["in_region_samples"]
    clocks["window"] = "timed region" if n_extra == 0 else f"timed region + {n_extra} identical untimed steps run back-to-back after it"
    value = T["value"]
    num_groups = last.tables[0].num_groups
    docs_matched = last.tables[0].stats["num_docs_scanned"]
    d2h_bytes = int(num_groups * (16 + 16 * len(q.aggregations)) + 64)
    last.free()

    # ---- the 25 % selectivity variant of the same query (IN list of 500 values: loads the aggregation phase) ----
    sel25 = None
    if not args.no_variants:
        w25 = w.with_query(datagen.config2_sql(segs, 500))
        p25 = parity_check(w25, dist, oracle_threads)
        T25 = run_timed(w25, max(3, min(args.steps, 10)), 3, torch, dist)
        T25["last"].free()
        alg25 = algorithmic_bytes(segs, w25.q, "all") * world
        sel25 = {"workload": "same table, c1 IN(500 values) AND c2 < k: ~25 % of the rows pass the filter", "ms_per_step": T25["ms_per_step"],
                 "value": T25["value"], "filter_kernel_ms": T25["filter_ms"], "agg_kernel_ms": T25["agg_ms"], "docs_matched": p25["docs_matched"],
                 "parity_checked": True,
                 "whole_query_frac_on_step_time": alg25 / (T25["ms_per_step"] * 1e-3) / 1e9 / (measured_peak_gbs()[0] * world),
                 "whole_query_frac_on_kernel_time": (algorithmic_bytes(segs, w25.q, "all") / ((T25["filter_ms"] + T25["agg_ms"]) * 1e-3) / 1e9 / measured_peak_gbs()[0]
                                                     if T25["filter_ms"] + T25["agg_ms"] > 0 else None)}

    # ---- the other scaling curve (both are reported at every N; `scaling` names the headline's) ----
    other = None
    other_name = "strong" if head_scaling == "weak" else "weak"
    w2 = None
    if not args.no_variants:
        w2 = Workload(args, rank, world, other_name, dist)
        parity[other_name] = parity_check(w2, dist, oracle_threads)
        T2 = run_timed(w2, args.steps, args.warmup, torch, dist)
        T2["last"].free()
        other = {"scaling": other_name, "ms_per_step": T2["ms_per_step"], "value": T2["value"], "rows_total": w2.rows_rank * world,
                 "segments_per_gpu": len(w2.segs), "rows_per_segment": w2.segs[0].num_docs,
                 "breakdown_ms": {"filter_kernel": T2["filter_ms"], "agg_kernel": T2["agg_ms"], "nccl_merge": T2["comm_ms"],
                                  "device_total": T2["device_ms"], "host_and_gaps": T2["ms_per_step"] - (T2["device_ms"] or 0.0)},
                 "parity_checked": True}

    # ---- e2e: same call sequence from HOST buffers (stage + execute + read-back) ----
    e2e = None
    rows_total = w.rows_rank * world
    if not args.no_e2e:
        e2e_steps = max(2, min(args.steps, 5))
        docs_matched_rank = docs_matched // max(world, 1)       # merged statistics are totals over ranks; per-rank data is iid

        def barrier():
            if world > 1:
                dist.barrier()

        def e2e_leg(in_place):
            """stage from the page-locked host buffers + execute + read the result back, K times.  in_place: only the
            predicate columns are copied to HBM; the group-by / aggregation columns are gathered over PCIe from the
            mapped host buffers for the matching rows (PB_Q_GATHER_IN_PLACE)."""
            staged_bytes, in_place_cols = 0, 0

            def e2e_step():
                nonlocal staged_bytes, in_place_cols
                st = [native.StagedSegment(s) for s in segs]
                g2 = native.SegmentGroup(st)
                if world > 1:
                    for col in q.group_by:
                        g2.set_global_dictionary(col, w.group.export_dictionary(col))
                r2 = w.step(g2, native.PB_Q_GATHER_IN_PLACE if in_place else 0)
                _ = r2.tables[0].num_groups if r2.tables else 0      # result read-back
                staged_bytes = sum(s.device_bytes() for s in st)
                in_place_cols = r2.in_place_columns
                r2.free()
                g2.release()
                for s in st:
                    s.release()

            e2e_step()   # warm
            barrier()
            torch.cuda.synchronize()
            t1 = time.perf_counter()
            for _ in range(e2e_steps):
                e2e_step()
            torch.cuda.synchronize()
            barrier()
            el = time.perf_counter() - t1
            if world > 1:
                t = torch.tensor([el], dtype=torch.float64, device="cuda")
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
                el = float(t.item())
            # in place: every gathered value is one or two 4-byte words; PCIe moves them as 32-byte sectors
            gather_values = docs_matched_rank * in_place_cols // max(len(segs), 1)     # matching rows x columns read in place
            h2d = int(staged_bytes + 32 * gather_values)
            return {"value": rows_total * e2e_steps / el, "ms_per_step": 1000 * el / e2e_steps, "h2d_bytes_per_step": h2d,
                    "staged_bytes_per_step": int(staged_bytes), "in_place_columns": int(in_place_cols)}

        legs = {"stage_all": e2e_leg(False)}
        if args.e2e_policy == "in_place":
            legs["gather_in_place"] = e2e_leg(True)
        head = legs["gather_in_place"] if "gather_in_place" in legs else legs["stage_all"]
        e2e = {"value": head["value"], "unit": "rows/s", "h2d_bytes_per_step": head["h2d_bytes_per_step"],
               "d2h_bytes_per_step": int(d2h_bytes), "steps": e2e_steps, "ms_per_step": head["ms_per_step"],
               "policy": "gather_in_place" if "gather_in_place" in legs else "stage_all", "legs": legs,
               "note": "per step: pb_segment_stage from page-locked host buffers + execute + result read-back.  stage_all copies every "
                       "touched column to HBM; gather_in_place (PB_Q_GATHER_IN_PLACE) copies the predicate columns and gathers the "
                       "group-by/aggregation columns of the matching rows over PCIe from the mapped host buffers "
                       "(h2d = staged bytes + 32-byte sectors x gathered values)"}

    if rank != 0:
        if world > 1:
            _teardown(native, dist)
        return 0

    # ---- roofline: the longer of the two hot kernels is the dominant one; CUDA events on the call's own stream ----
    peak, peak_src = measured_peak_gbs()
    f_mean, a_mean = T["filter_ms"], T["agg_ms"]
    alg_filter = algorithmic_bytes(segs, q, "filter")
    alg_agg = algorithmic_bytes(segs, q, "agg")
    alg_all = algorithmic_bytes(segs, q, "all")
    dom = "pb_filter_kernel" if f_mean >= a_mean else "pb_agg_kernel"
    dom_ms, dom_alg = (f_mean, alg_filter) if dom == "pb_filter_kernel" else (a_mean, alg_agg)
    achieved = dom_alg / (dom_ms * 1e-3) / 1e9 if dom_ms > 0 else 0.0
    traffic, traffic_src = None, None
    tp = os.path.join(ROOT, "profiles", "scan_kernel_traffic.json")
    if os.path.exists(tp):
        try:
            tj = json.load(open(tp))
            traffic = tj.get(dom + "_dram_bytes_per_launch")
            traffic_src = f"static: ncu --set full capture committed as profiles/scan_kernel_traffic.json ({tj.get('captured', 'date unknown')}), not measured by this run"
        except Exception:
            traffic = None
    step_ms = 1000 * elapsed / args.steps
    roofline = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": traffic,
                "kernel": dom, "kernel_ms": dom_ms, "algorithmic_bytes_per_launch": dom_alg, "peak_source": peak_src,
                "traffic_source": traffic_src,
                "kernels": {"pb_filter_kernel": {"ms": f_mean, "algorithmic_bytes": alg_filter, "frac": alg_filter / (f_mean * 1e-3) / 1e9 / peak if f_mean else None},
                            "pb_agg_kernel": {"ms": a_mean, "algorithmic_bytes": alg_agg, "frac": alg_agg / (a_mean * 1e-3) / 1e9 / peak if a_mean else None,
                                              "note": "full-scan convention; the kernel only touches the sectors of rows that pass the filter, so this "
                                                      "fraction is not a bandwidth utilisation at low selectivity"}},
                "whole_query": {"algorithmic_bytes": alg_all * world, "step_ms": step_ms,
                                "frac_on_step_time": alg_all * world / (step_ms * 1e-3) / 1e9 / (peak * world),
                                "kernel_ms": f_mean + a_mean, "frac_on_kernel_time": alg_all / ((f_mean + a_mean) * 1e-3) / 1e9 / peak if f_mean + a_mean > 0 else None,
                                "note": "BASELINE.md full-scan convention (87 bits/row); frac_on_step_time divides by the driver-visible step "
                                        "(launch gaps, finalize, host and the NCCL merge included)"}}

    # ---- CPU baseline: the oracle (port of the reference algorithm) on this box's host cores ----
    cpu, cpu_all = None, None
    if world == 1 and not args.no_cpu_baseline:
        from oracle import oracle
        oracle.build()

        def time_oracle(osegs, oq, threads, budget_s):
            oracle_query_all_threads(osegs[:1], oq, 1)   # warm
            reps, t2 = 0, time.perf_counter()
            while True:
                oracle_query_all_threads(osegs, oq, threads)
                reps += 1
                if time.perf_counter() - t2 > budget_s or reps >= 5000:
                    break
            return reps, time.perf_counter() - t2

        threads = min(len(segs), os.cpu_count() or 1)
        reps, cdt = time_oracle(segs, q, threads, 10.0)
        cpu = {"value": w.rows_rank * reps / cdt, "unit": "rows/s", "cores": threads, "kind": "port",
               "sample": f"{reps} passes of the full {w.rows_rank}-row query, one thread per segment ({threads} threads of {os.cpu_count()} cores: "
                         f"how GroupByCombineOperator parallelises 8 segments), {cdt:.1f} s"}
        if w2 is not None and other_name == "strong":
            # the same 100 M rows cut into 64 segments so that up to 64 host cores work at once
            threads2 = min(len(w2.segs), os.cpu_count() or 1)
            reps2, cdt2 = time_oracle(w2.segs, w2.q, threads2, 10.0)
            cpu_all = {"value": w2.rows_rank * reps2 / cdt2, "unit": "rows/s", "cores": threads2, "kind": "port",
                       "sample": f"{reps2} passes of the {w2.rows_rank}-row table as {len(w2.segs)} segments on {threads2} threads "
                                 f"({os.cpu_count()} cores on the box), {cdt2:.1f} s"}

    line = {"metric": METRIC, "value": value, "unit": "rows/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": max(args.warmup, 3),
            "ms_per_step": step_ms, "higher_is_better": True, "scaling": head_scaling, "vs_baseline": None,
            "dtype": "f64", "data": "synthetic", "config": workload_config(args, segs, w),
            "clocks": clocks, "e2e": e2e, "gpu_launches": T["launches"], "roofline": roofline, "cpu_baseline": cpu,
            "cpu_baseline_all_cores": cpu_all, "parity_checked": True, "parity": parity,
            other_name: other, "selectivity_25pct": sel25,
            "device_ms_per_step": T["device_ms"], "scan_kernel_ms": T["scan_ms"], "filter_kernel_ms": f_mean, "agg_kernel_ms": a_mean,
            "nccl_merge_ms": T["comm_ms"],
            "step_wall_ms": {"min": float(np.min(T["step_wall"])), "median": float(np.median(T["step_wall"])), "max": float(np.max(T["step_wall"])),
                             "all": [round(float(x), 3) for x in T["step_wall"]]}, "host_us_by_phase": T["host_us"],
            "num_groups": int(num_groups), "docs_matched": int(docs_matched),
            "kernel_variant": {0: "tma+width-specialised", 4: "tma+generic", 8: "ldg+width-specialised", 12: "ldg+generic"}.get(args.flags & 12)}
    if outputs is not None:
        os.makedirs(args.dump_outputs, exist_ok=True)
        for name, arr in outputs.items():
            np.save(os.path.join(args.dump_outputs, name + ".npy"), arr)
    _emit(line)
    if world > 1:
        _teardown(native, dist)
    return 0


def lib_launches(r):
    from pinot_b200 import native
    return native.lib().pb_result_kernel_launches(r._rh)


if __name__ == "__main__":
    sys.exit(main())
