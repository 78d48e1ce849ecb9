#!/usr/bin/env python
"""bench.py -- the hot path of BASELINE.json at the sizes it names, one JSON line per run.

  python bench.py --gpus N --steps K --warmup W            (N>1 via torch.distributed.run, one rank per GPU)
  python bench.py --impl reference ...                     (CPU arm: one worker per host core over the same files)
  python bench.py --workload scan_agg|join|sort_shuffle|all   (default all: the headline + the other configs as sub-results)
  python bench.py --dump-outputs DIR ...                   (also write every leg's last timed result as DIR/<leg>.<column>.npy)

Headline (`metric`, `value`, `e2e`, `roofline`): BASELINE configs[1] -- ParquetScan -> Filter -> HashAggregate (GROUP BY int64,
SUM/COUNT) over a synthetic TPC-DS SF100 `store_sales` (287,997,024 rows); one step = one pass of the whole plan.
  `value`  : rows/s with the Parquet file images already resident in HBM.
  `e2e`    : rows/s through the C ABI from HOST inputs, H2D of the encoded column chunks and D2H of the result inside the timed
             region.  The headline e2e reads plain files through the engine's reader (the path the JVM drives: page cache ->
             pinned staging -> H2D); `e2e.pinned_images` is the same plan over file images registered in pinned host memory.
`workloads.join` (configs[2]) and `workloads.sort_shuffle` (configs[3]) carry the same fields for HashJoin store_sales x date_dim
and for SortExec + ShuffleWriterExec; at N > 1 the shuffle's hash repartition is an NCCL all-to-all-v inside the timed region.
The oracle is used only by the cpu_baseline / --impl reference legs (as the timed CPU arm), never by the product path.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import sys
import tempfile
import threading
import time
from concurrent.futures import ProcessPoolExecutor, ThreadPoolExecutor

import numpy as np
import pyarrow as pa
import pyarrow.compute as pc
import pyarrow.parquet as pq

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True          # the bench writes nothing into the source tree, which may be read-only

SF100_ROWS = 287_997_024
ROWS_PER_FILE = 16_000_000
DATE_LO, DATE_HI = 2450816, 2452642          # ss_sold_date_sk window (~5 years)
FILTER_LO, FILTER_HI = 2451000, 2452000      # WHERE ss_sold_date_sk >= lo AND < hi
N_ITEMS = 204_000                            # item cardinality at SF100
CODEC = os.environ.get("AURON_BENCH_CODEC", "SNAPPY")   # page compression of the synthetic files (SNAPPY = Spark default; NONE = uncompressed)
SCHEMA = pa.schema([("ss_item_sk", pa.int32()), ("ss_quantity", pa.int32()), ("ss_sold_date_sk", pa.int32())])
PARITY_NOTE = ("results are checked in tests/ against the pinned oracle port and Arrow C++ (the reference's Rust build is not runnable "
               "here: arithmetic / Parquet decode / row order / shuffle bytes are pinned by those, see DESIGN.md)")


def gen_file(path: str, rows: int, seed: int):
    rng = np.random.default_rng(seed)
    t = pa.table({
        "ss_item_sk": pa.array(rng.integers(1, N_ITEMS + 1, rows, dtype=np.int32)),
        "ss_quantity": pa.array(rng.integers(1, 101, rows, dtype=np.int32), mask=rng.random(rows) < 0.03),
        "ss_sold_date_sk": pa.array(rng.integers(DATE_LO, DATE_HI, rows, dtype=np.int32), mask=rng.random(rows) < 0.04),
    }, schema=SCHEMA)
    # Spark's writer defaults: SNAPPY pages, dictionary encoding, ~128 MB row groups (8M rows x 3 projected columns)
    # written under a temporary name and renamed: a run that dies mid-write leaves no partial file for later runs to reuse as input
    tmp = f"{path}.{os.getpid()}.tmp"
    pq.write_table(t, tmp, compression=CODEC, use_dictionary=True, row_group_size=8_000_000, data_page_size=1 << 20)
    os.replace(tmp, path)


def gen_dataset(directory: str, total_rows: int) -> list[tuple[str, int]]:
    os.makedirs(directory, exist_ok=True)
    specs, left, i = [], total_rows, 0
    while left > 0:
        r = min(ROWS_PER_FILE, left)
        specs.append((os.path.join(directory, f"store_sales_{CODEC.lower()}_{i:03d}.parquet"), r, 42 + i))
        left -= r
        i += 1
    with ThreadPoolExecutor(max_workers=min(8, os.cpu_count() or 1)) as ex:
        list(ex.map(lambda s: gen_file(*s) if not os.path.exists(s[0]) else None, specs))
    return [(p, r) for p, r, _ in specs]


def build_plan(P, files: list[str], sizes: list[int]) -> bytes:
    scan = P.parquet_scan(SCHEMA, list(zip(files, sizes)), [0, 1, 2])
    flt = P.filter_(scan, [P.binary("GtEq", P.col("ss_sold_date_sk"), P.lit(FILTER_LO, pa.int32())),
                           P.binary("Lt", P.col("ss_sold_date_sk"), P.lit(FILTER_HI, pa.int32()))])
    agg = P.agg(flt, [P.try_cast(P.col("ss_item_sk"), pa.int64())], ["ss_item_sk"],
                [P.agg_expr("SUM", [P.col("ss_quantity")], pa.int64()), P.agg_expr("COUNT", [P.col("ss_quantity")], pa.int64())],
                ["sum_qty", "cnt_qty"], ["PARTIAL", "PARTIAL"])
    return P.task_definition(agg)


def bind_to_gpu_numa_node(torch, gpu_index: int):
    """One process per GPU: run on the cores of the GPU's NUMA node, so that the pinned host buffers (first touch) and the
    scan's worker threads sit next to the PCIe root the GPU hangs off.  Returns the node id or None."""
    try:
        p = torch.cuda.get_device_properties(gpu_index)
        if hasattr(p, "pci_bus_id"):
            bdf = f"{p.pci_domain_id:04x}:{p.pci_bus_id:02x}:{p.pci_device_id:02x}.0"
        else:   # older torch: NVML reports the same bus id string
            import pynvml
            pynvml.nvmlInit()
            bus = pynvml.nvmlDeviceGetPciInfo(pynvml.nvmlDeviceGetHandleByIndex(gpu_index)).busId
            bus = bus.decode() if isinstance(bus, bytes) else bus
            bdf = bus[-12:].lower()
        base = f"/sys/bus/pci/devices/{bdf}"
        node = int(open(base + "/numa_node").read())
        cpus = set()
        for part in open(base + "/local_cpulist").read().strip().split(","):
            lo, _, hi = part.partition("-")
            cpus.update(range(int(lo), int(hi or lo) + 1))
        cpus &= os.sched_getaffinity(0)
        if node >= 0 and cpus:
            os.sched_setaffinity(0, cpus)
            return node
    except Exception:
        pass
    return None


class ClockSampler:
    """SM clock + throttle reasons sampled DURING the timed region (profiling recipe), through NVML in a background thread
    (the same counters `nvidia-smi --query-gpu=clocks.sm,clocks_event_reasons.*` prints, without a subprocess per sample)."""
    REASONS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap"}

    def __init__(self, gpu_index: int, period_s: float = 0.02):
        self.sm, self.mx, self.reasons, self.idx, self.period = [], None, set(), gpu_index, period_s
        self._stop = threading.Event()
        self._thr = None

    def __enter__(self):
        try:
            if os.environ.get("AURON_BENCH_NO_CLOCKS"):
                raise RuntimeError("sampling disabled")
            import pynvml
            pynvml.nvmlInit()
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            phys = int(vis.split(",")[self.idx]) if vis and vis.split(",")[self.idx].isdigit() else self.idx
            h = pynvml.nvmlDeviceGetHandleByIndex(phys)
            self.mx = float(pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM))

            def loop():
                while not self._stop.is_set():
                    try:
                        self.sm.append(float(pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM)))
                        mask = pynvml.nvmlDeviceGetCurrentClocksEventReasons(h)
                        for bit, name in self.REASONS.items():
                            if mask & bit:
                                self.reasons.add(name)
                    except Exception:
                        pass
                    self._stop.wait(self.period)

            self._thr = threading.Thread(target=loop, daemon=True)
            self._thr.start()
        except Exception:
            self._thr = None
        return self

    def __exit__(self, *a):
        self._stop.set()
        if self._thr:
            self._thr.join(timeout=1)

    def summary(self):
        return {"sm_mhz": statistics.median(self.sm) if self.sm else None, "sm_max_mhz": self.mx, "reasons": sorted(self.reasons),
                "samples": len(self.sm)}


# ------------------------------------------------------------------------------------------------ CPU arm (config 2)
def _cpu_one_split(split):
    """One Spark task's worth of the reference pipeline on ONE core: Arrow C++ Parquet reader + filter (stand-in for the parquet
    crate / arrow-rs kernels the reference delegates to) feeding the oracle's C hash aggregate (port of agg_hash_map.rs / sum.rs /
    count.rs).  A split is one row group of one file (Spark cuts input splits at row-group boundaries: 128 MB); Auron runs one
    such task per core, so does this arm."""
    import oracle
    path, rg = split
    pa.set_cpu_count(1)
    pa.set_io_thread_count(1)
    t = pq.ParquetFile(path).read_row_group(rg, columns=["ss_item_sk", "ss_quantity", "ss_sold_date_sk"], use_threads=False)
    d = t["ss_sold_date_sk"]
    mask = pc.and_kleene(pc.greater_equal(d, FILTER_LO), pc.less(d, FILTER_HI))
    ft = t.filter(mask)
    r = oracle.agg_sum_count_i64(ft["ss_item_sk"].combine_chunks().cast(pa.int64()), ft["ss_quantity"].combine_chunks().cast(pa.int64()))
    return t.num_rows, r["k"].to_numpy(zero_copy_only=False), r["sum"].to_numpy(zero_copy_only=False), r["cnt"].to_numpy(zero_copy_only=False)


def _cpu_warm(_):
    import oracle  # noqa: F401
    return 0


class CpuArm:
    """All host cores, one split (row group) per worker at a time, partial aggregates merged at the end (the final merge a Spark stage
    does).  The table has fewer splits (36) than a big host has cores, so one step runs `passes` passes over the table concurrently --
    every core holds a task, rows/s counts every row processed."""

    def __init__(self, files: list[str], cores: int):
        self.cores = cores
        splits = []
        for f in files:
            splits += [(f, g) for g in range(pq.ParquetFile(f).metadata.num_row_groups)]
        self.passes = max(1, -(-cores // len(splits)))
        self.splits = splits * self.passes
        import multiprocessing
        # spawn, not fork: the GPU arm calls this from a process that holds a CUDA context and worker threads
        self.pool = ProcessPoolExecutor(max_workers=cores, mp_context=multiprocessing.get_context("spawn"))
        list(self.pool.map(_cpu_warm, range(cores)))

    def run(self) -> tuple[int, float]:
        t0 = time.perf_counter()
        rows = 0
        sums = np.zeros(N_ITEMS + 2, dtype=np.int64)
        cnts = np.zeros(N_ITEMS + 2, dtype=np.int64)
        for n, k, s, c in self.pool.map(_cpu_one_split, self.splits):
            rows += n
            kk = np.nan_to_num(k.astype(np.float64), nan=N_ITEMS + 1).astype(np.int64)
            np.add.at(sums, kk, np.nan_to_num(s.astype(np.float64)).astype(np.int64))
            np.add.at(cnts, kk, c.astype(np.int64))
        return rows, time.perf_counter() - t0

    def describe(self, nfiles: int) -> str:
        return (f"{self.passes} concurrent pass(es) over all {nfiles} files = {len(self.splits)} row-group splits per step, one single-threaded worker "
                "process per core: Arrow C++ scan+filter, oracle C hash aggregate, partials merged")

    def close(self):
        self.pool.shutdown()


# ------------------------------------------------------------------------------------------------ helpers
def pinned_array(torch, vals: np.ndarray, typ: pa.DataType, null_mask: np.ndarray | None, keep: list) -> pa.Array:
    """Arrow array whose value buffer lives in pinned host memory (the e2e legs copy from it)."""
    raw = vals.view(np.uint8).reshape(-1)
    tb = torch.empty(raw.size, dtype=torch.uint8).pin_memory()
    tb.numpy()[:] = raw
    keep.append(tb)
    n = len(vals) // 2 if pa.types.is_decimal(typ) else len(vals)
    vbuf = pa.py_buffer(np.packbits(~null_mask, bitorder="little").tobytes()) if null_mask is not None else None
    return pa.Array.from_buffers(typ, n, [vbuf, pa.py_buffer(tb.numpy())], null_count=int(null_mask.sum()) if null_mask is not None else 0)


def decimal_words(unscaled: np.ndarray) -> np.ndarray:
    """int64 unscaled values -> the two little-endian 64-bit words of decimal128 (sign-extended)"""
    out = np.empty(2 * len(unscaled), dtype=np.uint64)
    out[0::2] = unscaled.view(np.uint64)
    out[1::2] = np.where(unscaled < 0, np.uint64(0xFFFFFFFFFFFFFFFF), np.uint64(0))
    return out


def do_workload(args, w: str) -> bool:
    return args.workload in ("all", w)


def dump_outputs(directory: str, outputs: dict[str, pa.Table]):
    """--dump-outputs: every column of every leg's last timed result as <directory>/<leg>.<column>.npy in float64 (NULL is NaN,
    decimals by value).  Rows are sorted by all columns: the engine's row order is unspecified, the rows are what two builds must agree on.
    A column whose name is empty or repeated (the state columns of a PARTIAL aggregate) is named col<position>."""
    os.makedirs(directory, exist_ok=True)
    for leg, t in outputs.items():
        names = t.column_names
        t = t.rename_columns([n if n and names.count(n) == 1 else f"col{i}" for i, n in enumerate(names)])
        if t.num_rows:
            t = t.take(pc.sort_indices(t, sort_keys=[(n, "ascending") for n in t.column_names], null_placement="at_start"))
        for name, col in zip(t.column_names, t.columns):
            np.save(os.path.join(directory, f"{leg}.{name}.npy"), pc.cast(col, pa.float64()).to_numpy().astype(np.float64))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="auron")
    ap.add_argument("--workload", default="all", choices=["all", "scan_agg", "join", "sort_shuffle"])
    ap.add_argument("--rows", type=int, default=SF100_ROWS)
    ap.add_argument("--op-rows", type=int, default=int(os.environ.get("AURON_BENCH_OP_ROWS", 64_000_000)), help="rows per GPU of the sort/shuffle workload")
    # per user: on a shared host another user's directory of the same name is not writable
    ap.add_argument("--data-dir", default=os.path.join(tempfile.gettempdir(), f"auron_b200_bench_{os.getuid()}"))
    ap.add_argument("--skip-e2e", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write the result arrays of the last timed step of every GPU leg "
                                                          "as DIR/<leg>.<column name or col<position>>.npy (float64, rows in a canonical order; rank 0's results when N > 1)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    cores = len(os.sched_getaffinity(0))
    config = {"workload": "BASELINE configs[1]: ParquetScan->Filter->HashAggregate(GROUP BY int64 ss_item_sk, SUM/COUNT ss_quantity), "
                          "synthetic TPC-DS SF100 store_sales", "rows": args.rows, "groups": N_ITEMS, "filter_selectivity": "~0.53",
              "parquet": f"3 INT32 columns, RLE_DICTIONARY + PLAIN fallback pages, 8M-row (~128 MB) row groups, {CODEC} pages "
                         "(decompressed on the GPU)",
              "l2_policy": "inputs (>=1.4 GB encoded per step) are far larger than the 126 MB L2",
              "parallelism": f"dp{args.gpus}: table partitions sharded per GPU, no data-path collective in the scan/aggregate step; one process per GPU "
                             "bound to the GPU's NUMA node",
              "parity": PARITY_NOTE}

    if args.impl == "reference":
        if rank != 0:
            return
        files = gen_dataset(args.data_dir, args.rows)
        paths = [f for f, _ in files]
        arm = CpuArm(paths, cores)
        warm = min(args.warmup, 1)
        for _ in range(warm):
            arm.run()
        rows, secs = 0, 0.0
        steps = args.steps                               # every step is the WHOLE table (all files) at least once
        for _ in range(steps):
            r, s = arm.run()
            rows += r
            secs += s
        arm.close()
        v = rows / secs
        print(json.dumps({"impl": "reference", "metric": "rows_per_sec", "value": v, "unit": "rows/s", "n_gpus": args.gpus, "steps": steps,
                          "warmup": warm, "ms_per_step": 1000 * secs / steps, "higher_is_better": True, "scaling": "weak",
                          "vs_baseline": None, "dtype": "int64", "data": "synthetic", "config": config,
                          "cpu_baseline": {"value": v, "unit": "rows/s", "cores": cores, "kind": "port",
                                           "sample": arm.describe(len(files))},
                          "e2e": {"value": v, "unit": "rows/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))
        return

    cpu_line = None
    if world == 1 and rank == 0 and do_workload(args, "scan_agg") and not os.environ.get("AURON_BENCH_NO_CPU"):
        # the CPU baseline of the headline runs first, before this process owns a CUDA context (worker processes, all cores)
        files0 = gen_dataset(args.data_dir, args.rows)
        arm = CpuArm([f for f, _ in files0], cores)
        r, s = arm.run()
        arm.close()
        cpu_line = {"value": r / s, "unit": "rows/s", "cores": cores, "kind": "port", "sample": arm.describe(len(files0))}

    import torch
    import torch.distributed as dist
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    torch.cuda.set_device(local_rank)
    numa = bind_to_gpu_numa_node(torch, local_rank)    # before any pinned allocation / worker thread exists
    config["numa_node"] = numa
    # host worker threads of this rank: its share of the CPUs it is bound to (ranks on the same NUMA node share them)
    bound = len(os.sched_getaffinity(0))
    nodes = max(1, len([d for d in os.listdir("/sys/devices/system/node") if d.startswith("node")])) if os.path.isdir("/sys/devices/system/node") else 1
    ranks_per_node = max(1, -(-world // nodes))
    os.environ.setdefault("AURON_SCAN_THREADS", str(max(4, min(32, bound // ranks_per_node))))
    config["host_threads_per_rank"] = int(os.environ["AURON_SCAN_THREADS"])
    from auron_b200 import proto as P
    from auron_b200 import runtime

    os.environ["AURON_PROFILE"] = "1"
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    peak_src = "measured (MEASURED_PEAKS.json hbm_gbs)" if "hbm_gbs" in peaks else "fallback 6.65 TB/s"

    def barrier_sync():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(make_task, steps: int, collect: bool):
        """`steps` runs of one task each, bracketed by barrier + synchronize, max over ranks.  Returns (seconds, kernel timers,
        last result table, per-step ms)."""
        kern, step_ms, out = {}, [], None
        import gc
        gc.collect()
        gc.disable()          # (a collection inside a 5 ms step is a 30 % outlier)
        barrier_sync()
        t0 = time.perf_counter()
        for _ in range(steps):
            ts = time.perf_counter()
            with make_task() as task:
                out = pa.Table.from_batches(list(task), schema=task.schema)
                if collect or os.environ.get("AURON_BENCH_VERBOSE"):
                    for depth, op, name, v in task.metrics():
                        if op == "__kernels__":
                            if collect:
                                kern[name] = kern.get(name, 0) + v
                        elif os.environ.get("AURON_BENCH_VERBOSE"):
                            print(f"[metric] {op}.{name} = {v}", file=sys.stderr)
            step_ms.append(1000 * (time.perf_counter() - ts))
        barrier_sync()
        dt = time.perf_counter() - t0
        gc.enable()
        if world > 1:
            tt = torch.tensor([dt], device="cuda", dtype=torch.float64)
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            dt = float(tt.item())
        v = sorted(step_ms)
        return dt, kern, out, {"min": v[0], "median": v[len(v) // 2], "max": v[-1], "all": [round(x, 3) for x in step_ms]}

    def roofline_of(kern: dict, steps: int, dt: float, alg: dict, traffic_key: str | None = None, isolated: dict | None = None):
        names = sorted({k.rsplit(".", 1)[0] for k in kern if k.endswith(".device_us")}, key=lambda n: -kern[n + ".device_us"])
        roofs = []
        for n in names:
            us = kern[n + ".device_us"] / steps
            r = {"kernel": n, "device_ms_per_step": us / 1000.0, "launches_per_step": kern[n + ".launches"] / steps, "share_of_step": (us / 1e6) / (dt / steps)}
            if alg.get(n) and us > 0:
                r["algorithmic_bytes_per_step"] = alg[n]
                r["achieved_gbs"] = alg[n] / (us * 1e-6) / 1e9
                r["frac_of_peak"] = r["achieved_gbs"] / peak
            roofs.append(r)
        # the roofline's kernel: the launch site with the most device time among those the step's data flows through (an
        # algorithmic-byte figure exists); sites without one (the latency-bound Snappy walk of the level prefixes) stay in `kernels`
        with_bytes = [n for n in names if alg.get(n)]
        dom = with_bytes[0] if with_bytes else (names[0] if names else None)
        dom_us = kern[dom + ".device_us"] / steps if dom else None
        dom_bytes = alg.get(dom) if dom else None
        traffic, traffic_src = None, None
        try:
            tj = json.load(open(os.path.join(ROOT, "profiles", "r02_traffic.json")))
            if traffic_key and traffic_key in tj and tj[traffic_key].get("kernel") == dom:
                traffic, traffic_src = tj[traffic_key]["dram_bytes_per_step"], tj[traffic_key]["source"]
        except Exception:
            pass
        res = {"bound": "hbm", "kernel": dom, "achieved": (dom_bytes / (dom_us * 1e-6) / 1e9) if dom_bytes and dom_us else None, "peak": peak, "unit": "GB/s",
               "frac": (dom_bytes / (dom_us * 1e-6) / 1e9 / peak) if dom_bytes and dom_us else None, "traffic": traffic, "traffic_source": traffic_src,
               "peak_source": peak_src, "algorithmic_bytes_per_step": dom_bytes, "kernels": roofs,
               "note": "kernel times are CUDA-event intervals on the launching streams inside the timed region; the kernels of the batches in flight share the "
                       "SMs (decompression / scout of batch k+1 next to the scan kernel of batch k), so an interval is longer than the kernel would run alone "
                       "and the intervals sum to more than the step"}
        if isolated and dom and isolated.get(dom + ".device_us"):
            iso_us = isolated[dom + ".device_us"] / max(1, isolated.get("_steps", 1))
            res["alone"] = {"device_ms_per_step": iso_us / 1000.0, "achieved": dom_bytes / (iso_us * 1e-6) / 1e9 if dom_bytes else None,
                            "frac": dom_bytes / (iso_us * 1e-6) / 1e9 / peak if dom_bytes else None,
                            "how": "the same kernel timed by the same events in extra untimed steps with one batch in flight at a time (AURON_FUSED_ONE_LANE=1)"}
        return res

    outputs: dict[str, pa.Table] = {}      # leg -> result of its last timed step (--dump-outputs)
    ctx = dict(args=args, torch=torch, dist=dist, P=P, runtime=runtime, timed=timed, roofline_of=roofline_of, world=world, rank=rank, local_rank=local_rank, cores=cores,
               outputs=outputs)
    do = (lambda w: do_workload(args, w))
    line = None

    # ================================================================================================ config 2: scan -> filter -> aggregate
    if do("scan_agg"):
        if rank == 0:
            gen_dataset(args.data_dir, args.rows)
        if world > 1:
            dist.barrier()
        files = gen_dataset(args.data_dir, args.rows)       # no-op when the files exist
        paths = [f for f, _ in files]
        if world > 1 and rank > 0:
            # every rank scans its OWN copy of the table partition (as every executor scans its own files): written by this process, bound to
            # its GPU's NUMA node, so the page-cache pages of the e2e leg are node-local instead of all ranks reading rank 0's pages
            # across the socket (2 ranks on one copy: 17 GB/s of page-cache reads each)
            import shutil
            rd = os.path.join(args.data_dir, f"rank{rank}")
            os.makedirs(rd, exist_ok=True)
            mine = []
            for f in paths:
                g = os.path.join(rd, os.path.basename(f))
                if not (os.path.exists(g) and os.path.getsize(g) == os.path.getsize(f)):
                    shutil.copyfile(f, g + ".tmp")
                    os.replace(g + ".tmp", g)
                mine.append(g)
            paths = mine
        sizes = [os.path.getsize(f) for f in paths]
        total_rows = sum(r for _, r in files)
        h2d_bytes = unc_bytes = 0      # column-chunk bytes as stored (what crosses PCIe) / after page decompression
        for f in paths:
            md = pq.ParquetFile(f).metadata
            for g in range(md.num_row_groups):
                for c in range(md.num_columns):
                    cc = md.row_group(g).column(c)
                    h2d_bytes += cc.total_compressed_size
                    unc_bytes += cc.total_uncompressed_size
        # device batches of 6 files (96M rows = 12 row groups): the host prepares batch k+1 while the GPU works on batch k; measured on
        # B200: 5.6 ms per step at 96M, 5.9 ms at 72M, 5.7 ms at 144M, 6.5 ms with the whole table as one batch
        os.environ.setdefault("AURON_GPU_CHUNK_ROWS", str(96_000_000))
        # ---- value: file images resident in HBM
        hbm_paths = [f"hbm://{os.path.basename(p)}@{local_rank}" for p in paths]
        for p, hp in zip(paths, hbm_paths):
            with open(p, "rb") as fh:
                runtime.put_device_file(hp, fh.read(), device=local_rank)
        plan_hbm = build_plan(P, hbm_paths, sizes)
        mk = lambda plan: (lambda: runtime.Task(plan, device=local_rank))
        timed(mk(plan_hbm), args.warmup, False)
        with ClockSampler(local_rank) as cs:
            dt, kern, out, value_spread = timed(mk(plan_hbm), args.steps, True)
        clocks = cs.summary()
        outputs["scan_agg"] = out
        value = world * total_rows * args.steps / dt
        os.environ["AURON_FUSED_ONE_LANE"] = "1"      # two untimed steps without overlap between batches: the kernels' own durations
        _, kern_alone, _, _ = timed(mk(plan_hbm), 2, True)
        kern_alone["_steps"] = 2
        del os.environ["AURON_FUSED_ONE_LANE"]
        for hp in hbm_paths:
            runtime.drop_device_file(hp)
        # ---- e2e: the same call with HOST inputs; every step uploads the projected column chunks inside the timed region
        e2e = None
        if not args.skip_e2e:
            plan_host = build_plan(P, paths, sizes)
            timed(mk(plan_host), max(1, min(args.warmup, 2)), False)
            dtf, _, out_f, sp = timed(mk(plan_host), args.steps, False)
            outputs["scan_agg_e2e"] = out_f
            e2e = {"value": world * total_rows * args.steps / dtf, "unit": "rows/s", "h2d_bytes_per_step": h2d_bytes, "d2h_bytes_per_step": out_f.nbytes,
                   "ms_per_step": 1000 * dtf / args.steps, "step_ms": sp,
                   "input": "parquet files read by the engine (OS page cache -> pread into pinned staging -> H2D): the path a JVM host drives"}
            pin_paths = [f"pinned://{os.path.basename(p)}@{local_rank}" for p in paths]
            keep = []
            for p, hp, sz in zip(paths, pin_paths, sizes):
                buf = torch.empty(sz, dtype=torch.uint8).pin_memory()
                with open(p, "rb") as fh:
                    fh.readinto(memoryview(buf.numpy()))
                runtime.put_host_file(hp, buf)
                keep.append(buf)
            plan_pin = build_plan(P, pin_paths, sizes)
            timed(mk(plan_pin), 1, False)
            dte, _, out_e, sp = timed(mk(plan_pin), args.steps, False)
            outputs["scan_agg_e2e_pinned"] = out_e
            e2e["pinned_images"] = {"value": world * total_rows * args.steps / dte, "ms_per_step": 1000 * dte / args.steps, "step_ms": sp,
                                    "input": "parquet file images registered in pinned host memory (auron_b200_put_host_file): H2D per column chunk, no pread"}
            for hp in pin_paths:
                runtime.drop_host_file(hp)
            del keep
        sel_rows = int(out.column(2).to_numpy().sum() / 0.97) if out.num_rows else 0        # filtered rows reaching the aggregate (approx)
        val_bits = 2 * (total_rows // 8)                                                    # validity bitmaps of the two nullable columns
        alg = {   # algorithmic bytes per step of every launch site (DESIGN.md section 3: inputs once + outputs once)
            "fz_scan_filter_agg": unc_bytes + val_bits + out.nbytes,     # encoded page bytes + validity in, groups out (nothing else leaves the chip)
            "fz_scout": val_bits * 2,                                    # definition levels in (~1 bit/row run-length coded), validity bitmaps out
            "fz_merge": 2 * len(paths) * 2 * N_ITEMS * 8,                # dictionary-space accumulators in, direct table out
            # pq_decompress: only the level prefixes of the nullable v1 pages run through the Snappy decoder (the value sections are single
            # literals read in place): no algorithmic-byte figure is claimed for it
        }
        roofline = roofline_of(kern, args.steps, dt, alg, "scan_agg", kern_alone)
        line = {"metric": "rows_per_sec", "value": value, "unit": "rows/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": 1000 * dt / args.steps, "step_ms": value_spread, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "int64",
                "data": "synthetic", "config": config, "clocks": clocks, "e2e": e2e,
                "gpu_launches": int(kern.get("total_launches", 0)), "roofline": roofline, "cpu_baseline": None,
                "result_groups": out.num_rows, "selected_rows_est": sel_rows}
        line["cpu_baseline"] = cpu_line

    # ================================================================================================ config 3 / 4 sub-results
    workloads = {}
    if do("join"):
        workloads["join"] = bench_join(**ctx)
    if do("sort_shuffle"):
        workloads["sort_shuffle"] = bench_sort_shuffle(**ctx)

    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    if rank != 0:
        return
    if line is None:   # a single sub-workload was asked for: its result is the line
        w = next(iter(workloads.values()))
        line = {"metric": "rows_per_sec", "unit": "rows/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "higher_is_better": True,
                "scaling": "weak", "vs_baseline": None, "data": "synthetic", **w}
    else:
        line["workloads"] = workloads
    print(json.dumps(line))
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, outputs)


# ================================================================================================ config 3: HashJoin store_sales x date_dim
def bench_join(args, torch, dist, P, runtime, timed, roofline_of, world, rank, local_rank, cores, outputs):
    """BASELINE configs[2]: inner hash join, build = date_dim (73,049 rows: d_date_sk int32, d_year int32), probe = store_sales SF100
    (287,997,024 rows: ss_sold_date_sk int32 drawn from a ~1,800-day window, 4 % NULL; payload ss_ext_sales_price decimal(7,2)).  The joined
    rows stay on the device: a global SUM/COUNT over them is the result that leaves (so the measurement is the join, not a 6 GB D2H)."""
    n = args.rows
    rng = np.random.default_rng(7 + rank)
    dkey = np.arange(2415022, 2415022 + 73049, dtype=np.int32)
    dyear = (1900 + np.arange(73049) // 365).astype(np.int32)
    dd = pa.table({"d_date_sk": pa.array(dkey), "d_year": pa.array(dyear)})
    sold = rng.integers(DATE_LO, DATE_HI, n, dtype=np.int32)
    null = rng.random(n) < 0.04
    price = rng.integers(0, 2_000_000, n, dtype=np.int64)
    keep: list = []
    ss = pa.table({"ss_sold_date_sk": pinned_array(torch, sold, pa.int32(), null, keep),
                   "ss_ext_sales_price": pinned_array(torch, decimal_words(price), pa.decimal128(7, 2), None, keep)})
    chunk = 24_000_000
    rid_ss, rid_dd = f"bj_ss{rank}", f"bj_dd{rank}"
    for b in ss.to_batches(max_chunksize=chunk):
        runtime.put_device_batch(rid_ss, b, device=local_rank)
    runtime.put_device_batch(rid_dd, dd.to_batches()[0], device=local_rank)
    out_schema = pa.schema(list(dd.schema) + list(ss.schema))

    def plan(ss_id, dd_id):
        j = P.hash_join(out_schema, P.ffi_reader(dd.schema, dd_id), P.ffi_reader(ss.schema, ss_id), [(P.col("d_date_sk"), P.col("ss_sold_date_sk"))], "INNER", "LEFT")
        return P.task_definition(P.agg(j, [], [], [P.agg_expr("SUM", [P.col("d_year")], pa.int64()), P.agg_expr("SUM", [P.col("ss_ext_sales_price")], pa.decimal128(17, 2)),
                                                   P.agg_expr("COUNT", [P.col("ss_sold_date_sk")], pa.int64())], ["y", "p", "c"], ["PARTIAL"] * 3))

    steps, warm = args.steps, max(1, min(args.warmup, 2))
    td = plan(rid_ss, rid_dd)
    mk = lambda: runtime.Task(td, device=local_rank)
    timed(mk, warm, False)
    dt, kern, out, spread = timed(mk, steps, True)
    outputs["join"] = out
    matched = int((~null).sum())
    exp_year = int(dyear[sold[~null] - 2415022].astype(np.int64).sum())
    ok = out.column(2)[0].as_py() == matched and out.column(0)[0].as_py() == exp_year
    value = world * n * steps / dt
    e2e = None
    if not args.skip_e2e:
        td_h = plan("host_ss", "host_dd")
        mkh = lambda: runtime.Task(td_h, {"host_ss": ss.to_batches(max_chunksize=chunk), "host_dd": dd.to_batches()}, device=local_rank)
        timed(mkh, 1, False)
        dth, _, outh, sp = timed(mkh, steps, False)
        outputs["join_e2e"] = outh
        e2e = {"value": world * n * steps / dth, "unit": "rows/s", "h2d_bytes_per_step": ss.nbytes + dd.nbytes, "d2h_bytes_per_step": outh.nbytes,
               "ms_per_step": 1000 * dth / steps, "step_ms": sp, "input": "Arrow batches in pinned host memory exported through the FFI reader (24M-row batches)"}
    alg = {"join_probe": n * 4 + n // 8 + matched * 8,        # probe keys + validity in, (probe row, build row) pairs out
           "take": matched * 2 * (4 + 4 + 4 + 16),            # output columns gathered: row bytes in + out
           "join_build": 73049 * 4 * 2}
    res = {"value": value, "ms_per_step": 1000 * dt / steps, "step_ms": spread, "steps": steps, "dtype": "int32 keys / decimal128 payload", "result_ok": bool(ok),
           "config": {"workload": "BASELINE configs[2]: HashJoinExec store_sales x date_dim SF100, build + probe + global SUM/COUNT of the joined rows", "rows": n,
                      "build_rows": 73049, "matched_rows": matched, "l2_policy": "probe side (5.8 GB of Arrow columns) is far larger than the 126 MB L2"},
           "e2e": e2e, "roofline": roofline_of(kern, steps, dt, alg), "gpu_launches": int(kern.get("total_launches", 0))}
    if world == 1:
        m = min(n, 32_000_000)
        sl = ss.slice(0, m)
        t0 = time.perf_counter()
        j = sl.join(dd, keys="ss_sold_date_sk", right_keys="d_date_sk", join_type="inner", use_threads=True)
        pc.sum(j["d_year"])
        s = time.perf_counter() - t0
        res["cpu_baseline"] = {"value": m / s, "unit": "rows/s", "cores": cores, "kind": "port",
                               "sample": f"first {m} probe rows: Arrow C++ (Acero) hash join + SUM, all host threads (stand-in: the reference's join cannot be built here)"}
    runtime.drop_device_resource(rid_ss)
    runtime.drop_device_resource(rid_dd)
    del keep
    return res


# ================================================================================================ config 4: SortExec + ShuffleWriterExec
def bench_sort_shuffle(args, torch, dist, P, runtime, timed, roofline_of, world, rank, local_rank, cores, outputs):
    """BASELINE configs[3]: every GPU holds a shard of store_sales projected to (ss_item_sk int32, ss_ticket_number int64, ss_ext_sales_price
    decimal(7,2)) = 28 B/row.  Leg 1: SortExec ORDER BY ss_item_sk.  Leg 2: ShuffleWriterExec hash(ss_item_sk) into 200 Spark partitions --
    N = 1: Auron's compacted shuffle format (.data + .index) written to tmpfs; N > 1: the hash repartition is exchanged between the GPUs
    with an NCCL all-to-all-v (exchange.cu) inside the timed region and every rank reduces the rows of the partitions it owns."""
    n = args.op_rows
    rng = np.random.default_rng(100 + rank)
    item = rng.integers(1, N_ITEMS + 1, n, dtype=np.int32)
    ticket = rng.integers(1, 240_000_000, n, dtype=np.int64)
    price = rng.integers(0, 2_000_000, n, dtype=np.int64)
    keep: list = []
    t4 = pa.table({"ss_item_sk": pinned_array(torch, item, pa.int32(), None, keep), "ss_ticket_number": pinned_array(torch, ticket, pa.int64(), None, keep),
                   "ss_ext_sales_price": pinned_array(torch, decimal_words(price), pa.decimal128(7, 2), None, keep)})
    rid = f"bs_t4_{rank}"
    for b in t4.to_batches(max_chunksize=16_000_000):
        runtime.put_device_batch(rid, b, device=local_rank)
    steps, warm = args.steps, max(1, min(args.warmup, 2))
    res = {"steps": steps,
           "config": {"workload": "BASELINE configs[3]: SortExec + ShuffleWriterExec hash(ss_item_sk) -> 200 partitions, store_sales projected to 28 B/row",
                      "rows_per_gpu": n, "full_share_rows_per_gpu_at_sf1000_8gpu": 359_998_500, "partitions": 200,
                      "l2_policy": f"shard ({n * 28 / 1e9:.1f} GB of Arrow columns) is far larger than the 126 MB L2"}}
    # ---- leg 1: sort (COUNT on top so that one row leaves the GPU)
    td_sort = P.task_definition(P.agg(P.sort(P.ffi_reader(t4.schema, rid), [P.sort_expr(P.col("ss_item_sk"))]), [], [],
                                      [P.agg_expr("COUNT", [P.col("ss_item_sk")], pa.int64())], ["c"], ["PARTIAL"]))
    mk = lambda: runtime.Task(td_sort, device=local_rank)
    timed(mk, warm, False)
    dt, kern, out, spread = timed(mk, steps, True)
    outputs["sort"] = out
    res["sort"] = {"value": world * n * steps / dt, "unit": "rows/s", "ms_per_step": 1000 * dt / steps, "step_ms": spread,
                   "roofline": roofline_of(kern, steps, dt, {"radix_sort": 3 * 2 * 12 * n, "take": 2 * 28 * n}), "result_ok": out.column(0)[0].as_py() == n}
    # ---- leg 2: shuffle write / exchange
    if world == 1:
        # a directory of this run's own on tmpfs: on a shared host a fixed path may belong to another user
        d = tempfile.mkdtemp(prefix="auron_bench_shuffle_", dir="/dev/shm" if os.path.isdir("/dev/shm") else None)
        # every map task writes its own new .data / .index pair (as in Spark): rewriting one path would charge the release of the old
        # file's pages to the step
        import itertools
        import shutil
        serial = itertools.count()

        def mk():
            k = next(serial)
            return runtime.Task(P.task_definition(P.shuffle_writer(P.ffi_reader(t4.schema, rid), P.hash_repartition([P.col("ss_item_sk")], 200),
                                                                   f"{d}/s{k}.data", f"{d}/s{k}.index")), device=local_rank)

        try:
            timed(mk, warm, False)
            dt, kern, out, spread = timed(mk, steps, True)
            fsz = os.path.getsize(f"{d}/s0.data")
            with open(f"{d}/s{next(serial) - 1}.index", "rb") as fh:          # the .index of the last timed step: per-partition byte offsets
                outputs["shuffle"] = pa.table({"index_offsets": np.frombuffer(fh.read(), dtype="<i8")})
        finally:
            shutil.rmtree(d)
        res["shuffle"] = {"value": n * steps / dt, "unit": "rows/s", "ms_per_step": 1000 * dt / steps, "step_ms": spread, "file_bytes": fsz,
                          "file_gbs": fsz * steps / dt / 1e9, "mode": "ShuffleWriterExec -> .data/.index on tmpfs (LZ4 frames, Auron compacted format)",
                          "roofline": roofline_of(kern, steps, dt, {"murmur3_partition_ids": 8 * n, "partition_rows": 8 * n, "take": 2 * 28 * n, "serde_write": 2 * 28 * n,
                                                                    "lz4_compress": 28 * n + fsz})}
    else:
        ids = [runtime.nccl_unique_id() if rank == 0 else None]
        dist.broadcast_object_list(ids, src=0)
        runtime.nccl_init(ids[0], rank, world, local_rank)
        exch = P.shuffle_writer(P.ffi_reader(t4.schema, rid), P.hash_repartition([P.col("ss_item_sk")], 200), "nccl://bench", "")
        td_x = P.task_definition(P.agg(exch, [], [], [P.agg_expr("COUNT", [P.col("ss_item_sk")], pa.int64()), P.agg_expr("SUM", [P.col("ss_ticket_number")], pa.int64())],
                                       ["c", "s"], ["PARTIAL"] * 2), stage_id=1, partition_id=rank)
        mk = lambda: runtime.Task(td_x, device=local_rank)
        timed(mk, warm, False)
        dt, kern, out, spread = timed(mk, steps, True)
        outputs["shuffle"] = out
        cnt = torch.tensor([out.column(0)[0].as_py(), out.column(1)[0].as_py(), int(ticket.sum())], device="cuda", dtype=torch.int64)
        dist.all_reduce(cnt)
        comm = n * 28 * (world - 1) // world            # bytes this rank sends (= receives) per step
        res["shuffle"] = {"value": world * n * steps / dt, "unit": "rows/s", "ms_per_step": 1000 * dt / steps, "step_ms": spread,
                          "mode": "ShuffleWriterExec[nccl://]: murmur3 partition ids -> partition-contiguous gather -> NCCL all-to-all-v over NVLink -> owner-side COUNT/SUM",
                          "collective": "ncclSend/ncclRecv grouped all-to-all-v (exchange.cu), inside the timed region",
                          "comm_bytes_per_rank_per_step": comm, "alltoall_gbs_per_rank": comm * steps / dt / 1e9, "nvlink_peak_gbs_per_direction": 900,
                          "exchange_ok": bool(int(cnt[0]) == n * world and int(cnt[1]) == int(cnt[2])),
                          "roofline": roofline_of(kern, steps, dt, {"murmur3_partition_ids": 8 * n, "partition_rows": 8 * n, "take": 2 * 28 * n})}
        runtime.nccl_finalize()
    res["value"], res["ms_per_step"] = res["shuffle"]["value"], res["shuffle"]["ms_per_step"]
    if world == 1:
        import oracle
        m = min(n, 16_000_000)
        sl = t4.slice(0, m)
        t0 = time.perf_counter()
        idx = pc.sort_indices(sl, sort_keys=[("ss_item_sk", "ascending")])
        sl.take(idx)
        s_sort = time.perf_counter() - t0
        t0 = time.perf_counter()
        oracle.partition_ids([sl["ss_item_sk"].combine_chunks()], 200)
        s_part = time.perf_counter() - t0
        res["cpu_baseline"] = {"sort_rows_per_sec": m / s_sort, "partition_ids_rows_per_sec": m / s_part, "unit": "rows/s", "cores": cores, "kind": "port",
                               "sample": f"first {m} rows: Arrow C++ sort_indices + take (all host threads); oracle C murmur3 partition ids (1 thread)"}
    runtime.drop_device_resource(rid)
    del keep
    return res


def _json_only_stdout():
    """Everything libraries print to stdout while the bench runs (NCCL's "NCCL version ..." banner comes from C code) is sent
    to stderr; only the JSON line reaches the real stdout."""
    sys.stdout.flush()
    real = os.dup(1)
    os.dup2(2, 1)
    sys.stdout = os.fdopen(real, "w", buffering=1)


if __name__ == "__main__":
    _json_only_stdout()
    main()
