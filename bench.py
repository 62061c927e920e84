#!/usr/bin/env python
"""bench.py — rows/s of the Parseable query hot path on B200 (BASELINE.json metric).

Headline workload (BASELINE.json configs[3], "C4"), weak scaling, one rank per GPU:
    SELECT host, status, COUNT(*), SUM(bytes), MIN(latency_ms), MAX(latency_ms), SUM(duration_s), MAX(cpu)
    FROM logs GROUP BY host, status          (+ the injected p_timestamp range, which footer statistics decide)
over RGS_PER_GPU row groups (125.8 M rows) PER GPU -> 1.007 B rows at 8 GPUs.  Every rank scans its own
files (file i -> rank i % N, the reference's partitioned_files round-robin, stream_schema_provider.rs:351-364)
and the partial tables meet in one grouped NCCL all-reduce INSIDE the timed step (PQ_QUERY_ALLREDUCE).
A "step" is one pass of the hot path over the whole table.

value  = total rows / step time with the encoded column chunks already resident in HBM (decode ->
         group-by -> all-reduce -> result batches on the host); steps are timed on the host around a
         device-synchronising call, max over ranks; the scan kernel is timed with CUDA events on its stream.
e2e    = the same query through the same C-ABI call with the Parquet file images in page-locked HOST
         memory: footer parse, page walk, H2D of the referenced chunks, flat-store build, kernels,
         all-reduce, D2H every step.
c2     = second workload on the same line (BASELINE.json configs[1]): WHERE level='ERROR' AND
         latency_ms>100 -> selected row ordinals, per rank over the same files (no collective in a filter scan).
--impl reference: the declared CPU stand-in for the reference's DataFusion path (BASELINE.md §3):
         pyarrow/Acero, all host threads, same files, same query, on rank 0's shard.

Launch: python bench.py [--gpus N --steps K --warmup W] [--dump-outputs DIR]; under torchrun one rank per GPU.
--steps K is the number of timed steps of every timed loop (resident, e2e, C2, reference arm).
--dump-outputs DIR: rank 0 writes what the last timed steps returned, as float64 .npy files (see dump_outputs).
"""
from __future__ import annotations

import argparse
import atexit
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

ROW_GROUP = 262_144
RGS_PER_FILE = 16                  # one Parquet file per ingest minute batch in Parseable
RGS_PER_GPU = 480                  # 125 829 120 rows per GPU; 8 GPUs: 1 006 632 960 rows ("1B")
# the generated tables are cached between runs, one directory per user: on a shared host another user's directory is
# neither writable nor known to hold complete files
DATA_DIR = os.environ.get("PQB_DATA_DIR") or os.path.join(tempfile.gettempdir(), f"pqb_bench_{os.getuid()}")
# the columns the two workloads reference (logs16 has 16; an unreferenced column is never read by either arm)
COLS = ["p_timestamp", "level", "latency_ms", "host", "bytes", "status", "duration_s", "cpu"]
C4_COLS = ["p_timestamp", "host", "status", "bytes", "latency_ms", "duration_s", "cpu"]
C2_COLS = ["p_timestamp", "level", "latency_ms"]
METRIC = "rows/sec filter+group-by over 1B-row synthetic log Parquet; % HBM roofline"
WORKLOAD = ("C4 group-by: GROUP BY host,status -> COUNT(*), SUM(bytes), MIN/MAX(latency_ms), SUM(duration_s), MAX(cpu); "
            "125.8M rows per GPU (1.007B at 8), file-sharded, one grouped NCCL all-reduce of the partial tables per step")
C2_WORKLOAD = "C2 scan+filter: WHERE level='ERROR' AND latency_ms>100 -> row ids, same files, per GPU"


# ------------------------------------------------------------------ data
# Headline files are UNCOMPRESSED (SURVEY §8d; north_star's decode list); PQB_BENCH_CODEC=LZ4 writes the same row groups
# with Parseable's default codec (LZ4_RAW, src/cli.rs:441-448) for development probes (tests/scripts/open_probe.py)
CODEC = os.environ.get("PQB_BENCH_CODEC", "NONE").upper()
def _gen_one(args):
    path, first, n = args
    from parseable_b200 import synth
    if not os.path.exists(path):
        synth.write_logs16(path, n_row_groups=n, first_rg=first, columns=COLS, compression=CODEC)
    return path


def file_jobs(n_row_groups: int):
    jobs, g = [], 0
    while g < n_row_groups:
        n = min(RGS_PER_FILE, n_row_groups - g)
        jobs.append((os.path.join(DATA_DIR, f"logs8_{g:06d}_{n}{'' if CODEC == 'NONE' else '_' + CODEC.lower()}.parquet"), g, n))
        g += n
    return jobs


def ensure_data(n_row_groups: int, rank: int = 0, world: int = 1, all_workers: bool = False) -> list[str]:
    """Row groups [0, n_row_groups) of the seeded logs16 generator (SURVEY §8d), generated on this box;
    rank r writes the files r, r + world, ... (its own shard)."""
    os.makedirs(DATA_DIR, exist_ok=True)
    jobs = file_jobs(n_row_groups)
    mine = [j for i, j in enumerate(jobs) if i % world == rank and not os.path.exists(j[0])]
    if mine:
        import multiprocessing as mp
        workers = max(1, min(len(mine), ((os.cpu_count() or 2) - 2) // (1 if all_workers else world)))
        t = time.time()
        with mp.get_context("spawn").Pool(workers) as pool:
            pool.map(_gen_one, mine, chunksize=1)
        print(f"[bench] rank {rank}: generated {len(mine)} files with {workers} workers in {time.time() - t:.1f}s", file=sys.stderr)
    return [j[0] for j in jobs]


class ClockSampler:
    """nvidia-smi clocks / throttle reasons, sampled from before the warm-up to the end of the timed regions
    (B200_PROFILING.md); the summary only keeps the samples taken inside a timed region."""

    def __init__(self, gpu_index: int):
        self.rows = []
        self.proc = None
        self.idx = gpu_index
        self.windows = []

    def start(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-i", str(self.idx), "-lms", "10"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            atexit.register(self._terminate)          # a run that fails before stop() must not leave the sampler running
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.perf_counter(), [x.strip() for x in line.split(",")]))

    def window(self, t0, t1):
        self.windows.append((t0, t1))

    def _terminate(self):
        if self.proc and self.proc.poll() is None:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()
                self.proc.wait()

    def stop(self) -> dict:
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"], "samples": 0}
        time.sleep(0.05)
        self._terminate()
        # a sample describes the ~10 ms before it was printed
        inside = [r for (t, r) in self.rows if any(a <= t <= b + 0.03 for a, b in self.windows)]
        sm = sorted(int(r[0]) for r in inside if r and r[0].isdigit())
        mx = [int(r[1]) for _, r in self.rows if len(r) > 1 and r[1].isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[i] for r in inside if len(r) >= 6 for i in range(4) if r[2 + i] == "Active"})
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons,
                "samples": len(sm), "samples_total": len(self.rows)}


# ------------------------------------------------------------------ queries
def c4_query():
    from parseable_b200.query import count_star, max_, min_, sum_
    return ["host", "status"], [count_star(), sum_("bytes"), min_("latency_ms"), max_("latency_ms"), sum_("duration_s"), max_("cpu")]


def c2_filters():
    from parseable_b200.query import col
    return [(col("level") == "ERROR") & (col("latency_ms") > 100)]


def time_filters(n_row_groups: int):
    """The range Query::final_logical_plan injects (src/query/mod.rs:774-833): here it covers every row, so
    footer statistics decide it, like a dashboard query over "the last N hours"."""
    from parseable_b200 import synth
    from parseable_b200.query import DEFAULT_TIMESTAMP_KEY, Timestamp, col
    lo = synth.TS_BASE - (n_row_groups + 2) * synth.RG_TS_STRIDE_MS
    hi = synth.TS_BASE + 1
    return [col(DEFAULT_TIMESTAMP_KEY) >= Timestamp(lo), col(DEFAULT_TIMESTAMP_KEY) < Timestamp(hi)], (lo, hi)


def schema():
    import pyarrow as pa
    return {"p_timestamp": pa.timestamp("ms"), "level": pa.string(), "latency_ms": pa.int64(), "host": pa.string(),
            "bytes": pa.int64(), "status": pa.int64(), "duration_s": pa.float64(), "cpu": pa.float64()}


C4_NAMES = ["host", "status", "count(*)", "sum(bytes)", "min(latency_ms)", "max(latency_ms)", "sum(duration_s)", "max(cpu)"]


def canon(tbl):
    """Group-by result in a canonical form: our column names, sorted by the keys."""
    import pyarrow as pa
    tbl = tbl.select(C4_NAMES).cast(pa.schema([("host", pa.string()), ("status", pa.int64()), ("count(*)", pa.int64()), ("sum(bytes)", pa.int64()),
                                               ("min(latency_ms)", pa.int64()), ("max(latency_ms)", pa.int64()), ("sum(duration_s)", pa.float64()),
                                               ("max(cpu)", pa.float64())]))
    return tbl.sort_by([("host", "ascending"), ("status", "ascending")])


def tables_agree(a, b, what: str):
    """COUNT / integer aggregates / MIN / MAX bit-exact, f64 SUM within 1e-9 relative (north_star)."""
    import numpy as np
    a, b = canon(a), canon(b)
    assert a.num_rows == b.num_rows, f"{what}: {a.num_rows} groups vs {b.num_rows}"
    for name in C4_NAMES:
        x, y = a[name].combine_chunks(), b[name].combine_chunks()
        if name == "sum(duration_s)":
            xv, yv = x.to_numpy(zero_copy_only=False), y.to_numpy(zero_copy_only=False)
            rel = np.abs(xv - yv) / np.maximum(np.abs(yv), 1e-300)
            assert float(rel.max(initial=0.0)) <= 1e-9, f"{what}: {name} differs by {rel.max():.3e} relative"
        else:
            assert x.equals(y), f"{what}: column {name} differs"
    return True


DUMP_BYTES = 64_000_000            # all arrays of one --dump-outputs directory together
DUMP_SEED = 20260922


def _utf8_codes(arr):
    """Utf8 values as float64: the top 53 bits of a BLAKE2b digest of the UTF-8 bytes (a float64 holds such an integer
    exactly), NaN for NULL. Equal strings give equal codes, so two builds' key columns compare as numbers."""
    import hashlib
    import numpy as np
    return np.array([np.nan if v is None else float(int.from_bytes(hashlib.blake2b(v.encode(), digest_size=8).digest(), "little") >> 11)
                     for v in arr.to_pylist()], dtype=np.float64)


def dump_outputs(out_dir: str, c4_table, c2_ids) -> dict:
    """Write what the last timed steps returned as out_dir/<name>.npy, float64 (integers are exact below 2**53, NULL is NaN):
    c4_<column>: the C4 result table in canonical order (canon: sorted by host, status), host as _utf8_codes;
    c2_row_ids: the C2 row ids as returned (ascending); when they do not fit in DUMP_BYTES next to the C4 arrays, a sample
    at positions drawn with DUMP_SEED, kept in order.  The tables are the seeded ones ensure_data writes, so two builds run
    with the same arguments can be compared array for array.  Returns {name: length}."""
    import numpy as np
    arrays = {}
    t = canon(c4_table)
    for name, short in zip(C4_NAMES, ["host", "status", "count", "sum_bytes", "min_latency_ms", "max_latency_ms",
                                      "sum_duration_s", "max_cpu"]):
        c = t[name]
        arrays["c4_" + short] = _utf8_codes(c) if name == "host" else np.asarray(c.to_numpy(zero_copy_only=False), dtype=np.float64)
    if c2_ids is not None:
        room = (DUMP_BYTES - sum(a.nbytes + 128 for a in arrays.values()) - 128) // 8     # 128: the .npy header
        if len(c2_ids) > room:
            keep = np.sort(np.random.default_rng(DUMP_SEED).choice(len(c2_ids), size=room, replace=False))
            c2_ids = c2_ids[keep]
        arrays["c2_row_ids"] = c2_ids.astype(np.float64)
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)
    return {name: len(a) for name, a in arrays.items()}


def plain_schema():
    """Utf8 columns as plain strings: the files' embedded Arrow schema says dictionary<int32, string> (one dictionary
    per row group), which Acero cannot group across fragments."""
    import pyarrow as pa
    return pa.schema(list(schema().items()))


def acero_groupby(files, n_row_groups):
    """The declared CPU stand-in (BASELINE.md §3): pyarrow dataset scan + Acero hash aggregate, all threads."""
    import pyarrow as pa
    import pyarrow.compute as pc
    import pyarrow.dataset as ds
    _, (lo, hi) = time_filters(n_row_groups)
    d = ds.dataset(files, format="parquet", schema=plain_schema())
    expr = (pc.field("p_timestamp") >= pa.scalar(lo, pa.timestamp("ms"))) & (pc.field("p_timestamp") < pa.scalar(hi, pa.timestamp("ms")))
    t = d.to_table(columns=["host", "status", "bytes", "latency_ms", "duration_s", "cpu"], filter=expr)
    g = t.group_by(["host", "status"]).aggregate([([], "count_all"), ("bytes", "sum"), ("latency_ms", "min"), ("latency_ms", "max"),
                                                  ("duration_s", "sum"), ("cpu", "max")])
    g = g.rename_columns([{"count_all": "count(*)", "bytes_sum": "sum(bytes)", "latency_ms_min": "min(latency_ms)",
                           "latency_ms_max": "max(latency_ms)", "duration_s_sum": "sum(duration_s)", "cpu_max": "max(cpu)"}.get(c, c)
                          for c in g.column_names])
    return g, t.num_rows


def acero_c2(files, n_row_groups):
    import pyarrow as pa
    import pyarrow.compute as pc
    import pyarrow.dataset as ds
    _, (lo, hi) = time_filters(n_row_groups)
    d = ds.dataset(files, format="parquet", schema=plain_schema())
    expr = ((pc.field("level") == "ERROR") & (pc.field("latency_ms") > 100) &
            (pc.field("p_timestamp") >= pa.scalar(lo, pa.timestamp("ms"))) & (pc.field("p_timestamp") < pa.scalar(hi, pa.timestamp("ms"))))
    tb = d.to_table(columns=["latency_ms"], filter=expr)
    return tb.num_rows


# ------------------------------------------------------------------ CPU legs
def _port_worker(args):
    path, nrg = args
    from oracle.oracle import Oracle
    o = Oracle.from_parquet(path, columns=C4_COLS)
    keys, aggs = c4_query()
    tf, _ = time_filters(nrg)
    g = o.group_by(keys, aggs, tf)
    return o.n, g.num_rows


def port_throughput(files: list[str], workers: int, nrg: int):
    """oracle port (pyarrow decode + oracle.c scalar semantics), one process per file; (rows/s, rows, seconds)."""
    import multiprocessing as mp
    with mp.get_context("spawn").Pool(workers) as pool:
        pool.map(_port_worker, [(files[0], nrg)])            # warm the pool / page cache / imports
        t = time.time()
        res = pool.map(_port_worker, [(f, nrg) for f in files], chunksize=1)
        dt = time.time() - t
    rows = sum(r[0] for r in res)
    return rows / dt, rows, dt


def run_reference(args, rank: int, world: int):
    if rank != 0:
        return
    import pyarrow as pa
    nrg = args.row_groups * world
    files = ensure_data(nrg, 0, world, all_workers=True)  # only rank 0's files are needed (the other ranks do not run)
    shard = files[0::world]                               # rank 0's files: the same bytes the GPU arm's rank 0 scans
    cores = os.cpu_count() or 1
    pa.set_cpu_count(cores)
    pa.set_io_thread_count(cores)
    vals = []
    acero_groupby(shard, nrg)                             # warm: page cache, thread pools
    for _ in range(args.steps):
        t = time.time()
        g, rows = acero_groupby(shard, nrg)
        vals.append((rows / (time.time() - t), rows, time.time() - t))
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, g, None)
    vs = sorted(v[0] for v in vals)
    v = vs[len(vs) // 2]                                  # median
    ms = 1000.0 * sorted(x[2] for x in vals)[len(vals) // 2]
    line = {
        "impl": "reference", "metric": METRIC, "value": v, "unit": "rows/s",
        "n_gpus": args.gpus, "steps": len(vals), "steps_requested": args.steps, "warmup": 1, "ms_per_step": ms,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "i64/f64/utf8-dictionary", "data": "synthetic",
        "config": {"workload": WORKLOAD, "rows_per_step": vals[-1][1],
                   "note": "one host: the CPU arm scans ONE GPU's shard with all host threads; its rows/s does not grow with N"},
        "cpu_baseline": {"value": v, "unit": "rows/s", "cores": cores, "kind": "port",
                         "standin": "pyarrow 24 / Acero dataset scan + hash aggregate, declared stand-in for the reference's DataFusion path "
                                    "(BASELINE.md §3: no cargo in this image); median of %d passes" % len(vals),
                         "sample": f"{len(shard)} files = {vals[-1][1]} rows (one GPU's shard), all {cores} host threads"},
        "e2e": {"value": v, "unit": "rows/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------ GPU arm
def pin_to_gpu_numa(local_rank: int) -> dict:
    """Bind this rank to the CPU NUMA node its GPU hangs off, before any pinned host buffer is allocated
    (first touch puts the file images on that node): at N > 1 the ranks' H2D copies then do not cross sockets."""
    try:
        import torch
        pr = torch.cuda.get_device_properties(local_rank)
        bdf = f"{getattr(pr, 'pci_domain_id', 0):04x}:{pr.pci_bus_id:02x}:{pr.pci_device_id:02x}.0"
        node = int(open(f"/sys/bus/pci/devices/{bdf}/numa_node").read())
        if node < 0:
            return {"numa_node": None, "why": "no NUMA information for the GPU"}
        cpus = set()
        for part in open(f"/sys/devices/system/node/node{node}/cpulist").read().strip().split(","):
            lo, _, hi = part.partition("-")
            cpus.update(range(int(lo), int(hi or lo) + 1))
        cpus &= os.sched_getaffinity(0)
        if not cpus:
            return {"numa_node": node, "why": "no allowed CPU on that node"}
        os.sched_setaffinity(0, cpus)
        return {"numa_node": node, "cpus": len(cpus), "gpu": bdf}
    except Exception as e:                               # best effort: never fail the bench over placement
        return {"numa_node": None, "why": f"{type(e).__name__}: {e}"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=30, help="timed steps of every timed loop")
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--row-groups", type=int, default=RGS_PER_GPU, help="row groups PER GPU (smaller tables for development runs)")
    ap.add_argument("--skip-cpu", action="store_true")
    ap.add_argument("--skip-e2e", action="store_true")
    ap.add_argument("--skip-c2", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the results of the last timed steps to DIR/<name>.npy (dump_outputs)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.warmup < 3:
        args.warmup = 3

    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import numpy as np
    import pyarrow as pa
    import torch
    import torch.distributed as dist
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the GPU arm has no CPU fallback")
    torch.cuda.set_device(local_rank)
    gloo = None
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
        gloo = dist.new_group(backend="gloo")       # host-side barriers / gathers: no kernel spinning on the GPU while rank 0 works

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier(group=gloo)

    def max_over_ranks(x: float) -> float:
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX, group=gloo)
        return float(t.item())

    nrg_total = args.row_groups * world
    all_files = ensure_data(nrg_total, rank, world)
    barrier()
    files = all_files[rank::world]                    # file i -> rank i % N (partitioned_files, stream_schema_provider.rs:351-364)

    import ctypes as C
    from oracle.oracle import Oracle                   # checker only (tests / smoke / this file's parity checks and CPU legs)
    from parseable_b200 import _lib as L
    from parseable_b200.query import DeviceTable, HostFile, StandardTableProvider
    lib = L.load()
    dev = (C.c_int * 1)(local_rank)
    if lib.pq_init(dev, 1) != 0:
        raise SystemExit(f"pq_init failed: {lib.pq_last_error(None)}")
    if world > 1:
        ident = [None]
        if rank == 0:
            buf = C.create_string_buffer(L.PQ_COMM_ID_BYTES)
            assert lib.pq_comm_unique_id(buf) == 0
            ident[0] = buf.raw
        dist.broadcast_object_list(ident, src=0, group=gloo)
        assert lib.pq_comm_init_rank(ident[0], world, rank) == 0, lib.pq_last_error(None)

    sch = schema()
    keys, aggs = c4_query()
    tf, _ = time_filters(nrg_total)
    ar_flag = L.PQ_QUERY_ALLREDUCE if world > 1 else 0
    checks = {}
    clocks = ClockSampler(local_rank)
    clocks.start()

    # ================= headline: C4 group-by, table resident =================
    t0 = time.perf_counter()
    table = DeviceTable(files, C4_COLS)
    open_s = time.perf_counter() - t0
    prov = StandardTableProvider(table, schema=sch)
    rows_per_gpu = table.rows
    r = prov.aggregate(keys, aggs, tf, flags=ar_flag)          # first answer: what the parity checks below look at
    result = r.table()
    groups = result.num_rows
    # ---- parity the driver can see ----
    local = prov.aggregate(keys, aggs, tf).table()            # this rank's partial answer, no collective
    if world > 1:
        # (1) every rank holds the same all-reduced table; (2) it equals the merge of the per-rank partial tables
        parts = [None] * world
        dist.gather_object(local.to_pydict(), parts if rank == 0 else None, dst=0, group=gloo)
        mine = [None] * world
        dist.gather_object(canon(result).to_pydict(), mine if rank == 0 else None, dst=0, group=gloo)
        if rank == 0:
            for r_i in range(1, world):
                tables_agree(pa.table(mine[r_i]), result, f"rank {r_i} vs rank 0 after the all-reduce")
            merged = pa.concat_tables([pa.table(p) for p in parts]).group_by(["host", "status"]).aggregate(
                [("count(*)", "sum"), ("sum(bytes)", "sum"), ("min(latency_ms)", "min"), ("max(latency_ms)", "max"),
                 ("sum(duration_s)", "sum"), ("max(cpu)", "max")])
            merged = merged.rename_columns([c[:-4] if c.endswith(("_sum", "_min", "_max")) else c for c in merged.column_names])
            tables_agree(result, merged, "all-reduced table vs merge of the per-rank partial tables")
            checks["allreduce_parity"] = True
            checks["allreduce_ranks_identical"] = True
    if rank == 0:
        assert int(np.sum(local["count(*)"].to_numpy())) == rows_per_gpu
        checks["count_star_total_equals_rows"] = True
        # the oracle (pyarrow decode + oracle.c) on one whole file of this shard
        ora = Oracle.from_parquet(files[0], columns=C4_COLS)
        one = StandardTableProvider([files[0]], schema=sch).aggregate(keys, aggs, tf).table()
        tables_agree(one, ora.group_by(keys, aggs, tf), "GPU vs oracle, group-by over one whole file")
        checks["oracle_groupby_one_file"] = {"rows": ora.n, "groups": one.num_rows, "agrees": True}
        del ora
    # the W warm-up steps come right before the timed ones (the checks above open other tables, run other queries and,
    # on rank 0 only, keep the host busy for seconds)
    barrier()
    for _ in range(args.warmup):
        r = prov.aggregate(keys, aggs, tf, flags=ar_flag)
    barrier()
    step_ms, scan_ms, dev_ms, host_ms, ar_ms = [], [], [], [], []
    launches = 0
    t_a = time.perf_counter()
    for _ in range(args.steps):
        ts = time.perf_counter()
        r = prov.aggregate(keys, aggs, tf, flags=ar_flag)
        step_ms.append(1000.0 * (time.perf_counter() - ts))
        m = r.metrics
        launches += m["kernel_launches"]
        scan_ms.append(m["scan_kernel_ms"]); dev_ms.append(m["device_ms"]); host_ms.append(m["host_ms"]); ar_ms.append(m["allreduce_ms"])
    barrier()
    t_b = time.perf_counter()
    clocks.window(t_a, t_b)
    dt = max_over_ranks(t_b - t_a)
    ms_per_step = 1000.0 * dt / args.steps
    value = rows_per_gpu * world / (dt / args.steps)
    algo_bytes = r.metrics["algorithmic_bytes"]
    d2h_res = r.metrics["d2h_bytes"]
    c4_last = r.table()                                # the last timed step's answer (--dump-outputs)
    assert c4_last.num_rows == groups
    if rank == 0:
        print(f"[bench] C4 resident step: wall {ms_per_step:.3f} ms = pq_query_open {sum(host_ms) / len(host_ms):.3f} ms (device {sum(dev_ms) / len(dev_ms):.3f} ms, "
              f"scan kernels {sum(scan_ms) / len(scan_ms):.3f} ms, all-reduce {sum(ar_ms) / len(ar_ms):.3f} ms) + binding/Arrow import; table open {open_s:.2f} s",
              file=sys.stderr)
    table.close()

    # ================= e2e: host buffers (page-locked file images), H2D + D2H inside every step =================
    e2e = None
    hfs = None
    numa = None
    if not args.skip_e2e:
        # the pinned file images are filled (first touch) from the NUMA node of this rank's GPU; the thread's affinity is
        # restored right after, so that the CPU legs further down keep every core
        aff = os.sched_getaffinity(0)
        numa = pin_to_gpu_numa(local_rank)
        hfs = [HostFile(path=p, pinned=True) for p in files]
        os.sched_setaffinity(0, aff)
        prov_e = StandardTableProvider(hfs, schema=sch)
        for _ in range(2):
            re_ = prov_e.aggregate(keys, aggs, tf, flags=ar_flag)
        barrier()
        k = args.steps
        t_a = time.perf_counter()
        for _ in range(k):
            re_ = prov_e.aggregate(keys, aggs, tf, flags=ar_flag)
        barrier()
        t_b = time.perf_counter()
        clocks.window(t_a, t_b)
        dte = max_over_ranks(t_b - t_a)
        if rank == 0:
            tables_agree(re_.table(), result, "e2e result vs resident result")
            checks["e2e_result_equals_resident"] = True
            print(f"[bench] C4 e2e step: wall {1000.0 * dte / k:.2f} ms = pq_query_open {re_.metrics['host_ms']:.2f} ms "
                  f"(footers+page walk+H2D+flat store {re_.metrics['upload_ms']:.2f} ms, device {re_.metrics['device_ms']:.2f} ms) + binding", file=sys.stderr)
        e2e = {"value": rows_per_gpu * world / (dte / k), "unit": "rows/s", "h2d_bytes_per_step": re_.metrics["h2d_bytes"],
               "d2h_bytes_per_step": re_.metrics["d2h_bytes"], "ms_per_step": 1000.0 * dte / k, "steps": k,
               "what": "pinned host file images -> footer parse -> H2D of the referenced chunks -> flat store -> kernels -> all-reduce -> result on host"}

    # ================= second workload: C2 scan + filter =================
    c2 = None
    c2_last_ids = None
    if not args.skip_c2:
        flt = c2_filters() + tf
        tbl2 = DeviceTable(files, C2_COLS)
        prov2 = StandardTableProvider(tbl2, schema=sch)
        for _ in range(args.warmup):
            r2 = prov2.scan(filters=flt)
        sel = sum(b.num_rows for b in r2.batches)
        if rank == 0:
            ids = np.concatenate([b.column(0).to_numpy() for b in r2.batches]) if r2.batches else np.array([], np.int64)
            assert len(ids) == sel and (sel == 0 or (ids[0] >= 0 and ids[-1] < rows_per_gpu)) and bool(np.all(np.diff(ids) > 0))
            assert prov2.scan(filters=flt, count_only=True).metrics["rows_selected"] == sel
            # full-size row-id equality against the oracle on one whole file (the first file holds row ordinals [0, rows))
            ora = Oracle.from_parquet(files[0], columns=C2_COLS)
            want = ora.row_ids(flt)
            assert np.array_equal(ids[: len(want)], want) and (len(ids) == len(want) or ids[len(want)] >= ora.n), "C2 row ids differ from the oracle"
            checks["c2_row_ids_equal_oracle_one_file"] = {"rows": ora.n, "selected": int(len(want)), "agrees": True}
            checks["c2_row_ids_strictly_ascending"] = True
            del ora
        barrier()
        s_ms, k_ms2 = [], []
        l2 = 0
        t_a = time.perf_counter()
        for _ in range(args.steps):
            ts = time.perf_counter()
            r2 = prov2.scan(filters=flt)
            s_ms.append(1000.0 * (time.perf_counter() - ts))
            k_ms2.append(r2.metrics["scan_kernel_ms"])
            l2 += r2.metrics["kernel_launches"]
        barrier()
        t_b = time.perf_counter()
        clocks.window(t_a, t_b)
        dt2 = max_over_ranks(t_b - t_a)
        launches += l2
        if args.dump_outputs and rank == 0:
            c2_last_ids = np.concatenate([b.column(0).to_numpy() for b in r2.batches]) if r2.batches else np.array([], np.int64)
        c2 = {"workload": C2_WORKLOAD, "value": rows_per_gpu * world / (dt2 / args.steps), "unit": "rows/s", "ms_per_step": 1000.0 * dt2 / args.steps,
              "selected_rows_per_gpu": sel, "kernel": "k_flat_filter", "kernel_ms": sum(k_ms2) / len(k_ms2),
              "algorithmic_bytes": r2.metrics["algorithmic_bytes"], "d2h_bytes_per_step": r2.metrics["d2h_bytes"],
              "device_ms_per_step": r2.metrics["device_ms"], "gpu_launches": l2}
        tbl2.close()
        if hfs is not None:
            prov2e = StandardTableProvider(hfs, schema=sch)
            for _ in range(2):
                r2e = prov2e.scan(filters=flt)
            barrier()
            k = args.steps
            t_a = time.perf_counter()
            for _ in range(k):
                r2e = prov2e.scan(filters=flt)
            barrier()
            t_b = time.perf_counter()
            clocks.window(t_a, t_b)
            dt2e = max_over_ranks(t_b - t_a)
            assert sum(b.num_rows for b in r2e.batches) == sel
            c2["e2e"] = {"value": rows_per_gpu * world / (dt2e / k), "unit": "rows/s", "ms_per_step": 1000.0 * dt2e / k,
                         "h2d_bytes_per_step": r2e.metrics["h2d_bytes"], "d2h_bytes_per_step": r2e.metrics["d2h_bytes"], "steps": k}
    if hfs is not None:
        for h in hfs:
            h.close()
    clk = clocks.stop()

    if rank != 0:
        if world > 1:
            dist.barrier(group=gloo)
            dist.destroy_process_group()
        return

    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    peak_kind = "measured (MEASURED_PEAKS.json hbm_gbs)" if "hbm_gbs" in peaks else "fallback 6.65 TB/s (B200_PROFILING.md)"
    traffic = {}
    try:
        traffic = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
    except Exception:
        pass

    def roof(kernel, kernel_ms, bytes_, traffic_key):
        ach = bytes_ / (kernel_ms * 1e-3) / 1e9 if kernel_ms > 0 else 0.0
        # the ncu capture was taken at the default size: no figure for other table sizes
        return {"bound": "hbm", "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak,
                "traffic": traffic.get(traffic_key) if args.row_groups == RGS_PER_GPU else None,
                "kernel": kernel, "kernel_ms": kernel_ms, "algorithmic_bytes": bytes_, "peak_kind": peak_kind}

    if c2 is not None:
        c2["roofline"] = roof("k_flat_filter", c2["kernel_ms"], c2["algorithmic_bytes"], "k_flat_filter_dram_bytes_per_launch")
    cpu_baseline = None
    if not args.skip_cpu:
        cores = os.cpu_count() or 1
        # the oracle port (the checker) timed on a bounded sample of the same files, one process per file
        sample = files[: max(1, min(len(files), cores // 4 if cores >= 8 else 2, 16))]
        v, rows, secs = port_throughput(sample, workers=min(cores, len(sample)), nrg=nrg_total)
        cpu_baseline = {"value": v, "unit": "rows/s", "cores": min(cores, len(sample)), "kind": "port",
                        "sample": f"{len(sample)} of {len(files)} files ({rows} rows, {secs:.1f} s): pyarrow decode + oracle.c group-by, one process per file"}
        try:
            pa.set_cpu_count(cores)
            pa.set_io_thread_count(cores)
            acero_groupby(files, nrg_total)
            ta = time.time()
            ag, arows = acero_groupby(files, nrg_total)
            asecs = time.time() - ta
            # the independent engine's answer over this rank's WHOLE shard is also a full-size parity check
            tables_agree(local, ag, "GPU vs Acero over the whole shard")
            checks["acero_whole_shard_agrees"] = {"rows": arows, "groups": ag.num_rows, "agrees": True}
            cpu_baseline["acero_standin"] = {"value": arows / asecs, "unit": "rows/s", "cores": cores, "rows": arows, "seconds": asecs,
                                             "note": "pyarrow/Acero dataset scan + hash aggregate over one GPU's shard, not DataFusion (BASELINE.md §3)"}
            if c2 is not None:
                acero_c2(files, nrg_total)
                ta = time.time()
                asel = acero_c2(files, nrg_total)
                asecs = time.time() - ta
                assert asel == c2["selected_rows_per_gpu"], (asel, c2["selected_rows_per_gpu"])
                checks["c2_acero_count_agrees"] = True
                c2["acero_standin"] = {"value": rows_per_gpu / asecs, "unit": "rows/s", "cores": cores, "seconds": asecs}
        except AssertionError:
            raise
        except Exception as e:  # pragma: no cover
            cpu_baseline["acero_standin"] = {"error": repr(e)}
    k_ms = sum(scan_ms) / len(scan_ms)
    line = {
        "metric": METRIC,
        "value": value, "unit": "rows/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "i64/f64/utf8-dictionary (bit-packed indices)", "data": "synthetic",
        "config": {"workload": WORKLOAD, "rows_per_gpu": rows_per_gpu, "rows_total": rows_per_gpu * world, "row_groups_per_gpu": args.row_groups,
                   "groups": groups, "l2": "inputs (encoded chunks read per step) larger than L2; no explicit flush",
                   "parallelism": f"file shards x{world} (file i -> rank i % N), one grouped ncclAllReduce of the partial tables per step" if world > 1
                   else "1 GPU, no collective"},
        "roofline": roof("k_flat_agg (+k_acc_reduce)", k_ms, algo_bytes, "k_flat_agg_dram_bytes_per_launch"),
        "allreduce_ms": sum(ar_ms) / len(ar_ms), "device_ms_per_step": sum(dev_ms) / len(dev_ms),
        "e2e": e2e, "gpu_launches": launches, "clocks": clk, "cpu_baseline": cpu_baseline,
        "d2h_bytes_per_step_resident": d2h_res, "c2": c2, "numa": numa,
    }
    q = sorted(step_ms)
    line["step_ms_quantiles"] = {"p10": q[len(q) // 10], "p50": q[len(q) // 2], "p90": q[(len(q) * 9) // 10], "max": q[-1]}
    line["step_ms"] = [round(x, 3) for x in step_ms]      # rank 0's wall time of every timed step, in order
    line["checks"] = checks
    if args.dump_outputs:
        lens = dump_outputs(args.dump_outputs, c4_last, c2_last_ids)
        print(f"[bench] --dump-outputs: {lens} -> {args.dump_outputs}", file=sys.stderr)
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier(group=gloo)
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
