#!/usr/bin/env python
"""bench.py — the measurement contract of the csvplus_b200 hot path.

Headline workload = BASELINE.json configs[3] (north_star's target), the reference README's own pattern
(/root/reference/README.md:34-56, csvplus.go:545-583):
    customers (100 M rows, 6 cols) -> SelectColumns(id,name,surname)        -> UniqueIndexOn("id")
    products  (  1 M rows, 3 cols) -> SelectColumns(prod_id,product,price)  -> UniqueIndexOn("prod_id")
    orders (125 M rows PER GPU, 5 cols) -> SelectColumns(cust_id,prod_id,qty,ts).Join(custIdx,"cust_id").Join(prodIdx)
one "step" = one full pass of that pipeline over synthetic CSV (SURVEY §8d shapes).  At --gpus 8 the job is exactly
the config (1 B orders x 100 M customers x 1 M products); the build sides have the config's size at every N, the probe
stream is sharded by row range (weak scaling).
  value = probe rows/s with the CSV bytes already resident in HBM (whole job, all ranks);
  e2e   = the same through the public API from HOST (pinned) CSV buffers, H2D inside the timed region, ending in the
          README's sink: ToCsv(name,surname,qty,product,price,ts) of every joined row, copied back to pinned host
          memory inside the timed region (probe file streamed in batches over two contexts, H2D/compute/D2H overlapped).
Also timed in the same run:
  csv_parse  BASELINE configs[1]: people 100 M rows x 6 cols, parse + SelectColumns(name,surname,id) + Filter(Like name=Amelia)
  index_on   BASELINE configs[4]: 10 M rows, IndexOn("cust_id","prod_id") (composite key, ~50 % of the rows in duplicate
             groups) + ResolveDuplicates(keep the bytewise smallest order_id), both §Q1 tail shapes
"roofline" describes the dominant kernel of the step (csv_scan).
--dump-outputs DIR writes a fixed sample of the tables the last timed step of the join, csv_parse and index_on legs returned
(dump_table); the inputs come from SEED, so two builds run with the same arguments can be compared output for output.

Multi-GPU (torchrun, one rank per GPU): every rank parses 1/N of the customers file; the parsed columns are
all-gathered (NCCL) and every rank builds the full index; products (25 MB) are parsed by every rank.

--impl reference: the reference (pure Go) cannot be built here (no Go toolchain), so the arm times the CPU oracle port
of the same pipeline (oracle/, kind "port") on a bounded sample whose sizes are printed in its `config`, single-threaded
because the reference is strictly single-threaded (csvplus.go has no goroutines).
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

SEED = 0xC5B200
CUST_COLS = [("id", -1), ("name", -1), ("surname", -1)]
PROD_COLS = [("prod_id", -1), ("product", -1), ("price", -1)]
ORDER_COLS = [("cust_id", -1), ("prod_id", -1), ("qty", -1), ("ts", -1)]
PEOPLE_COLS = [("name", -1), ("surname", -1), ("id", -1)]
INDEX_COLS = [("order_id", -1), ("cust_id", -1), ("prod_id", -1), ("qty", -1)]
SINK_COLS = ("name", "surname", "qty", "product", "price", "ts")  # README.md:59-64

ORD_ROWS = 125_000_000      # per GPU
CUST_ROWS = 100_000_000     # whole job
PROD_ROWS = 1_000_000
PEOPLE_ROWS = 100_000_000   # per GPU
INDEX_ROWS = 10_000_000


def hbm_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured"
        except Exception:
            pass
    return 6650.0, "fallback"


class ClockSampler:
    """nvidia-smi polled every 100 ms in the background (a 20 ms poll measurably slows the step: its NVML queries
    contend with the launches); stop(t0, t1) keeps the samples whose timestamps fall inside the timed region
    [t0, t1] (wall clock), so that it may be started early (nvidia-smi needs ~0.1 s to start)"""

    def __init__(self, index: int):
        self.p = None
        try:
            self.p = subprocess.Popen(
                ["nvidia-smi", f"--id={index}",
                 "--query-gpu=timestamp,clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,"
                 "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
                 "clocks_event_reasons.sw_power_cap", "--format=csv,noheader,nounits", "-lms", "100"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.p = None

    def stop(self, t0: float | None = None, t1: float | None = None):
        import datetime
        if self.p is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.p.terminate()
        try:
            out, _ = self.p.communicate(timeout=5)
        except Exception:
            self.p.kill(); out = ""
        rows = []
        for ln in out.splitlines():
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 7:
                continue
            try:
                ts = datetime.datetime.strptime(f[0], "%Y/%m/%d %H:%M:%S.%f").timestamp()
                rows.append((ts, float(f[1]), float(f[2]), f[3:7]))
            except ValueError:
                continue
        inside = [r for r in rows if t0 is not None and t1 is not None and t0 - 0.01 <= r[0] <= t1 + 0.01]
        window = "timed region" if inside else "whole run (no sample fell inside the timed region)"
        use = inside or rows
        reasons = set()
        for r in use:
            for name, v in zip(["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"], r[3]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median([r[1] for r in use]) if use else None,
                "sm_max_mhz": max(r[2] for r in use) if use else None,
                "reasons": sorted(reasons), "samples": len(use), "window": window}


def index_sides(n_rows: int) -> int:
    """cust/prod id ranges of the index_on workload: n_cust = n_prod = sqrt(1.44 n) so that ~50 % of the rows share
    their (cust_id, prod_id) key with another row (Poisson, mean 0.69 extra rows per key)"""
    return max(2, int((1.44 * n_rows) ** 0.5))


# ------------------------------------------------------------------ reference arm / cpu baseline (oracle port)
def cpu_join3_sample(n_orders: int, n_cust: int, n_prod: int, ctx=None, data=None):
    """the three-way join pipeline in the CPU oracle, single thread; returns (rows/s, seconds, sample text)"""
    from oracle import oracle as orc
    if data is None:
        cust = ctx.gen_csv("customers", (0, n_cust), seed=SEED, n_cust=n_cust, permute=True).to_host()
        prod = ctx.gen_csv("products", (0, n_prod), seed=SEED, n_prod=n_prod, permute=True).to_host()
        orders = ctx.gen_csv("orders", (0, n_orders), seed=SEED, n_cust=n_cust, n_prod=n_prod).to_host()
    else:
        cust, prod, orders = data
    t0 = time.perf_counter()
    cidx = orc.reader_rows(cust, select=[c for c, _ in CUST_COLS]).unique_index_on("id", stable=False)
    pidx = orc.reader_rows(prod, select=[c for c, _ in PROD_COLS]).unique_index_on("prod_id", stable=False)
    joined = orc.reader_rows(orders, select=[c for c, _ in ORDER_COLS]).join(cidx, "cust_id").join(pidx)
    n = len(joined)
    dt = time.perf_counter() - t0
    assert n == n_orders, (n, n_orders)
    return n_orders / dt, dt, f"orders {n_orders} x customers {n_cust} x products {n_prod} rows, same generator, 1 thread"


def cpu_parse_sample(n_rows: int, ctx):
    from oracle import oracle as orc
    people = ctx.gen_csv("people", (0, n_rows), seed=SEED).to_host()
    t0 = time.perf_counter()
    r = orc.reader_rows(people, select=[c for c, _ in PEOPLE_COLS], pred=orc.Like({"name": "Amelia"}))
    n = len(r)
    dt = time.perf_counter() - t0
    return people.size / dt / 1e9, n_rows / dt, dt, n


def cpu_index_sample(n_rows: int, ctx):
    """IndexOn(cust_id, prod_id) + ResolveDuplicates(min order_id) in the oracle (std::sort with the reference's
    map-lookup comparator standing in for sort.Sort), 1 thread"""
    from oracle import oracle as orc
    side = index_sides(n_rows)
    raw = ctx.gen_csv("orders", (0, n_rows), seed=SEED, n_cust=side, n_prod=side).to_host()
    rows = orc.reader_rows(raw, select=[c for c, _ in INDEX_COLS])
    t0 = time.perf_counter()
    ix = rows.index_on("cust_id", "prod_id", stable=False)
    t1 = time.perf_counter()
    ix.dedup("min", "order_id")
    t2 = time.perf_counter()
    return n_rows / (t1 - t0), t1 - t0, t2 - t1, len(ix)


def workload_config(world, ref=None):
    if ref is not None:
        return {"workload": "three-way Join (BASELINE configs[3] pattern) on the reference arm's bounded sample",
                "orders_rows_per_gpu": ref[0], "customers_rows": ref[1], "products_rows": ref[2],
                "parallelism": "1 CPU thread (the reference is single-threaded)",
                "note": "the b200 arm runs orders %d/GPU x customers %d x products %d; a CPU step at that size would take "
                        "~15 min, so the arm times this sample of the same generator and pipeline" % (ORD_ROWS, CUST_ROWS, PROD_ROWS)}
    return {"workload": "orders(%d M rows/GPU) x customers(%d M) x products(%d M): parse+SelectColumns, UniqueIndexOn(id), "
                        "UniqueIndexOn(prod_id), Join(custIdx,cust_id).Join(prodIdx) [BASELINE configs[3]; configs[1] under "
                        "csv_parse, configs[4] under index_on]" % (ORD_ROWS // 10**6, CUST_ROWS // 10**6, max(1, PROD_ROWS // 10**6)),
            "orders_rows_per_gpu": ORD_ROWS, "customers_rows": CUST_ROWS, "products_rows": PROD_ROWS,
            "people_rows_per_gpu": PEOPLE_ROWS, "index_rows": INDEX_ROWS,
            "parallelism": f"probe row-range shards x{world}; customers parsed 1/{world} per rank and all-gathered (NCCL); "
                           "index built on every rank" if world > 1 else "single GPU",
            "l2": "inputs (>= 25 MB products, otherwise >= 0.5 GB per pass) exceed or stream through the 126 MB L2; no flush needed"}


def run_reference(args, rank):
    if rank != 0:
        return
    import csvplus_b200 as cp
    ctx = cp.Context(int(os.environ.get("LOCAL_RANK", "0")))  # (generates the sample inputs; nothing on this arm's timed path)
    n_orders, n_cust, n_prod = args.ref_orders, args.ref_customers, args.ref_products
    cust = ctx.gen_csv("customers", (0, n_cust), seed=SEED, n_cust=n_cust, permute=True).to_host()
    prod = ctx.gen_csv("products", (0, n_prod), seed=SEED, n_prod=n_prod, permute=True).to_host()
    orders = ctx.gen_csv("orders", (0, n_orders), seed=SEED, n_cust=n_cust, n_prod=n_prod).to_host()
    times = []
    sample = ""
    for i in range(args.warmup + args.steps):
        _, dt, sample = cpu_join3_sample(n_orders, n_cust, n_prod, data=(cust, prod, orders))
        if i >= args.warmup:
            times.append(dt)
    ms = 1e3 * sum(times) / len(times)
    value = n_orders / (ms / 1e3)
    line = {
        "impl": "reference", "metric": "rows/sec end-to-end Join", "value": value, "unit": "rows/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "u8", "data": "synthetic",
        "config": workload_config(args.gpus, ref=(n_orders, n_cust, n_prod)),
        "cpu_baseline": {"value": value, "unit": "rows/s", "cores": 1, "kind": "port",
                         "sample": sample + " (oracle/ C++ restatement of csvplus; the Go reference has no toolchain here)"},
        "e2e": {"value": value, "unit": "rows/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


def ncu_traffic(paths):
    """mean dram__bytes_read.sum + dram__bytes_write.sum per csv_scan launch from the committed ncu metrics pass of this
    bench command's join step; (None, None) if no file is present"""
    import csv
    for path in paths:
        try:
            per_id = {}
            with open(path) as f:
                rows = [r for r in csv.reader(f) if len(r) > 14]
            hdr = rows[0]
            ki, mi, ui, vi, ii = (hdr.index(x) for x in ("Kernel Name", "Metric Name", "Metric Unit", "Metric Value", "ID"))
            for r in rows[1:]:
                if "csv_scan" in r[ki] and r[mi] in ("dram__bytes_read.sum", "dram__bytes_write.sum"):
                    scale = {"byte": 1, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9}[r[ui]]
                    per_id[r[ii]] = per_id.get(r[ii], 0.0) + float(r[vi].replace(",", "")) * scale
            if per_id:
                return sum(per_id.values()) / len(per_id), os.path.relpath(path, ROOT)
        except Exception:
            continue
    return None, None


def bind_to_gpu_numa_node(local: int):
    """Pin this process (and the pinned host buffers it allocates afterwards) to the NUMA node the GPU hangs off,
    so that H2D copies do not cross the socket interconnect.  Best effort: silently skipped where /sys is not
    available.  Returns the node id or None."""
    try:
        import torch
        pr = torch.cuda.get_device_properties(local)
        bdf = "%04x:%02x:%02x.0" % (pr.pci_domain_id, pr.pci_bus_id, pr.pci_device_id)
        node = int(open(f"/sys/bus/pci/devices/{bdf}/numa_node").read().strip())
        if node < 0:
            return None
        cpus = set()
        for part in open(f"/sys/devices/system/node/node{node}/cpulist").read().strip().split(","):
            a, _, b = part.partition("-")
            cpus.update(range(int(a), int(b or a) + 1))
        allowed = cpus & os.sched_getaffinity(0)
        if allowed:
            os.sched_setaffinity(0, allowed)
        return node
    except Exception:
        return None


def without_greatest_key(table, key_cols):
    """the table minus every row that carries the greatest key (the last row of the sorted order): used to reach the
    other §Q1 tail shape — the last sorted row a singleton / a member of a duplicate group"""
    import csvplus_b200 as cp
    ix = table.index_on(*key_cols)
    st = ix.table()
    last = st.rows(len(st) - 1, len(st))[0]
    return table.filter(cp.Not(cp.Like({c: last[c] for c in key_cols})))


def min_id_resolver(table, lo, hi):
    """the tie-order-independent resolver of SURVEY §8d cfg 5, vectorised (host user code, like the Go closure the
    reference calls once per group): for every duplicate group keep the row whose order_id is bytewise smallest"""
    import numpy as np
    if len(lo) == 0:
        return np.empty(0, np.int64)
    off, data = table.column("order_id")
    cnt = hi - lo
    starts = np.zeros(len(lo), np.int64); starts[1:] = np.cumsum(cnt)[:-1]
    rows = np.repeat(lo - starts, cnt) + np.arange(int(cnt.sum()), dtype=np.int64)   # sorted positions of all grouped rows
    b0, ln = off[rows], off[rows + 1] - off[rows]
    assert int(ln.max()) <= 8
    key = np.zeros(len(rows), np.uint64)  # value left-aligned, zero padded: integer order == bytewise string order
    for b in range(8):
        m = ln > b
        key[m] |= data[b0[m] + b].astype(np.uint64) << np.uint64(8 * (7 - b))
    gmin = np.minimum.reduceat(key, starts)
    is_min = key == np.repeat(gmin, cnt)
    first = np.flatnonzero(is_min)
    gid = np.repeat(np.arange(len(lo)), cnt)[first]
    keep = np.full(len(lo), -1, np.int64)
    keep[gid[::-1]] = rows[first[::-1]]  # the lowest position among equal minima (values equal => same row content for the key)
    return keep


DUMP_BLOCKS, DUMP_BLOCK_ROWS = 32, 256  # rows of each table --dump-outputs writes: at most 32 blocks of 256
DUMP_LIMIT_BYTES = 64 << 20            # all files of one run together


def dump_sample_blocks(n_rows: int):
    """[lo, hi) row ranges --dump-outputs samples from a table of n_rows rows: the first and the last block and seeded
    blocks between them, in row order; the same n_rows always gives the same ranges"""
    import numpy as np
    b = DUMP_BLOCK_ROWS
    nblocks = -(-n_rows // b)
    if nblocks <= DUMP_BLOCKS:
        picks = np.arange(nblocks)
    else:
        inner = np.random.default_rng(SEED).choice(np.arange(1, nblocks - 1), DUMP_BLOCKS - 2, replace=False)
        picks = np.sort(np.concatenate([[0, nblocks - 1], inner]))
    return [(int(k) * b, min(n_rows, (int(k) + 1) * b)) for k in picks]


def dump_table(out_dir: str, name: str, table) -> int:
    """Writes a fixed sample of a table's rows as float arrays: <name>.num_rows.npy (the table's row count),
    <name>.sample_rows.npy (the sampled row positions) and per column <name>.<column>.npy, float32 [rows, width],
    the field's bytes followed by -1 up to the width of the longest sampled field.  Returns the bytes written."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    n = len(table)
    blocks = dump_sample_blocks(n)
    arrays = {"num_rows": np.array([n], np.float64),
              "sample_rows": np.concatenate([np.arange(lo, hi) for lo, hi in blocks] or [[]]).astype(np.float64)}
    for c in table.columns:
        parts = [table.column(c, lo, hi) for lo, hi in blocks]
        lens = np.concatenate([np.diff(off) for off, _ in parts] or [[]]).astype(np.int64)
        data = np.concatenate([d for _, d in parts] or [[]]).astype(np.float32)
        width = int(lens.max()) if len(lens) else 0
        m = np.full((len(lens), width), -1, np.float32)
        m[np.arange(width) < lens[:, None]] = data  # row-major order of the mask is the order of the bytes
        arrays[c] = m
    written = 0
    for k, a in arrays.items():
        path = os.path.join(out_dir, f"{name}.{k}.npy")
        np.save(path, a)
        written += os.path.getsize(path)
    return written


def main():
    global ORD_ROWS, CUST_ROWS, PROD_ROWS, PEOPLE_ROWS, INDEX_ROWS
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--orders", type=int, default=ORD_ROWS, help="probe rows per GPU")
    ap.add_argument("--customers", type=int, default=CUST_ROWS)
    ap.add_argument("--products", type=int, default=PROD_ROWS)
    ap.add_argument("--people", type=int, default=PEOPLE_ROWS)
    ap.add_argument("--index-rows", type=int, default=INDEX_ROWS)
    ap.add_argument("--ref-orders", type=int, default=2_000_000)
    ap.add_argument("--ref-customers", type=int, default=1_600_000)
    ap.add_argument("--ref-products", type=int, default=100_000)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--e2e-batches", type=int, default=24)
    ap.add_argument("--e2e-workers", type=int, default=8)
    ap.add_argument("--e2e-sweep", default="", help="e.g. 8x4,16x8: time these (batches x workers) settings of the e2e leg, report the best")
    ap.add_argument("--dump-outputs", metavar="DIR", default="",
                    help="write a fixed sample of the tables the last timed step of each device-resident leg returned as DIR/*.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs applies to --impl b200")
    ORD_ROWS, CUST_ROWS, PROD_ROWS, PEOPLE_ROWS, INDEX_ROWS = args.orders, args.customers, args.products, args.people, args.index_rows
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank)
        return

    import numpy as np
    import torch
    import torch.distributed as dist

    import csvplus_b200 as cp
    torch.cuda.set_device(local)
    numa_node = bind_to_gpu_numa_node(local)
    # (NCCL prints its version banner on stdout when the first communicator comes up: stdout carries the JSON line only)
    saved_stdout = os.dup(1)
    os.dup2(2, 1)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    ctx = cp.Context(local)
    stream = torch.cuda.ExternalStream(ctx.stream, device=torch.device("cuda", local))

    # ---------------- synthetic inputs (device resident; pinned host copies for the e2e leg)
    cust_lo, cust_hi = rank * CUST_ROWS // world, (rank + 1) * CUST_ROWS // world
    d_cust = ctx.gen_csv("customers", (cust_lo, cust_hi), seed=SEED, n_cust=CUST_ROWS, permute=True, header=True)
    d_prod = ctx.gen_csv("products", (0, PROD_ROWS), seed=SEED, n_prod=PROD_ROWS, permute=True, header=True)
    d_orders = ctx.gen_csv("orders", (rank * ORD_ROWS, (rank + 1) * ORD_ROWS), seed=SEED, n_cust=CUST_ROWS, n_prod=PROD_ROWS, header=True)
    d_people = ctx.gen_csv("people", (rank * PEOPLE_ROWS, (rank + 1) * PEOPLE_ROWS), seed=SEED, header=True)
    ctx.sync()
    # the step's tables, index structures and scratch (~35 GB at the default sizes, more with the gathered build side) come
    # out of memory the pool maps once, here, instead of growing it over the first iterations (measured at N = 2 without
    # it: steps of 200 ms until the sixth iteration, 56 ms after)
    free_b, _total_b = torch.cuda.mem_get_info(local)
    reserve_b = int(min(0.45 * free_b, 56e9))
    reserved = ctx.reserve(reserve_b)

    # Python's cyclic collector: a full collection walks every object torch's import created (hundreds of ms) and its
    # schedule depends only on allocation counts, so it hits every rank at the same step (measured at N = 2: steps of
    # 55 ms with one of 150-780 ms every ~14 calls).  Everything alive now is long-lived: park it where collections
    # do not look.
    import gc
    gc.collect()
    gc.freeze()

    from csvplus_b200.dist import allgather_table_nccl, init_comm
    if world > 1:
        init_comm(ctx, dist)  # the library's own communicator: the build-side all-gather runs inside the C ABI
        dist.barrier()

    dbg = bool(os.environ.get("BENCH_DEBUG")) and rank == 0

    def join_step(cust_src, prod_src, orders_src):
        marks = []

        def mark(name):
            if dbg:
                ctx.sync(); torch.cuda.synchronize()
                marks.append((name, time.perf_counter()))
        mark("start")
        tc, err = cp.parse_csv(ctx, cust_src, spec=CUST_COLS)
        assert err is None
        mark("parse_cust")
        if world > 1:  # the build-side all-gather (cpb_allgather_table: NCCL on the ctx stream, one host sync for the sizes)
            tc = allgather_table_nccl(ctx, tc)
            mark("allgather")
        tp, err = cp.parse_csv(ctx, prod_src, spec=PROD_COLS)
        assert err is None
        pidx = tp.index_on("prod_id", unique=True)
        mark("products")
        to, err = cp.parse_csv(ctx, orders_src, spec=ORDER_COLS)
        assert err is None
        mark("parse_orders")
        cidx = tc.index_on("id", unique=True)
        mark("index")
        j = to.join(cidx, "cust_id").join(pidx)
        mark("join")
        if dbg:
            print("phases(ms): " + " ".join("%s=%.2f" % (marks[i][0], (marks[i][1] - marks[i - 1][1]) * 1e3)
                                           for i in range(1, len(marks))), file=sys.stderr)
        return j

    def parse_step(people_src):
        t, err = cp.parse_csv(ctx, people_src, spec=PEOPLE_COLS, pred=cp.Like({"name": "Amelia"}))
        assert err is None
        return t

    sync0 = [0, 0]
    per_step = []

    def timed(fn, steps, warmup, sampler_dev=None):
        sampler = ClockSampler(sampler_dev) if sampler_dev is not None and not os.environ.get("BENCH_NO_SAMPLER") else None  # polls through warm-up + timed steps
        for _ in range(warmup):
            r = fn(); del r
        ctx.sync(); torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        ctx.stats(enable=True, reset=True)
        l0 = ctx.kernel_launches()
        sync0[0] = ctx.host_syncs()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t_begin = time.time()
        e0.record(stream)
        rows = 0
        marks = []
        for i in range(steps):
            r = fn(); rows = len(r)
            if i + 1 < steps:  # the last step's result is returned to the caller
                del r
            ev = torch.cuda.Event(enable_timing=True); ev.record(stream); marks.append(ev)
        e1.record(stream)
        sync0[1] = ctx.host_syncs() - sync0[0]
        ctx.sync(); torch.cuda.synchronize()
        t_end = time.time()
        ms = e0.elapsed_time(e1)
        per_step[:] = [round((e0 if i == 0 else marks[i - 1]).elapsed_time(marks[i]), 3) for i in range(steps)]
        if os.environ.get("BENCH_DEBUG") or os.environ.get("BENCH_PER_STEP"):
            print("rank %d per-step ms: %s" % (rank, per_step), file=sys.stderr)
        if world > 1:
            dist.barrier()
            tms = torch.tensor([ms], device="cuda", dtype=torch.float64)
            dist.all_reduce(tms, op=dist.ReduceOp.MAX)
            ms = float(tms.item())
        stats = ctx.stats()
        ctx.stats(enable=False)
        clocks = sampler.stop(t_begin, t_end) if sampler else None
        return ms / steps, rows, stats, ctx.kernel_launches() - l0, clocks, r

    dumped = [0]

    def dump(name, table):
        if args.dump_outputs and rank == 0:
            dumped[0] += dump_table(args.dump_outputs, name, table)
            assert dumped[0] <= DUMP_LIMIT_BYTES, f"--dump-outputs wrote {dumped[0]} bytes"

    # ---------------- device-resident timing (value)
    ms_join, out_rows, st_join, launches, clocks, last = timed(lambda: join_step(d_cust, d_prod, d_orders), args.steps, args.warmup, local)
    dump("join", last)
    del last
    join_syncs = sync0[1] / args.steps
    join_per_step = list(per_step)
    assert out_rows == ORD_ROWS, (out_rows, ORD_ROWS)  # every order matches exactly one customer and one product
    ms_parse, parse_rows, st_parse, _, _, last = timed(lambda: parse_step(d_people), args.steps, args.warmup)
    dump("csv_parse", last)
    del last
    peak, peak_kind = hbm_peak()
    traffic, traffic_src = ncu_traffic([os.path.join(ROOT, "profiles", f) for f in ("r2_traffic_csv_scan.csv", "r1_traffic_csv_scan.csv")])

    def roof(st, traffic=None):
        s = st.get("csv_scan")
        if not s or not s["launches"]:
            return None
        per_launch_bytes = s["algo_bytes"] / s["launches"]
        per_launch_ms = s["ms"] / s["launches"]
        ach = per_launch_bytes / (per_launch_ms * 1e-3) / 1e9
        return {"bound": "hbm", "kernel": "csv_scan", "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak,
                "traffic": traffic, "traffic_unit": "bytes/launch (ncu dram read+write, %s)" % traffic_src if traffic else None,
                "peak_kind": f"of {peak_kind}", "launches": s["launches"], "ms_per_launch": per_launch_ms,
                "algo_bytes_per_launch": per_launch_bytes}

    # ---------------- config 5: IndexOn(composite key) + ResolveDuplicates
    index_on = None
    if INDEX_ROWS > 0:
        side = index_sides(INDEX_ROWS)

        def index_input(n):
            return ctx.gen_csv("orders", (0, n), seed=SEED, n_cust=side, n_prod=side, header=True)

        def build(n, d):
            t, err = cp.parse_csv(ctx, d, nbytes=None, spec=INDEX_COLS)
            assert err is None and len(t) == n
            return t

        d_ix = index_input(INDEX_ROWS)
        t_ix = build(INDEX_ROWS, d_ix)

        def tail_in_group(ix):
            lo, hi = ix.dup_groups()
            return len(hi) > 0 and int(hi[-1]) == len(ix)

        # the second §Q1 shape: drop the rows of the greatest key until the last sorted row falls on the other side
        shape_a = tail_in_group(t_ix.index_on("cust_id", "prod_id"))
        t_b, cand = None, t_ix
        for _ in range(40):
            cand = without_greatest_key(cand, ("cust_id", "prod_id"))
            if tail_in_group(cand.index_on("cust_id", "prod_id")) != shape_a:
                t_b = cand
                break

        def index_step(tab):  # the reference's index IS the sorted rows: materialise them inside the timed step
            ix = tab.index_on("cust_id", "prod_id")
            ix.table()
            return ix

        ms_ix, ix_rows, st_ix, _, _, last = timed(lambda: index_step(t_ix), args.steps, args.warmup)
        dump("index_on", last.table())
        del last

        def resolve_path(tab):
            w0 = time.perf_counter()
            ix = tab.index_on("cust_id", "prod_id")
            ctx.sync(); w1 = time.perf_counter()
            lo, hi = ix.dup_groups()
            w2 = time.perf_counter()
            keep = min_id_resolver(ix.table(), lo, hi)
            w3 = time.perf_counter()
            n_before = len(ix)
            ix.dedup_apply(keep)
            ctx.sync(); w4 = time.perf_counter()
            grouped = int((hi - lo).sum())
            return {"rows": n_before, "groups": int(len(lo)), "rows_in_groups": grouped, "rows_after": len(ix),
                    "last_row_in_group": bool(len(hi) and int(hi[-1]) == n_before),
                    "ms": {"index_on": (w1 - w0) * 1e3, "dup_groups": (w2 - w1) * 1e3, "resolver_host_callback": (w3 - w2) * 1e3,
                           "dedup_apply": (w4 - w3) * 1e3}}

        resolve_path(t_ix)  # warm-up
        shapes = [resolve_path(t_ix)]
        if t_b is not None:
            shapes.append(resolve_path(t_b))
        for s in shapes:  # §Q1 (csvplus.go:851-864): a trailing singleton is lost iff at least one group exists
            lost = 0 if s["last_row_in_group"] or s["groups"] == 0 else 1
            assert s["rows_after"] == s["rows"] - s["rows_in_groups"] + s["groups"] - lost, s
        # algorithmic bytes (SURVEY §8d): R*(k + 4) + 2*P, k = mean key bytes per row, P = payload (all columns, data + offsets)
        P = 0
        for c in t_ix.columns:
            nb = C_u64()
            ctx.lib.cpb_table_col_bytes(ctx.h, t_ix.h, t_ix.columns.index(c), 0, len(t_ix), nb.ref())
            P += nb.value + 4 * (len(t_ix) + 1)
        kb = 0
        for c in ("cust_id", "prod_id"):
            nb = C_u64()
            ctx.lib.cpb_table_col_bytes(ctx.h, t_ix.h, t_ix.columns.index(c), 0, len(t_ix), nb.ref())
            kb += nb.value
        algo = kb + 4 * INDEX_ROWS + 2 * P
        index_on = {"metric": "IndexOn rows/s (configs[4]: 10 M rows, composite key cust_id,prod_id; then ResolveDuplicates)",
                    "value": INDEX_ROWS / (ms_ix * 1e-3), "unit": "rows/s", "ms_per_step": ms_ix, "rows": INDEX_ROWS,
                    "key_space": "%d x %d" % (side, side),
                    "roofline": {"bound": "hbm", "achieved": algo / (ms_ix * 1e-3) / 1e9, "peak": peak, "unit": "GB/s",
                                 "frac": algo / (ms_ix * 1e-3) / 1e9 / peak, "algo_bytes": algo,
                                 "formula": "R*(k+4) + 2*P, k = key bytes/row, P = payload (data + offsets of all 4 columns)"},
                    "kernels": {k: {"launches": v["launches"], "ms": round(v["ms"], 4)} for k, v in sorted(st_ix.items())},
                    "resolve_duplicates": shapes}
        del t_ix, t_b, d_ix

    # ---------------- end-to-end timing from pinned host buffers
    e2e = None
    parse_e2e = None
    if not args.no_e2e:
        import threading
        h_cust, h_prod, h_orders, h_people = (ctx.host_alloc(d.nbytes) for d in (d_cust, d_prod, d_orders, d_people))
        for h, d in ((h_cust, d_cust), (h_prod, d_prod), (h_orders, d_orders), (h_people, d_people)):
            ctx.lib.cpb_memcpy_d2h(ctx.h, h.ptr, d.ptr, d.nbytes)
        # e2e is a streaming pipeline, as a csvplus user would run large files: one uploader thread copies products,
        # customers and then the probe CSV in batches of complete records (pinned host -> device staging,
        # cpb_memcpy_h2d), so the H2D engine never idles; the main context parses / indexes the build sides as they
        # arrive; --e2e-workers contexts (one CUDA stream each) parse, join and serialise the probe batches and copy the
        # CSV text back (cpb_table_to_csv_into) — D2H runs on the other DMA engine, concurrently with the uploads.
        def e2e_config(nbatch, nwork):
            nbatch = max(2, nbatch)
            oview = h_orders.array()
            bounds = [0]
            for b in range(1, nbatch):
                pos = b * h_orders.nbytes // nbatch
                nl = int(np.flatnonzero(oview[pos:pos + 4096] == 10)[0])  # synthetic rows hold no quoted newlines
                bounds.append(pos + nl + 1)
            bounds.append(h_orders.nbytes)
            # sink buffer: the README's six output columns as CSV; sized from one probe batch (+ 10 %)
            t0, _ = cp.parse_csv(ctx, h_orders.ptr, nbytes=bounds[1], spec=ORDER_COLS)
            tc0, _ = cp.parse_csv(ctx, d_cust, spec=CUST_COLS)
            tp0, _ = cp.parse_csv(ctx, d_prod, spec=PROD_COLS)
            per_row = 0  # mean output bytes per joined row: the six sink columns + separators
            for tab, cols in ((t0, ("qty", "ts")), (tc0, ("name", "surname")), (tp0, ("product", "price"))):
                for c in cols:
                    nb = C_u64()
                    ctx.lib.cpb_table_col_bytes(ctx.h, tab.h, tab.columns.index(c), 0, len(tab), nb.ref())
                    per_row += nb.value / max(1, len(tab)) + 1
            del t0, tc0, tp0
            out_cap = int(ORD_ROWS * per_row * 1.05) + (1 << 20)
            h_out = ctx.host_alloc(out_cap)
            out_slots = [(b * (out_cap // nbatch)) & ~15 for b in range(nbatch)] + [out_cap]
            nwork = max(1, nwork)
            workers = [cp.Context(local) for _ in range(nwork)]
            wstreams = [torch.cuda.ExternalStream(w.stream, device=torch.device("cuda", local)) for w in workers]
            ORDER_ASSUME = [("cust_id", 1), ("prod_id", 2), ("qty", 3), ("ts", 4)]
            out_bytes = [0]

            # device staging the uploader fills (allocated once, like the pinned buffers): build sides + one 16-byte aligned
            # slot per probe batch
            up = cp.Context(local)
            dv_cust, dv_prod = up.device_alloc(h_cust.nbytes), up.device_alloc(h_prod.nbytes)
            dv_off = [0]
            for b in range(nbatch):
                dv_off.append((dv_off[-1] + (bounds[b + 1] - bounds[b]) + 255) & ~255)
            dv_orders = up.device_alloc(dv_off[-1] + 256)
            up.sync()

            DEBUG = bool(os.environ.get("BENCH_DEBUG"))

            def join_e2e():
                t_a = time.perf_counter()
                written = [0] * nbatch
                rows_out = [0] * nbatch
                ready = threading.Event()
                got_prod, got_cust = threading.Event(), threading.Event()
                got = [threading.Event() for _ in range(nbatch)]
                box = {}
                errs = []
                tmarks = {}

                def fail(ex):
                    errs.append(ex)
                    for ev in [ready, got_prod, got_cust] + got:
                        ev.set()

                def upload():  # one thread keeps the H2D engine busy from the first byte to the last
                    try:
                        up.lib.cpb_memcpy_h2d(up.h, dv_prod.ptr, h_prod.ptr, h_prod.nbytes); got_prod.set()
                        up.lib.cpb_memcpy_h2d(up.h, dv_cust.ptr, h_cust.ptr, h_cust.nbytes); got_cust.set()
                        for b in range(nbatch):
                            up.lib.cpb_memcpy_h2d(up.h, dv_orders.ptr + dv_off[b], h_orders.ptr + bounds[b], bounds[b + 1] - bounds[b])
                            got[b].set()
                        tmarks["upload_done"] = time.perf_counter() - t_a
                    except Exception as ex:
                        fail(ex)

                def work(wi):
                    try:
                        w = workers[wi]
                        for b in range(wi, nbatch, nwork):
                            got[b].wait()
                            nb = bounds[b + 1] - bounds[b]
                            if b == 0:
                                t, e = cp.parse_csv(w, dv_orders.ptr + dv_off[b], on_device=True, nbytes=nb, spec=ORDER_COLS)
                            else:
                                t, e = cp.parse_csv(w, dv_orders.ptr + dv_off[b], on_device=True, nbytes=nb, spec=ORDER_ASSUME,
                                                    header_from_first_row=False, num_fields=5)
                            assert e is None
                            ready.wait()  # the build sides are parsed / indexed concurrently on the main context
                            if errs:
                                return
                            w0 = time.perf_counter()
                            j = t.join(box["cidx"], "cust_id").join(box["pidx"])
                            rows_out[b] = len(j)
                            if DEBUG:  # (the split join / sink timing needs a sync the pipeline itself does not)
                                w.sync()
                            w1 = time.perf_counter()
                            written[b] = j.to_csv_into(h_out, out_slots[b], *SINK_COLS, header=(b == 0))
                            w2 = time.perf_counter()
                            tmarks.setdefault("join_ms", []).append((w1 - w0) * 1e3); tmarks.setdefault("sink_ms", []).append((w2 - w1) * 1e3)
                            assert out_slots[b] + written[b] <= out_slots[b + 1]
                            del j, t
                        tmarks["worker%d_done" % wi] = time.perf_counter() - t_a
                    except Exception as ex:  # surfaced by the main thread
                        fail(ex)
                th = [threading.Thread(target=upload)] + [threading.Thread(target=work, args=(i,)) for i in range(nwork)]
                for t in th:
                    t.start()
                try:
                    got_prod.wait()
                    tp, err = cp.parse_csv(ctx, dv_prod, spec=PROD_COLS)
                    assert err is None
                    pidx = tp.index_on("prod_id", unique=True)
                    got_cust.wait()
                    tc, err = cp.parse_csv(ctx, dv_cust, spec=CUST_COLS)
                    assert err is None
                    if world > 1:
                        tc = allgather_table_nccl(ctx, tc)
                    cidx = tc.index_on("id", unique=True)
                    warm, _ = cp.parse_csv(ctx, b"cust_id,prod_id\n0,0\n")
                    warm.join(cidx, "cust_id").join(pidx)  # builds the probe tables once, before the workers share the indices
                    ctx.sync()
                    box["cidx"], box["pidx"] = cidx, pidx
                    ready.set()
                except Exception as ex:
                    fail(ex)
                t_b = time.perf_counter()
                for t in th:
                    t.join()
                if errs:
                    raise errs[0]
                out_bytes[0] = sum(written)
                if DEBUG:
                    print("e2e step: build %.1f ms, probe+sink tail %.1f ms; upload done %.1f, workers done %.1f / %.1f; per batch join %.1f sink %.1f ms"
                          % ((t_b - t_a) * 1e3, (time.perf_counter() - t_b) * 1e3, tmarks.get("upload_done", 0) * 1e3, min(v for k, v in tmarks.items() if k.startswith("worker")) * 1e3,
                             max(v for k, v in tmarks.items() if k.startswith("worker")) * 1e3, sum(tmarks.get("join_ms", [0])) / max(1, len(tmarks.get("join_ms", [0]))),
                             sum(tmarks.get("sink_ms", [0])) / max(1, len(tmarks.get("sink_ms", [0])))), file=sys.stderr)
                return sum(rows_out)

            def timed_multi(fn, steps, warmup):
                for _ in range(warmup):
                    fn()
                for w in [ctx] + workers:
                    w.sync()
                torch.cuda.synchronize()
                if world > 1:
                    dist.barrier()
                e0 = torch.cuda.Event(enable_timing=True)
                ends = [torch.cuda.Event(enable_timing=True) for _ in range(1 + len(wstreams))]
                e0.record(stream)
                rows = 0
                for _ in range(steps):
                    rows = fn()
                ends[0].record(stream)
                for e, ws in zip(ends[1:], wstreams):
                    e.record(ws)
                for w in [ctx] + workers:
                    w.sync()
                torch.cuda.synchronize()
                ms = max(e0.elapsed_time(e) for e in ends)
                if world > 1:
                    dist.barrier()
                    tms = torch.tensor([ms], device="cuda", dtype=torch.float64)
                    dist.all_reduce(tms, op=dist.ReduceOp.MAX)
                    ms = float(tms.item())
                return ms / steps, rows

            ms, rows = timed_multi(join_e2e, args.steps, args.warmup)
            first = bytes(h_out.array()[:64])
            for w in workers + [up]:
                w.sync()
            return ms, rows, out_bytes[0], first, nbatch, nwork

        # --e2e-sweep "8x4,16x8": time several (batches x workers) settings, report the best one (stderr lists them all)
        configs = [(args.e2e_batches, args.e2e_workers)]
        if args.e2e_sweep:
            configs = [tuple(int(x) for x in c.split("x")) for c in args.e2e_sweep.split(",")]
        best = None
        for nb_, nw_ in configs:
            r = e2e_config(nb_, nw_)
            if rank == 0 and len(configs) > 1:
                print("e2e sweep: batches %d workers %d -> %.1f ms/step" % (r[4], r[5], r[0]), file=sys.stderr)
            if best is None or r[0] < best[0]:
                best = r
        ms_e2e, e2e_rows, out_bytes_best, first, nbatch, nwork = best
        assert e2e_rows == out_rows, (e2e_rows, out_rows)
        # the sink really holds the result: header + one line per joined row
        assert first.startswith(b"name,surname,qty,product,price,ts\n"), first
        e2e = {"value": world * ORD_ROWS / (ms_e2e * 1e-3), "unit": "rows/s", "ms_per_step": ms_e2e,
               "h2d_bytes_per_step": h_cust.nbytes + h_prod.nbytes + h_orders.nbytes, "d2h_bytes_per_step": out_bytes_best,
               "batches": nbatch, "workers": nwork, "host_numa_node": numa_node, "sink": "ToCsv(%s)" % ",".join(SINK_COLS),
               "note": "pinned host CSV -> H2D (one uploader, cpb_memcpy_h2d) -> parse/index/join/join/ToCsv on the GPU through the "
                       "public API -> D2H of the CSV text of every joined row into pinned host memory; the probe file is streamed "
                       "in %d batches of complete records over %d contexts so H2D, compute and D2H overlap" % (nbatch, nwork)}
        ms_pe2e = timed(lambda: parse_step(h_people), args.steps, args.warmup)[0]
        parse_e2e = {"value": world * h_people.nbytes / (ms_pe2e * 1e-3) / 1e9, "unit": "GB/s", "ms_per_step": ms_pe2e,
                     "h2d_bytes_per_step": h_people.nbytes}

    # ---------------- CPU baseline beside it (rank 0, N=1 only)
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        v, dt, sample = cpu_join3_sample(args.ref_orders, args.ref_customers, args.ref_products, ctx=ctx)
        pg, pr, pdt, _ = cpu_parse_sample(4_000_000, ctx)
        iv, it_sort, it_dedup, _ = cpu_index_sample(1_000_000, ctx)
        cpu = {"value": v, "unit": "rows/s", "cores": 1, "kind": "port", "seconds": dt,
               "sample": sample + "; C++ restatement proxy of the Go reference (single-threaded like it), host cores: %d" % (os.cpu_count() or 0),
               "csv_parse": {"value": pg, "unit": "GB/s", "rows_per_s": pr, "sample": "people 4 M rows, parse+select+filter, 1 thread"},
               "index_on": {"value": iv, "unit": "rows/s", "sort_seconds": it_sort, "resolve_seconds": it_dedup,
                            "sample": "1 M rows, IndexOn(cust_id,prod_id) + ResolveDuplicates(min order_id), 1 thread"}}

    sys.stdout.flush()
    os.dup2(saved_stdout, 1)
    if rank == 0:
        kernel_ms = sum(v["ms"] for k, v in st_join.items() if not k.startswith(("h2d", "d2h")))
        line = {
            "metric": "rows/sec end-to-end Join", "value": world * ORD_ROWS / (ms_join * 1e-3), "unit": "rows/s",
            "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_join, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
            "config": dict(workload_config(world), pool_reserved_bytes=reserve_b if reserved else 0),
            "clocks": clocks, "gpu_launches": launches, "out_rows_per_gpu": out_rows,
            "kernel_ms_per_step": kernel_ms / args.steps, "host_gap_ms_per_step": ms_join - kernel_ms / args.steps,
            "host_syncs_per_step": join_syncs, "per_step_ms_rank0": join_per_step,
            "e2e": e2e,
            "roofline": roof(st_join, traffic if world == 1 else None),
            "csv_parse": {"metric": "CSV parse GB/s (configs[1]: parse+SelectColumns(name,surname,id)+Filter(Like name=Amelia))",
                          "value": world * d_people.nbytes / (ms_parse * 1e-3) / 1e9, "unit": "GB/s", "ms_per_step": ms_parse,
                          "rows_per_s": world * PEOPLE_ROWS / (ms_parse * 1e-3), "rows_out_per_gpu": parse_rows,
                          "input_bytes_per_gpu": d_people.nbytes, "roofline": roof(st_parse), "e2e": parse_e2e},
            "index_on": index_on,
            "cpu_baseline": cpu,
            "kernels": {k: {"launches": v["launches"], "ms": round(v["ms"], 4)} for k, v in sorted(st_join.items())},
        }
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


class C_u64:
    """tiny ctypes out-parameter helper"""

    def __init__(self):
        import ctypes
        self._c = ctypes.c_uint64()
        self._ctypes = ctypes

    def ref(self):
        return self._ctypes.byref(self._c)

    @property
    def value(self):
        return self._c.value


if __name__ == "__main__":
    main()
