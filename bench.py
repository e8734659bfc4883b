#!/usr/bin/env python
"""bench.py — headline benchmark of the hot path (contract in the task statement).

Workload (default): BASELINE.json configs[2], "TPC-H SF100 q3 (3-way hash join + sort) single B200" — the largest
single-GPU configuration the metric is quoted on — run through the operator layer (csrc/exec.cu, the C++ mirror of the
reference's GpuExec nodes) behind the C ABI:

    customer -> Filter(c_mktsegment = 'BUILDING')                       \
    orders   -> Filter(o_orderdate < 1995-03-15) -> [exchange o_custkey] -> ShuffledHashJoin -> [exchange o_orderkey] \
    lineitem -> Filter(l_shipdate > 1995-03-15)  -> [exchange l_orderkey] ------------------------> ShuffledHashJoin
             -> HashAggregate(l_orderkey, o_orderdate, o_shippriority; sum(l_extendedprice * (1 - l_discount)))
             -> TopN(10; revenue desc, o_orderdate) -> [exchange single] -> TopN(10)

At N GPUs the SAME job is strong-scaled: every rank owns 1/N of each table and the bracketed exchanges are real
hash-partitioned all-to-alls of row payloads over NVLink (fused partition -> peer-store kernel, csrc/exchange.cu).
A "step" is one pass of the whole query.  The result is asserted against the numpy restatement at every N.

value   : lineitem rows/s, whole job, input batches already resident in HBM.
e2e     : same metric through the operator layer with HOST (pinned) column batches: the H2D copies of every input batch
          (HostColumnarToGpu) and the D2H of the result are inside the timed region.
roofline: dominant kernel by CUDA-event share; achieved = algorithmic bytes (SURVEY §8d formulas) / its event time.
--impl reference: the CPU restatement of the same plan (oracle/tpch.py q3_cpu: pyarrow Acero, all host cores; no JVM/Spark
          exists in this image) on a bounded sample (the SF10 instance of the same generator).
--workload q6: the round-1 configuration (BASELINE configs[1], SF10 q6 from Parquet); also reported under `extra` at N=1.
--dump-outputs DIR: after the timed steps, rank 0 writes the result of the last timed step, one column per file, as
          DIR/<column>.npy (float64; decimals as their value, dates as days since 1970-01-01).  The inputs are seeded, so two
          builds run with the same arguments can be compared output for output.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

SF10_ROWS = 59_986_052
COLS = ["l_shipdate", "l_discount", "l_quantity", "l_extendedprice"]
# generated Parquet inputs are cached per user: a shared host's temporary directory may hold another user's cache
CACHE = os.environ.get("B2_BENCH_CACHE", os.path.join(tempfile.gettempdir(), "b2_bench_cache_%d" % os.getuid()))
NVLINK_GBS = 900.0   # NVLink 5 per direction per GPU (SURVEY §8d exchange roofline)
Q3_WORKLOAD = "TPC-H SF%g q3 (3 filters, customer JOIN orders JOIN lineitem, group-by (l_orderkey, o_orderdate, o_shippriority), top-10)"


def hbm_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


def dump_outputs(path, columns):
    """columns: {name: values} -> path/<name>.npy as float64"""
    os.makedirs(path, exist_ok=True)
    for name, vals in columns.items():
        np.save(os.path.join(path, name + ".npy"), np.asarray(vals, dtype=np.float64))


class ClockSampler:
    """SM clock + throttle reasons DURING the timed region.  NVML in a thread (a query costs microseconds, so even a 40 ms
    region at N = 8 gets dozens of samples; one is taken synchronously at start and one at stop); `nvidia-smi -lms` (first
    sample after ~50 ms) only when the NVML binding is missing."""
    Q = "index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown," \
        "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
    BITS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap"}

    def __init__(self, gpu):
        self.gpu, self.proc, self.nv, self.h = gpu, None, None, None
        self.sm, self.reasons, self.mx = [], set(), None
        self.thread, self.stop_flag = None, False

    def _nvml_sample(self):
        nv, h = self.nv, self.h
        self.sm.append(float(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)))
        try:
            r = nv.nvmlDeviceGetCurrentClocksEventReasons(h)
        except Exception:
            r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(h)
        for bit, name in self.BITS.items():
            if r & bit:
                self.reasons.add(name)

    def _loop(self):
        import time as _t
        while not self.stop_flag:
            try:
                self._nvml_sample()
            except Exception:
                return
            _t.sleep(0.002)

    def start(self):
        try:
            import pynvml as nv
            nv.nvmlInit()
            h = None
            try:
                import torch
                u = str(torch.cuda.get_device_properties(self.gpu).uuid)
                h = nv.nvmlDeviceGetHandleByUUID(("GPU-" + u if not u.startswith("GPU-") else u).encode())
            except Exception:
                h = nv.nvmlDeviceGetHandleByIndex(self.gpu)
            self.nv, self.h = nv, h
            self.mx = float(nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM))
            self._nvml_sample()
            import threading
            self.thread = threading.Thread(target=self._loop, daemon=True)
            self.thread.start()
            return
        except Exception:
            self.nv = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits", "-lms", "20"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except OSError:
            self.proc = None

    def stop(self):
        if self.nv is not None:
            self.stop_flag = True
            if self.thread:
                self.thread.join(timeout=1)
            try:
                self._nvml_sample()
            except Exception:
                pass
            return {"sm_mhz": statistics.median(self.sm) if self.sm else None, "sm_max_mhz": self.mx, "reasons": sorted(self.reasons),
                    "samples": len(self.sm), "source": "nvml"}
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            out, _ = self.proc.communicate(timeout=5)
        except Exception:
            self.proc.kill()
            out = ""
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in out.strip().splitlines():
            f = [x.strip() for x in line.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for k, nme in enumerate(names):
                if f[5 + k].lower().startswith("active"):
                    reasons.add(nme)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": sorted(reasons),
                "samples": len(sm), "source": "nvidia-smi"}


# ------------------------------------------------------------------------------------------------------------------------
# q6 (BASELINE configs[1])
def build_q6(m):
    c_ship = m.col(0, m.DATE32, nullable=False)
    c_disc, c_qty, c_price = (m.col(i, m.DECIMAL64, 12, 2, nullable=False) for i in (1, 2, 3))
    from benchdata import tpch
    pred = ((c_ship >= m.lit(tpch.Q6_DATE_LO, m.DATE32)) & (c_ship < m.lit(tpch.Q6_DATE_HI, m.DATE32)) & (c_disc >= m.lit(5, m.DECIMAL64, 3, 2))
            & (c_disc <= m.lit(7, m.DECIMAL64, 3, 2)) & (c_qty < m.lit(2400, m.DECIMAL64, 12, 2)))
    rev = c_price * c_disc
    return m.Program([pred, rev]), [(m.AGG_SUM, 0, m.DECIMAL128, 4, 35)]


# ------------------------------------------------------------------------------------------------------------------------
# q3 (BASELINE configs[2] at N = 1, strong-scaled with hash exchanges at N > 1)
Q3_SCHEMA = {
    "customer": ["c_custkey", "c_mktsegment"],
    "orders": ["o_orderkey", "o_custkey", "o_orderdate", "o_shippriority"],
    "lineitem": ["l_orderkey", "l_extendedprice", "l_discount", "l_shipdate"],
}
Q3_WIDTH = {"c_custkey": 8, "o_orderkey": 8, "o_custkey": 8, "o_orderdate": 4, "o_shippriority": 4, "l_orderkey": 8, "l_extendedprice": 8,
            "l_discount": 8, "l_shipdate": 4}


def q3_dtype(m, name):
    return {"c_custkey": (m.INT64, 0), "c_mktsegment": (m.STRING, 0), "o_orderkey": (m.INT64, 0), "o_custkey": (m.INT64, 0), "o_orderdate": (m.DATE32, 0),
            "o_shippriority": (m.INT32, 0), "l_orderkey": (m.INT64, 0), "l_extendedprice": (m.DECIMAL64, 2), "l_discount": (m.DECIMAL64, 2),
            "l_shipdate": (m.DATE32, 0)}[name]


def q3_programs(m):
    """the bound expressions of the plan, compiled once (Spark binds and compiles per plan, not per batch)"""
    from benchdata import tpch
    D = tpch.Q3_DATE
    one = m.lit(1, m.DECIMAL32, 1, 0)
    price, disc = m.col(1, m.DECIMAL64, 12, 2, nullable=False), m.col(2, m.DECIMAL64, 12, 2, nullable=False)
    return {
        "cust_pred": m.Program([m.col(1, m.STRING, nullable=False) == m.strlit(tpch.Q3_SEGMENT)]),
        "ord_pred": m.Program([m.col(2, m.DATE32, nullable=False) < m.lit(D, m.DATE32)]),
        "line_pred": m.Program([m.col(3, m.DATE32, nullable=False) > m.lit(D, m.DATE32)]),
        # pre-step projection of the aggregate over the join output [l_orderkey, l_extendedprice, l_discount, o_orderdate, o_shippriority]
        "agg_pre": m.Program([m.col(0, m.INT64, nullable=False), m.col(3, m.DATE32, nullable=False), m.col(4, m.INT32, nullable=False),
                              price * (one - disc)]),
    }


def build_q3_plan(m, E, progs, sources, comm=None, rank=0, world=1):
    """sources: {"customer": exec, "orders": exec, "lineitem": exec} yielding batches in Q3_SCHEMA column order.
    Returns (root exec, {name: exec}) — the named nodes are the operators reported per step."""
    X = (lambda child, keys: E.GpuShuffleExchangeExec(child, keys, comm, world)) if world > 1 else (lambda child, keys: child)
    n = {}
    n["filter_customer"] = E.GpuFilterExec(progs["cust_pred"], sources["customer"], output=[0])           # -> [c_custkey]
    n["filter_orders"] = E.GpuFilterExec(progs["ord_pred"], sources["orders"])                            # all 4 columns
    n["filter_lineitem"] = E.GpuFilterExec(progs["line_pred"], sources["lineitem"], output=[0, 1, 2])     # -> [l_orderkey, price, disc]
    if world > 1:
        n["exchange_customer"] = X(n["filter_customer"], [0])
        n["exchange_orders"] = X(n["filter_orders"], [1])
        n["exchange_lineitem"] = X(n["filter_lineitem"], [0])
    cust, ords, line = (n.get("exchange_" + t, n["filter_" + t]) for t in ("customer", "orders", "lineitem"))
    # orders JOIN customer on o_custkey = c_custkey -> [o_orderkey, o_orderdate, o_shippriority]
    n["join_orders_customer"] = E.GpuShuffledHashJoinExec([1], [0], m.JOIN_INNER, ords, cust, stream_out=[0, 2, 3], build_out=[])
    j1 = n["join_orders_customer"]
    if world > 1:
        n["exchange_join1"] = X(j1, [0])
        j1 = n["exchange_join1"]
    # lineitem JOIN that on l_orderkey = o_orderkey -> [l_orderkey, price, disc, o_orderdate, o_shippriority]
    n["join_lineitem_orders"] = E.GpuShuffledHashJoinExec([0], [0], m.JOIN_INNER, line, j1, stream_out=[0, 1, 2], build_out=[1, 2])
    n["coalesce"] = E.GpuCoalesceBatches(n["join_lineitem_orders"], 1 << 30)
    n["aggregate"] = E.GpuHashAggregateExec(n["coalesce"], [0, 1, 2], [(m.AGG_SUM, 3, m.DECIMAL128, 4, 36)], pre_project=progs["agg_pre"], mode="complete")
    order = [(3, 0, 0), (1, 1, 1)]     # revenue desc nulls last, o_orderdate asc nulls first
    n["topn"] = E.GpuTopN(10, order, n["aggregate"])
    root = n["topn"]
    if world > 1:
        n["exchange_topn"] = X(root, [])
        n["topn_final"] = E.GpuTopN(10, order, n["exchange_topn"])
        root = n["topn_final"]
    return root, n


def q3_rows_of(table):
    """result batch -> [(l_orderkey, revenue, o_orderdate, o_shippriority)] (the oracle's tuple order)"""
    if table is None:
        return []
    return [(r[0], r[3], r[1], r[2]) for r in table.to_rows()]


def q3_columns(rows):
    """q3 result rows -> output columns (revenue: DECIMAL(36, 4) as its value)"""
    return {"l_orderkey": [r[0] for r in rows], "revenue": [r[1] / 10**4 for r in rows], "o_orderdate": [r[2] for r in rows],
            "o_shippriority": [r[3] for r in rows]}


def q6_columns(res):
    """q6 result (unscaled DECIMAL(35, 4) sum, or None) -> output column"""
    return {"revenue": [np.nan if res is None else res / 10**4]}


def q3_host_chunks(sf, rank, world, seed=42):
    """this rank's share of the synthetic tables: {table: [chunk dict]} (numpy, generated on host threads)"""
    from concurrent.futures import ThreadPoolExecutor
    from benchdata import tpch
    out = {}
    with ThreadPoolExecutor(max_workers=min(32, os.cpu_count() or 4)) as ex:
        for t in ("customer", "orders", "lineitem"):
            out[t] = list(ex.map(lambda i, t=t: tpch.q3_chunk(t, sf, i, seed), tpch.q3_chunks_of_rank(t, rank, world)))
    return out


def q3_host_batches(m, chunks):
    """{table: [host column lists for GpuHostBatchSource]} over the numpy chunks (no copies)"""
    out = {}
    for t, cols in Q3_SCHEMA.items():
        out[t] = []
        for ch in chunks[t]:
            out[t].append([(q3_dtype(m, c)[0], q3_dtype(m, c)[1], ch[c], None) for c in cols])
    return out


def q3_device_batches(m, chunks):
    out = {}
    for t, cols in Q3_SCHEMA.items():
        out[t] = []
        for ch in chunks[t]:
            dev = []
            for c in cols:
                dt, scale = q3_dtype(m, c)
                if dt == m.STRING:
                    dev.append(m.Column.from_string_buffers(*ch[c]))
                else:
                    dev.append(m.Column.from_numpy(ch[c], dtype=dt, scale=scale))
            out[t].append(m.Table.from_columns(dev))
    return out


def q3_input_bytes(chunks):
    b = 0
    for t, cols in Q3_SCHEMA.items():
        for ch in chunks[t]:
            for c in cols:
                b += (ch[c][0].nbytes + ch[c][1].nbytes) if c == "c_mktsegment" else ch[c].nbytes
    return b


def run_reference(args, rank, world):
    """CPU arm: rank 0 only.  q3 on the SF`--ref-sf` instance of the same generator (bounded sample), pyarrow on all cores."""
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    if args.workload == "q6":
        from benchdata import tpch as gen
        from oracle import tpch
        raw = gen.lineitem_q6_parquet(args.rows, 42, CACHE)
        for _ in range(args.warmup):
            res = tpch.q6_cpu(raw, cores)
        t0 = time.perf_counter()
        for _ in range(args.steps):
            res = tpch.q6_cpu(raw, cores)
        dt = time.perf_counter() - t0
        outputs = q6_columns(res)
        rows, name, cfg = args.rows, "tpch_q6_rows_per_sec", {"workload": "TPC-H SF10 q6 (scan+filter+agg), Parquet source (snappy, dictionary, INT64 decimals)", "rows": args.rows, "result": res}
        sample = "full %d-row partition per step; pyarrow %d threads (CPU restatement, NOT Spark)" % (rows, cores)
    else:
        from benchdata import tpch as gen
        from oracle import tpch   # the CPU arm IS the restatement (no JVM/Spark on the box)
        sf = args.ref_sf
        tabs = tpch.q3_arrow_tables(sf, 42, threads=min(32, cores))
        rows = gen.q3_rows(sf)["lineitem"]
        for _ in range(min(args.warmup, 1)):
            res = tpch.q3_cpu(*tabs, threads=cores)
        t0 = time.perf_counter()
        for _ in range(args.steps):
            res = tpch.q3_cpu(*tabs, threads=cores)
        dt = time.perf_counter() - t0
        outputs = q3_columns(res)
        name = "tpch_q3_rows_per_sec"
        cfg = {"workload": Q3_WORKLOAD % args.sf, "sf": args.sf, "cpu_plan": "pyarrow Acero on all host cores over the SF%g instance of the same generator (bounded sample)" % sf,
               "sample_sf": sf, "lineitem_rows_per_step": rows, "result_top1": res[0] if res else None}
        sample = "SF%g instance of the synthetic q3 tables (%d lineitem rows) per step, columns cached in host memory; pyarrow Acero on %d threads " \
                 "(CPU restatement, NOT Spark)" % (sf, rows, cores)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, outputs)
    val = rows * args.steps / dt
    line = {"impl": "reference", "metric": name, "value": val, "unit": "rows/s", "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1000 * dt / args.steps, "higher_is_better": True, "scaling": "strong" if args.workload == "q3" else "weak",
            "vs_baseline": None, "dtype": "int64/decimal128", "data": "synthetic", "config": cfg,
            "cpu_baseline": {"value": val, "unit": "rows/s", "cores": cores, "kind": "port", "sample": sample},
            "e2e": {"value": val, "unit": "rows/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200")
    ap.add_argument("--workload", default="q3", choices=["q3", "q6"])
    ap.add_argument("--sf", type=float, default=100.0, help="q3: TPC-H scale factor (default: SF100)")
    ap.add_argument("--ref-sf", type=float, default=10.0, help="q3 CPU arm / cpu_baseline: scale factor of the bounded sample")
    ap.add_argument("--rows", type=int, default=SF10_ROWS, help="q6: lineitem rows per GPU (default: SF10)")
    ap.add_argument("--cpu-baseline", type=int, default=1)
    ap.add_argument("--extra-q6", type=int, default=1, help="q3 at N=1: also report the SF10 q6 step under `extra`")
    ap.add_argument("--check", type=int, default=1, help="assert the result against the numpy restatement")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None, help="write the last timed step's result columns to DIR/<column>.npy")
    args = ap.parse_args()
    if args.steps is None:
        args.steps = 10 if args.workload == "q3" else 30
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.sf == int(args.sf):
        args.sf = int(args.sf)
    if args.ref_sf == int(args.ref_sf):
        args.ref_sf = int(args.ref_sf)
    rank = int(os.environ.get("RANK", "0")); world = int(os.environ.get("WORLD_SIZE", "1")); local = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    if args.warmup < 3:
        args.warmup = 3
    # stdout carries exactly one JSON line: anything a library prints (NCCL's version banner) goes to stderr
    sys.stdout.flush()
    saved_stdout = os.dup(1)
    os.dup2(2, 1)

    import torch  # plumbing only: rendezvous, barrier, max-over-ranks
    import torch.distributed as dist
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    import spark_rapids_b200 as m
    comm = None
    if args.workload == "q6":
        m.init(local, 8 << 30)
    else:
        m.init(local, int(min(64, max(8, args.sf * 0.5 / world + 8))) << 30)   # Rmm.initialize analogue: pre-grown stream-ordered pool
    if world > 1:
        uid = [m.Comm.unique_id() if rank == 0 else None]
        dist.broadcast_object_list(uid, src=0)
        comm = m.Comm(uid[0], rank, world)

    def barrier():
        m.sync(); torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        m.sync()

    def max_over_ranks(ms):
        if world > 1:
            tt = torch.tensor([ms], device="cuda"); dist.all_reduce(tt, op=dist.ReduceOp.MAX); return float(tt.item())
        return ms

    ctx = {"args": args, "rank": rank, "world": world, "local": local, "m": m, "comm": comm, "barrier": barrier, "max_over_ranks": max_over_ranks, "dist": dist}
    line = bench_q6(ctx) if args.workload == "q6" else bench_q3(ctx)
    if rank == 0:
        sys.stdout.flush()
        os.dup2(saved_stdout, 1)
        print(json.dumps(line), flush=True)
        os.dup2(2, 1)
    if comm:
        comm.close()
    if world > 1:
        dist.destroy_process_group()


# ------------------------------------------------------------------------------------------------------------------------
def bench_q3(ctx):
    args, rank, world, local, m, comm = ctx["args"], ctx["rank"], ctx["world"], ctx["local"], ctx["m"], ctx["comm"]
    barrier, max_over_ranks = ctx["barrier"], ctx["max_over_ranks"]
    from benchdata import tpch
    from spark_rapids_b200 import execs as E
    sf = args.sf
    rows_all = tpch.q3_rows(sf)
    t_gen = time.perf_counter()
    chunks = q3_host_chunks(sf, rank, world)
    gen_s = time.perf_counter() - t_gen
    in_bytes = q3_input_bytes(chunks)
    dev = q3_device_batches(m, chunks)      # `value` leg: the input batches are resident in HBM
    progs = q3_programs(m)

    def plan(resident):
        if resident:
            src = {t: E.GpuBatchSource(dev[t]) for t in Q3_SCHEMA}
        else:
            hb = q3_host_batches(m, chunks)
            src = {t: E.GpuHostBatchSource(hb[t]) for t in Q3_SCHEMA}
        return build_q3_plan(m, E, progs, src, comm, rank, world)

    def step(resident):
        root, nodes = plan(resident)
        out = root.collect()
        return q3_rows_of(out), nodes     # to_rows(): D2H of the result

    def timed(resident, steps, profile=False):
        barrier()
        if profile:
            m.profile_enable(True)
        l0 = m.kernel_launch_count()
        e0, e1 = m.Event(), m.Event()
        w0 = time.perf_counter()
        e0.record()
        ops = {} if profile else None
        for _ in range(steps):
            res, nodes = step(resident)
            if profile:   # per-operator device time of this step (the step already ended in the D2H of its result)
                for name, node in nodes.items():
                    self_ms, _ = node.device_time()
                    mt = node.metrics
                    o = ops.setdefault(name, {"ms": 0.0, "rows_out": 0, "batches": 0})
                    o["ms"] += self_ms; o["rows_out"] += mt["numOutputRows"]; o["batches"] += mt["numOutputBatches"]
            del nodes
        e1.record()
        m.sync()
        ms = e0.elapsed_ms(e1)
        wall = (time.perf_counter() - w0) * 1000
        launches = m.kernel_launch_count() - l0
        prof = m.profile_report() if profile else None
        if profile:
            for o in ops.values():
                o["ms"] /= steps; o["rows_out"] //= steps; o["batches"] //= steps
            m.profile_enable(False)
        barrier()
        return max_over_ranks(ms), wall, launches, prof, ops, res

    for _ in range(args.warmup):
        res_w, _ = step(True)
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    ms, wall, launches, prof, ops, res = timed(True, args.steps, profile=True)
    clocks = sampler.stop() if rank == 0 else None
    if rank == 0 and args.dump_outputs:
        dump_outputs(args.dump_outputs, q3_columns(res))
    xstats0 = comm.stats() if comm else None
    # e2e: pinned host batches -> HostColumnarToGpu inside the timed region
    pinned = []
    for t, cols in Q3_SCHEMA.items():
        for ch in chunks[t]:
            for c in cols:
                for a in (ch[c] if c == "c_mktsegment" else (ch[c],)):
                    if a.nbytes:
                        m.host_register(a); pinned.append(a)
    for _ in range(2):
        step(False)
    ms_e2e, wall_e2e, _, _, _, res_e2e = timed(False, args.steps)
    for a in pinned:
        m.host_unregister(a)

    exch = None
    if comm:
        st = comm.stats()
        sent = [None] * world
        ctx["dist"].all_gather_object(sent, st["bytes_sent"])
        exch = {"bytes_sent_per_step_all_ranks": int(sum(sent) / (args.warmup + 2 * args.steps + 2)), "path": "fused partition->peer-store (NVLink)" if st["arena_bytes"] else "NCCL grouped send/recv",
                "arena_bytes": st["arena_bytes"]}
    if rank != 0:
        return None
    assert res_w == res and res_e2e == res, ("q3 result differs between steps", res_w, res, res_e2e)
    n_line = rows_all["lineitem"]
    value = n_line * args.steps / (ms / 1000)
    e2e = n_line * args.steps / (ms_e2e / 1000)
    peak, peak_src = hbm_peak()

    # ---- per-operator rows/s and roofline (algorithmic bytes: SURVEY §8d config 3 formulas; rank 0's share at N > 1)
    share = 1.0 / world
    def rows_in(t):
        return rows_all[t] * share
    r = {k: v["rows_out"] for k, v in ops.items()}
    K = 8
    alg = {
        "filter_customer": rows_in("customer") * (8 + 4 + 10) + r["filter_customer"] * 8,          # key + offsets + ~10 chars read, key written
        "filter_orders": rows_in("orders") * 24 + r["filter_orders"] * 24,
        "filter_lineitem": rows_in("lineitem") * 28 + r["filter_lineitem"] * 24,
    }
    b1 = r.get("exchange_customer", r["filter_customer"]); s1 = r.get("exchange_orders", r["filter_orders"]); m1 = r["join_orders_customer"]
    b2 = r.get("exchange_join1", m1); s2 = r.get("exchange_lineitem", r["filter_lineitem"]); m2 = r["join_lineitem_orders"]
    # join: build B*(k+4) table write + B*k read; probe S*k read + M*8 maps; gather M*(8 + 2*W)
    alg["join_orders_customer"] = b1 * (K + 4) + b1 * K + s1 * K + m1 * 8 + m1 * (8 + 2 * 16)
    alg["join_lineitem_orders"] = b2 * (K + 4) + b2 * K + s2 * K + m2 * 8 + m2 * (8 + 2 * 32)
    g = r["aggregate"]
    alg["aggregate"] = m2 * (16 + 16) + g * (16 + 16)        # N*(k+v) read + G*(k+v) written, k = 8+4+4, v = 2 x dec64 in / dec128 out
    alg["topn"] = g * (16 + 4)
    in_rows = {"filter_customer": rows_in("customer"), "filter_orders": rows_in("orders"), "filter_lineitem": rows_in("lineitem"),
               "join_orders_customer": s1, "join_lineitem_orders": s2, "aggregate": m2, "topn": g}
    operators = []
    for name, o in ops.items():
        ent = {"name": name, "ms_per_step": o["ms"], "rows_out": o["rows_out"], "batches": o["batches"]}
        if name in in_rows and o["ms"] > 0:
            ent["rows_in"] = int(in_rows[name]); ent["rows_per_sec"] = in_rows[name] / (o["ms"] / 1000)
        if name in alg and o["ms"] > 0:
            ent["alg_GBps"] = alg[name] / 1e9 / (o["ms"] / 1000); ent["hbm_frac"] = ent["alg_GBps"] / peak
        if name.startswith("exchange") and exch and o["ms"] > 0:
            ent["note"] = "device time incl. the header all-gather wait for the slowest rank"
        operators.append(ent)
    operators.sort(key=lambda e: -e["ms_per_step"])
    # ---- per-kernel shares; the dominant kernel's roofline
    tot_k = sum(k["ms"] for k in prof) or 1.0
    # algorithmic bytes per kernel NAME, summed over the step (the kernels are shared by the operators)
    kalg = {
        "filter_kernel": alg["filter_customer"] + alg["filter_orders"] + alg["filter_lineitem"],
        "join_build_kernel": (b1 + b2) * (K + 4 + K),
        "join_probe_distinct_kernel": (s1 + s2) * K + (m1 + m2) * 8,
        "join_probe_distinct1_kernel": (s1 + s2) * K + (m1 + m2) * 8,      # S*k read + M*8 maps written (SURVEY 8d)
        # selection vectors: the predicate column (DATE32) read + 4 B per selected row written
        "simple_filter_ids_kernel": (rows_in("orders") + rows_in("lineitem")) * 4 + (r["filter_orders"] + r["filter_lineitem"]) * 4,
        "filter_staged_kernel": alg["filter_customer"],
        "radix_rows_kernel": m2 * (32 + 28),                                 # join output row in, packed (hash, key, value) row out
        "part_scatter2_kernel": 2 * m2 * 28 * 2,                             # two 8-bit passes, each reads and writes 28 B per row
        "radix_agg_kernel": alg["aggregate"],
        "gather_fixed_kernel": m1 * (4 + 2 * 16) + m2 * (4 + 2 * 24) + m2 * (4 + 2 * 8) + g * (4 + 2 * 16),
        "aggregate_global_kernel": alg["aggregate"], "aggregate_smem_kernel": alg["aggregate"],
        "xchg_scatter_kernel": (r.get("filter_customer", 0) * 8 + r.get("filter_orders", 0) * 24 + m1 * 16 + r.get("filter_lineitem", 0) * 24) * 2,
    }
    kernels = []
    for k in prof:
        per = k["ms"] / max(1, k["launches"])
        ent = {"name": k["name"], "launches_per_step": k["launches"] / args.steps, "ms_per_launch": per, "ms_per_step": k["ms"] / args.steps, "share": k["ms"] / tot_k}
        if k["name"] in kalg and k["ms"] > 0:
            ent["alg_bytes_per_step"] = kalg[k["name"]]
            ent["alg_GBps"] = kalg[k["name"]] / 1e9 / (k["ms"] / args.steps / 1000)
        kernels.append(ent)
    kernels.sort(key=lambda e: -e["share"])
    dom = next((k for k in kernels if "alg_GBps" in k), kernels[0] if kernels else {"name": None})
    traffic = None
    try:
        tj = json.load(open(os.path.join(ROOT, "profiles", "r2_ncu_q3_traffic.json")))
        if sf == 100 and world == 1:
            traffic = tj[dom["name"]]["traffic_bytes_per_launch"]
    except Exception:
        traffic = None
    lp = max(1.0, dom.get("launches_per_step", 1.0))
    roof = {"bound": "hbm", "kernel": dom["name"], "achieved": dom.get("alg_GBps", 0.0), "peak": peak, "unit": "GB/s", "frac": dom.get("alg_GBps", 0.0) / peak,
            "traffic": traffic, "algorithmic_bytes": dom.get("alg_bytes_per_step", 0) / lp, "launches_per_step": dom.get("launches_per_step"),
            "traffic_source": "profiles/r2_ncu_q3_traffic.json (dram__bytes_read.sum + dram__bytes_write.sum per launch)" if traffic else None,
            "peak_source": peak_src, "note": "dominant kernel by CUDA-event share of the step among the kernels with a §8d byte formula; achieved = "
                                              "algorithmic bytes of all its launches in a step / their summed event time; per-kernel list in `kernels`"}
    line = {"metric": "tpch_q3_rows_per_sec", "value": value, "unit": "rows/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms / args.steps, "query_sec": ms / args.steps / 1000, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "int64/decimal128", "data": "synthetic",
            "config": {"workload": Q3_WORKLOAD % sf,
                       "sf": sf, "rows": rows_all, "input_bytes_per_gpu": int(in_bytes), "batches_per_gpu": {t: len(chunks[t]) for t in chunks},
                       "l2": "inputs larger than L2 (%.1f GB of input columns per GPU per step)" % (in_bytes / 1e9),
                       "result_top1": res[0] if res else None, "datagen_s": gen_s,
                       "parallelism": ("%d GPUs, strong scaling: 1/%d of every table per rank, hash exchange on the join keys" % (world, world)) if world > 1 else "1 GPU"},
            "e2e": {"value": e2e, "unit": "rows/s", "h2d_bytes_per_step": int(in_bytes) * world, "d2h_bytes_per_step": 10 * 32, "ms_per_step": ms_e2e / args.steps,
                    "note": "host column batches (pinned) -> HostColumnarToGpu -> same plan; result rows copied back"},
            "gpu_launches": int(launches), "wall_ms_per_step": wall / args.steps, "clocks": clocks, "roofline": roof, "operators": operators, "kernels": kernels[:12]}
    if exch:
        xms = sum(o["ms"] for n, o in ops.items() if n.startswith("exchange"))
        exch["exchange_ms_per_step_rank0"] = xms
        per_gpu = exch["bytes_sent_per_step_all_ranks"] / world
        exch["GBps_per_gpu"] = per_gpu / 1e9 / (xms / 1000) if xms > 0 else None
        exch["nvlink_frac"] = exch["GBps_per_gpu"] / NVLINK_GBS if exch["GBps_per_gpu"] else None
        line["exchange"] = exch
    if args.check:
        from oracle import tpch as cpu    # checker: the only use of oracle/ in this arm besides cpu_baseline
        t0 = time.perf_counter()
        expect = cpu.q3_expected(sf, 42, threads=min(16, os.cpu_count() or 4))
        line["config"]["check_s"] = time.perf_counter() - t0
        assert [(x[1], x[2]) for x in res] == [(x[1], x[2]) for x in expect], ("q3 order (revenue desc, o_orderdate) differs from the numpy restatement", res, expect)
        assert sorted(res) == sorted(expect), ("q3 result differs from the numpy restatement", res, expect)
        line["config"]["checked"] = "result == numpy restatement over all %d lineitem rows (oracle/tpch.py q3_numpy)" % n_line
    if args.cpu_baseline:
        from oracle import tpch as cpu
        cores = os.cpu_count() or 1
        rsf = min(args.ref_sf, sf)
        tabs = cpu.q3_arrow_tables(rsf, 42, threads=min(32, cores))
        cres = cpu.q3_cpu(*tabs, threads=cores)
        t0 = time.perf_counter(); reps = 2
        for _ in range(reps):
            cres = cpu.q3_cpu(*tabs, threads=cores)
        dt = (time.perf_counter() - t0) / reps
        if rsf == sf and args.check:
            assert cres == expect, ("CPU plan disagrees with the numpy restatement", cres, expect)
        crows = tpch.q3_rows(rsf)["lineitem"]
        line["cpu_baseline"] = {"value": crows / dt, "unit": "rows/s", "cores": cores, "kind": "port",
                                "sample": "SF%g instance of the same generator (%d lineitem rows), %d reps, columns cached in host memory; pyarrow Acero filter/join/group-by/top-k "
                                          "on %d threads (CPU restatement, NOT Spark)" % (rsf, crows, reps, cores)}
    if args.extra_q6 and world == 1:
        try:
            dev.clear()
            line["extra"] = {"tpch_sf10_q6": extra_q6(m, args)}
        except Exception as ex:  # the headline must survive a failure of the extra leg
            line["extra"] = {"tpch_sf10_q6": {"error": repr(ex)[:300]}}
    return line


def extra_q6(m, args):
    """BASELINE configs[1] (round 1's headline): SF10 q6 from Parquet, bytes resident in HBM, 5 steps"""
    from benchdata import tpch
    raw = tpch.lineitem_q6_parquet(SF10_ROWS, 42, CACHE)
    devb = m.DeviceBuffer(raw.nbytes + 64)
    devb.copy_from_host(raw)
    prog, spec = build_q6(m)

    def step():
        t = m.parquet_decode_device(raw, devb.ptr, COLS)
        return m.scan_aggregate(prog, True, t, [], spec).to_rows()[0][0]
    for _ in range(3):
        res = step()
    m.sync()
    e0, e1 = m.Event(), m.Event()
    e0.record()
    for _ in range(5):
        res = step()
    e1.record(); m.sync()
    ms = e0.elapsed_ms(e1) / 5
    from oracle import tpch as cpu
    assert res == cpu.q6_numpy_chunks(tpch.lineitem_q6_chunks(SF10_ROWS, 42)), "q6 result mismatch"
    return {"ms_per_step": ms, "rows_per_sec": SF10_ROWS / (ms / 1000), "rows": SF10_ROWS, "parquet_bytes": int(raw.nbytes), "checked": True}


# ------------------------------------------------------------------------------------------------------------------------
def bench_q6(ctx):
    """round-1 workload: weak-scaled SF10 q6 from Parquet per GPU (kept for `--workload q6`)"""
    args, rank, world, local, m, comm = ctx["args"], ctx["rank"], ctx["world"], ctx["local"], ctx["m"], ctx["comm"]
    barrier, max_over_ranks = ctx["barrier"], ctx["max_over_ranks"]
    from benchdata import tpch
    rows = args.rows
    raw = tpch.lineitem_q6_parquet(rows, 42 + rank, CACHE)
    nbytes = raw.nbytes
    m.host_register(raw)
    dev = m.DeviceBuffer(nbytes + 64)
    dev.copy_from_host(raw)
    prog, spec = build_q6(m)

    def step(resident, dev_ptr=None):
        if dev_ptr is not None:
            t = m.parquet_decode_device(raw, dev_ptr, COLS)
        else:
            t = m.parquet_decode_device(raw, dev.ptr, COLS) if resident else m.parquet_decode(raw, COLS)
        part = m.scan_aggregate(prog, True, t, [], spec)
        if comm is not None:
            got, _ = comm.exchange_hash(part, [])            # SinglePartition -> rank 0 owns the final aggregate
            part = m.reduce(got, [(m.AGG_SUM, 0, m.DECIMAL128, 4, 35)]) if got is not None and got.num_rows else part
        return part.to_rows()[0][0]

    def timed(resident, steps, profile=False):
        barrier()
        if profile:
            m.profile_enable(True)
        l0 = m.kernel_launch_count()
        e0, e1 = m.Event(), m.Event()
        w0 = time.perf_counter()
        e0.record()
        if resident:
            for _ in range(steps):
                res = step(True)
        else:
            nxt = m.AsyncUpload(raw)
            for k in range(steps):
                cur, nxt = nxt, (m.AsyncUpload(raw) if k + 1 < steps else None)
                res = step(False, cur.wait())
                cur.free()
        e1.record()
        m.sync()
        ms = e0.elapsed_ms(e1)
        wall = (time.perf_counter() - w0) * 1000
        launches = m.kernel_launch_count() - l0
        prof = m.profile_report() if profile else None
        if profile:
            m.profile_enable(False)
        barrier()
        return max_over_ranks(ms), wall, launches, prof, res

    for _ in range(args.warmup):
        res_w = step(True)
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    ms, wall, launches, prof, res = timed(True, args.steps, profile=True)
    clocks = sampler.stop() if rank == 0 else None
    if rank == 0 and args.dump_outputs:
        dump_outputs(args.dump_outputs, q6_columns(res))
    for _ in range(2):
        step(False)
    ms_e2e, wall_e2e, _, _, res_e2e = timed(False, args.steps)
    # the merged result at N > 1: every rank's partition is checked on rank 0 against the exact integer restatement
    expect_all = None
    if world > 1 and args.check:
        from oracle import tpch as cpu
        mine = cpu.q6_numpy_chunks(tpch.lineitem_q6_chunks(rows, 42 + rank))
        allv = [None] * world
        ctx["dist"].all_gather_object(allv, mine)
        expect_all = sum(v for v in allv if v is not None)
    if rank != 0:
        return None
    total_rows = rows * world
    value = total_rows * args.steps / (ms / 1000)
    e2e = total_rows * args.steps / (ms_e2e / 1000)
    peak, peak_src = hbm_peak()
    tot_k = sum(k["ms"] for k in prof) or 1.0
    st = m.parquet_last_stats()
    alg = {"snappy_kernel": st["compressed_in"] + st["decompressed_out"], "values_kernel": st["page_bytes"] + st["column_bytes"],
           "aggregate_smem_kernel": rows * 28.0}
    kernels = []
    for k in prof:
        per = k["ms"] / max(1, k["launches"])
        ent = {"name": k["name"], "launches_per_step": k["launches"] / args.steps, "ms_per_launch": per, "share": k["ms"] / tot_k}
        if k["name"] in alg:
            ent["alg_GBps"] = alg[k["name"]] / 1e9 / (per / 1000)
        kernels.append(ent)
    kernels.sort(key=lambda e: -e["share"])
    dom = kernels[0] if kernels else {"name": None, "alg_GBps": 0.0}
    traffic = None
    try:
        if rows == SF10_ROWS:
            traffic = json.load(open(os.path.join(ROOT, "profiles", "r1_ncu_sf10_traffic.json")))[dom["name"]]["traffic_bytes_per_launch"]
    except Exception:
        traffic = None
    roof = {"bound": "hbm", "kernel": dom["name"], "achieved": dom.get("alg_GBps", 0.0), "peak": peak, "unit": "GB/s",
            "frac": dom.get("alg_GBps", 0.0) / peak, "traffic": traffic, "algorithmic_bytes": alg.get(dom["name"]),
            "traffic_source": "profiles/r1_ncu_sf10_traffic.json (dram__bytes_read.sum + dram__bytes_write.sum, one launch)" if traffic else None,
            "peak_source": peak_src, "note": "dominant kernel by CUDA-event share of the step; per-kernel list in `kernels`"}
    line = {"metric": "tpch_q6_rows_per_sec", "value": value, "unit": "rows/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms / args.steps, "query_sec": ms / args.steps / 1000, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "int64/decimal128", "data": "synthetic",
            "config": {"workload": "TPC-H SF10 q6 (scan+filter+agg), Parquet source (snappy, dictionary, INT64 decimals)", "rows_per_gpu": rows,
                       "parquet_bytes_per_gpu": int(nbytes), "l2": "inputs larger than L2 (parquet %.0f MB + 1.68 GB decoded per step)" % (nbytes / 1e6),
                       "result_unscaled_dec25_4": res, "parallelism": "partition per GPU, exchange of partial aggregates" if world > 1 else "1 GPU"},
            "e2e": {"value": e2e, "unit": "rows/s", "h2d_bytes_per_step": int(nbytes) * world, "d2h_bytes_per_step": 16 * world,
                    "ms_per_step": ms_e2e / args.steps},
            "parquet_stats": st, "gpu_launches": int(launches), "wall_ms_per_step": wall / args.steps, "clocks": clocks, "roofline": roof, "kernels": kernels[:8]}
    assert res_w == res and res_e2e == res, ("q6 result differs between steps", res_w, res, res_e2e)
    if expect_all is not None:
        assert res == expect_all, ("merged q6 result differs from the exact restatement over every rank's partition", res, expect_all)
    if args.cpu_baseline:
        from oracle import tpch as cpu
        cores = os.cpu_count() or 1
        cpu.q6_cpu(raw, cores)
        t0 = time.perf_counter(); reps = 2
        for _ in range(reps):
            cres = cpu.q6_cpu(raw, cores)
        dt = (time.perf_counter() - t0) / reps
        if world == 1:
            assert cres == res, ("CPU restatement disagrees with the GPU result", cres, res)
            if rows <= SF10_ROWS and args.check:
                expect = cpu.q6_numpy_chunks(tpch.lineitem_q6_chunks(rows, 42 + rank))
                assert res == expect, ("q6 result mismatch", res, expect)
        line["cpu_baseline"] = {"value": rows / dt, "unit": "rows/s", "cores": cores, "kind": "port",
                                "sample": "one full %d-row partition, %d reps; pyarrow scan+compute on %d threads (CPU restatement, NOT Spark)" % (rows, reps, cores)}
    return line


if __name__ == "__main__":
    main()
