#!/usr/bin/env python
"""bench.py -- TPC-H Q1/Q6/Q3 lineitem rows/s + HBM roofline fraction at SF100 on N B200s.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--sf 100] [--queries q6,q1,q3] [--dump-outputs DIR]
  python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...
  python bench.py --impl reference ...      # the reference's CPU path (oracle port) on host cores

A "step" = one execution of every query of the workload over the (row-range sharded)
SF100 tables resident in HBM.  `value` = lineitem rows scanned by all queries of a step,
over all ranks, per second (barrier + device sync on both sides, max over ranks).
`e2e` = the same with HOST column buffers: pg_table_create/append/seal (H2D) + execute +
result fetch inside the timed region.  `roofline` is for the dominant kernel (the Q1
scan): algorithmic bytes / CUDA-event duration measured by the library on its own stream.
One JSON line on stdout (rank 0).
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

LINEITEM_ROWS_PER_SF = 6_000_000   # nominal; the exact generated count is reported


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--sf", type=float, default=100.0)
    ap.add_argument("--queries", default="q6,q1,q3")
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--e2e-steps", type=int, default=2)
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--e2e-native", action="store_true", help="e2e leg with native-width host buffers (int64 DECIMALs) instead of narrow ones")
    ap.add_argument("--no-extra", action="store_true", help="skip the Q18 / group-by timings reported beside the metric")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-chunked-e2e", action="store_true", help="skip the 2048-row-chunk pageable-memory e2e leg (C++ host shim subprocess)")
    ap.add_argument("--cpu-sample-sf", type=float, default=None,
                    help="CPU sample: this SF worth of rows (default: 4 for the cpu_baseline leg, 10 for --impl reference, shrunk to fit the time bound)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the result columns of the last timed step as DIR/<query>_col<i>.npy (float64), so that two builds "
                         "can be compared output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the results of the GPU path (--impl ours)")
    return args


def measured_peak_gbs():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, device):
        self.device, self.proc, self.path = device, None, None

    def start(self):
        try:
            fd, self.path = tempfile.mkstemp(suffix=".csv")
            os.close(fd)
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.device), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=open(self.path, "w"), stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if not self.proc:
            return out
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, reasons, smax = [], set(), None
        for line in open(self.path):
            f = [x.strip() for x in line.split(",")]
            if len(f) < 8:
                continue
            try:
                sm.append(float(f[1]))
                smax = float(f[2])
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        os.unlink(self.path)
        if sm:
            sm.sort()
            out.update(sm_mhz=sm[len(sm) // 2], sm_max_mhz=smax, reasons=sorted(reasons), samples=len(sm))
        return out


# ----------------------------------------------------------------------------------------
# parity: every bench run re-checks its own results (untimed) against the committed fixtures
# ----------------------------------------------------------------------------------------

GOLDEN = os.path.join(ROOT, "tests", "golden")
# query -> (ORDER BY applied by the host parents that stay in Go, number of columns)
PARITY_RENDER = {"q6": ([], 1), "q1": ([(0, False), (1, False)], 10), "q3": ([], 4), "q9": ([], 3), "q18": ([], 6)}


def parity_fixture(q, sf):
    """Path of the committed oracle result for query q at this scale factor, or None.  The fixtures were
    produced once on the CPU by tests/golden/make_sf100*_fixture*.py (the oracle over the same dbgen-equivalent
    data); bench.py only reads the text files, it never runs the oracle in this arm."""
    if sf != int(sf):
        return None
    p = os.path.join(GOLDEN, "oracle_sf%d_%s.txt" % (int(sf), q))
    return p if os.path.exists(p) else None


def parity_check(X, q, chunks, sf):
    """True / False (byte-for-byte equality of the rendered rows with the fixture) or None (no fixture)."""
    fx = parity_fixture(q, sf)
    if fx is None or q not in PARITY_RENDER:
        return None
    order, ncols = PARITY_RENDER[q]
    return X.rows_text(X.order_limit(chunks, order), ncols) == open(fx).read()


# ----------------------------------------------------------------------------------------
# --dump-outputs: the result columns of the last timed step, as numbers
# ----------------------------------------------------------------------------------------

DUMP_LIMIT_BYTES = 64 << 20


def column_values(vec):
    """One result vector as float64: DECIMAL / HUGEINT records as their numeric value, codes of CHAR / DICT columns as
    numbers, NULL as NaN."""
    import numpy as np
    d = vec.Data
    if d.dtype.names == ("coef", "scale", "neg"):
        x = d["coef"].astype(np.float64) / 10.0 ** d["scale"].astype(np.float64)
        x = np.where(d["neg"] != 0, -x, x)
    elif d.dtype.names == ("lower", "upper"):
        x = d["upper"].astype(np.float64) * 2.0 ** 64 + d["lower"].astype(np.float64)
    else:
        x = d.astype(np.float64)
    if vec.Mask is not None:
        valid = np.unpackbits(vec.Mask, bitorder="little")[:len(x)].astype(bool)
        x = np.where(valid, x, np.nan)
    return x


def dump_outputs(path, results):
    """results: {query: (chunks, number of result columns)}.  Rows are put in the order of the host ORDER BY that stays in
    Go (PARITY_RENDER), so that the files do not depend on the order in which the device emitted groups.  Above
    DUMP_LIMIT_BYTES in all, every query keeps the same fixed, seeded sample fraction of its rows."""
    import numpy as np
    cols = {}
    for q, (chunks, ncols) in results.items():
        qc = [np.concatenate([column_values(c.Data[i]) for c in chunks]) if chunks else np.zeros(0) for i in range(ncols)]
        order = PARITY_RENDER.get(q, ([], 0))[0]
        if order and qc and len(qc[0]):
            idx = np.lexsort([-qc[i] if desc else qc[i] for i, desc in reversed(order)])
            qc = [c[idx] for c in qc]
        cols[q] = qc
    total = sum(c.nbytes for qc in cols.values() for c in qc)
    rng = np.random.default_rng(0)
    os.makedirs(path, exist_ok=True)
    for q, qc in cols.items():
        n = len(qc[0]) if qc else 0
        if total > DUMP_LIMIT_BYTES:
            keep = np.sort(rng.choice(n, n * DUMP_LIMIT_BYTES // total, replace=False))
            qc = [c[keep] for c in qc]
        for i, c in enumerate(qc):
            np.save(os.path.join(path, "%s_col%d.npy" % (q, i)), c)


# ----------------------------------------------------------------------------------------
# reference arm: the reference's own CPU implementation of the path = the oracle port
# ----------------------------------------------------------------------------------------

def cpu_reference_run(queries, sample_sf, steps, warmup):
    """Time the C restatement of the reference executor (oracle/refexec.c), single thread
    (the reference executes on one goroutine), on a bounded dbgen-equivalent sample."""
    from oracle import oracle as O
    O.build()
    orders, line = O.gen_orders_lineitem(sample_sf)
    cust = O.gen_customer(sample_sf)
    nline = len(line["l_orderkey"])

    def step():
        for q in queries:
            if q == "q6":
                O.q6(line)
            elif q == "q1":
                O.q1(line)
            elif q == "q3":
                O.q3(cust, orders, line, capacity=16)
    for _ in range(warmup):
        step()
    per_q = {}
    t0 = time.perf_counter()
    for _ in range(steps):
        for q in queries:
            t = time.perf_counter()
            {"q6": lambda: O.q6(line), "q1": lambda: O.q1(line),
             "q3": lambda: O.q3(cust, orders, line, capacity=16)}[q]()
            per_q[q] = per_q.get(q, 0.0) + (time.perf_counter() - t)
    dt = time.perf_counter() - t0
    rows = nline * len(queries) * steps
    return {"rows_per_s": rows / dt, "ms_per_step": dt / steps * 1e3, "lineitem_rows": nline,
            "per_query_rows_per_s": {q: nline * steps / per_q[q] for q in queries}}


def run_reference_arm(args, queries):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    sample_sf = min(args.cpu_sample_sf if args.cpu_sample_sf else 10.0, args.sf)
    steps, warmup = max(1, args.steps), max(0, args.warmup)          # the same warm-up as our arm
    # bound the whole run to a few minutes: ~3.2-4 s per SF1 step for q6+q1+q3 on one core (the reference executes on one
    # goroutine), plus ~2.5 s per SF1 to generate the sample
    while (steps + warmup) * sample_sf * 4.0 + sample_sf * 2.5 > 400 and sample_sf > 0.05:
        sample_sf /= 2
    r = cpu_reference_run(queries, sample_sf, steps, warmup)
    sample = "dbgen-equivalent SF%g sample (%d lineitem rows) of the SF%g workload, per step" % (
        sample_sf, r["lineitem_rows"], args.sf)
    line = {
        "impl": "reference", "metric": "tpch_q1_q6_q3_lineitem_rows_per_s", "value": r["rows_per_s"],
        "unit": "rows/s", "n_gpus": args.gpus, "steps": steps, "warmup": warmup, "ms_per_step": r["ms_per_step"],
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "int64/decimal(19)",
        "data": "synthetic (dbgen-equivalent generator, in-box)",
        "config": {"workload": "TPC-H " + "+".join(q.upper() for q in queries) + " at SF%g" % args.sf,
                   "queries": queries, "sf": args.sf, "sample": sample, "kind": "port",
                   "implementation": "oracle/refexec.c: C restatement of the reference's Go executor for this path, 2048-row chunks, "
                                     "govalues-equivalent decimals, 1 thread (the Go toolchain is absent on the box)"},
        "cpu_baseline": {"value": r["rows_per_s"], "unit": "rows/s", "cores": 1, "kind": "port", "sample": sample,
                         "note": "C restatement of the reference's single-goroutine executor (no Go toolchain on "
                                 "the box); per query: " + json.dumps(r["per_query_rows_per_s"])},
        "e2e": {"value": r["rows_per_s"], "unit": "rows/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


# ----------------------------------------------------------------------------------------
# our arm
# ----------------------------------------------------------------------------------------

def main():
    args = parse_args()
    queries = [q.strip() for q in args.queries.split(",") if q.strip()]
    if args.impl == "reference":
        run_reference_arm(args, queries)
        return

    import numpy as np
    import torch
    import torch.distributed as dist

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus and world > 1:
        raise SystemExit("WORLD_SIZE %d != --gpus %d" % (world, args.gpus))
    torch.cuda.set_device(local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    from plan_b200 import _lib as L
    from plan_b200 import compute as X
    from plan_b200 import tpch as T
    import ctypes as C
    lib = L.lib()
    L.check(lib.pg_init(local_rank))
    if world > 1:
        from plan_b200 import dist as D
        D.init_comm(lib, L.check)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def min_over_ranks(x):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MIN)
        return float(t.item())

    def sum_over_ranks(x):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        return float(t.item())

    # ---- data: this rank's contiguous order range, generated in HBM -------------------------
    n_orders = lib.pg_tpch_num_orders(args.sf)
    o_lo, o_hi = n_orders * rank // world, n_orders * (rank + 1) // world
    want = ["lineitem"] + (["orders", "customer"] if "q3" in queries else [])
    t_gen = time.perf_counter()
    tables = T.generate_device_tables(args.sf, o_lo, o_hi, want=tuple(want))
    if "customer" in tables:
        tables["customer"].set_replicated()        # small dimension table: whole copy on every rank
    gen_s = time.perf_counter() - t_gen
    local_rows = tables["lineitem"].rows()
    total_rows = int(sum_over_ranks(float(local_rows)))

    # Q3 runs with its ORDER BY revenue desc, o_orderdate LIMIT 10 tail fused (device top-k), which is
    # the query BASELINE names; Q1/Q6 return their few groups to the host Order/Project parents
    plans = {"q6": T.q6_plan, "q1": T.q1_plan, "q3": lambda **kw: T.q3_topk_plan(10, **kw)}
    execs = {}
    for q in queries:
        ex = X.gpuPipelineExec(plans[q](), tables)
        ex.Init()
        execs[q] = ex

    def run_query(q):
        ex = execs[q]
        ex.Reset()
        chunks = X.drain(ex)
        return chunks, ex.stats

    def step(acc=None):
        results = {}
        for q in queries:
            chunks, st = run_query(q)
            results[q] = chunks
            if acc is not None:
                a = acc.setdefault(q, {"kernel_ms": 0.0, "main_ms": 0.0, "exec_ms": 0.0, "launches": 0, "n": 0,
                                       "bytes": st.algorithmic_bytes, "main_bytes": st.main_kernel_bytes})
                a["kernel_ms"] += st.kernel_ms
                a["main_ms"] += st.main_kernel_ms
                a["exec_ms"] += st.exec_ms
                a["launches"] += st.kernel_launches
                a["n"] += 1
        return results

    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
        t_wait = time.perf_counter()          # nvidia-smi needs a moment before its first sample
        while time.perf_counter() - t_wait < 3.0 and not (os.path.exists(sampler.path) and os.path.getsize(sampler.path) > 0):
            time.sleep(0.05)
    for _ in range(max(args.warmup, 3)):
        step()
    acc = {}
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        last = step(acc)
    barrier()
    dt = max_over_ranks(time.perf_counter() - t0)
    # the timed region can be a few milliseconds: keep the same steps running (untimed) until the
    # 100 ms sampler has seen the GPU under this load a few times
    t_keep = time.perf_counter()
    while time.perf_counter() - t_keep < 0.6:
        step()
    clocks = sampler.stop() if rank == 0 else None
    if clocks is not None:
        clocks["note"] = "sampled every 100 ms from warm-up through the timed steps and 0.6 s of the same steps after"
    ms_per_step = dt / args.steps * 1e3
    value = total_rows * len(queries) * args.steps / dt
    if rank == 0 and args.dump_outputs:
        dump_outputs(args.dump_outputs, {q: (last[q], len(execs[q].coltypes)) for q in queries})

    # ---- parity (untimed): the results of THIS run, on every rank, against the committed fixtures --------
    def all_ranks_agree(flag):
        """None stays None; otherwise True only if every rank's rendered result equals the fixture."""
        if flag is None:
            return None
        return bool(min_over_ranks(1.0 if flag else 0.0) > 0.5)

    parity = {}
    for q in queries:
        chunks, _ = run_query(q)
        parity[q] = all_ranks_agree(parity_check(X, q, chunks, args.sf))

    # ---- roofline of the dominant kernel (largest share of device time) ---------------------
    peak, peak_src = measured_peak_gbs()
    per_query = {}
    for q in queries:
        a = acc[q]
        main_ms = max_over_ranks(a["main_ms"] / a["n"])
        kern_ms = max_over_ranks(a["kernel_ms"] / a["n"])
        exec_ms = max_over_ranks(a["exec_ms"] / a["n"])
        gbs = a["main_bytes"] / (a["main_ms"] / a["n"] * 1e-3) / 1e9 if a["main_ms"] > 0 else 0.0
        per_query[q] = {"rows_per_s": total_rows / (exec_ms * 1e-3), "exec_ms": exec_ms, "kernel_ms": kern_ms,
                        "main_kernel_ms": main_ms, "main_kernel_bytes": a["main_bytes"],
                        "achieved_gbs_per_gpu": gbs, "frac_of_measured_peak": gbs / peak}
    dom = max(queries, key=lambda q: per_query[q]["main_kernel_ms"])
    roofline = {"bound": "hbm", "achieved": per_query[dom]["achieved_gbs_per_gpu"], "peak": peak, "unit": "GB/s",
                "frac": per_query[dom]["achieved_gbs_per_gpu"] / peak, "traffic": None,
                "kernel": execs[dom].Explain().split(" kernel=")[1].split(" ")[0] if " kernel=" in execs[dom].Explain() else dom,
                "query": dom, "peak_source": peak_src,
                "algorithmic_bytes_per_launch": per_query[dom]["main_kernel_bytes"],
                "avg_launch_ms": per_query[dom]["main_kernel_ms"]}
    # DRAM traffic of the dominant kernel: ncu's dram bytes per launch relative to the algorithmic bytes,
    # from the committed capture of the same kernel (profiles/traffic_ratio.json), scaled to this launch
    try:
        tr = json.load(open(os.path.join(ROOT, "profiles", "traffic_ratio.json")))
        for kname, info in tr["kernels"].items():
            if kname in roofline["kernel"]:
                roofline["traffic"] = info["ratio"] * roofline["algorithmic_bytes_per_launch"]
                roofline["traffic_source"] = tr["source"] + "; ratio %.5f applied to this launch's algorithmic bytes" % info["ratio"]
    except Exception:
        pass
    launches = sum(a["launches"] for a in acc.values())

    # ---- beside the metric (NOT part of `value`): the next queries SURVEY.md 8(d) names -----------
    also = {}
    if "q3" in queries and not args.no_extra:
        extra_tables = dict(tables)
        try:
            extra_tables.update(T.generate_device_tables(args.sf, want=("part", "supplier", "partsupp", "nation")))
            for name in ("part", "supplier", "partsupp", "nation"):
                extra_tables[name].set_replicated()
        except Exception as e:
            also["q9_tables"] = {"error": str(e)[:200]}
        extra_plans = {"q9": T.q9_plan, "q18": T.q18_plan,
                       "groupby_l_orderkey_having": lambda: T.groupby_plan(key="l_orderkey", value="l_quantity", having_gt=314, topk=100)}
        for name, mk in extra_plans.items():
            try:
                ex = X.gpuPipelineExec(mk(), extra_tables)
                ex.Init()
                for _ in range(2):
                    ex.Reset(); chunks = X.drain(ex)
                if name in PARITY_RENDER:
                    parity[name] = all_ranks_agree(parity_check(X, name, chunks, args.sf))
                tot = 0.0
                for _ in range(5):
                    barrier()
                    ex.Reset(); X.drain(ex)
                    tot += ex.stats.exec_ms
                also[name] = {"exec_ms": max_over_ranks(tot / 5), "rows_scanned_per_gpu": int(ex.stats.rows_scanned),
                              "pipeline": ex.Explain()[:160]}
                ex.Close()
            except Exception as e:      # reported, never fatal for the metric line
                also[name] = {"error": str(e)[:200]}

        # BASELINE config 5 as written: partsupp SHARDED by row range, so Q9's lineitem x partsupp join has its two sides
        # on different ranks and runs through the all-to-all hash-partitioned ROW exchange (exchange.cuh).  On one rank
        # the same path is forced (PG_FORCE_EXCHANGE) and the exchange degenerates to a device copy.
        if "partsupp" in extra_tables:
            try:
                xt = dict(extra_tables)
                if world > 1:
                    xt["partsupp"] = T.generate_device_tables(args.sf, want=("partsupp",), partsupp_shard=(rank, world))["partsupp"]
                os.environ["PG_FORCE_EXCHANGE"] = "1"
                ex = X.gpuPipelineExec(T.q9_plan(), xt)
                ex.Init()
                os.environ.pop("PG_FORCE_EXCHANGE")
                for _ in range(2):
                    ex.Reset(); chunks = X.drain(ex)
                parity["q9_row_exchange"] = all_ranks_agree(parity_check(X, "q9", chunks, args.sf))
                tot = comm = 0.0
                for _ in range(5):
                    barrier()
                    ex.Reset(); X.drain(ex)
                    tot += ex.stats.exec_ms
                    comm += ex.stats.comm_ms
                sent_b, sent_r = float(ex.stats.aux[5]), float(ex.stats.aux[7])
                comm_ms = max_over_ranks(comm / 5)
                also["q9_row_exchange"] = {"exec_ms": max_over_ranks(tot / 5), "exchange_ms": comm_ms,
                                           "rows_sent_to_other_ranks": int(sum_over_ranks(sent_r)), "bytes_sent_to_other_ranks": int(sum_over_ranks(sent_b)),
                                           "nvlink_gbs_per_rank": (sum_over_ranks(sent_b) / world) / (comm_ms * 1e-3) / 1e9 if comm_ms > 0 and world > 1 else None,
                                           "explain": "ROW EXCHANGE" in ex.Explain(), "partsupp": "row-range sharded" if world > 1 else "whole (exchange forced)"}
                ex.Close()
                if world > 1:
                    xt["partsupp"].free()
            except Exception as e:
                os.environ.pop("PG_FORCE_EXCHANGE", None)
                also["q9_row_exchange"] = {"error": str(e)[:300]}

    # ---- e2e: host buffers through the C ABI (H2D inside the timed region) -------------------
    e2e = None
    if not args.no_e2e:
        need = {"lineitem": ["l_quantity", "l_extendedprice", "l_discount", "l_tax", "l_returnflag", "l_linestatus",
                             "l_shipdate"] + (["l_orderkey"] if "q3" in queries else [])}
        if "q3" in queries:
            need["orders"] = ["o_orderkey", "o_custkey", "o_orderdate", "o_shippriority"]
            need["customer"] = ["c_custkey", "c_mktsegment"]
        schemas = {"lineitem": T.LINEITEM, "orders": T.ORDERS, "customer": T.CUSTOMER}
        # HOST buffers = the flattened column buffers the Go shim hands over: one array per column at the narrowest
        # width its value range allows (frame of reference: value = base + stored; the shim walks every vector to
        # flatten govalues Decimals / Dates anyway and so knows the range).  They are exported once, untimed, from
        # the resident tables in their stored encoding (pg_table_read_column_stored) into pinned host memory.
        host = {}
        h2d_bytes = 0
        native_bytes = 0
        for tname, cols in need.items():
            host[tname] = {}
            for cdef in schemas[tname]:
                if cdef[0] in cols:
                    dt_ = np.dtype(__import__("plan_b200.chunk", fromlist=["x"]).native_dtype(cdef[1]))
                    n = tables[tname].rows()
                    w, base = tables[tname].column_encoding(cdef[0])
                    if args.e2e_native:
                        w, base = dt_.itemsize, 0
                    pinned = torch.empty(max(n, 1) * w, dtype=torch.uint8, pin_memory=True)
                    ci = [c[0] for c in schemas[tname]].index(cdef[0])
                    if args.e2e_native:
                        L.check(lib.pg_table_read_column(tables[tname].handle, ci, 0, n, pinned.data_ptr()))
                    else:
                        L.check(lib.pg_table_read_column_stored(tables[tname].handle, ci, 0, n, pinned.data_ptr()))
                    host[tname][cdef[0]] = (pinned.data_ptr(), w if w != dt_.itemsize or base != 0 else 0, base, pinned)
                    h2d_bytes += n * w
                    native_bytes += n * dt_.itemsize
        # the e2e tables carry only the referenced columns; plans are built on that pruned schema
        sub = T.FULL.pruned(need)
        sub_schema = sub.tables
        offsets = {"lineitem": 0, "orders": o_lo, "customer": 0}
        e_plans = {q: plans[q](schema=sub) for q in queries}
        # free the resident tables' HBM is not needed: 180 GB holds both copies at SF100

        def e2e_step():
            d2h = 0
            tabs = {}
            for tname in need:
                t = X.DeviceTable.create(tname, sub_schema[tname])
                t.append_cols([host[tname][c[0]][:3] for c in sub_schema[tname]], tables[tname].rows())
                t.seal(offsets[tname])
                if tname == "customer":
                    t.set_replicated()
                tabs[tname] = t
            for q in queries:
                ex = X.gpuPipelineExec(e_plans[q], tabs)
                ex.Init()
                chunks = X.drain(ex)
                d2h += sum(v.Data.nbytes for c in chunks for v in c.Data)
                ex.Close()
            for t in tabs.values():
                t.free()
            return d2h
        e2e_step()                                  # warm-up (allocator, pinned paths)
        barrier()
        t0 = time.perf_counter()
        d2h = 0
        for _ in range(max(1, args.e2e_steps)):
            d2h = e2e_step()
        barrier()
        edt = max_over_ranks(time.perf_counter() - t0)
        e2e = {"value": total_rows * len(queries) * max(1, args.e2e_steps) / edt, "unit": "rows/s",
               "h2d_bytes_per_step": int(sum_over_ranks(float(h2d_bytes))), "d2h_bytes_per_step": int(sum_over_ranks(float(d2h))),
               "ms_per_step": edt / max(1, args.e2e_steps) * 1e3, "steps": max(1, args.e2e_steps),
               "native_width_bytes_per_step": int(sum_over_ranks(float(native_bytes))),
               "host_buffers": "native widths (int64 DECIMAL, int32 DATE/INT)" if args.e2e_native else
                               "narrow frame-of-reference column buffers (pg_table_append_cols), pinned",
               "includes": "pg_table_create+append_cols(H2D from pinned host, device widening)+seal(stats, packing)+plan compile/execute+result fetch"}

    # ---- the same e2e step the way the reference's executor would feed it (rank 0, N=1 only): 2048-row chunks from
    # PAGEABLE host memory, one pg_table_append_cols call per chunk, through the C++ host shim (plan_b200/host/
    # append_bench.cc); its Q6 / Q1 / Q3 results are checked against the same fixtures
    if e2e is not None and rank == 0 and world == 1 and not args.no_chunked_e2e and queries == ["q6", "q1", "q3"]:
        exe = os.path.join(ROOT, "plan_b200", "host", "planhost_append")
        try:
            r = subprocess.run([exe, "%g" % args.sf, "2048", "narrow", "1"], capture_output=True, text=True, timeout=600)
            if r.returncode != 0:
                raise RuntimeError(r.stderr[-300:])
            ch = json.loads(r.stdout.strip().splitlines()[-1])
            texts = {}
            for part in r.stderr.split("== ")[1:]:
                name, _, body = part.partition("\n")
                texts[name.strip()] = body
            ok = {}
            for q in ("q6", "q1", "q3"):
                fx = parity_fixture(q, args.sf)
                ok[q] = None if fx is None else (texts.get(q) == open(fx).read())
            parity["chunked_e2e"] = None if any(v is None for v in ok.values()) else all(ok.values())
            e2e["chunked_pageable"] = {"value": total_rows * 3 / (ch["ms_per_step"] * 1e-3), "unit": "rows/s", "ms_per_step": ch["ms_per_step"],
                                       "append_calls_per_step": ch["append_calls_per_step"], "chunk_rows": ch["chunk_rows"],
                                       "h2d_bytes_per_step": ch["h2d_bytes_per_step"], "host_memory": ch["host_memory"],
                                       "note": "what a per-chunk shim costs: one append call per 2048-row scan chunk from pageable memory, "
                                               "gathered in pinned staging inside the library; `e2e.value` above is the bulk export path (f2)"}
        except Exception as ex_:      # reported, never fatal for the metric line
            e2e["chunked_pageable"] = {"error": str(ex_)[:300]}

    # ---- CPU baseline beside it (rank 0, N=1 only) -------------------------------------------
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        sample_sf = min(args.cpu_sample_sf if args.cpu_sample_sf else 4.0, args.sf)
        r = cpu_reference_run(queries, sample_sf, 1, 0)
        cpu = {"value": r["rows_per_s"], "unit": "rows/s", "cores": 1, "kind": "port",
               "sample": "dbgen-equivalent SF%g sample (%d lineitem rows), one pass of %s" % (
                   sample_sf, r["lineitem_rows"], "+".join(queries)),
               "host_cores": os.cpu_count(), "per_query_rows_per_s": r["per_query_rows_per_s"]}

    if rank == 0:
        out = {
            "metric": "tpch_q1_q6_q3_lineitem_rows_per_s", "value": value, "unit": "rows/s", "n_gpus": world,
            "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": ms_per_step, "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "int64 fixed-point (128-bit merge)",
            "data": "synthetic (dbgen-equivalent TPC-H generator, in HBM)",
            "config": {"workload": "TPC-H " + "+".join(q.upper() for q in queries) + " at SF%g, lineitem/orders row-range "
                                   "sharded over %d GPU(s)" % (args.sf, world),
                       "queries": queries, "sf": args.sf, "lineitem_rows": total_rows,
                       "l2": "inputs larger than L2 (%.1f GB of columns per GPU vs 126 MB)" % (
                           per_query[dom]["main_kernel_bytes"] / 1e9),
                       "parallelism": "row-range shard x%d, NCCL all-gather merge of partial aggregates" % world},
            "parity": parity, "parity_source": "rendered rows == tests/golden/oracle_sf%g_<query>.txt byte for byte, checked on every "
                                               "rank after the timed loop (null: no fixture at this SF)" % args.sf,
            "queries": per_query, "also_measured": also, "roofline": roofline, "cpu_baseline": cpu, "e2e": e2e, "gpu_launches": launches,
            "clocks": clocks, "datagen_s": gen_s,
        }
        print(json.dumps(out))
    for ex in execs.values():
        ex.Close()
    for t in tables.values():
        t.free()
    if world > 1:
        lib.pg_comm_destroy()
        dist.destroy_process_group()
    bad = sorted(q for q, ok in parity.items() if ok is False)
    if bad:
        sys.stderr.write("bench.py: PARITY MISMATCH against tests/golden fixtures for %s\n" % ", ".join(bad))
        sys.exit(3)


if __name__ == "__main__":
    main()
