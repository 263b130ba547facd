"""Measurement (not a test): TPC-H Q10 at SF100 on one GPU -- lineitem / orders / nation generated in HBM, the customer table
uploaded (c_custkey / c_nationkey read back from the generated one, c_acctbal from the oracle's generator, the VARCHARs from the
oracle's generators or, with --text placeholder, seeded placeholder strings of dbgen's lengths; only the k + ties result rows
ever read the string bytes).  Prints the card, its power limit, the median and spread of kernel_ms (CUDA events) and exec_ms
over the timed executions, then one PG_TRACE=1 execution for the per-phase split (on stderr).

    python tests/q10_sf100.py [--sf 100] [--steps 20] [--warmup 3] [--text oracle|placeholder]
"""
import argparse
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def placeholder_text(n, seed=10):
    """c_address 10..40 bytes, c_phone 15, c_comment 29..116 (dbgen's lengths), cut from a seeded random letter pool"""
    import numpy as np
    rng = np.random.default_rng(seed)
    pool = bytes(rng.integers(97, 123, size=1 << 16, dtype=np.uint8))
    off = rng.integers(0, (1 << 16) - 128, size=n)

    def cut(lens):
        return np.array([pool[o:o + k] for o, k in zip(off.tolist(), lens.tolist())], dtype=object)
    return cut(rng.integers(10, 41, size=n)), cut(np.full(n, 15)), cut(rng.integers(29, 117, size=n))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sf", type=float, default=100.0)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--text", choices=["oracle", "placeholder"], default="oracle")
    a = ap.parse_args()
    import numpy as np
    from oracle import oracle as O
    from plan_b200 import _lib as L, compute as X, tpch as T
    O.build()
    L.check(L.lib().pg_init(0))
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()
    print("card: %s" % smi, flush=True)
    t0 = time.time()
    tables = T.generate_device_tables(a.sf, want=("lineitem", "orders", "customer", "nation"))
    gen = tables.pop("customer")
    custkey, nationkey = gen.read_column("c_custkey"), gen.read_column("c_nationkey")
    gen.free()
    n = len(custkey)
    t1 = time.time()
    acct = O.gen_q11_q22_columns(a.sf)["c_acctbal"]
    assert len(acct) == n
    name = np.array([b"Customer#%09d" % k for k in custkey.tolist()], dtype=object)
    if a.text == "oracle":
        cust = {"c_custkey": custkey, "c_nationkey": nationkey}
        ct = O.gen_customer_text(a.sf, cust)
        obj = lambda xs: np.array([x.encode() for x in xs], dtype=object)   # noqa: E731
        addr, phone, comment = obj(ct["c_address"]), obj(ct["c_phone"]), obj(O.comments("c_comment", range(n)))
    else:
        addr, phone, comment = placeholder_text(n)
    t2 = time.time()
    cx = {"c_custkey": custkey, "c_name": name, "c_acctbal": acct, "c_nationkey": nationkey, "c_address": addr, "c_phone": phone, "c_comment": comment}
    tables.update(T.upload_tables({"customer": cx}, schema=T.Schema(customer=T.Q10_CUSTOMER)))
    del cx, name, addr, phone, comment
    t3 = time.time()
    print("SF%g: lineitem %d rows, customer %d rows; VARCHAR columns from the %s; device generation %.1f s, customer columns %.1f s, upload %.1f s"
          % (a.sf, tables["lineitem"].rows(), n, "oracle's generators" if a.text == "oracle" else "seeded placeholders of dbgen's lengths",
             t1 - t0, t2 - t1, t3 - t2), flush=True)
    ex = X.gpuPipelineExec(T.q10_plan(), tables)
    ex.Init()
    print("explain: %s" % ex.Explain(), flush=True)
    kms, ems = [], []
    for it in range(a.warmup + a.steps):
        ex.Reset()
        chunks = X.drain(ex)
        if it >= a.warmup:
            kms.append(ex.stats.kernel_ms)
            ems.append(ex.stats.exec_ms)
    rows = X.order_limit(chunks, [])
    print("joined rows %d, groups before LIMIT %d, rows out %d" % (ex.stats.aux[1], ex.stats.aux[6], len(rows)))
    for r in rows[:3]:
        print("  " + "|".join(v.String() for v in r[:5]))

    def spread(xs):
        xs = np.array(xs)
        return "median %.3f ms, min %.3f, max %.3f, p10-p90 %.3f-%.3f" % (np.median(xs), xs.min(), xs.max(), np.percentile(xs, 10), np.percentile(xs, 90))
    print("%d timed executions after %d warm-up" % (a.steps, a.warmup))
    print("kernel_ms (CUDA events, whole pipeline): %s" % spread(kms))
    print("exec_ms (host clock around pg_plan_execute): %s" % spread(ems), flush=True)
    os.environ["PG_TRACE"] = "1"            # syncs at every mark: diagnosis only, after the timed runs
    ex.Reset()
    X.drain(ex)
    os.environ["PG_TRACE"] = "0"
    sys.stderr.flush()
    ex.Close()
    for x in tables.values():
        x.free()


if __name__ == "__main__":
    main()
