"""Measurement (not a test): TPC-H Q13 at SF100 on one GPU.  o_orderkey / o_custkey come from the device generator (read back),
the customer keys likewise; o_comment is the real generated text (tests/comment_text.py), uploaded in chunks as (blob, offsets).
Prints the card and its power limit, the median and spread of kernel_ms (CUDA events, whole pipeline), main_kernel_ms
(left_count_kernel) and exec_ms over the timed executions, the bytes the count pass must read over its kernel time, the
word-at-a-time matcher against PG_LIKE_BYTEWISE=1 (alternating executions), one PG_TRACE=1 execution for the per-phase split
(on stderr), and parity with oracle.q13.

    python tests/q13_sf100.py [--sf 100] [--steps 20] [--warmup 3] [--chunk 5000000] [--no-parity]
"""
import argparse
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

HBM_BYTES_PER_S = 7.7e12          # B200 data sheet (one GPU of an HGX B200)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sf", type=float, default=100.0)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--chunk", type=int, default=5000000)
    ap.add_argument("--no-parity", action="store_true")
    a = ap.parse_args()
    import numpy as np
    from oracle import oracle as O
    from comment_text import comment_blob
    from plan_b200 import _lib as L, compute as X, tpch as T
    O.build()
    L.check(L.lib().pg_init(0))
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()
    print("card: %s" % smi, flush=True)
    t0 = time.time()
    gen = T.generate_device_tables(a.sf, want=("orders", "customer"))
    okey, ocust = gen["orders"].read_column("o_orderkey"), gen["orders"].read_column("o_custkey")
    custkey = gen["customer"].read_column("c_custkey")
    for x in gen.values():
        x.free()
    n = len(okey)
    t1 = time.time()
    cust = X.DeviceTable.create("customer", T.Q13_CUSTOMER)
    cust.append([custkey])
    cust.seal(0)
    orders = X.DeviceTable.create("orders", T.Q13_ORDERS)
    text_bytes = 0
    for lo in range(0, n, a.chunk):
        hi = min(n, lo + a.chunk)
        blob, off = comment_blob(O, "o_comment", lo, hi)
        text_bytes += len(blob)
        orders.append([okey[lo:hi], ocust[lo:hi], (blob, off)])
        del blob, off
    orders.seal(0)
    tables = {"customer": cust, "orders": orders}
    t2 = time.time()
    ck_width = orders.column_encoding("o_custkey")[0]
    pass_bytes = text_bytes + (n + 1) * 8 + n * ck_width
    print("SF%g: orders %d rows (o_comment %.2f GB), customer %d rows; device generation + read-back %.1f s, text + upload %.1f s"
          % (a.sf, n, text_bytes / 1e9, len(custkey), t1 - t0, t2 - t1), flush=True)
    print("count pass reads %.2f GB: o_comment bytes, offsets (8 B/row), o_custkey (%d B/row stored)" % (pass_bytes / 1e9, ck_width), flush=True)

    def prepared(bytewise):
        os.environ["PG_LIKE_BYTEWISE"] = "1" if bytewise else "0"
        ex = X.gpuPipelineExec(T.q13_plan(), tables)
        ex.Init()
        os.environ["PG_LIKE_BYTEWISE"] = "0"
        return ex

    word, byte = prepared(False), prepared(True)
    print("explain: %s" % word.Explain())
    print("explain (PG_LIKE_BYTEWISE=1): %s" % byte.Explain(), flush=True)
    res = {"word": ([], [], []), "byte": ([], [], [])}
    out = {}
    for it in range(a.warmup + a.steps):
        for name, ex in (("word", word), ("byte", byte)):
            ex.Reset()
            out[name] = X.drain(ex)
            if it >= a.warmup:
                res[name][0].append(ex.stats.kernel_ms)
                res[name][1].append(ex.stats.main_kernel_ms)
                res[name][2].append(ex.stats.exec_ms)

    def spread(xs):
        xs = np.array(xs)
        return "median %.3f ms, min %.3f, max %.3f" % (np.median(xs), xs.min(), xs.max())
    print("%d timed executions after %d warm-up, word-at-a-time and byte-wise alternating" % (a.steps, a.warmup))
    for name in ("word", "byte"):
        k, m, e = res[name]
        print("[%s] kernel_ms (whole pipeline): %s" % (name, spread(k)))
        print("[%s] main_kernel_ms (left_count_kernel): %s  -> %.2f TB/s over the count pass = %.2f of 7.7 TB/s"
              % (name, spread(m), pass_bytes / (np.median(m) * 1e-3) / 1e12, pass_bytes / (np.median(m) * 1e-3) / HBM_BYTES_PER_S))
        print("[%s] exec_ms (host clock around pg_plan_execute): %s" % (name, spread(e)))
    print("byte-wise / word-at-a-time, median left_count_kernel: %.2fx" % (np.median(res["byte"][1]) / np.median(res["word"][1])))
    print("counters: build rows passing %d, rows counted %d, distinct counts %d" % (word.stats.aux[0], word.stats.aux[1], word.stats.aux[6]), flush=True)
    rows = lambda ch: [tuple(v.String() for v in r) for r in X.order_limit(ch, [(1, True), (0, True)])]   # noqa: E731
    assert rows(out["word"]) == rows(out["byte"]), "the two matchers disagree"
    os.environ["PG_TRACE"] = "1"            # syncs at every mark: diagnosis only, after the timed runs
    word.Reset()
    X.drain(word)
    os.environ["PG_TRACE"] = "0"
    sys.stderr.flush()
    if not a.no_parity:
        t3 = time.time()
        want = O.q13({"o_custkey": ocust}, len(custkey))
        ok = rows(out["word"]) == [("NULL" if c is None else str(c), str(d)) for c, d in want]
        print("parity with oracle.q13 at SF%g: %s (%d rows; oracle %.1f s)" % (a.sf, ok, len(want), time.time() - t3), flush=True)
        assert ok
    word.Close()
    byte.Close()
    for x in tables.values():
        x.free()


if __name__ == "__main__":
    main()
