import os, sys, time, numpy as np, torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from plan_b200 import _lib as L, compute as X, tpch as T, chunk as K
sf = float(sys.argv[1])
lib = L.lib(); L.check(lib.pg_init(0))
tables = T.generate_device_tables(sf)
need = {"lineitem": ["l_quantity", "l_extendedprice", "l_discount", "l_tax", "l_returnflag", "l_linestatus", "l_shipdate", "l_orderkey"],
        "orders": ["o_orderkey", "o_custkey", "o_orderdate", "o_shippriority"], "customer": ["c_custkey", "c_mktsegment"]}
schemas = {"lineitem": T.LINEITEM, "orders": T.ORDERS, "customer": T.CUSTOMER}
host = {}; nbytes = 0
for tname, cols in need.items():
    host[tname] = {}
    for cdef in schemas[tname]:
        if cdef[0] in cols:
            dt_ = np.dtype(K.native_dtype(cdef[1])); n = tables[tname].rows()
            pinned = torch.empty(max(n, 1) * dt_.itemsize, dtype=torch.uint8, pin_memory=True)
            arr = pinned.numpy()[:n * dt_.itemsize].view(dt_)
            ci = [c[0] for c in schemas[tname]].index(cdef[0])
            L.check(lib.pg_table_read_column(tables[tname].handle, ci, 0, n, arr.ctypes.data))
            host[tname][cdef[0]] = (arr, pinned); nbytes += n * dt_.itemsize
sub = T.FULL.pruned(need)
plans = {"q6": T.q6_plan(schema=sub), "q1": T.q1_plan(schema=sub), "q3": T.q3_topk_plan(schema=sub)}
for it in range(3):
    ts = [time.perf_counter()]
    tabs = {}
    for tname in need:
        t = X.DeviceTable.create(tname, sub.tables[tname]); tabs[tname] = t
    ts.append(time.perf_counter())
    for tname in need:
        tabs[tname].append([host[tname][c[0]][0] for c in sub.tables[tname]])
    ts.append(time.perf_counter())
    for tname in need:
        tabs[tname].seal(0)
    tabs["customer"].set_replicated()
    ts.append(time.perf_counter())
    for q, p in plans.items():
        ex = X.gpuPipelineExec(p, tabs); ex.Init(); X.drain(ex); ex.Close()
    ts.append(time.perf_counter())
    for t in tabs.values(): t.free()
    ts.append(time.perf_counter())
    d = [1e3 * (b - a) for a, b in zip(ts, ts[1:])]
    print("iter %d: create %.1f append %.1f (%.1f GB/s) seal %.1f queries %.1f free %.1f total %.1f ms" % (it, d[0], d[1], nbytes / d[1] / 1e6, d[2], d[3], d[4], sum(d)))
