"""GPU runs of TPC-H Q10: a star join (lineitem x orders x customer x nation) grouped by customer ROWS.  The seven group keys
depend on the customer row (n_name through c_nationkey), four of them are VARCHARs, and ORDER BY revenue ... LIMIT is
pre-selected on the device.  Checked against the reference's q10.txt, oracle.q10 and the tree-walking row oracle."""
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

GOLDEN = os.path.join(os.path.dirname(__file__), "golden")
EVERY = 10 ** 9                       # oracle.q10's limit for "every group"


def _run(plan, tables):
    from plan_b200 import compute as X
    ex = X.gpuPipelineExec(plan, tables)
    ex.Init()
    chunks = X.drain(ex)
    stats, explain = ex.stats, ex.Explain()
    ex.Close()
    return chunks, stats, explain


def _refused(plan, tables):
    """prepare refuses the plan: returns the message"""
    from plan_b200 import _lib as L, compute as X
    ex = X.gpuPipelineExec(plan, tables)
    with pytest.raises(L.PlanGpuError) as ei:
        ex.Init()
    ex.Close()
    assert ei.value.status == L.PG_EUNSUPPORTED
    return str(ei.value)


def _customer(oracle, sf, cust):
    """the Q10 customer table from the oracle's generators (the device generator has no address / phone / comment / acctbal)"""
    ct, x22 = oracle.gen_customer_text(sf, cust), oracle.gen_q11_q22_columns(sf)
    obj = lambda xs: np.array([x.encode() for x in xs], dtype=object)   # noqa: E731
    cx = {"c_custkey": cust["c_custkey"], "c_name": cust["c_name"], "c_acctbal": x22["c_acctbal"], "c_nationkey": cust["c_nationkey"],
          "c_address": obj(ct["c_address"]), "c_phone": obj(ct["c_phone"]),
          "c_comment": obj(oracle.comments("c_comment", range(len(cust["c_custkey"]))))}
    return cx, ct, x22


def _nation(keys=range(25)):
    k = np.array(list(keys), dtype=np.int32)
    return {"n_nationkey": k, "n_name": k.astype(np.uint8)}


def _upload(host):
    from plan_b200 import tpch as T
    return T.upload_tables(host, schema=T.Schema(customer=T.Q10_CUSTOMER))


def _free(t):
    for x in t.values():
        x.free()


def _rows(chunks):
    """(c_custkey, c_name, revenue at scale 4, c_acctbal at scale 2, n_name, c_address, c_phone, c_comment): oracle.q10's rows"""
    out = []
    for c in chunks:
        k, name, rev, bal, nat, addr, ph, cm = c.Data[:8]
        for r in range(c.Card()):
            x = rev.Data[r]
            out.append((int(k.Data[r]), name.Data[r].decode(), (-1 if x["neg"] else 1) * int(x["coef"]) * 10 ** (4 - int(x["scale"])),
                        int(bal.Data[r]), nat.Dict[int(nat.Data[r])], addr.Data[r].decode(), ph.Data[r].decode(), cm.Data[r].decode()))
    return out


def _rnd2(v):
    """a scale-4 revenue as the ORDER BY compares it: Int64(2), rounded half-even to two fractional digits (v >= 0)"""
    q, r = divmod(v, 100)
    return q + 1 if r > 50 or (r == 50 and q % 2) else q


def _check_topk(got, full, limit):
    """got: the GPU rows in output order; full: every group.  ORDER BY compares revenue rounded to two digits and ties come
    out in any order: the rows above the k-th rounded key must be exactly the oracle's, the rows at the cut among its ties."""
    assert len(got) == min(limit, len(full))
    if not got:
        return
    keys = [_rnd2(r[2]) for r in got]
    assert keys == sorted(keys, reverse=True)
    cut = keys[-1]
    assert sorted(r for r in got if _rnd2(r[2]) > cut) == sorted(r for r in full if _rnd2(r[2]) > cut)
    at = [r for r in got if _rnd2(r[2]) == cut]
    assert len(set(at)) == len(at) and set(at) <= {r for r in full if _rnd2(r[2]) == cut}


@pytest.fixture(scope="module")
def q10(pg, oracle, sf01_host):
    """SF0.1 lineitem / orders (CPU generator), nation and the Q10 customer table, uploaded; oracle.q10 per date window"""
    cx, ct, x22 = _customer(oracle, 0.1, sf01_host["customer"])
    host = {"lineitem": sf01_host["lineitem"], "orders": sf01_host["orders"], "customer": cx, "nation": _nation()}
    t = _upload(host)
    cache = {}

    def full(date_lo=None, date_hi=None):
        if (date_lo, date_hi) not in cache:
            cache[(date_lo, date_hi)] = oracle.q10(sf01_host["customer"], sf01_host["orders"], sf01_host["lineitem"], x22, ct,
                                                   date_lo=date_lo, date_hi=date_hi, limit=EVERY)
        return cache[(date_lo, date_hi)]
    yield t, host, full
    _free(t)


@pytest.fixture(scope="module")
def small(pg, oracle):
    """SF0.02 host tables (CPU generator) for the variants, refusals and edges"""
    orders, line = oracle.gen_orders_lineitem(0.02)
    cust = oracle.gen_customer(0.02)
    cx, ct, x22 = _customer(oracle, 0.02, cust)
    return {"lineitem": line, "orders": orders, "customer": cx, "nation": _nation()}, cust, ct, x22


def test_q10_reproduces_the_reference_golden_file_sf1(pg, oracle):
    """cases/tpch/1g/plan/q10.txt byte for byte: SF1 lineitem / orders / nation generated in HBM, the customer table uploaded.
    The 20 rows carry negative balances and comments cut from across the text pool."""
    from plan_b200 import compute as X, tpch as T
    t = T.generate_device_tables(1.0, want=("lineitem", "orders", "nation"))
    try:
        cx, _, _ = _customer(oracle, 1.0, oracle.gen_customer(1.0))
        t.update(_upload({"customer": cx}))
        chunks, _, explain = _run(T.q10_plan(), t)
        assert "hits_star_rows_kernel" in explain
        assert X.rows_text(X.order_limit(chunks, []), 8) == open(os.path.join(GOLDEN, "ref_sf1_q10.txt")).read()
    finally:
        _free(t)


def test_q10_explain_and_counters(q10):
    """Explain names the new mode; joined rows and groups before LIMIT equal numpy counts from the oracle's columns"""
    from plan_b200 import tpch as T
    t, host, full = q10
    chunks, stats, explain = _run(T.q10_plan(), t)
    assert "groups=rows of customer (dependent keys fetched per group)" in explain
    assert "kernel=filter_hits_kernel+hits_star_rows_kernel" in explain and "top-k=device" in explain and "ROW EXCHANGE" not in explain
    orders, line = host["orders"], host["lineitem"]
    oidx = np.searchsorted(orders["o_orderkey"], line["l_orderkey"])
    od = orders["o_orderdate"][oidx]
    m = (od >= T.days(1993, 3, 1)) & (od < T.days(1993, 6, 1)) & (line["l_returnflag"] == ord("R"))
    assert stats.aux[1] == int(m.sum())
    assert stats.aux[6] == len(np.unique(orders["o_custkey"][oidx][m])) == len(full())
    _check_topk(_rows(chunks), full(), 20)


WINDOWS = {"quarter": (None, None), "no_orders": (-3650, -3000), "everything": (-3650, 20000)}


@pytest.mark.parametrize("limit", [0, 1, 20, 128, 129, 1000])
@pytest.mark.parametrize("window", list(WINDOWS))
def test_q10_top_k_matches_the_oracle(q10, window, limit):
    """limit <= 128 takes the single-message device select, 129 and 1000 the host-driven radix select"""
    from plan_b200 import tpch as T
    t, _, full = q10
    lo, hi = WINDOWS[window]
    chunks, stats, _ = _run(T.q10_plan(date_lo=lo, date_hi=hi, limit=limit), t)
    want = full(lo, hi)
    assert stats.aux[6] == len(want)
    assert (len(want) == 0) == (window == "no_orders") and (window != "everything" or len(want) > 5000)
    _check_topk(_rows(chunks), want, limit)


def test_q10_bare_aggregate_is_every_group(q10):
    from plan_b200 import tpch as T
    t, _, full = q10
    chunks, _, _ = _run(T.q10_plan(limit=None), t)
    assert sorted(_rows(chunks)) == sorted(full())


@pytest.mark.parametrize("env", ["PG_TOPK_HOST", "PG_JOIN_NO_RANK_INDEX", "PG_JOIN_NO_BITMAP_BUILD", "PG_FORCE_EXCHANGE"])
def test_q10_switches_give_the_same_result(q10, env, monkeypatch):
    from plan_b200 import tpch as T
    t, _, full = q10
    base, _, _ = _run(T.q10_plan(limit=129), t)
    monkeypatch.setenv(env, "1")
    chunks, _, explain = _run(T.q10_plan(limit=129), t)
    assert "ROW EXCHANGE" not in explain and "hits_star_rows_kernel" in explain
    assert _rows(chunks) == _rows(base) or sorted(_rows(chunks)) == sorted(_rows(base))      # ties at the cut in any order
    _check_topk(_rows(chunks), full(), 129)
    chunks, _, _ = _run(T.q10_plan(limit=None), t)
    assert sorted(_rows(chunks)) == sorted(full())


def _variant(kind):
    """the bare Q10 aggregate as avg(...) + count(*), as sum(...) + count(*), or as count(*) alone"""
    from plan_b200 import chunk as K, compute as X, tpch as T
    H = K.HugeintType()
    if kind == "avg":
        return T.q10_plan(limit=None, agg="avg")
    node = T.q10_plan(limit=None)
    cnt = X.func("count", H, node.Info.GroupBys[0])          # count(*) -> count(a non-null column), as the binder plans it
    if kind == "sum+count":
        node.Info.Aggs.append(cnt)
        node.Outputs.append(X.col(1, 1, H))
    else:                                                    # count only: the sum plane is carried as zeros nobody reads
        node.Info.Aggs = [cnt]
        node.Outputs = [o if o.ColRef[0] == 0 else X.col(1, 0, H) for o in node.Outputs]
    return node


@pytest.mark.parametrize("kind", ["avg", "sum+count", "count"])
def test_q10_variants_match_the_row_oracle(pg, oracle, small, kind):
    """avg(DECIMAL) = sum.Quo(count) bit for bit, and count(*) beside or instead of the sum, against rowexec on the same tree"""
    from oracle import rowexec as R
    from plan_b200 import tpch as T
    host = small[0]
    plan = _variant(kind)
    t = _upload(host)
    try:
        chunks, _, explain = _run(plan, t)
    finally:
        _free(t)
    assert "hits_star_rows_kernel" in explain
    tabs = {"lineitem": R.table_rows(host["lineitem"], T.LINEITEM), "orders": R.table_rows(host["orders"], T.ORDERS),
            "customer": R.table_rows(host["customer"], T.Q10_CUSTOMER), "nation": R.table_rows(host["nation"], T.NATION)}

    def norm(v):
        return (v.coef, v.scale, bool(v.neg)) if isinstance(v, R.Dec) else v
    want = sorted(tuple(norm(v) for v in r) for r in R.execute(plan, tabs))
    got = []
    for c in chunks:
        for r in range(c.Card()):
            row = []
            for v in c.Data:
                x = v.Data[r]
                if v.Dict is not None:
                    row.append(v.Dict[int(x)])
                elif isinstance(x, bytes):
                    row.append(x.decode())
                elif getattr(x, "dtype", None) is not None and x.dtype.names and "coef" in x.dtype.names:
                    row.append((int(x["coef"]), int(x["scale"]), bool(x["neg"]) and int(x["coef"]) != 0))
                elif getattr(x, "dtype", None) is not None and x.dtype.names:
                    row.append((int(x["upper"]) << 64) + int(x["lower"]))
                else:
                    row.append(int(x))
            got.append(row)
    acct = [o.ColRef for o in plan.Outputs].index((0, 2))            # c_acctbal: DECIMAL64, the raw coefficient at scale 2
    for row in got:
        row[acct] = (abs(row[acct]), 2, row[acct] < 0)
    assert len(want) > 100 and sorted(tuple(r) for r in got) == want


def test_q10_refuses_duplicate_customer_keys(pg, small):
    from plan_b200 import tpch as T
    host = dict(small[0])
    host["customer"] = {k: np.concatenate([v, v]) for k, v in host["customer"].items()}
    t = _upload(host)
    try:
        assert "build key of customer is not unique" in _refused(T.q10_plan(), t)
    finally:
        _free(t)


def test_q10_refuses_keys_without_the_anchor(pg, small):
    """without c_custkey two customers could carry equal keys and would have to merge: refused, not grouped by row"""
    from plan_b200 import compute as X, tpch as T
    node = T.q10_plan(limit=None)
    node.Info.GroupBys = node.Info.GroupBys[1:]
    node.Outputs = [X.col(0, o.ColRef[1] - 1, o.DataTyp) if o.ColRef[0] == 0 else o for o in node.Outputs if o.ColRef != (0, 0)]
    t = _upload(small[0])
    try:
        assert "anchor" in _refused(node, t)
    finally:
        _free(t)


def test_q10_refuses_a_sum_that_could_exceed_int64(pg, small):
    from plan_b200 import tpch as T
    host = dict(small[0])
    host["lineitem"] = dict(host["lineitem"], l_extendedprice=host["lineitem"]["l_extendedprice"] * 100000)
    t = _upload(host)
    try:
        assert "exceed int64" in _refused(T.q10_plan(), t)
    finally:
        _free(t)


@pytest.mark.parametrize("case", ["empty_lineitem", "empty_customer", "no_returns"])
def test_q10_empty_inputs_give_an_empty_result(pg, small, case):
    from plan_b200 import tpch as T
    host = dict(small[0])
    if case == "empty_lineitem":
        host["lineitem"] = {k: v[:0] for k, v in host["lineitem"].items()}
    elif case == "empty_customer":
        host["customer"] = {k: v[:0] for k, v in host["customer"].items()}
    else:
        host["lineitem"] = dict(host["lineitem"], l_returnflag=np.where(host["lineitem"]["l_returnflag"] == ord("R"), ord("A"),
                                                                         host["lineitem"]["l_returnflag"]).astype(host["lineitem"]["l_returnflag"].dtype))
    t = _upload(host)
    try:
        for limit in (20, None):
            chunks, stats, explain = _run(T.q10_plan(limit=limit), t)
            assert "hits_star_rows_kernel" in explain and chunks == [] and stats.aux[6] == 0
    finally:
        _free(t)


def test_q10_customers_without_a_nation_row_drop_out(pg, oracle, small):
    """INNER join: the rows of customers whose nation is missing are not joined (numpy: the same window, nation >= 5)"""
    from plan_b200 import tpch as T
    host, cust, ct, x22 = small
    host = dict(host, nation=_nation(range(5, 25)))
    t = _upload(host)
    try:
        chunks, stats, _ = _run(T.q10_plan(limit=None), t)
    finally:
        _free(t)
    full = oracle.q10(cust, host["orders"], host["lineitem"], x22, ct, limit=EVERY)
    want = [r for r in full if r[4] not in T.NATIONS[:5]]
    assert 0 < len(want) < len(full) and sorted(_rows(chunks)) == sorted(want)
    orders, line = host["orders"], host["lineitem"]
    oidx = np.searchsorted(orders["o_orderkey"], line["l_orderkey"])
    od = orders["o_orderdate"][oidx]
    m = (od >= T.days(1993, 3, 1)) & (od < T.days(1993, 6, 1)) & (line["l_returnflag"] == ord("R"))
    m &= cust["c_nationkey"][orders["o_custkey"][oidx] - 1] >= 5
    assert stats.aux[1] == int(m.sum()) and stats.aux[6] == len(want)
