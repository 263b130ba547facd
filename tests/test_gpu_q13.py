"""GPU runs of TPC-H Q13: customers LEFT JOIN orders (o_comment not like '%pending%accounts%'), count(o_orderkey) per customer,
then customers per count.  The GPU runs it as a grouped LEFT-join count: the orders are streamed once into a count per customer
row, and the outer aggregate is a histogram of those counts.  Checked against the reference's q13.txt, numpy, the tree-walking
row oracle and oracle.wildcard_match."""
import collections
import os

import numpy as np
import pytest

from comment_text import comment_blob

pytestmark = pytest.mark.gpu

GOLDEN = os.path.join(os.path.dirname(__file__), "golden")
KERNEL_OUTER = "kernel=left_count_kernel+count_hist_kernel"
KERNEL_INNER = "kernel=left_count_kernel+left_compact_kernel"


def _pack(v):
    return np.packbits(np.asarray(v, dtype=np.uint8), bitorder="little")


def _tables(cust_keys, okey, ocust, text, valid=None):
    """customer (c_custkey) and orders (o_orderkey, o_custkey, o_comment) uploaded; text: (blob, offsets) or a list of bytes;
    valid: {column: bool array} of the orders"""
    from plan_b200 import compute as X, tpch as T
    c = X.DeviceTable.create("customer", T.Q13_CUSTOMER)
    c.append([np.asarray(cust_keys, np.int32)])
    c.seal(0)
    o = X.DeviceTable.create("orders", T.Q13_ORDERS)
    vl = None if not valid else [(_pack(valid[n]) if n in valid else None) for n, *_ in T.Q13_ORDERS]
    o.append([np.asarray(okey, np.int64), np.asarray(ocust, np.int32), text], valid=vl)
    o.seal(0)
    return {"customer": c, "orders": o}


def _free(t):
    for x in t.values():
        x.free()


def _run(plan, tables, env=None):
    from plan_b200 import compute as X
    old = {k: os.environ.get(k) for k in (env or {})}
    os.environ.update(env or {})
    try:
        ex = X.gpuPipelineExec(plan, tables)
        ex.Init()
        chunks = X.drain(ex)
        stats, explain = ex.stats, ex.Explain()
        ex.Close()
    finally:
        for k, v in old.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v
    return chunks, stats, explain


def _refused(plan, tables, at_run=False):
    from plan_b200 import _lib as L, compute as X
    ex = X.gpuPipelineExec(plan, tables)
    with pytest.raises(L.PlanGpuError) as ei:
        ex.Init()
        if at_run:
            X.drain(ex)
    ex.Close()
    assert ei.value.status == L.PG_EUNSUPPORTED
    return str(ei.value)


def _val(v):
    return None if v.IsNull else int(v.String())


def _rows(chunks):
    return [tuple(_val(c.Data[i].GetValue(r)) for i in range(len(c.Data))) for c in chunks for r in range(c.Card())]


def _outer_want(counts, null_if_empty=True):
    """(c_count, custdist) rows, sorted, from the per-customer counts"""
    vals = counts if null_if_empty else np.maximum(counts, 1)
    d = collections.Counter(int(x) for x in vals)
    return _sorted([((None if k == 0 else k), n) for k, n in d.items()])


def _inner_want(keys, counts, null_if_empty=True):
    vals = counts if null_if_empty else np.maximum(counts, 1)
    return sorted((int(k), (None if v == 0 else int(v))) for k, v in zip(keys, vals))


def _counts(cust_keys, ocust, flags):
    """per customer (in cust_keys order) the number of orders with flags set; unknown customers count nowhere"""
    idx = np.searchsorted(cust_keys, ocust)
    idx = np.minimum(idx, len(cust_keys) - 1)
    ok = flags & (cust_keys[idx] == ocust) if len(cust_keys) else np.zeros(0, bool)
    return np.bincount(idx[ok], minlength=len(cust_keys))[:len(cust_keys)] if len(cust_keys) else np.zeros(0, np.int64)


def _like2(oracle, n):
    """flags of `o_comment like '%pending%accounts%'` for the first n orders (oracle/tpchgen.c tg_comments_like2)"""
    import ctypes as C
    L = oracle.lib()
    L.tg_comments_like2.argtypes = [C.c_int64, C.c_int, C.c_int64, C.c_int64, C.c_char_p, C.c_char_p, C.c_void_p]
    like = np.empty(n, np.uint8)
    seed, avg = oracle.COMMENT_STREAMS["o_comment"]
    assert L.tg_comments_like2(seed, avg, 0, n, b"pending", b"accounts", like.ctypes.data_as(C.c_void_p)) == 0
    return like


def _skey(r):
    return (r[0] is not None, r[0] or 0, r[1] if len(r) > 1 else 0)


def _sorted(rows):
    return sorted(rows, key=_skey)


@pytest.fixture(scope="module")
def sf005(pg, oracle):
    """SF0.05 customer / orders with the generated o_comment text, uploaded"""
    orders, _ = oracle.gen_orders_lineitem(0.05, lineitem_cols=[], orders_cols=["o_orderkey", "o_custkey"])
    cust = oracle.gen_customer(0.05)
    blob, off = comment_blob(oracle, "o_comment", 0, len(orders["o_orderkey"]))
    text = [bytes(blob[off[i]:off[i + 1]]) for i in range(len(off) - 1)]
    t = _tables(cust["c_custkey"], orders["o_orderkey"], orders["o_custkey"], (blob, off))
    yield t, cust["c_custkey"], orders, text
    _free(t)


def test_q13_reproduces_the_reference_golden_file_sf1(pg, oracle):
    """cases/tpch/1g/plan/q13.txt byte for byte (the NULL row included), Explain, and the counters against numpy"""
    from plan_b200 import compute as X, tpch as T
    orders, _ = oracle.gen_orders_lineitem(1.0, lineitem_cols=[], orders_cols=["o_orderkey", "o_custkey"])
    ck = oracle.gen_customer(1.0)["c_custkey"]
    blob, off = comment_blob(oracle, "o_comment", 0, len(orders["o_orderkey"]))
    t = _tables(ck, orders["o_orderkey"], orders["o_custkey"], (blob, off))
    try:
        chunks, stats, explain = _run(T.q13_plan(), t)
    finally:
        _free(t)
    got = X.rows_text(X.order_limit(chunks, [(1, True), (0, True)]), 2)
    assert got == open(os.path.join(GOLDEN, "ref_sf1_q13.txt")).read()
    assert explain == ("left-join count: groups=rows of customer; orders pass like=2-segment word search; " + KERNEL_OUTER)
    keep = _like2(oracle, len(orders["o_custkey"])) == 0
    counts = _counts(ck, orders["o_custkey"], keep)
    assert stats.aux[0] == int(keep.sum()) and stats.aux[1] == int(counts.sum())
    assert stats.aux[6] == len(np.unique(counts)) == got.count("\n") - 1


def test_inner_aggregate_alone_sf01(pg, oracle, sf01_host):
    """per-customer counts = bincount over the tg_comments_like2 flags, NULL exactly where the count is 0; count(*) gives
    max(m, 1) as the row oracle computes it"""
    from oracle import rowexec as R
    from plan_b200 import compute as X, tpch as T
    orders, ck = sf01_host["orders"], sf01_host["customer"]["c_custkey"]
    blob, off = comment_blob(oracle, "o_comment", 0, len(orders["o_orderkey"]))
    like = _like2(oracle, len(orders["o_custkey"]))
    counts = np.bincount(orders["o_custkey"][like == 0], minlength=len(ck) + 1)[1:]
    t = _tables(ck, orders["o_orderkey"], orders["o_custkey"], (blob, off))
    try:
        chunks, stats, explain = _run(T.q13_plan(outer=False), t)
        assert explain.endswith(KERNEL_INNER)
        got = _rows(chunks)
        assert sorted(got) == _inner_want(ck, counts) and stats.aux[6] == len(ck)
        assert any(v is None for _, v in got)
        # count(*) over the LEFT join: the NULL-padded row counts once
        plan = T.q13_plan(outer=False)
        plan.Info.Aggs = [X.func("count", plan.Info.Aggs[0].DataTyp)]
        chunks, _, _ = _run(plan, t)
        got = sorted(_rows(chunks))
        assert got == _inner_want(ck, counts, null_if_empty=False)
        text = [bytes(blob[off[i]:off[i + 1]]) for i in range(len(off) - 1)]
        n = 3000                                                   # the row oracle over the first customers' orders
        sel = orders["o_custkey"] <= n
        oc = {"o_orderkey": orders["o_orderkey"][sel], "o_custkey": orders["o_custkey"][sel],
              "o_comment": np.array([x for x, s in zip(text, sel) if s], dtype=object)}
        tabs = {"customer": R.table_rows({"c_custkey": ck[:n]}, T.Q13_CUSTOMER), "orders": R.table_rows(oc, T.Q13_ORDERS)}
        want = sorted((r[0], r[1]) for r in R.execute(plan, tabs))
        assert [r for r in got if r[0] <= n] == want
    finally:
        _free(t)


PATTERNS = [("%pending%accounts%", "2-segment word search"), ("%special%requests%", "2-segment word search"),
            ("%ly%final%deposits%", "3-segment word search"), ("%%pending%%accounts%%", "2-segment word search"),
            ("%accounts%", "1-segment word search"), ("%furiously%", "byte-wise wildcard match"),
            ("%pend_ng%", "byte-wise wildcard match"), ("pending%", "byte-wise wildcard match")]


@pytest.mark.parametrize("bytewise", [False, True])
@pytest.mark.parametrize("negate", [False, True])
@pytest.mark.parametrize("pattern,kind", PATTERNS)
def test_patterns_both_levels(sf005, oracle, pattern, kind, negate, bytewise):
    """LIKE and NOT LIKE, with and without PG_LIKE_BYTEWISE=1, both aggregate levels, against oracle.wildcard_match"""
    from plan_b200 import tpch as T
    t, ck, orders, text = sf005
    m = np.array([oracle.wildcard_match(pattern.encode(), x) for x in text], bool)
    keep = m if negate else ~m
    counts = _counts(ck, orders["o_custkey"], keep)
    env = {"PG_LIKE_BYTEWISE": "1" if bytewise else "0"}
    for outer in (True, False):
        plan = T.q13_plan(pattern=pattern, outer=outer)
        if negate:      # `o_comment like pattern`
            plan_scan = (plan.Children[0] if outer else plan).Children[0].Children[1]
            plan_scan.Filters[0].FunImpl = "like"
        chunks, stats, explain = _run(plan, t, env)
        want_kind = "byte-wise wildcard match" if bytewise else kind
        assert "orders pass like=" + want_kind + ";" in explain, explain
        if outer:
            assert _sorted(_rows(chunks)) == _sorted(_outer_want(counts))
        else:
            assert sorted(_rows(chunks)) == _inner_want(ck, counts)
        assert stats.aux[0] == int(keep.sum()) and stats.aux[1] == int(counts.sum())


CRAFTED = [b"", b"p", b"pending", b"accounts", b"pendingaccounts", b"xxxxxxxpending accounts", b"accounts pending",
           b"pendpendingaccounts", b"1234567pending12345accounts", b"pending\x80\xffaccounts", b"\x80\x81\x82pending accounts\xfe",
           b"pendin accounts", b"ly", b"lyly", b"lly", b"yl ly", b"l\x80ly" + b"y" * 30, b"x" * 63 + b"pending" + b"accounts",
           b"accountspending", b"pending" + b"a" * 200 + b"accounts", b"special requests", b"specialrequests", b"requests special"]


@pytest.mark.parametrize("pattern", ["%pending%accounts%", "%ly%ly%", "%special%requests%", "%pend%pending%"])
def test_crafted_strings(pg, oracle, pattern):
    """one order per customer, so each count shows one row's match: matches ending on the last byte, straddling 8-byte words,
    overlapping candidates, the second word only before the first, empty / short strings, bytes >= 0x80"""
    from plan_b200 import tpch as T
    n = len(CRAFTED)
    keys = np.arange(1, n + 1, dtype=np.int32)
    for shift in range(8):      # every alignment of the strings inside the 8-byte words
        text = [b"#" * ((i * 3 + shift) % 8) + s if i % 2 else s for i, s in enumerate(CRAFTED)]
        m = np.array([oracle.wildcard_match(pattern.encode(), x) for x in text], bool)
        t = _tables(keys, keys.astype(np.int64), keys, text)
        try:
            for neg in (False, True):
                plan = T.q13_plan(pattern=pattern, outer=False)
                if neg:
                    plan.Children[0].Children[1].Filters[0].FunImpl = "like"
                chunks, _, _ = _run(plan, t)
                keep = m if neg else ~m
                assert sorted(_rows(chunks)) == [(int(k), 1 if f else None) for k, f in zip(keys, keep)], (pattern, shift, neg)
        finally:
            _free(t)


@pytest.mark.parametrize("env", [{"PG_JOIN_NO_RANK_INDEX": "1"}, {"PG_JOIN_NO_BITMAP_BUILD": "1"}])
def test_switches_give_the_same_result(sf005, env):
    from plan_b200 import tpch as T
    t = sf005[0]
    for outer in (True, False):
        a, sa, _ = _run(T.q13_plan(outer=outer), t)
        b, sb, _ = _run(T.q13_plan(outer=outer), t, env)
        assert sorted(_rows(a), key=_skey) == sorted(_rows(b), key=_skey)
        assert list(sa.aux[:2]) == list(sb.aux[:2])


def test_edges(pg, oracle):
    """empty orders, empty customer, unknown customers, NULL o_custkey / o_orderkey, a hot customer, a preserved-side filter"""
    from plan_b200 import compute as X, tpch as T
    ck = np.arange(1, 1001, dtype=np.int32)
    none = (np.zeros(0, np.uint8), np.zeros(1, np.int64))
    t = _tables(ck, np.zeros(0, np.int64), np.zeros(0, np.int32), none)
    try:
        assert _rows(_run(T.q13_plan(), t)[0]) == [(None, 1000)]
        assert sorted(_rows(_run(T.q13_plan(outer=False), t)[0])) == [(int(k), None) for k in ck]
    finally:
        _free(t)
    t = _tables(np.zeros(0, np.int32), np.arange(5, dtype=np.int64), np.arange(5, dtype=np.int32), [b"x"] * 5)
    try:
        assert _rows(_run(T.q13_plan(), t)[0]) == []
        assert _rows(_run(T.q13_plan(outer=False), t)[0]) == []
    finally:
        _free(t)
    # unknown customers (0, 1001.., negative), NULL keys and NULL o_orderkey, a customer holding 70 001 orders
    rng = np.random.default_rng(5)
    n = 200000
    ocust = rng.integers(-50, 1100, n).astype(np.int32)
    ocust[:80000] = 7
    okey = np.arange(n, dtype=np.int64)
    v_ck = (rng.random(n) > 0.05) | (np.arange(n) < 80000)
    v_ok = (rng.random(n) > 0.05) | (np.arange(n) < 80000)
    text = [b"pending accounts" if i % 11 == 0 else b"regular" for i in range(n)]
    keep = np.array([i % 11 != 0 for i in range(n)])
    t = _tables(ck, okey, ocust, text, valid={"o_custkey": v_ck, "o_orderkey": v_ok})
    try:
        counts = _counts(ck, ocust, keep & v_ck & v_ok)
        assert counts[6] > 70000 and sorted(counts)[-2] < 1024         # the hot customer is a group of its own
        chunks, stats, _ = _run(T.q13_plan(), t)
        assert _sorted(_rows(chunks)) == _sorted(_outer_want(counts))
        assert stats.aux[0] == int(keep.sum()) and stats.aux[1] == int(counts.sum())
        assert sorted(_rows(_run(T.q13_plan(outer=False), t)[0])) == _inner_want(ck, counts)
        # count(*): NULL o_orderkey rows count too, a customer without orders counts once
        plan = T.q13_plan(outer=False)
        plan.Info.Aggs = [X.func("count", plan.Info.Aggs[0].DataTyp)]
        star = _counts(ck, ocust, keep & v_ck)
        assert sorted(_rows(_run(plan, t)[0])) == _inner_want(ck, star, null_if_empty=False)
        # a range filter on the preserved side: only customers 100..499 are groups (under both lookup builds)
        plan = T.q13_plan()
        scan = plan.Children[0].Children[0].Children[0]
        B, I = X.K.LType(X.K.LTID_BOOLEAN), X.K.IntegerType()
        scan.Filters = [X.func(">=", B, X.col(0, 0, I), X.const(100, I)), X.func("<", B, X.col(0, 0, I), X.const(500, I))]
        for env in (None, {"PG_JOIN_NO_RANK_INDEX": "1"}):
            chunks, stats, _ = _run(plan, t, env)
            assert _sorted(_rows(chunks)) == _sorted(_outer_want(counts[99:499]))
            assert stats.aux[1] == int(counts[99:499].sum())
    finally:
        _free(t)


def test_refusals(pg, oracle):
    """each refusal one GPU can reach, with its reason"""
    from plan_b200 import compute as X, tpch as T
    H, B, I = X.K.HugeintType(), X.K.LType(X.K.LTID_BOOLEAN), X.K.IntegerType()
    keys = np.arange(1, 101, dtype=np.int32)
    text = [b"x"] * 100
    t = _tables(keys, keys.astype(np.int64), keys, text)
    try:
        plan = T.q13_plan(outer=False)
        plan.Info.Aggs = [X.func("sum", H, X.col(0, 1, X.K.BigintType()))]
        assert "the per-group aggregate is not exactly one count" in _refused(plan, t)
        plan = T.q13_plan()
        plan.Info.Aggs = [X.func("sum", H, X.col(0, 1, H))]
        assert "the outer aggregate is not count(*)" in _refused(plan, t)
        plan = T.q13_plan()
        plan.Info.GroupBys = [X.col(0, 0, I)]
        assert "the outer aggregate is not grouped by the per-group count alone" in _refused(plan, t)
        plan = T.q13_plan(outer=False)
        plan.Filters = [X.func(">", B, X.col(1, 0, H), X.const(1, H))]
        assert "HAVING on the per-group count" in _refused(plan, t)
        plan = T.q13_plan()
        plan.Filters = [X.func(">", B, X.col(1, 0, H), X.const(1, H))]
        assert "HAVING on the outer aggregate" in _refused(plan, t)
        plan = T.q13_plan(outer=False)
        plan.Info.GroupBys = [X.col(0, 1, X.K.BigintType())]
        assert "the group key is not the anchor" in _refused(plan, t)
    finally:
        _free(t)
    # a nullable anchor key
    from plan_b200 import tpch as T2
    c = X.DeviceTable.create("customer", T2.Q13_CUSTOMER)
    c.append([keys], valid=[_pack(keys != 50)])
    c.seal(0)
    o = _tables(keys, keys.astype(np.int64), keys, text)
    o["customer"].free()
    o["customer"] = c
    try:
        assert "the anchor key c_custkey is nullable" in _refused(T.q13_plan(), o)
    finally:
        _free(o)
    # duplicate customers: refused when the pipeline runs
    dup = np.array([1, 2, 3, 3, 4], np.int32)
    t = _tables(dup, np.arange(5, dtype=np.int64), np.array([1, 2, 3, 4, 5], np.int32), [b"x"] * 5)
    try:
        for env in (None, {"PG_JOIN_NO_RANK_INDEX": "1"}):
            os.environ.update(env or {})
            try:
                assert "holds a key more than once" in _refused(T.q13_plan(), t, at_run=True)
            finally:
                for k in env or {}:
                    os.environ.pop(k, None)
    finally:
        _free(t)
