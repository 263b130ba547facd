"""CPU: the oracle (C restatement of the reference executor + dbgen-equivalent generator) is
pinned against the reference's own SF1 golden result files and known official dbgen rows."""
import os

import numpy as np
import pytest

GOLDEN = os.path.join(os.path.dirname(__file__), "golden")


@pytest.fixture(scope="module")
def sf1(oracle):
    orders, line = oracle.gen_orders_lineitem(1.0)
    return {"orders": orders, "lineitem": line, "customer": oracle.gen_customer(1.0)}


def test_generator_row_counts_match_official_dbgen(oracle):
    L = oracle.lib()
    assert L.tg_count_lineitems(1.0, 0, 1500000) == 6001215       # official SF1 lineitem cardinality
    assert L.tg_count_lineitems(10.0, 0, 15000000) == 59986052    # SF10


def test_generator_first_rows_match_official_dbgen(oracle, sf1):
    """First rows of the official SF1 lineitem.tbl / orders.tbl / customer.tbl."""
    l, o, c = sf1["lineitem"], sf1["orders"], sf1["customer"]
    d = oracle.days
    want = [  # orderkey partkey suppkey line qty extprice disc tax rf ls ship commit receipt
        (1, 155190, 7706, 1, 17, 2116823, 4, 2, "N", "O", d(1996, 3, 13), d(1996, 2, 12), d(1996, 3, 22)),
        (1, 67310, 7311, 2, 36, 4598316, 9, 6, "N", "O", d(1996, 4, 12), d(1996, 2, 28), d(1996, 4, 20)),
        (1, 63700, 3701, 3, 8, 1330960, 10, 2, "N", "O", d(1996, 1, 29), d(1996, 3, 5), d(1996, 1, 31)),
        (1, 2132, 4633, 4, 28, 2895564, 9, 6, "N", "O", d(1996, 4, 21), d(1996, 3, 30), d(1996, 5, 16)),
        (1, 24027, 1534, 5, 24, 2282448, 10, 4, "N", "O", d(1996, 3, 30), d(1996, 3, 14), d(1996, 4, 1)),
        (1, 15635, 638, 6, 32, 4962016, 7, 2, "N", "O", d(1996, 1, 30), d(1996, 2, 7), d(1996, 2, 3)),
        (2, 106170, 1191, 1, 38, 4469446, 0, 5, "N", "O", d(1997, 1, 28), d(1997, 1, 14), d(1997, 2, 2)),
        (3, 4297, 1798, 1, 45, 5405805, 6, 0, "R", "F", d(1994, 2, 2), d(1994, 1, 4), d(1994, 2, 23)),
        (3, 19036, 6540, 2, 49, 4679647, 10, 0, "R", "F", d(1993, 11, 9), d(1993, 12, 20), d(1993, 11, 24)),
        (3, 128449, 3474, 3, 27, 3989088, 6, 7, "A", "F", d(1994, 1, 16), d(1993, 11, 22), d(1994, 1, 23)),
    ]
    cols = ["l_orderkey", "l_partkey", "l_suppkey", "l_linenumber", "l_quantity", "l_extendedprice", "l_discount",
            "l_tax", "l_returnflag", "l_linestatus", "l_shipdate", "l_commitdate", "l_receiptdate"]
    for r, row in enumerate(want):
        got = tuple(chr(int(l[cn][r])) if cn in ("l_returnflag", "l_linestatus") else int(l[cn][r]) for cn in cols)
        assert got == row, (r, got, row)
    # orders.tbl: 1|36901|O|173665.47|1996-01-02 ; 2|78002|O|46929.18|1996-12-01 ; 3|123314|F|193846.25|1993-10-14
    assert [int(x) for x in o["o_orderkey"][:9]] == [1, 2, 3, 4, 5, 6, 7, 32, 33]
    assert [int(x) for x in o["o_custkey"][:3]] == [36901, 78002, 123314]
    assert [int(x) for x in o["o_totalprice"][:3]] == [17366547, 4692918, 19384625]
    assert [chr(int(x)) for x in o["o_orderstatus"][:3]] == ["O", "O", "F"]
    assert [int(x) for x in o["o_orderdate"][:3]] == [d(1996, 1, 2), d(1996, 12, 1), d(1993, 10, 14)]
    segs = [oracle.SEGMENTS[int(x)] for x in c["c_mktsegment"][:10]]
    assert segs == ["BUILDING", "AUTOMOBILE", "AUTOMOBILE", "MACHINERY", "HOUSEHOLD", "AUTOMOBILE", "AUTOMOBILE",
                    "BUILDING", "FURNITURE", "HOUSEHOLD"]


def test_generator_ranges_are_independent(oracle, sf1):
    o2, l2 = oracle.gen_orders_lineitem(1.0, 700000, 700100)
    first = int(np.searchsorted(sf1["lineitem"]["l_orderkey"], l2["l_orderkey"][0]))
    for k, v in l2.items():
        assert np.array_equal(v, sf1["lineitem"][k][first:first + len(v)]), k
    for k, v in o2.items():
        assert np.array_equal(v, sf1["orders"][k][700000:700100]), k


def test_golden_copies_are_the_reference_files():
    """the ref_sf1_* fixtures are verbatim copies of the reference's own result files (cases/tpch/1g/plan/q*.txt): their
    SHA-256 digests are stored in golden/ref_sf1_sha256.txt, in `sha256sum` format, so that the same list also checks a
    checkout of the reference (`sha256sum -c` in its cases/tpch/1g/plan)"""
    import gzip
    import hashlib
    want = {}
    for line in open(os.path.join(GOLDEN, "ref_sf1_sha256.txt")):
        digest, name = line.split()
        want[name] = digest
    assert sorted(want) == sorted("q%d.txt" % q for q in range(1, 23))
    for q in range(1, 23):
        if q == 16:
            data = gzip.open(os.path.join(GOLDEN, "ref_sf1_q16.txt.gz"), "rb").read()
        else:
            data = open(os.path.join(GOLDEN, "ref_sf1_q%d.txt" % q), "rb").read()
        assert hashlib.sha256(data).hexdigest() == want["q%d.txt" % q], q


def test_q6_reproduces_reference_golden(oracle, sf1):
    assert oracle.q6_text(oracle.q6(sf1["lineitem"])) == open(os.path.join(GOLDEN, "ref_sf1_q6.txt")).read()


def test_q1_reproduces_reference_golden(oracle, sf1):
    res = oracle.q1(sf1["lineitem"])
    assert oracle.q1_text(res) == open(os.path.join(GOLDEN, "ref_sf1_q1.txt")).read()
    assert res["rows_selected"] == 1478493 + 38854 + 2874145 + 1478870
    for g in res["groups"]:        # data-independent KATs of SURVEY.md 8c: avg = sum / count
        assert repr(g["avg_qty"]) == repr(float(g["sum_qty"]) / float(g["count_order"]))


def test_q18_reproduces_reference_golden(oracle, sf1):
    """cases/tpch/1g/plan/q18.txt: HAVING on a HUGEINT sum, SEMI join, 5-key group-by, DECIMAL sort key, LIMIT."""
    rows = oracle.q18(sf1["customer"], sf1["orders"], sf1["lineitem"])
    assert oracle.q18_text(rows) == open(os.path.join(GOLDEN, "ref_sf1_q18.txt")).read()


def test_part_supplier_partsupp_first_rows_match_official_dbgen(oracle):
    """First rows of the official SF1 part.tbl / supplier.tbl / partsupp.tbl."""
    part = oracle.gen_part(0.01)
    assert [n.decode() for n in part["p_name"][:5]] == [
        "goldenrod lavender spring chocolate lace", "blush thistle blue yellow saddle", "spring green yellow purple cornsilk",
        "cornflower chocolate smoke green pink", "forest brown coral puff cream"]
    sup = oracle.gen_supplier(1.0)
    assert list(sup["s_nationkey"][:5]) == [17, 5, 1, 15, 11] and len(sup["s_suppkey"]) == 10000
    ps = oracle.gen_partsupp(1.0)
    assert list(ps["ps_suppkey"][:5]) == [2, 2502, 5002, 7502, 3]
    assert list(ps["ps_supplycost"][:5]) == [77164, 99349, 33709, 35784, 37849] and len(ps["ps_partkey"]) == 800000


def test_q9_reproduces_reference_golden(oracle, sf1):
    """cases/tpch/1g/plan/q9.txt: 175 (nation, year) groups of a six-way join with LIKE and EXTRACT(year)."""
    line = sf1["lineitem"]
    rows = oracle.q9(oracle.gen_part(1.0, "pink"), oracle.gen_supplier(1.0), oracle.gen_partsupp(1.0), sf1["orders"], line)
    assert oracle.q9_text(rows) == open(os.path.join(GOLDEN, "ref_sf1_q9.txt")).read()


def test_q4_q12_q14_q19_reproduce_reference_golden(oracle, sf1):
    """cases/tpch/1g/plan/q4.txt, q12.txt, q14.txt and q19.txt: pin l_shipmode / o_orderpriority / p_type of the generator (dbgen streams
    L_SMODE_SD, O_PRIO_SD, P_TYPE_SD and the member order of the smode / o_oprio / p_types distributions) and, through
    Q14, the reference's float32 arithmetic above the aggregate -- the known answers the CASE / aggregate-over-join GPU
    path is checked against (tests/test_gpu_rows.py)."""
    orders, line = sf1["orders"], sf1["lineitem"]
    extra = oracle.gen_q12_q14_columns(1.0)
    assert oracle.q12_text(oracle.q12(orders, line, extra)) == open(os.path.join(GOLDEN, "ref_sf1_q12.txt")).read()
    assert oracle.q4_text(oracle.q4(orders, line, extra)) == open(os.path.join(GOLDEN, "ref_sf1_q4.txt")).read()
    r19 = oracle.q19(line, extra, oracle.gen_q19_columns(1.0))      # cases/tpch/1g/plan/q19.txt: pins p_brand / p_size / p_container / l_shipinstruct
    assert "#\n" + oracle.fmt_decimal((r19["revenue"], 4, 0), 4) + "\n" == open(os.path.join(GOLDEN, "ref_sf1_q19.txt")).read()
    r = oracle.q14(line, extra)
    assert "#\n" + oracle.q14_promo_revenue(r["promo"], r["total"]) + "\n" == open(os.path.join(GOLDEN, "ref_sf1_q14.txt")).read()


def test_q5_q7_q8_q11_q17_q21_q22_reproduce_reference_golden(oracle, sf1):
    """Seven more of the reference's SF1 result files (cases/tpch/1g/plan/q{5,7,8,11,17,21,22}.txt), byte for byte.  They pin what
    the earlier files do not reach: the c_nationkey stream (Q5 / Q7 / Q8 / Q22), l_suppkey joined to s_nationkey on the lineitem
    side (Q5 / Q7 / Q21), c_acctbal and ps_availqty (Q22, Q11), o_orderstatus and the commit / receipt dates per order (Q21),
    a DECIMAL quotient printed at scale 4 (Q8) and a DECIMAL sum divided by a FLOAT literal in float32 (Q17)."""
    orders, line, cust = sf1["orders"], sf1["lineitem"], sf1["customer"]
    supp, ps = oracle.gen_supplier(1.0), oracle.gen_partsupp(1.0)
    e12, e19, e22 = oracle.gen_q12_q14_columns(1.0), oracle.gen_q19_columns(1.0), oracle.gen_q11_q22_columns(1.0)
    # first rows of the official customer.tbl / partsupp.tbl
    assert e22["c_acctbal"][:5].tolist() == [71156, 12165, 749812, 286683, 79447]
    assert e22["ps_availqty"][:4].tolist() == [3325, 8076, 3956, 4069]
    gold = lambda q: open(os.path.join(GOLDEN, "ref_sf1_q%d.txt" % q)).read()   # noqa: E731
    dec = lambda v, s: oracle.fmt_decimal((v, s, 0), s)                          # noqa: E731
    assert oracle.rows_text(1, [(n, dec(v, 4)) for n, v in oracle.q5(cust, supp, orders, line)]) == gold(5)
    assert oracle.rows_text(3, [(a, b, y, dec(v, 4)) for a, b, y, v in oracle.q7(cust, supp, orders, line)]) == gold(7)
    assert oracle.rows_text(1, [(y, oracle.fmt_decimal(q, 4)) for y, q, _a, _b in oracle.q8(cust, supp, orders, line, e12)]) == gold(8)
    assert oracle.rows_text(1, [(k, dec(v, 2)) for k, v in oracle.q11(supp, ps, e22)]) == gold(11)
    r17 = oracle.q17(line, e19)
    assert r17["rows"] == 558 and oracle.rows_text(0, [(r17["avg_yearly"],)]) == gold(17)
    assert oracle.rows_text(1, oracle.q21(supp, orders, line)) == gold(21)
    assert oracle.rows_text(2, [(c, n, dec(v, 2)) for c, n, v in oracle.q22(cust, orders, e22)]) == gold(22)


def test_q15_q16_q20_reproduce_reference_golden(oracle, sf1):
    """cases/tpch/1g/plan/q15.txt, q16.txt (18341 rows, kept gzipped) and q20.txt (177 rows), byte for byte: they pin dbgen's
    generated supplier TEXT -- s_address (a_rnd over the 64-character alphabet, with dbgen's wrapped int32 range), s_phone, and the
    suppliers whose comment holds "Customer ... Complaints" (BBB streams) -- plus p_name prefixes and ps_availqty against the
    per-(part, supplier) shipped quantity."""
    import gzip
    line = sf1["lineitem"]
    supp, ps, part = oracle.gen_supplier(1.0), oracle.gen_partsupp(1.0), oracle.gen_part(1.0)
    e12, e19, e22, st = oracle.gen_q12_q14_columns(1.0), oracle.gen_q19_columns(1.0), oracle.gen_q11_q22_columns(1.0), oracle.gen_supplier_text(1.0)
    assert st["s_address"][0] == " N kD4on9OM Ipw3,gf0JBoQDd7tgrzrddZ" and st["s_phone"][0] == "27-918-335-1736"      # official supplier.tbl row 1
    assert (np.nonzero(st["complaint"])[0] + 1).tolist() == [358, 2820, 3804, 9504]
    gold = lambda q: open(os.path.join(GOLDEN, "ref_sf1_q%d.txt" % q)).read()   # noqa: E731
    rows = [(k, n, a, p, oracle.fmt_decimal((v, 4, 0), 4)) for k, n, a, p, v in oracle.q15(line, st)]
    assert oracle.rows_text(4, rows) == gold(15)
    assert oracle.rows_text(3, oracle.q16(ps, e12, e19, st)) == gzip.open(os.path.join(GOLDEN, "ref_sf1_q16.txt.gz"), "rt").read()
    assert oracle.rows_text(1, oracle.q20(part, supp, ps, line, e22, st)) == gold(20)


def test_q2_q10_q13_reproduce_reference_golden(oracle, sf1):
    """cases/tpch/1g/plan/q2.txt (100 rows), q10.txt (20 rows) and q13.txt, byte for byte.  Q2 / Q10 print generated addresses, phone
    numbers, signed balances and a COMMENT column; Q13 filters 1.5 M orders on `o_comment not like '%pending%accounts%'` under a LEFT
    join.  Comments are cut from dbgen's 300 MiB grammar-generated text pool, restated in oracle/tpchgen.c: the 120 printed comments
    sit at offsets spread over the whole pool and all match."""
    orders, line, cust = sf1["orders"], sf1["lineitem"], sf1["customer"]
    supp, ps = oracle.gen_supplier(1.0), oracle.gen_partsupp(1.0)
    e12, e19, e22 = oracle.gen_q12_q14_columns(1.0), oracle.gen_q19_columns(1.0), oracle.gen_q11_q22_columns(1.0)
    st, ct = oracle.gen_supplier_text(1.0), oracle.gen_customer_text(1.0, cust)
    assert ct["c_address"][0] == "IVhzIApeRb ot,c,E" and ct["c_phone"][0] == "25-989-741-2988"                # official customer.tbl row 1
    assert st["s_acctbal"][:3].tolist() == [575594, 403268, 419240]                                           # official supplier.tbl rows 1-3
    assert oracle.comments("c_comment", [0]) == ["to the even, regular platelets. regular, ironic epitaphs nag e"]    # customer.tbl row 1
    gold = lambda q: open(os.path.join(GOLDEN, "ref_sf1_q%d.txt" % q)).read()   # noqa: E731
    sdec = lambda v, s: oracle.fmt_decimal((abs(v), s, int(v < 0)), s)          # noqa: E731
    rows = [(k, n, sdec(r, 4), sdec(b, 2), nn, a, p, c) for k, n, r, b, nn, a, p, c in oracle.q10(cust, orders, line, e22, ct)]
    assert len(rows) == 20 and oracle.rows_text(7, rows) == gold(10)
    rows = [(sdec(b, 2), sn, nn, p, mf, a, ph, c) for b, sn, nn, p, mf, a, ph, c in oracle.q2(supp, ps, e12, e19, st)]
    assert len(rows) == 100 and oracle.rows_text(7, rows) == gold(2)
    rows = [("NULL" if c is None else c, n) for c, n in oracle.q13(orders, len(cust["c_custkey"]))]
    assert rows[0] == ("NULL", 50005) and oracle.rows_text(1, rows) == gold(13)


def test_q3_reproduces_reference_golden(oracle, sf1):
    res = oracle.q3(sf1["customer"], sf1["orders"], sf1["lineitem"])
    assert oracle.q3_text(res) == open(os.path.join(GOLDEN, "ref_sf1_q3.txt")).read()


def test_decimal_contract(oracle):
    """govalues contract points the restatement relies on."""
    import ctypes as C
    L = oracle.lib()

    def op(name, a, b):
        oc, os_, on = C.c_uint64(), C.c_int(), C.c_int()
        rc = getattr(L, name)(a[0], a[1], a[2], b[0], b[1], b[2], C.byref(oc), C.byref(os_), C.byref(on))
        return rc, (oc.value, os_.value, on.value)
    assert op("orc_dec_add", (150, 2, 0), (25, 1, 0)) == (0, (400, 2, 0))                 # scale = max
    assert op("orc_dec_mul", (150, 2, 0), (25, 1, 0)) == (0, (3750, 3, 0))                # scale = sum
    assert op("orc_dec_add", (100, 2, 0), (250, 2, 1)) == (0, (150, 2, 1))                # sign
    # 20-digit result: keep 19 digits, half-even
    assert op("orc_dec_add", (9999999999999999999, 6, 0), (6, 6, 0)) == (0, (1000000000000000000, 5, 0))
    assert op("orc_dec_add", (9999999999999999990, 6, 0), (15, 6, 0)) == (0, (1000000000000000000, 5, 0))   # tie -> even
    assert op("orc_dec_add", (9999999999999999990, 6, 0), (25, 6, 0)) == (0, (1000000000000000002, 5, 0))   # tie -> even
    assert op("orc_dec_add", (9999999999999999999, 0, 0), (1, 0, 0))[0] != 0              # integer part overflows
    # Quo: exact when it terminates, else 19 significant digits; trailing zeros trimmed
    assert op("orc_dec_quo", (100, 2, 0), (4, 0, 0)) == (0, (25, 2, 0))
    assert op("orc_dec_quo", (1, 0, 0), (3, 0, 0)) == (0, (3333333333333333333, 19, 0))
    rc, (coef, scale, neg) = op("orc_dec_quo", (5658655440073, 2, 0), (1478493, 0, 0))            # 38273.1297...
    assert rc == 0 and neg == 0 and str(coef).startswith("3827312973462167") and coef * 10 ** (19 - scale) // 10 ** 19 == 38273
    # formatting: Int64(scale) rounds half-even, NewFromInt64 strips trailing zeros
    assert oracle.fmt_decimal((5656804138090, 2, 0), 2) == "56568041380.9"
    assert oracle.fmt_decimal((3827312915, 5, 0), 2) == "38273.13"
    assert oracle.fmt_decimal((125, 3, 0), 2) == "0.12" and oracle.fmt_decimal((135, 3, 0), 2) == "0.14"
    assert oracle.fmt_double(25.522005853257337) == "25.522005853257337"
    assert oracle.fmt_double(1e21) == "1e+21" and oracle.fmt_double(100.0) == "100"
    assert oracle.fmt_double(1e9) == "1e+09" and oracle.fmt_double(16777216.0) == "1.6777216e+07" and oracle.fmt_double(343478.59375) == "343478.59375"
    # the float32 cast the reference applies to DECIMAL columns in range predicates
    f = np.float32
    lo, hi = f(0.03) - f(0.01), f(0.03) + f(0.01)
    passing = [c for c in range(0, 11) if lo <= f(L.orc_dec_float64(c, 2, 0)) <= hi]
    assert passing == [2, 3, 4]


def test_wildcard_match_restatement(oracle):
    """Truth table of the reference's LIKE matcher (wildcardMatch, function_operator_boolean.go:336-377)."""
    cases = [("%pink%", "cornflower chocolate smoke green pink", True), ("%pink%", "forest brown coral puff cream", False),
             ("", "", True), ("", "a", False), ("%", "", True), ("%", "abc", True), ("_", "", False), ("_", "a", True), ("_", "ab", False),
             ("a%b", "ab", True), ("a%b", "axxb", True), ("a%b", "axxbc", False), ("a%b%", "axxbc", True), ("%a%a%", "banana", True),
             ("%a_a%", "banana", True), ("%ab", "aab", True), ("%ab", "aba", False), ("a_c", "abc", True), ("a_c", "ac", False),
             ("%%", "x", True), ("%_", "", False), ("abc", "abc", True), ("abc", "abd", False), ("abc%", "ab", False)]
    for pat, tgt, want in cases:
        assert oracle.wildcard_match(pat.encode(), tgt.encode()) is want, (pat, tgt)


def test_row_oracle_agrees_with_the_golden_pinned_restatements(oracle):
    """oracle/rowexec.py (the tree-walking oracle the GPU row tests are checked against) evaluates the reference's Q4 / Q12 / Q14 /
    Q19 PLANS -- MARK join + mark filter, CASE / OR / IN / LIKE inside aggregates over a join, a three-branch OR above a join --
    and must give what the numpy restatements give, which are pinned by the reference's golden files at SF1.  This ties the row
    oracle's join / aggregate / CASE / string-predicate semantics to the reference's own answers."""
    import numpy as np
    from oracle import rowexec as R
    from plan_b200 import chunk as K, tpch as T
    sf = 0.01
    orders, line = oracle.gen_orders_lineitem(sf)
    x12, x19 = oracle.gen_q12_q14_columns(sf), oracle.gen_q19_columns(sf)
    npart = len(x12["p_type"])
    part = {"p_partkey": np.arange(1, npart + 1, dtype=np.int32), "p_type": x12["p_type"], "p_brand": x19["p_brand"], "p_size": x19["p_size"],
            "p_container": x19["p_container"]}
    lx = dict(line, l_shipmode=x12["l_shipmode"], l_shipinstruct=x19["l_shipinstruct"])
    ox = dict(orders, o_orderpriority=x12["o_orderpriority"])

    def rows(cols, sch):
        return R.table_rows(cols, sch)
    # Q12 (the SF0.01 sample has few FOB / TRUCK rows in 1996: use every year by widening the plan's year to the data's bulk)
    for year in (1994, 1996):
        got = R.execute(T.q12_plan(year=year), {"lineitem": rows(lx, T.Q12_LINEITEM), "orders": rows(ox, T.Q12_ORDERS)})
        want = oracle.q12(orders, line, x12, year=year)
        assert sorted((r[0], r[1], r[2]) for r in got) == sorted(want)
    # Q4
    got = R.execute(T.q4_plan(), {"orders": rows(ox, T.Q4_ORDERS), "lineitem": rows(line, T.Q4_LINEITEM)})
    assert sorted((r[0], r[1]) for r in got) == sorted(oracle.q4(orders, line, x12))
    # Q14: the two exact sums
    got = R.execute(T.q14_plan(), {"lineitem": rows(line, T.Q14_LINEITEM), "part": rows(part, T.Q14_PART)})
    ref = oracle.q14(line, x12)
    assert len(got) == 1 and [v.signed() * 10 ** (4 - v.scale) for v in got[0]] == [ref["promo"], ref["total"]]
    # Q19 over a whole-year-free sample is tiny at SF0.01: loosen nothing, just require equality (possibly of empty results)
    got = R.execute(T.q19_plan(), {"lineitem": rows(lx, T.Q19_LINEITEM), "part": rows(part, T.Q19_PART)})
    ref = oracle.q19(line, x12, x19)
    if ref["rows"] == 0:
        assert got == [] or got[0][0] is None
    else:
        assert got[0][0].signed() * 10 ** (4 - got[0][0].scale) == ref["revenue"]


def test_row_oracle_runs_the_q5_q7_q8_plans(oracle):
    """Six- to eight-table left-deep join stacks (a two-key join, the same dimension joined twice under two aliases, an OR of
    two-sided string equalities above the joins, CASE inside a sum, extract(year)) as PhysicalOperator trees through the tree-walking
    oracle: it must give what the numpy restatements give, which reproduce the reference's q5.txt / q7.txt / q8.txt at SF1."""
    import numpy as np
    from oracle import rowexec as R
    from plan_b200 import tpch as T
    sf = 0.02
    orders, line = oracle.gen_orders_lineitem(sf)
    cust, supp, x12 = oracle.gen_customer(sf), oracle.gen_supplier(sf), oracle.gen_q12_q14_columns(sf)
    assert T.NATION_REGION == oracle.NATION_REGION and T.REGIONS == oracle.REGIONS
    nation = {"n_nationkey": np.arange(25, dtype=np.int32), "n_name": np.arange(25, dtype=np.uint8), "n_regionkey": np.array(T.NATION_REGION, np.int32)}
    region = {"r_regionkey": np.arange(5, dtype=np.int32), "r_name": np.arange(5, dtype=np.uint8)}
    part = {"p_partkey": np.arange(1, len(x12["p_type"]) + 1, dtype=np.int32), "p_type": x12["p_type"]}
    rows = R.table_rows
    tabs = {"lineitem": rows(line, T.LINEITEM), "orders": rows(orders, T.ORDERS), "customer": rows(cust, T.CUSTOMER), "supplier": rows(supp, T.SUPPLIER),
            "nation": rows(nation, T.NATION_R), "region": rows(region, T.REGION), "part": rows(part, T.Q8_PART)}
    s4 = lambda v: v.signed() * 10 ** (4 - v.scale)   # noqa: E731
    want = oracle.q5(cust, supp, orders, line)
    assert len(want) == 5 and sorted((r[0], s4(r[1])) for r in R.execute(T.q5_plan(), tabs)) == sorted(want)
    want = oracle.q7(cust, supp, orders, line)
    assert len(want) == 4 and sorted((r[0], r[1], r[2], s4(r[3])) for r in R.execute(T.q7_plan(), tabs)) == want
    want = oracle.q8(cust, supp, orders, line, x12)
    got = sorted((r[0], s4(r[1]), s4(r[2])) for r in R.execute(T.q8_plan(), tabs))
    assert len(want) == 2 and got == [(y, a, b) for y, _q, a, b in want]
    for y, q, a, b in want:                                     # the host-side division above the aggregate: govalues Quo
        d = R.dec_quo(R.Dec(a, 4), R.Dec(b, 4))
        assert (d.coef, d.scale) == (q[0], q[1]) or (a == 0 and d.coef == 0)


def test_row_oracle_runs_the_q13_plan(oracle):
    """Q13 as the reference plans it -- Agg over Agg over a LEFT join whose build side carries `o_comment not like '%pending%accounts%'`
    -- through the tree-walking oracle: NULL padding of customers without a surviving order, count(o_orderkey) = NULL over them
    (CountOp.Finalize), NULL as a group key of the outer aggregate.  It must give what oracle.q13 gives, which reproduces q13.txt at SF1:
    this is what pins the row oracle's LEFT join."""
    import numpy as np
    from oracle import rowexec as R
    from plan_b200 import tpch as T
    sf = 0.02
    orders, _ = oracle.gen_orders_lineitem(sf, lineitem_cols=[])
    cust = oracle.gen_customer(sf)
    text = oracle.comments("o_comment", range(len(orders["o_orderkey"])))
    assert text[0] == "nstructions sleep furiously among " and text[1] == " foxes. pending accounts at the pending, silent asymptot"   # official orders.tbl rows 1-2
    oc = dict(orders, o_comment=np.array([c.encode() for c in text], dtype=object))
    tabs = {"customer": R.table_rows(cust, T.Q13_CUSTOMER), "orders": R.table_rows(oc, T.Q13_ORDERS)}
    want = oracle.q13(orders, len(cust["c_custkey"]))
    assert want[0] == (None, 1000) and sum(1 for t in text if oracle.wildcard_match(b"%pending%accounts%", t.encode())) > 100
    got = R.execute(T.q13_plan(), tabs)
    key = lambda r: (-r[1], -(r[0] or 0))   # noqa: E731
    assert sorted(((r[0], r[1]) for r in got), key=key) == want


def test_row_oracle_runs_the_q10_plan(oracle):
    """Q10's aggregate (seven group keys: INTEGER, four VARCHARs, a signed DECIMAL, a dictionary name) over a four-table join through
    the tree-walking oracle; ordered by revenue and cut to 20 rows it must equal oracle.q10, which reproduces q10.txt at SF1."""
    import numpy as np
    from oracle import rowexec as R
    from plan_b200 import tpch as T
    sf = 0.02
    orders, line = oracle.gen_orders_lineitem(sf)
    cust = oracle.gen_customer(sf)
    ct, x22 = oracle.gen_customer_text(sf, cust), oracle.gen_q11_q22_columns(sf)
    obj = lambda xs: np.array([x.encode() for x in xs], dtype=object)   # noqa: E731
    cx = {"c_custkey": cust["c_custkey"], "c_name": cust["c_name"], "c_acctbal": x22["c_acctbal"], "c_nationkey": cust["c_nationkey"],
          "c_address": obj(ct["c_address"]), "c_phone": obj(ct["c_phone"]), "c_comment": obj(oracle.comments("c_comment", range(len(cust["c_custkey"]))))}
    nation = {"n_nationkey": np.arange(25, dtype=np.int32), "n_name": np.arange(25, dtype=np.uint8)}
    tabs = {"lineitem": R.table_rows(line, T.LINEITEM), "orders": R.table_rows(orders, T.ORDERS), "customer": R.table_rows(cx, T.Q10_CUSTOMER),
            "nation": R.table_rows(nation, T.NATION)}
    plan = T.q10_plan()
    got = R.execute(plan.Children[0].Children[0], tabs)                 # the aggregate below Limit <- Order (host parents)
    s4 = lambda v: v.signed() * 10 ** (4 - v.scale)   # noqa: E731
    top = sorted((-s4(r[2]), r[0]) + tuple(r) for r in got)[:20]
    mine = [(r[2], r[3], s4(r[4]), r[5].signed() * 10 ** (2 - r[5].scale), r[6], r[7], r[8], r[9]) for r in top]
    assert len(got) > 500 and mine == oracle.q10(cust, orders, line, x22, ct)


def test_row_oracle_agrees_with_the_c_oracle_on_the_headline_plans(oracle):
    """The two oracles are independent restatements: oracle/refexec.c + numpy (pinned by q1 / q3 / q6 / q9 / q18.txt at SF1) and the
    tree-walking oracle/rowexec.py that executes PhysicalOperator trees.  Running the five headline PLANS (tpch.q6_plan ... q18_plan,
    the trees the GPU path is given) through rowexec must give the C oracle's answers exactly: Q6's float32 BETWEEN on a DECIMAL
    column, Q1's eight aggregates incl. avg(DECIMAL) as a 19-digit quotient and avg(INTEGER) as a double, Q3's three-table join, Q9's
    six-table star with LIKE and extract(year), Q18's join against a HAVING sub-aggregate."""
    import numpy as np
    from oracle import rowexec as R
    from plan_b200 import tpch as T
    sf = 0.01
    orders, line = oracle.gen_orders_lineitem(sf)
    cust, supp, ps, part = oracle.gen_customer(sf), oracle.gen_supplier(sf), oracle.gen_partsupp(sf), oracle.gen_part(sf, like_word="pink")
    nation = {"n_nationkey": np.arange(25, dtype=np.int32), "n_name": np.arange(25, dtype=np.uint8)}
    rows = R.table_rows
    tabs = {"lineitem": rows(line, T.LINEITEM), "orders": rows(orders, T.ORDERS), "customer": rows(cust, T.CUSTOMER),
            "part": rows({"p_partkey": part["p_partkey"], "p_name": part["p_name"]}, T.PART), "supplier": rows(supp, T.SUPPLIER),
            "partsupp": rows(ps, T.PARTSUPP), "nation": rows(nation, T.NATION)}
    s4 = lambda v: v.signed() * 10 ** (4 - v.scale)   # noqa: E731
    dec = lambda v: (v.coef, v.scale, int(v.neg))     # noqa: E731
    # Q6
    got = R.execute(T.q6_plan(), tabs)
    want = oracle.q6(line)
    assert want["rows_selected"] > 500 and len(got) == 1 and s4(got[0][0]) == want["exact"]
    # Q1
    got, want = R.execute(T.q1_plan(), tabs), oracle.q1(line)
    assert len(got) == len(want["groups"]) == 4
    for g in want["groups"]:
        r = [x for x in got if (x[0], x[1]) == (g["l_returnflag"], g["l_linestatus"])][0]
        assert (r[2], dec(r[3]), dec(r[4]), dec(r[5]), r[6], dec(r[7]), dec(r[8]), r[9]) == (
            g["sum_qty"], g["sum_base_price"], g["sum_disc_price"], g["sum_charge"], g["avg_qty"], g["avg_price"], g["avg_disc"], g["count_order"])
    # Q3 (every group, not only the top 10)
    want = sorted((g["l_orderkey"], g["x_revenue"], g["o_orderdate"], g["o_shippriority"]) for g in oracle.q3(cust, orders, line)["groups"])
    assert len(want) > 50 and sorted((r[0], s4(r[1]), r[2], r[3]) for r in R.execute(T.q3_plan(), tabs)) == want
    # Q9 (below its Order)
    want = sorted(oracle.q9(part, supp, ps, orders, line))
    assert len(want) > 100 and sorted((r[0], r[1], s4(r[2])) for r in R.execute(T.q9_plan().Children[0], tabs)) == want
    # Q18 (the aggregate below Limit <- Order; threshold lowered so the small sample has groups)
    node = T.q18_plan(qty_gt=150)
    while node.Typ != R.POT_Agg:
        node = node.Children[0]
    got = sorted((-r[4].signed(), r[3], r[0], r[1], r[2], r[5]) for r in R.execute(node, tabs))[:100]
    want = oracle.q18(cust, orders, line, qty_gt=150, limit=100)
    assert len(want) == 100 and [(a[2], a[3], a[4], a[1], -a[0], a[5]) for a in got] == [
        (g["c_name"], g["c_custkey"], g["o_orderkey"], g["o_orderdate"], g["o_totalprice"], g["sum_qty"]) for g in want]


def test_row_oracle_agrees_with_the_restatements_on_the_other_plan_builders(oracle):
    """The remaining plan builders the GPU tests use -- high-cardinality group-bys with HAVING, SEMI / ANTI joins, EXISTS / NOT EXISTS as
    MARK / AntiMARK joins under `mark = true / false`, string predicates, the wide min / max / sum / avg shape with NULLs -- through the
    tree-walking oracle against their numpy / C restatements: two independent statements of each."""
    import numpy as np
    from oracle import rowexec as R
    from plan_b200 import tpch as T
    sf = 0.01
    orders, line = oracle.gen_orders_lineitem(sf)
    cust = oracle.gen_customer(sf)
    tabs = {"lineitem": R.table_rows(line, T.LINEITEM), "orders": R.table_rows(orders, T.ORDERS), "customer": R.table_rows(cust, T.CUSTOMER)}

    def agg_node(p):
        while p.Typ != R.POT_Agg:
            p = p.Children[0]
        return p
    num = lambda v: v.signed() if isinstance(v, R.Dec) else v   # noqa: E731
    plain = lambda want: {int(k): (int(v[0]), int(v[1])) for k, v in want.items()}   # noqa: E731
    for kw in (dict(key="l_orderkey", value="l_quantity", having_gt=200), dict(key="l_partkey", value="l_quantity"),
               dict(key="l_suppkey", value="l_extendedprice", ship_le=9500)):
        got = {r[0]: (num(r[1]), r[2]) for r in R.execute(agg_node(T.groupby_plan(**kw)), tabs)}
        assert len(got) >= 100 and got == plain(oracle.groupby_sum(line, **kw)), kw
    for anti in (False, True):
        want = plain(oracle.semi_groupby(orders, line, anti=anti))
        assert len(want) > 400
        assert {r[0]: (num(r[1]), r[2]) for r in R.execute(agg_node(T.semi_plan(anti=anti)), tabs)} == want
        assert {r[0]: (num(r[1]), r[2]) for r in R.execute(agg_node(T.exists_plan(negated=anti)), tabs)} == want
    for fl in ([("c_name", "like", "%00001%")], [("c_mktsegment", "not like", "_U%"), ("c_name", "like", "Customer#0000005__")],
               [("c_mktsegment", "=", "BUILDING")], [("c_name", "like", "nothing%")]):
        got, want = R.execute(T.customer_filter_plan(fl), tabs), oracle.customer_filter(cust, fl, oracle.SEGMENTS)
        assert (got == [] and want is None) or tuple(got[0]) == want, fl
    # the wide shape, with NULLs in three columns: aggregates over no valid input are NULL
    rng = np.random.default_rng(5)
    n = len(line["l_orderkey"])
    valid = {"l_quantity": rng.random(n) >= 0.1, "l_extendedprice": rng.random(n) >= 0.3, "l_tax": rng.random(n) >= 0.2}
    valid["l_tax"][line["l_returnflag"] == ord("A")] = False                     # one group without any valid l_tax
    args = (T.days(1993, 1, 1), T.days(1997, 6, 30), T.days(1997, 9, 1), T.days(1993, 2, 1), 5, 45, 3)
    want = oracle.stats(line, *args, valid=valid)
    got = R.execute(T.stats_plan(*args), {"lineitem": R.table_rows(line, T.LINEITEM, valid=valid)})
    tup = lambda v: None if v is None else (v.coef, v.scale, int(v.neg))         # noqa: E731
    assert len(got) == len(want["groups"]) == 3
    for g in want["groups"]:
        r = [x for x in got if x[0] == g["l_returnflag"]][0]
        assert [tup(v) for v in r[1:7]] == [g["min_ext"], g["max_ext"], g["max_disc"], g["sum_tax"], g["avg_tax"], g["sum_taxed"]] and r[7] == g["count"]
    assert [g["sum_tax"] for g in want["groups"] if g["l_returnflag"] == "A"] == [None]
