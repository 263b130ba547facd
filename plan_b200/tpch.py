"""TPC-H physical plans as the reference's planner emits them (SURVEY.md 3.4), plus the
in-box generated tables.  The planner itself stays in Go; these builders stand in for
`genPhyPlan` (/root/reference/pkg/compute/executor.go:76-114) in tests and benchmarks.

Typing follows the reference binder (SURVEY.md 8c-1):
  - `1 - l_discount`: INTEGER literal cast to DECIMAL(15,2), DECIMAL subtract -> DECIMAL(16,2)
  - `a * b` on DECIMALs: scale = sum of scales (function_scalar.go:429-475)
  - `l_discount between 0.03-0.01 and 0.03+0.01`: FLOAT literals, folded in float32, column
    cast to FLOAT (builder_binder.go:517-580)
  - date +/- interval folded to a DATE constant (rule_constant_folding.go:34-100)
  - sum(DECIMAL(w,s)) -> DECIMAL(38,s); avg(INT) -> DOUBLE; sum(INT)/count -> HUGEINT
"""
import ctypes as C
import datetime

import numpy as np

from . import _lib as L
from . import chunk as K
from .compute import (JOIN_ANTI, JOIN_ANTI_MARK, JOIN_LEFT, JOIN_MARK, JOIN_SEMI, JOIN_INNER, POT_Filter, POT_Agg, POT_Join, POT_Limit, POT_Order, POT_Scan, AggOpInfo, DeviceTable, JoinOpInfo,
                      LimitOpInfo, OrderOpInfo, PhysicalOperator, ScanOpInfo, cast, col, const, func)

SEGMENTS = ["AUTOMOBILE", "BUILDING", "FURNITURE", "HOUSEHOLD", "MACHINERY"]

LINEITEM = [("l_orderkey", L.PG_T_INT64, 0, 0, None), ("l_partkey", L.PG_T_INT32, 0, 0, None),
            ("l_suppkey", L.PG_T_INT32, 0, 0, None), ("l_linenumber", L.PG_T_INT32, 0, 0, None),
            ("l_quantity", L.PG_T_INT32, 0, 0, None), ("l_extendedprice", L.PG_T_DECIMAL64, 15, 2, None),
            ("l_discount", L.PG_T_DECIMAL64, 15, 2, None), ("l_tax", L.PG_T_DECIMAL64, 15, 2, None),
            ("l_returnflag", L.PG_T_CHAR1, 0, 0, None), ("l_linestatus", L.PG_T_CHAR1, 0, 0, None),
            ("l_shipdate", L.PG_T_DATE32, 0, 0, None), ("l_commitdate", L.PG_T_DATE32, 0, 0, None),
            ("l_receiptdate", L.PG_T_DATE32, 0, 0, None)]
ORDERS = [("o_orderkey", L.PG_T_INT64, 0, 0, None), ("o_custkey", L.PG_T_INT32, 0, 0, None),
          ("o_orderdate", L.PG_T_DATE32, 0, 0, None), ("o_shippriority", L.PG_T_INT32, 0, 0, None),
          ("o_totalprice", L.PG_T_DECIMAL64, 15, 2, None), ("o_orderstatus", L.PG_T_CHAR1, 0, 0, None)]
CUSTOMER = [("c_custkey", L.PG_T_INT32, 0, 0, None), ("c_mktsegment", L.PG_T_DICT8, 0, 0, SEGMENTS),
            ("c_nationkey", L.PG_T_INT32, 0, 0, None), ("c_name", L.PG_T_VARCHAR, 25, 0, None)]

NATIONS = ["ALGERIA", "ARGENTINA", "BRAZIL", "CANADA", "EGYPT", "ETHIOPIA", "FRANCE", "GERMANY", "INDIA", "INDONESIA", "IRAN", "IRAQ",
           "JAPAN", "JORDAN", "KENYA", "MOROCCO", "MOZAMBIQUE", "PERU", "CHINA", "ROMANIA", "SAUDI ARABIA", "VIETNAM", "RUSSIA",
           "UNITED KINGDOM", "UNITED STATES"]          # n_nationkey order (dbgen nations distribution)
PART = [("p_partkey", L.PG_T_INT32, 0, 0, None), ("p_name", L.PG_T_VARCHAR, 55, 0, None)]
SUPPLIER = [("s_suppkey", L.PG_T_INT32, 0, 0, None), ("s_nationkey", L.PG_T_INT32, 0, 0, None)]
PARTSUPP = [("ps_partkey", L.PG_T_INT32, 0, 0, None), ("ps_suppkey", L.PG_T_INT32, 0, 0, None),
            ("ps_supplycost", L.PG_T_DECIMAL64, 15, 2, None)]
NATION = [("n_nationkey", L.PG_T_INT32, 0, 0, None), ("n_name", L.PG_T_DICT8, 0, 0, NATIONS)]

DEC15_2 = K.DecimalType(15, 2)


def days(y, m, d):
    return (datetime.date(y, m, d) - datetime.date(1970, 1, 1)).days


def _ltype_of(coldef):
    _, t, w, s, _ = coldef
    return {L.PG_T_INT32: K.IntegerType(), L.PG_T_INT64: K.BigintType(), L.PG_T_DATE32: K.DateType(),
            L.PG_T_DECIMAL64: K.DecimalType(w, s), L.PG_T_CHAR1: K.VarcharType(), L.PG_T_DICT8: K.VarcharType(),
            L.PG_T_VARCHAR: K.VarcharType()}[t]


class Schema:
    """Column layout of the bound tables (ScanOpInfo.Columns / ColName2Idx).  The default is
    the full generated tables; a caller that uploads only the referenced columns passes the
    pruned layout so column references index the right positions."""

    def __init__(self, lineitem=None, orders=None, customer=None, part=None, supplier=None, partsupp=None, nation=None):
        self.tables = {"lineitem": lineitem or LINEITEM, "orders": orders or ORDERS, "customer": customer or CUSTOMER,
                       "part": part or PART, "supplier": supplier or SUPPLIER, "partsupp": partsupp or PARTSUPP, "nation": nation or NATION}
        self.idx = {t: {c[0]: i for i, c in enumerate(cols)} for t, cols in self.tables.items()}

    def col(self, table, name, side=0):
        i = self.idx[table][name]
        return col(side, i, _ltype_of(self.tables[table][i]))

    def pruned(self, need):
        """need: {table: [column names]} -> Schema holding only those columns (original order)."""
        kw = {t: [c for c in self.tables[t] if c[0] in need[t]] for t in need}
        return Schema(**kw)


FULL = Schema()


# ------------------------------------------------------------------ plans --

def q6_plan(date_lo=None, date_hi=None, disc_lit=0.03, disc_eps=0.01, qty_lt=24, schema=FULL):
    """Agg(no group; sum(l_extendedprice*l_discount)) <- Scan(lineitem; 5 comparisons)."""
    S = schema
    date_lo = days(1994, 1, 1) if date_lo is None else date_lo
    date_hi = days(1995, 1, 1) if date_hi is None else date_hi
    B = K.LType(K.LTID_BOOLEAN)
    f32 = np.float32
    flo = float(f32(disc_lit) - f32(disc_eps))     # subFloat32 folded at plan time
    fhi = float(f32(disc_lit) + f32(disc_eps))
    discf = cast(S.col("lineitem", "l_discount"), K.FloatType())
    filters = [
        func(">=", B, S.col("lineitem", "l_shipdate"), const(date_lo, K.DateType())),
        func("<", B, S.col("lineitem", "l_shipdate"), const(date_hi, K.DateType())),
        func("and", B, func(">=", B, discf, const(flo, K.FloatType())),
             func("<=", B, discf, const(fhi, K.FloatType()))),
        func("<", B, S.col("lineitem", "l_quantity"), const(qty_lt, K.IntegerType())),
    ]
    scan = PhysicalOperator(POT_Scan, Filters=filters, Info=ScanOpInfo("lineitem"))
    arg = func("*", K.DecimalType(18, 4), S.col("lineitem", "l_extendedprice"), S.col("lineitem", "l_discount"))
    agg = func("sum", K.DecimalType(38, 4), arg)
    return PhysicalOperator(POT_Agg, Outputs=[col(1, 0, K.DecimalType(38, 4))], Children=[scan],
                            Info=AggOpInfo([agg], []))


def _disc_price(ext, disc):
    """l_extendedprice * (1 - l_discount): INTEGER 1 cast to DECIMAL(15,2), DECIMAL(16,2) subtract,
    left operand cast to DECIMAL(16,2), product DECIMAL(18,4)."""
    one = cast(const(1, K.IntegerType()), DEC15_2)
    return func("*", K.DecimalType(18, 4), cast(ext, K.DecimalType(16, 2)), func("-", K.DecimalType(16, 2), one, disc))


def q1_plan(ship_le=None, schema=FULL):
    """Agg(group by l_returnflag,l_linestatus; 8 aggregates) <- Scan(lineitem; l_shipdate <= c)."""
    S = schema
    lc = lambda n: S.col("lineitem", n)   # noqa: E731
    ship_le = days(1998, 8, 11) if ship_le is None else ship_le    # 1998-12-01 - 112 days, folded
    B = K.LType(K.LTID_BOOLEAN)
    scan = PhysicalOperator(POT_Scan, Filters=[func("<=", B, lc("l_shipdate"), const(ship_le, K.DateType()))],
                            Info=ScanOpInfo("lineitem"))
    one_plus_tax = func("+", K.DecimalType(16, 2), cast(const(1, K.IntegerType()), DEC15_2), lc("l_tax"))
    charge = func("*", K.DecimalType(18, 8), _disc_price(lc("l_extendedprice"), lc("l_discount")),
                  cast(one_plus_tax, K.DecimalType(18, 4)))
    count_col = S.tables["lineitem"][0]        # count(*) -> count(first column) (builder_binder.go:207-228)
    aggs = [
        func("sum", K.HugeintType(), lc("l_quantity")),
        func("sum", K.DecimalType(38, 2), lc("l_extendedprice")),
        func("sum", K.DecimalType(38, 4), _disc_price(lc("l_extendedprice"), lc("l_discount"))),
        func("sum", K.DecimalType(38, 8), charge),
        func("avg", K.DoubleType(), lc("l_quantity")),
        func("avg", K.DecimalType(38, 2), lc("l_extendedprice")),
        func("avg", K.DecimalType(38, 2), lc("l_discount")),
        func("count", K.HugeintType(), col(0, 0, _ltype_of(count_col))),
    ]
    groups = [lc("l_returnflag"), lc("l_linestatus")]
    outs = [col(0, 0, K.VarcharType()), col(0, 1, K.VarcharType())] + [col(1, i, a.DataTyp) for i, a in enumerate(aggs)]
    return PhysicalOperator(POT_Agg, Outputs=outs, Children=[scan], Info=AggOpInfo(aggs, groups))


def q3_plan(segment="HOUSEHOLD", odate_lt=None, ship_gt=None, schema=FULL, segment_in=None, segment_ne=None):
    """Agg(group by l_orderkey,o_orderdate,o_shippriority; sum(ext*(1-disc)))
         <- Join(l_orderkey = o_orderkey) <- { Scan(lineitem; l_shipdate > d),
              Join(o_custkey = c_custkey) <- { Scan(orders; o_orderdate < d),
                                               Scan(customer; c_mktsegment = seg) } }
    Probe/left = larger relation, build/right = Children[1] (optimizer_joinorder.go:1028-1030)."""
    S = schema
    odate_lt = days(1995, 3, 29) if odate_lt is None else odate_lt
    ship_gt = days(1995, 3, 29) if ship_gt is None else ship_gt
    B = K.LType(K.LTID_BOOLEAN)
    seg_col = S.col("customer", "c_mktsegment")
    if segment_in is not None:            # c_mktsegment in (...): a code set on the build-side scan
        seg_filter = func("in", B, seg_col, *[const(x, K.VarcharType()) for x in segment_in])
    elif segment_ne is not None:
        seg_filter = func("<>", B, seg_col, const(segment_ne, K.VarcharType()))
    else:
        seg_filter = func("=", B, seg_col, const(segment, K.VarcharType()))
    cust = PhysicalOperator(POT_Scan, Info=ScanOpInfo("customer"), Filters=[seg_filter])
    orders = PhysicalOperator(POT_Scan, Info=ScanOpInfo("orders"),
                              Filters=[func("<", B, S.col("orders", "o_orderdate"), const(odate_lt, K.DateType()))])
    line = PhysicalOperator(POT_Scan, Info=ScanOpInfo("lineitem"),
                            Filters=[func(">", B, S.col("lineitem", "l_shipdate"), const(ship_gt, K.DateType()))])
    OI, LI = S.idx["orders"], S.idx["lineitem"]
    j1 = PhysicalOperator(
        POT_Join, Children=[orders, cust],
        Outputs=[col(0, OI["o_orderkey"], K.BigintType()), col(0, OI["o_orderdate"], K.DateType()),
                 col(0, OI["o_shippriority"], K.IntegerType())],
        Info=JoinOpInfo(JOIN_INNER, [func("=", B, S.col("orders", "o_custkey", 0), S.col("customer", "c_custkey", 1))]))
    j2 = PhysicalOperator(
        POT_Join, Children=[line, j1],
        Outputs=[col(0, LI["l_orderkey"], K.BigintType()), col(0, LI["l_extendedprice"], DEC15_2),
                 col(0, LI["l_discount"], DEC15_2), col(1, 1, K.DateType()), col(1, 2, K.IntegerType())],
        Info=JoinOpInfo(JOIN_INNER, [func("=", B, S.col("lineitem", "l_orderkey", 0), col(1, 0, K.BigintType()))]))
    rev = _disc_price(col(0, 1, DEC15_2), col(0, 2, DEC15_2))
    agg = func("sum", K.DecimalType(38, 4), rev)
    groups = [col(0, 0, K.BigintType()), col(0, 3, K.DateType()), col(0, 4, K.IntegerType())]
    outs = [col(0, 0, K.BigintType()), col(1, 0, K.DecimalType(38, 4)), col(0, 1, K.DateType()),
            col(0, 2, K.IntegerType())]
    return PhysicalOperator(POT_Agg, Outputs=outs, Children=[j2], Info=AggOpInfo([agg], groups))


def stats_plan(d0, d1, d2, d3, q0, q1, disc_gt_cents, schema=FULL, linestatus_ne=None, returnflag_in=None, returnflag_or=None):
    """A wider scan-aggregate shape (no specialised kernel: runs on the generic one):
    select l_returnflag, min(l_extendedprice), max(l_extendedprice), max(l_discount), sum(l_tax), avg(l_tax),
           sum(l_extendedprice * (1 + l_tax)), count(*)
    from lineitem where l_shipdate between d0 and d1 and l_commitdate <= d2 and l_receiptdate >= d3
      and l_quantity between q0 and q1 and l_discount > <decimal> group by l_returnflag"""
    S = schema
    lc = lambda n: S.col("lineitem", n)   # noqa: E731
    B = K.LType(K.LTID_BOOLEAN)
    D, I = K.DateType(), K.IntegerType()
    filters = [func(">=", B, lc("l_shipdate"), const(d0, D)), func("<=", B, lc("l_shipdate"), const(d1, D)),
               func("<=", B, lc("l_commitdate"), const(d2, D)), func(">=", B, lc("l_receiptdate"), const(d3, D)),
               func(">=", B, lc("l_quantity"), const(q0, I)), func("<=", B, lc("l_quantity"), const(q1, I)),
               func(">", B, lc("l_discount"), const(disc_gt_cents, DEC15_2))]
    V = K.VarcharType()
    if linestatus_ne is not None:          # l_linestatus <> 'O'
        filters.append(func("<>", B, lc("l_linestatus"), const(linestatus_ne, V)))
    if returnflag_in is not None:          # l_returnflag in ('A', 'R')
        filters.append(func("in", B, lc("l_returnflag"), *[const(x, V) for x in returnflag_in]))
    if returnflag_or is not None:          # l_returnflag = 'A' or l_returnflag = 'N'
        e = func("=", B, lc("l_returnflag"), const(returnflag_or[0], V))
        for x in returnflag_or[1:]:
            e = func("or", B, e, func("=", B, lc("l_returnflag"), const(x, V)))
        filters.append(e)
    scan = PhysicalOperator(POT_Scan, Filters=filters, Info=ScanOpInfo("lineitem"))
    one_plus_tax = func("+", K.DecimalType(16, 2), cast(const(1, I), DEC15_2), lc("l_tax"))
    taxed = func("*", K.DecimalType(18, 4), cast(lc("l_extendedprice"), K.DecimalType(16, 2)), one_plus_tax)
    aggs = [func("min", DEC15_2, lc("l_extendedprice")), func("max", DEC15_2, lc("l_extendedprice")),
            func("max", DEC15_2, lc("l_discount")), func("sum", K.DecimalType(38, 2), lc("l_tax")),
            func("avg", K.DecimalType(38, 2), lc("l_tax")), func("sum", K.DecimalType(38, 4), taxed),
            func("count", K.HugeintType(), col(0, 0, _ltype_of(S.tables["lineitem"][0])))]
    outs = [col(0, 0, K.VarcharType())] + [col(1, i, a.DataTyp) for i, a in enumerate(aggs)]
    return PhysicalOperator(POT_Agg, Outputs=outs, Children=[scan], Info=AggOpInfo(aggs, [lc("l_returnflag")]))


def groupby_avg_plan(key="l_suppkey", value="l_extendedprice", schema=FULL):
    """select <key>, avg(<value>), count(*) from lineitem group by <key>  (high-cardinality aggregate with an average:
    avg(DECIMAL) = sum.Quo(count) -> DECIMAL(38,s), avg(INTEGER) -> DOUBLE; function_aggr.go:63-86,881-895)"""
    S = schema
    lc = lambda n: S.col("lineitem", n)   # noqa: E731
    vt = _ltype_of(S.tables["lineitem"][S.idx["lineitem"][value]])
    avg_t = K.DoubleType() if vt.Id in (K.LTID_INTEGER, K.LTID_BIGINT) else K.DecimalType(38, vt.Scale)
    kt = _ltype_of(S.tables["lineitem"][S.idx["lineitem"][key]])
    aggs = [func("avg", avg_t, lc(value)), func("count", K.HugeintType(), col(0, 0, _ltype_of(S.tables["lineitem"][0])))]
    outs = [col(0, 0, kt), col(1, 0, avg_t), col(1, 1, K.HugeintType())]
    scan = PhysicalOperator(POT_Scan, Info=ScanOpInfo("lineitem"))
    return PhysicalOperator(POT_Agg, Outputs=outs, Children=[scan], Info=AggOpInfo(aggs, [lc(key)]))


def groupby_plan(key="l_orderkey", value="l_quantity", having_gt=None, ship_le=None, topk=None, schema=FULL):
    """High-cardinality group-by straight over lineitem (the inner aggregate of TPC-H Q18 when
    key = l_orderkey, having_gt = 314):
        select <key>, sum(<value>), count(*) from lineitem [where l_shipdate <= d]
        group by <key> [having sum(<value>) > k] [order by 2 desc, 1 limit n]
    sum(INTEGER) -> HUGEINT; `sum > 314` compares HUGEINTs (greatHugeintOp,
    function_operator_boolean.go:255-263) after the literal is cast INTEGER -> HUGEINT."""
    S = schema
    lc = lambda n: S.col("lineitem", n)   # noqa: E731
    B = K.LType(K.LTID_BOOLEAN)
    filters = [] if ship_le is None else [func("<=", B, lc("l_shipdate"), const(ship_le, K.DateType()))]
    scan = PhysicalOperator(POT_Scan, Filters=filters, Info=ScanOpInfo("lineitem"))
    vt = _ltype_of(S.tables["lineitem"][S.idx["lineitem"][value]])
    sum_t = K.HugeintType() if vt.Id in (K.LTID_INTEGER, K.LTID_BIGINT) else K.DecimalType(38, vt.Scale)
    aggs = [func("sum", sum_t, lc(value)), func("count", K.HugeintType(), col(0, 0, _ltype_of(S.tables["lineitem"][0])))]
    kt = _ltype_of(S.tables["lineitem"][S.idx["lineitem"][key]])
    outs = [col(0, 0, kt), col(1, 0, sum_t), col(1, 1, K.HugeintType())]
    having = []
    if having_gt is not None:
        having = [func(">", B, col(1, 0, sum_t), cast(const(having_gt, K.IntegerType()), sum_t))]
    agg = PhysicalOperator(POT_Agg, Outputs=outs, Filters=having, Children=[scan], Info=AggOpInfo(aggs, [lc(key)]))
    if topk is None:
        return agg
    order = PhysicalOperator(POT_Order, Outputs=outs, Children=[agg],
                             Info=OrderOpInfo([(col(0, 1, sum_t), True), (col(0, 0, kt), False)]))
    return PhysicalOperator(POT_Limit, Outputs=outs, Children=[order], Info=LimitOpInfo(topk))


def semi_plan(anti=False, odate_lt=None, ship_gt=None, schema=FULL):
    """SEMI / ANTI hash join under an aggregate (the `IN (subquery)` / `NOT IN` shape of Q18 / Q4 / Q21/Q22):
        select o_custkey, sum(o_totalprice), count(*) from orders
        where o_orderdate < d and o_orderkey [NOT] IN (select l_orderkey from lineitem where l_shipdate > s)
        group by o_custkey
    The subquery becomes the build side (Children[1]) of a SEMI / ANTI join (join_scan.go:90-165)."""
    S = schema
    odate_lt = days(1995, 3, 29) if odate_lt is None else odate_lt
    ship_gt = days(1995, 3, 29) if ship_gt is None else ship_gt
    B = K.LType(K.LTID_BOOLEAN)
    orders = PhysicalOperator(POT_Scan, Info=ScanOpInfo("orders"),
                              Filters=[func("<", B, S.col("orders", "o_orderdate"), const(odate_lt, K.DateType()))])
    line = PhysicalOperator(POT_Scan, Info=ScanOpInfo("lineitem"),
                            Filters=[func(">", B, S.col("lineitem", "l_shipdate"), const(ship_gt, K.DateType()))])
    OI = S.idx["orders"]
    j = PhysicalOperator(
        POT_Join, Children=[orders, line],
        Outputs=[col(0, OI["o_custkey"], K.IntegerType()), col(0, OI["o_totalprice"], DEC15_2)],
        Info=JoinOpInfo(JOIN_ANTI if anti else JOIN_SEMI,
                        [func("=", B, S.col("orders", "o_orderkey", 0), S.col("lineitem", "l_orderkey", 1))]))
    aggs = [func("sum", K.DecimalType(38, 2), col(0, 1, DEC15_2)), func("count", K.HugeintType(), col(0, 0, K.IntegerType()))]
    outs = [col(0, 0, K.IntegerType()), col(1, 0, K.DecimalType(38, 2)), col(1, 1, K.HugeintType())]
    return PhysicalOperator(POT_Agg, Outputs=outs, Children=[j], Info=AggOpInfo(aggs, [col(0, 0, K.IntegerType())]))


def q18_plan(qty_gt=314, limit=100, schema=FULL):
    """TPC-H Q18 (cases/tpch/query/q18.sql) below its final Project:
      Limit <- Order(o_totalprice desc, o_orderdate)
        <- Agg(group by c_name, c_custkey, o_orderkey, o_orderdate, o_totalprice; sum(l_quantity))
          <- SEMI Join(o_orderkey = l_orderkey)                 # `o_orderkey IN (subquery)`: builder_plan.go:234-262
               <- { Join(l_orderkey = o_orderkey) <- { Scan(lineitem), Join(o_custkey = c_custkey) <- { Scan(orders), Scan(customer) } },
                    Agg(group by l_orderkey; HAVING sum(l_quantity) > k) <- Scan(lineitem) }
    The inner-join order follows Q3's (probe = larger relation, optimizer_joinorder.go:1028-1030)."""
    S = schema
    B = K.LType(K.LTID_BOOLEAN)
    I, BI, D, H, V = K.IntegerType(), K.BigintType(), K.DateType(), K.HugeintType(), K.VarcharType()
    OI, LI, CI = S.idx["orders"], S.idx["lineitem"], S.idx["customer"]
    cust = PhysicalOperator(POT_Scan, Info=ScanOpInfo("customer"))
    orders = PhysicalOperator(POT_Scan, Info=ScanOpInfo("orders"))
    line = PhysicalOperator(POT_Scan, Info=ScanOpInfo("lineitem"))
    j1 = PhysicalOperator(          # orders x customer -> o_orderkey, o_orderdate, o_totalprice, c_name, c_custkey
        POT_Join, Children=[orders, cust],
        Outputs=[col(0, OI["o_orderkey"], BI), col(0, OI["o_orderdate"], D), col(0, OI["o_totalprice"], DEC15_2),
                 col(1, CI["c_name"], V), col(1, CI["c_custkey"], I)],
        Info=JoinOpInfo(JOIN_INNER, [func("=", B, S.col("orders", "o_custkey", 0), S.col("customer", "c_custkey", 1))]))
    j2 = PhysicalOperator(          # lineitem x j1 -> l_quantity, then j1's five columns
        POT_Join, Children=[line, j1],
        Outputs=[col(0, LI["l_quantity"], I), col(1, 0, BI), col(1, 1, D), col(1, 2, DEC15_2), col(1, 3, V), col(1, 4, I)],
        Info=JoinOpInfo(JOIN_INNER, [func("=", B, S.col("lineitem", "l_orderkey", 0), col(1, 0, BI))]))
    sub_scan = PhysicalOperator(POT_Scan, Info=ScanOpInfo("lineitem"))
    sub = PhysicalOperator(         # select l_orderkey from lineitem group by l_orderkey having sum(l_quantity) > k
        POT_Agg, Outputs=[col(0, 0, BI)], Children=[sub_scan],
        Filters=[func(">", B, col(1, 0, H), cast(const(qty_gt, I), H))],
        Info=AggOpInfo([func("sum", H, S.col("lineitem", "l_quantity"))], [S.col("lineitem", "l_orderkey")]))
    semi = PhysicalOperator(
        POT_Join, Children=[j2, sub], Outputs=[col(0, i, t) for i, t in enumerate([I, BI, D, DEC15_2, V, I])],
        Info=JoinOpInfo(JOIN_SEMI, [func("=", B, col(0, 1, BI), col(1, 0, BI))]))
    groups = [col(0, 4, V), col(0, 5, I), col(0, 1, BI), col(0, 2, D), col(0, 3, DEC15_2)]
    outs = [col(0, 0, V), col(0, 1, I), col(0, 2, BI), col(0, 3, D), col(0, 4, DEC15_2), col(1, 0, H)]
    agg = PhysicalOperator(POT_Agg, Outputs=outs, Children=[semi], Info=AggOpInfo([func("sum", H, col(0, 0, I))], groups))
    if limit is None:
        return agg
    order = PhysicalOperator(POT_Order, Outputs=outs, Children=[agg], Info=OrderOpInfo([(col(0, 4, DEC15_2), True), (col(0, 3, D), False)]))
    return PhysicalOperator(POT_Limit, Outputs=outs, Children=[order], Info=LimitOpInfo(limit))


def q9_plan(word="pink", schema=FULL, agg="sum"):
    """TPC-H Q9 (cases/tpch/query/q9.sql) below its final Project, the subquery's expressions inlined in the aggregate:
      Order(nation, o_year desc)
        <- Agg(group by n_name, extract(year from o_orderdate); sum(l_extendedprice*(1-l_discount) - ps_supplycost*l_quantity))
          <- Join(s_nationkey = n_nationkey) <- { Join(l_orderkey = o_orderkey) <- { Join(l_suppkey = ps_suppkey and l_partkey = ps_partkey)
               <- { Join(l_suppkey = s_suppkey) <- { Join(l_partkey = p_partkey) <- { Scan(lineitem), Scan(part; p_name like '%word%') },
                    Scan(supplier) }, Scan(partsupp) }, Scan(orders) }, Scan(nation) }
    A left-deep stack with the fact table as the leftmost leaf (probe = larger side, optimizer_joinorder.go:1028-1030)."""
    S = schema
    B = K.LType(K.LTID_BOOLEAN)
    I, BI, D, V = K.IntegerType(), K.BigintType(), K.DateType(), K.VarcharType()
    LI = S.idx["lineitem"]
    scan = lambda name, fl=None: PhysicalOperator(POT_Scan, Filters=fl or [], Info=ScanOpInfo(name))   # noqa: E731
    line, supp, ps, orders, nation = scan("lineitem"), scan("supplier"), scan("partsupp"), scan("orders"), scan("nation")
    part = scan("part", [func("like", B, S.col("part", "p_name"), const("%" + word + "%", V))])
    base = [col(0, LI["l_orderkey"], BI), col(0, LI["l_partkey"], I), col(0, LI["l_suppkey"], I), col(0, LI["l_quantity"], I),
            col(0, LI["l_extendedprice"], DEC15_2), col(0, LI["l_discount"], DEC15_2)]
    types = [BI, I, I, I, DEC15_2, DEC15_2]
    eq = lambda a, b: func("=", B, a, b)   # noqa: E731
    j1 = PhysicalOperator(POT_Join, Children=[line, part], Outputs=list(base),
                          Info=JoinOpInfo(JOIN_INNER, [eq(S.col("lineitem", "l_partkey", 0), S.col("part", "p_partkey", 1))]))
    up = lambda ts: [col(0, i, t) for i, t in enumerate(ts)]   # noqa: E731
    j2 = PhysicalOperator(POT_Join, Children=[j1, supp], Outputs=up(types) + [S.col("supplier", "s_nationkey", 1)],
                          Info=JoinOpInfo(JOIN_INNER, [eq(col(0, 2, I), S.col("supplier", "s_suppkey", 1))]))
    types = types + [I]
    j3 = PhysicalOperator(POT_Join, Children=[j2, ps], Outputs=up(types) + [S.col("partsupp", "ps_supplycost", 1)],
                          Info=JoinOpInfo(JOIN_INNER, [eq(col(0, 2, I), S.col("partsupp", "ps_suppkey", 1)),
                                                       eq(col(0, 1, I), S.col("partsupp", "ps_partkey", 1))]))
    types = types + [DEC15_2]
    j4 = PhysicalOperator(POT_Join, Children=[j3, orders], Outputs=up(types) + [S.col("orders", "o_orderdate", 1)],
                          Info=JoinOpInfo(JOIN_INNER, [eq(col(0, 0, BI), S.col("orders", "o_orderkey", 1))]))
    types = types + [D]
    j5 = PhysicalOperator(POT_Join, Children=[j4, nation], Outputs=up(types) + [S.col("nation", "n_name", 1)],
                          Info=JoinOpInfo(JOIN_INNER, [eq(col(0, 6, I), S.col("nation", "n_nationkey", 1))]))
    # amount: DECIMAL(18,4) product minus DECIMAL x cast(INTEGER) product (value scale 2), Sub -> scale 4
    amount = func("-", K.DecimalType(18, 4), _disc_price(col(0, 4, DEC15_2), col(0, 5, DEC15_2)),
                  func("*", K.DecimalType(18, 4), col(0, 7, DEC15_2), cast(col(0, 3, I), DEC15_2)))
    sum_t = K.DecimalType(38, 4)
    groups = [col(0, 9, V), func("extract", I, const("year", V), col(0, 8, D))]
    outs = [col(0, 0, V), col(0, 1, I), col(1, 0, sum_t)]
    aggs = [func(agg, sum_t, amount)]            # agg="avg": avg(DECIMAL) = sum.Quo(count) -> DECIMAL(38,4)
    if agg == "avg":
        aggs.append(func("count", K.HugeintType(), col(0, 0, BI)))
        outs.append(col(1, 1, K.HugeintType()))
    node = PhysicalOperator(POT_Agg, Outputs=outs, Children=[j5], Info=AggOpInfo(aggs, groups))
    return PhysicalOperator(POT_Order, Outputs=outs, Children=[node], Info=OrderOpInfo([(col(0, 0, V), False), (col(0, 1, I), True)]))


def part_like_plan(pattern, schema=FULL):
    """select count(p_partkey), sum(p_partkey) from part where p_name like <pattern>"""
    S = schema
    H = K.HugeintType()
    scan = PhysicalOperator(POT_Scan, Info=ScanOpInfo("part"),
                            Filters=[func("like", K.LType(K.LTID_BOOLEAN), S.col("part", "p_name"), const(pattern, K.VarcharType()))])
    pk = S.col("part", "p_partkey")
    aggs = [func("count", H, pk), func("sum", H, pk)]
    return PhysicalOperator(POT_Agg, Outputs=[col(1, 0, H), col(1, 1, H)], Children=[scan], Info=AggOpInfo(aggs, []))


def customer_filter_plan(filters, schema=FULL):
    """select count(*), sum(c_nationkey), sum(c_custkey) from customer where <filters>:
    a scan-aggregate over customer used to exercise string predicates (LIKE / NOT LIKE / = / <> on the
    VARCHAR c_name, LIKE on the dictionary column c_mktsegment).  filters: list of (column, op, literal)."""
    S = schema
    B = K.LType(K.LTID_BOOLEAN)
    fl = [func(op, B, S.col("customer", cname), const(lit, K.VarcharType())) for cname, op, lit in filters]
    scan = PhysicalOperator(POT_Scan, Filters=fl, Info=ScanOpInfo("customer"))
    H = K.HugeintType()
    ck = S.col("customer", "c_custkey")
    aggs = [func("count", H, ck), func("sum", H, S.col("customer", "c_nationkey")), func("sum", H, ck)]
    outs = [col(1, i, a.DataTyp) for i, a in enumerate(aggs)]
    return PhysicalOperator(POT_Agg, Outputs=outs, Children=[scan], Info=AggOpInfo(aggs, []))


def exists_plan(negated=False, odate_lt=None, ship_gt=None, schema=FULL):
    """EXISTS / NOT EXISTS as the reference plans it (builder_plan.go:380-429): a MARK / AntiMARK join whose extra
    boolean output is filtered with `mark = true` / `mark = false` (the shape of TPC-H Q4, Q21, Q22):
        select o_custkey, sum(o_totalprice), count(*) from orders
        where o_orderdate < d and [not] exists (select * from lineitem where l_orderkey = o_orderkey and l_shipdate > s)
        group by o_custkey
    The same rows as semi_plan(anti=negated)."""
    S = schema
    odate_lt = days(1995, 3, 29) if odate_lt is None else odate_lt
    ship_gt = days(1995, 3, 29) if ship_gt is None else ship_gt
    B = K.LType(K.LTID_BOOLEAN)
    orders = PhysicalOperator(POT_Scan, Info=ScanOpInfo("orders"),
                              Filters=[func("<", B, S.col("orders", "o_orderdate"), const(odate_lt, K.DateType()))])
    line = PhysicalOperator(POT_Scan, Info=ScanOpInfo("lineitem"),
                            Filters=[func(">", B, S.col("lineitem", "l_shipdate"), const(ship_gt, K.DateType()))])
    OI = S.idx["orders"]
    j = PhysicalOperator(
        POT_Join, Children=[orders, line],
        Outputs=[col(0, OI["o_custkey"], K.IntegerType()), col(0, OI["o_totalprice"], DEC15_2), col(2, 0, B)],   # side 2: the mark column
        Info=JoinOpInfo(JOIN_ANTI_MARK if negated else JOIN_MARK,
                        [func("=", B, S.col("orders", "o_orderkey", 0), S.col("lineitem", "l_orderkey", 1))]))
    flt = PhysicalOperator(POT_Filter, Outputs=j.Outputs, Children=[j], Filters=[func("=", B, col(0, 2, B), const(0 if negated else 1, B))])
    aggs = [func("sum", K.DecimalType(38, 2), col(0, 1, DEC15_2)), func("count", K.HugeintType(), col(0, 0, K.IntegerType()))]
    outs = [col(0, 0, K.IntegerType()), col(1, 0, K.DecimalType(38, 2)), col(1, 1, K.HugeintType())]
    return PhysicalOperator(POT_Agg, Outputs=outs, Children=[flt], Info=AggOpInfo(aggs, [col(0, 0, K.IntegerType())]))


def q3_topk_plan(limit=10, **kw):
    """Limit <- Order(revenue desc, o_orderdate) <- Agg(...) : the whole Q3 tail below the final
    Project, fused into the GPU pipeline (device top-k; SURVEY.md 8f-1)."""
    agg = q3_plan(**kw)
    order = PhysicalOperator(POT_Order, Outputs=agg.Outputs, Children=[agg],
                             Info=OrderOpInfo([(col(0, 1, K.DecimalType(38, 4)), True), (col(0, 2, K.DateType()), False)]))
    return PhysicalOperator(POT_Limit, Outputs=agg.Outputs, Children=[order], Info=LimitOpInfo(limit))


# ----------------------------------------------------------------- tables --

def generate_device_tables(sf, order_lo=0, order_hi=None, want=("lineitem", "orders", "customer"), partsupp_shard=None):
    """dbgen-equivalent tables generated directly in HBM (plangpu_tpch.h).  partsupp_shard=(rank, world): only
    that rank's row range of partsupp is generated (a SHARDED build side keyed differently from the lineitem
    shards -- Q9 then takes the all-to-all row exchange instead of a replicated partsupp)."""
    lib = L.lib()
    if order_hi is None:
        order_hi = lib.pg_tpch_num_orders(sf)
    out = {}
    ho, hl = C.c_void_p(), C.c_void_p()
    if "lineitem" in want or "orders" in want:
        L.check(lib.pg_tpch_orders_lineitem(sf, order_lo, order_hi,
                                            C.byref(ho) if "orders" in want else None,
                                            C.byref(hl) if "lineitem" in want else None))
        if "orders" in want:
            out["orders"] = DeviceTable("orders", ho, ORDERS)
        if "lineitem" in want:
            out["lineitem"] = DeviceTable("lineitem", hl, LINEITEM)
    if "customer" in want:
        hc = C.c_void_p()
        L.check(lib.pg_tpch_customer(sf, 0, lib.pg_tpch_num_customers(sf), C.byref(hc)))
        out["customer"] = DeviceTable("customer", hc, CUSTOMER)
    for name, fn, schema in (("part", lib.pg_tpch_part, PART), ("supplier", lib.pg_tpch_supplier, SUPPLIER),
                             ("partsupp", lib.pg_tpch_partsupp, PARTSUPP)):
        if name in want:
            h = C.c_void_p()
            if name == "partsupp" and partsupp_shard is not None:
                r, w = partsupp_shard
                n = 4 * lib.pg_tpch_num_parts(sf)
                L.check(lib.pg_tpch_partsupp_range(sf, n * r // w, n * (r + 1) // w, C.byref(h)))
            else:
                L.check(fn(sf, C.byref(h)))
            out[name] = DeviceTable(name, h, schema)
    if "nation" in want:
        h = C.c_void_p()
        L.check(lib.pg_tpch_nation(C.byref(h)))
        out["nation"] = DeviceTable("nation", h, NATION)
    return out


ALL_TABLES = ("lineitem", "orders", "customer", "part", "supplier", "partsupp", "nation")


def upload_tables(host, global_offsets=None, schema=FULL):
    """host: {table: {column: numpy array}} (e.g. from the CPU generator) -> sealed DeviceTables."""
    schemas = schema.tables
    out = {}
    for name, cols in host.items():
        t = DeviceTable.create(name, schemas[name])
        t.append([cols[c[0]] for c in schemas[name]])
        t.seal((global_offsets or {}).get(name, 0))
        out[name] = t
    return out


# ---- TPC-H Q12 / Q14: CASE inside aggregates over a join (row programs over the joined rows, rows.cu aggregate mode) ----

SHIPMODES = ["REG AIR", "AIR", "RAIL", "TRUCK", "MAIL", "FOB", "SHIP"]           # dbgen smode / o_oprio / p_types member order
PRIORITIES = ["1-URGENT", "2-HIGH", "3-MEDIUM", "4-NOT SPECIFIED", "5-LOW"]
PTYPES = ["%s %s %s" % (a, b, c) for a in ("STANDARD", "SMALL", "MEDIUM", "LARGE", "ECONOMY", "PROMO")
          for b in ("ANODIZED", "BURNISHED", "PLATED", "POLISHED", "BRUSHED") for c in ("TIN", "NICKEL", "BRASS", "STEEL", "COPPER")]
Q12_LINEITEM = [("l_orderkey", L.PG_T_INT64, 0, 0, None), ("l_shipmode", L.PG_T_DICT8, 0, 0, SHIPMODES), ("l_shipdate", L.PG_T_DATE32, 0, 0, None),
                ("l_commitdate", L.PG_T_DATE32, 0, 0, None), ("l_receiptdate", L.PG_T_DATE32, 0, 0, None)]
Q12_ORDERS = [("o_orderkey", L.PG_T_INT64, 0, 0, None), ("o_orderpriority", L.PG_T_DICT8, 0, 0, PRIORITIES)]
Q14_LINEITEM = [("l_partkey", L.PG_T_INT32, 0, 0, None), ("l_extendedprice", L.PG_T_DECIMAL64, 15, 2, None),
                ("l_discount", L.PG_T_DECIMAL64, 15, 2, None), ("l_shipdate", L.PG_T_DATE32, 0, 0, None)]
Q14_PART = [("p_partkey", L.PG_T_INT32, 0, 0, None), ("p_type", L.PG_T_DICT8, 0, 0, PTYPES)]


def q12_plan(modes=("FOB", "TRUCK"), year=1996):
    """cases/tpch/query/q12.sql:  Agg(group by l_shipmode; sum(case when o_orderpriority = '1-URGENT' or o_orderpriority =
    '2-HIGH' then 1 else 0 end), sum(case when o_orderpriority <> '1-URGENT' and o_orderpriority <> '2-HIGH' then 1 else 0 end))
      <- Join(l_orderkey = o_orderkey) <- { Scan(lineitem; l_shipmode in (..), l_commitdate < l_receiptdate,
                                                 l_shipdate < l_commitdate, l_receiptdate in [year, year+1)), Scan(orders) }
    The ORDER BY l_shipmode stays with the host parents."""
    S = Schema(lineitem=Q12_LINEITEM, orders=Q12_ORDERS)
    B, V, I, H, D = K.LType(K.LTID_BOOLEAN), K.VarcharType(), K.IntegerType(), K.HugeintType(), K.DateType()
    lc = lambda n: S.col("lineitem", n)   # noqa: E731
    line = PhysicalOperator(POT_Scan, Info=ScanOpInfo("lineitem"), Filters=[
        func("in", B, lc("l_shipmode"), *[const(m, V) for m in modes]),
        func("<", B, lc("l_commitdate"), lc("l_receiptdate")),
        func("<", B, lc("l_shipdate"), lc("l_commitdate")),
        func(">=", B, lc("l_receiptdate"), const(days(year, 1, 1), D)),
        func("<", B, lc("l_receiptdate"), const(days(year + 1, 1, 1), D))])
    orders = PhysicalOperator(POT_Scan, Info=ScanOpInfo("orders"))
    LI, OI = S.idx["lineitem"], S.idx["orders"]
    j = PhysicalOperator(POT_Join, Children=[line, orders], Outputs=[col(0, LI["l_shipmode"], V), col(1, OI["o_orderpriority"], V)],
                         Info=JoinOpInfo(JOIN_INNER, [func("=", B, S.col("lineitem", "l_orderkey", 0), S.col("orders", "o_orderkey", 1))]))
    prio = col(0, 1, V)
    high = func("case", I, const(0, I), func("or", B, func("=", B, prio, const("1-URGENT", V)), func("=", B, prio, const("2-HIGH", V))), const(1, I))
    low = func("case", I, const(0, I), func("and", B, func("<>", B, prio, const("1-URGENT", V)), func("<>", B, prio, const("2-HIGH", V))), const(1, I))
    aggs = [func("sum", H, high), func("sum", H, low)]
    outs = [col(0, 0, V), col(1, 0, H), col(1, 1, H)]
    return PhysicalOperator(POT_Agg, Outputs=outs, Children=[j], Info=AggOpInfo(aggs, [col(0, 0, V)]))


def q14_plan(date_lo=None, date_hi=None, pattern="PROMO%"):
    """cases/tpch/query/q14.sql below its final projection:  Agg(sum(case when p_type like 'PROMO%' then l_extendedprice * (1 -
    l_discount) else 0 end), sum(l_extendedprice * (1 - l_discount))) <- Join(l_partkey = p_partkey) <- { Scan(lineitem; l_shipdate
    in [d, d + 1 month)), Scan(part) }.  `100.00 * a / b` is a FLOAT projection above the aggregate and stays with the host."""
    S = Schema(lineitem=Q14_LINEITEM, part=Q14_PART)
    B, V, I, D = K.LType(K.LTID_BOOLEAN), K.VarcharType(), K.IntegerType(), K.DateType()
    date_lo = days(1996, 4, 1) if date_lo is None else date_lo
    date_hi = days(1996, 5, 1) if date_hi is None else date_hi
    lc = lambda n: S.col("lineitem", n)   # noqa: E731
    line = PhysicalOperator(POT_Scan, Info=ScanOpInfo("lineitem"), Filters=[func(">=", B, lc("l_shipdate"), const(date_lo, D)),
                                                                           func("<", B, lc("l_shipdate"), const(date_hi, D))])
    part = PhysicalOperator(POT_Scan, Info=ScanOpInfo("part"))
    LI, PI = S.idx["lineitem"], S.idx["part"]
    j = PhysicalOperator(POT_Join, Children=[line, part],
                         Outputs=[col(0, LI["l_extendedprice"], DEC15_2), col(0, LI["l_discount"], DEC15_2), col(1, PI["p_type"], V)],
                         Info=JoinOpInfo(JOIN_INNER, [func("=", B, S.col("lineitem", "l_partkey", 0), S.col("part", "p_partkey", 1))]))
    rev = _disc_price(col(0, 0, DEC15_2), col(0, 1, DEC15_2))
    promo = func("case", K.DecimalType(18, 4), cast(const(0, I), K.DecimalType(18, 4)), func("like", B, col(0, 2, V), const(pattern, V)), rev)
    aggs = [func("sum", K.DecimalType(38, 4), promo), func("sum", K.DecimalType(38, 4), rev)]
    return PhysicalOperator(POT_Agg, Outputs=[col(1, 0, K.DecimalType(38, 4)), col(1, 1, K.DecimalType(38, 4))], Children=[j], Info=AggOpInfo(aggs, []))


Q4_ORDERS = [("o_orderkey", L.PG_T_INT64, 0, 0, None), ("o_orderdate", L.PG_T_DATE32, 0, 0, None), ("o_orderpriority", L.PG_T_DICT8, 0, 0, PRIORITIES)]
Q4_LINEITEM = [("l_orderkey", L.PG_T_INT64, 0, 0, None), ("l_commitdate", L.PG_T_DATE32, 0, 0, None), ("l_receiptdate", L.PG_T_DATE32, 0, 0, None)]


def q4_plan(date_lo=None, date_hi=None):
    """cases/tpch/query/q4.sql as the reference plans it: the EXISTS becomes a MARK join under Filter(mark = true)
    (builder_plan.go:380-429); the build side carries the column-to-column filter l_commitdate < l_receiptdate.
      Agg(group by o_orderpriority; count(*)) <- Filter(mark = true) <- MarkJoin(o_orderkey = l_orderkey)
          <- { Scan(orders; o_orderdate in [d, d + 3 months)), Scan(lineitem; l_commitdate < l_receiptdate) }"""
    S = Schema(orders=Q4_ORDERS, lineitem=Q4_LINEITEM)
    B, V, H, D = K.LType(K.LTID_BOOLEAN), K.VarcharType(), K.HugeintType(), K.DateType()
    date_lo = days(1997, 7, 1) if date_lo is None else date_lo
    date_hi = days(1997, 10, 1) if date_hi is None else date_hi
    orders = PhysicalOperator(POT_Scan, Info=ScanOpInfo("orders"), Filters=[func(">=", B, S.col("orders", "o_orderdate"), const(date_lo, D)),
                                                                           func("<", B, S.col("orders", "o_orderdate"), const(date_hi, D))])
    line = PhysicalOperator(POT_Scan, Info=ScanOpInfo("lineitem"), Filters=[func("<", B, S.col("lineitem", "l_commitdate"), S.col("lineitem", "l_receiptdate"))])
    OI = S.idx["orders"]
    j = PhysicalOperator(POT_Join, Children=[orders, line], Outputs=[col(0, OI["o_orderpriority"], V), col(0, OI["o_orderkey"], K.BigintType()), col(2, 0, B)],
                         Info=JoinOpInfo(JOIN_MARK, [func("=", B, S.col("orders", "o_orderkey", 0), S.col("lineitem", "l_orderkey", 1))]))
    flt = PhysicalOperator(POT_Filter, Outputs=j.Outputs, Children=[j], Filters=[func("=", B, col(0, 2, B), const(1, B))])
    aggs = [func("count", H, col(0, 1, K.BigintType()))]         # count(*) -> count(<first column>) (builder_binder.go:207-228)
    return PhysicalOperator(POT_Agg, Outputs=[col(0, 0, V), col(1, 0, H)], Children=[flt], Info=AggOpInfo(aggs, [col(0, 0, V)]))


BRANDS = ["Brand#%d%d" % (m, n) for m in range(1, 6) for n in range(1, 6)]
CONTAINERS = ["%s %s" % (a, b) for a in ("SM", "LG", "MED", "JUMBO", "WRAP") for b in ("CASE", "BOX", "BAG", "JAR", "PKG", "PACK", "CAN", "DRUM")]
SHIPINSTRUCT = ["DELIVER IN PERSON", "COLLECT COD", "NONE", "TAKE BACK RETURN"]
Q19_LINEITEM = [("l_partkey", L.PG_T_INT32, 0, 0, None), ("l_quantity", L.PG_T_INT32, 0, 0, None), ("l_extendedprice", L.PG_T_DECIMAL64, 15, 2, None),
                ("l_discount", L.PG_T_DECIMAL64, 15, 2, None), ("l_shipmode", L.PG_T_DICT8, 0, 0, SHIPMODES), ("l_shipinstruct", L.PG_T_DICT8, 0, 0, SHIPINSTRUCT)]
Q19_PART = [("p_partkey", L.PG_T_INT32, 0, 0, None), ("p_brand", L.PG_T_DICT8, 0, 0, BRANDS), ("p_size", L.PG_T_INT32, 0, 0, None),
            ("p_container", L.PG_T_DICT8, 0, 0, CONTAINERS)]
Q19_GROUPS = (("Brand#23", ("SM CASE", "SM BOX", "SM PACK", "SM PKG"), 5, 5), ("Brand#15", ("MED BAG", "MED BOX", "MED PKG", "MED PACK"), 14, 10),
              ("Brand#44", ("LG CASE", "LG BOX", "LG PACK", "LG PKG"), 28, 15))


def q19_plan():
    """cases/tpch/query/q19.sql with the join condition common to the three OR branches taken out (what lets the reference plan
    a hash join at all):  Agg(sum(l_extendedprice * (1 - l_discount))) <- Filter(g1 OR g2 OR g3) <- Join(l_partkey = p_partkey)
    <- { Scan(lineitem), Scan(part) }; every g_i is an AND of string equalities / IN lists on dictionary columns of BOTH sides and
    integer ranges -- a general OR above a join, evaluated per joined row."""
    S = Schema(lineitem=Q19_LINEITEM, part=Q19_PART)
    B, V, I = K.LType(K.LTID_BOOLEAN), K.VarcharType(), K.IntegerType()
    LI, PI = S.idx["lineitem"], S.idx["part"]
    line = PhysicalOperator(POT_Scan, Info=ScanOpInfo("lineitem"))
    part = PhysicalOperator(POT_Scan, Info=ScanOpInfo("part"))
    jouts = [col(0, LI["l_quantity"], I), col(0, LI["l_extendedprice"], DEC15_2), col(0, LI["l_discount"], DEC15_2), col(0, LI["l_shipmode"], V),
             col(0, LI["l_shipinstruct"], V), col(1, PI["p_brand"], V), col(1, PI["p_size"], I), col(1, PI["p_container"], V)]
    j = PhysicalOperator(POT_Join, Children=[line, part], Outputs=jouts,
                         Info=JoinOpInfo(JOIN_INNER, [func("=", B, S.col("lineitem", "l_partkey", 0), S.col("part", "p_partkey", 1))]))
    qty, mode, instr, brand, size, cont = col(0, 0, I), col(0, 3, V), col(0, 4, V), col(0, 5, V), col(0, 6, I), col(0, 7, V)
    groups = []
    for b, conts, q0, smax in Q19_GROUPS:
        groups.append(func("and", B, func("=", B, brand, const(b, V)), func("in", B, cont, *[const(c, V) for c in conts]),
                           func(">=", B, qty, const(q0, I)), func("<=", B, qty, const(q0 + 10, I)),
                           func(">=", B, size, const(1, I)), func("<=", B, size, const(smax, I)),          # between 1 and smax
                           func("in", B, mode, const("AIR", V), const("AIR REG", V)), func("=", B, instr, const("DELIVER IN PERSON", V))))
    flt = PhysicalOperator(POT_Filter, Outputs=jouts, Children=[j], Filters=[func("or", B, *groups)])
    agg = func("sum", K.DecimalType(38, 4), _disc_price(col(0, 1, DEC15_2), col(0, 2, DEC15_2)))
    return PhysicalOperator(POT_Agg, Outputs=[col(1, 0, K.DecimalType(38, 4))], Children=[flt], Info=AggOpInfo([agg], []))


# ---------------------------------------------------------------------------------------------------------------------
# Q5 / Q7 / Q8: multi-way joins through customer / supplier to nation (and region).  Plan trees only: they are executed by the
# tree-walking oracle on the CPU (tests/test_oracle_golden.py) and their descriptors compile on the CPU; they were written after
# the round's GPU budget was spent and have NOT been run through the GPU path.
REGIONS = ["AFRICA", "AMERICA", "ASIA", "EUROPE", "MIDDLE EAST"]
NATION_REGION = [0, 1, 1, 1, 4, 0, 3, 3, 2, 2, 4, 4, 2, 4, 0, 0, 0, 1, 2, 3, 4, 2, 3, 3, 1]          # n_regionkey by n_nationkey (dbgen)
NATION_R = NATION + [("n_regionkey", L.PG_T_INT32, 0, 0, None)]
REGION = [("r_regionkey", L.PG_T_INT32, 0, 0, None), ("r_name", L.PG_T_DICT8, 0, 0, REGIONS)]
Q8_PART = [("p_partkey", L.PG_T_INT32, 0, 0, None), ("p_type", L.PG_T_DICT8, 0, 0, PTYPES)]


class _Stack:
    """a left-deep join stack that keeps track of the running output layout by column NAME"""

    def __init__(self, table, cols, names, filters=None):
        self.cols = cols                                      # {table: schema}
        idx = {c[0]: i for i, c in enumerate(cols[table])}
        self.node = PhysicalOperator(POT_Scan, Info=ScanOpInfo(table), Filters=filters or [])
        self.layout = None                                    # None: the node is the bare scan, columns by table position
        self.table, self.idx0 = table, idx
        self.keep = list(names)

    def ref(self, name):
        if self.layout is None:
            i = self.idx0[name]
            return col(0, i, _ltype_of(self.cols[self.table][i]))
        i, t = self.layout[name]
        return col(0, i, t)

    def join(self, table, on, take, filters=None, alias=None, jt=JOIN_INNER):
        """on: [(left name, right column)], take: right columns appended to the layout (as alias + name when aliased)"""
        B = K.LType(K.LTID_BOOLEAN)
        sch = self.cols[table]
        ridx = {c[0]: i for i, c in enumerate(sch)}
        right = PhysicalOperator(POT_Scan, Info=ScanOpInfo(table), Filters=filters or [])
        rref = lambda n: col(1, ridx[n], _ltype_of(sch[ridx[n]]))   # noqa: E731
        conds = [func("=", B, self.ref(l), rref(r)) for l, r in on]
        names = self.keep if self.layout is None else list(self.layout)
        outs, layout = [], {}
        for n in names:
            e = self.ref(n)
            layout[n] = (len(outs), e.DataTyp)
            outs.append(e)
        for n in take:
            e = rref(n)
            layout[(alias or "") + n] = (len(outs), e.DataTyp)
            outs.append(e)
        self.node = PhysicalOperator(POT_Join, Children=[self.node, right], Outputs=outs, Info=JoinOpInfo(jt, conds))
        self.layout = layout
        return self


def q5_plan(region="AMERICA", year=1994):
    """cases/tpch/query/q5.sql:  Agg(group by n_name; sum(l_extendedprice * (1 - l_discount)))
      <- lineitem x orders[o_orderdate in year] x customer x supplier (l_suppkey = s_suppkey AND c_nationkey = s_nationkey)
         x nation x region[r_name = region], left-deep with the fact table leftmost.  ORDER BY revenue desc stays with the host."""
    B, V, D = K.LType(K.LTID_BOOLEAN), K.VarcharType(), K.DateType()
    cols = {"lineitem": LINEITEM, "orders": ORDERS, "customer": CUSTOMER, "supplier": SUPPLIER, "nation": NATION_R, "region": REGION}
    oi = {c[0]: i for i, c in enumerate(ORDERS)}
    od = col(0, oi["o_orderdate"], D)
    st = _Stack("lineitem", cols, ["l_orderkey", "l_suppkey", "l_extendedprice", "l_discount"])
    st.join("orders", [("l_orderkey", "o_orderkey")], ["o_custkey"],
            filters=[func(">=", B, od, const(days(year, 1, 1), D)), func("<", B, od, const(days(year + 1, 1, 1), D))])
    st.join("customer", [("o_custkey", "c_custkey")], ["c_nationkey"])
    st.join("supplier", [("l_suppkey", "s_suppkey"), ("c_nationkey", "s_nationkey")], ["s_nationkey"])
    st.join("nation", [("s_nationkey", "n_nationkey")], ["n_name", "n_regionkey"])
    st.join("region", [("n_regionkey", "r_regionkey")], [], filters=[func("=", B, col(0, 1, V), const(region, V))])
    sum_t = K.DecimalType(38, 4)
    agg = func("sum", sum_t, _disc_price(st.ref("l_extendedprice"), st.ref("l_discount")))
    return PhysicalOperator(POT_Agg, Outputs=[col(0, 0, V), col(1, 0, sum_t)], Children=[st.node], Info=AggOpInfo([agg], [st.ref("n_name")]))


def q7_plan(a="FRANCE", b="ARGENTINA"):
    """cases/tpch/query/q7.sql:  Agg(group by supp_nation, cust_nation, extract(year from l_shipdate); sum(volume))
      <- Filter((n1.n_name = a AND n2.n_name = b) OR (n1.n_name = b AND n2.n_name = a))
      <- lineitem[l_shipdate between 1995-01-01 and 1996-12-31] x supplier x orders x customer x nation n1 x nation n2."""
    B, V, I, D = K.LType(K.LTID_BOOLEAN), K.VarcharType(), K.IntegerType(), K.DateType()
    cols = {"lineitem": LINEITEM, "orders": ORDERS, "customer": CUSTOMER, "supplier": SUPPLIER, "nation": NATION}
    li = {c[0]: i for i, c in enumerate(LINEITEM)}
    sd = col(0, li["l_shipdate"], D)
    st = _Stack("lineitem", cols, ["l_orderkey", "l_suppkey", "l_extendedprice", "l_discount", "l_shipdate"],
                filters=[func(">=", B, sd, const(days(1995, 1, 1), D)), func("<=", B, sd, const(days(1996, 12, 31), D))])
    st.join("supplier", [("l_suppkey", "s_suppkey")], ["s_nationkey"])
    st.join("orders", [("l_orderkey", "o_orderkey")], ["o_custkey"])
    st.join("customer", [("o_custkey", "c_custkey")], ["c_nationkey"])
    st.join("nation", [("s_nationkey", "n_nationkey")], ["n_name"], alias="n1.")
    st.join("nation", [("c_nationkey", "n_nationkey")], ["n_name"], alias="n2.")
    n1, n2 = st.ref("n1.n_name"), st.ref("n2.n_name")
    pair = lambda x, y: func("and", B, func("=", B, n1, const(x, V)), func("=", B, n2, const(y, V)))   # noqa: E731
    flt = PhysicalOperator(POT_Filter, Outputs=list(st.node.Outputs), Children=[st.node], Filters=[func("or", B, pair(a, b), pair(b, a))])
    sum_t = K.DecimalType(38, 4)
    groups = [n1, n2, func("extract", I, const("year", V), st.ref("l_shipdate"))]
    agg = func("sum", sum_t, _disc_price(st.ref("l_extendedprice"), st.ref("l_discount")))
    outs = [col(0, 0, V), col(0, 1, V), col(0, 2, I), col(1, 0, sum_t)]
    return PhysicalOperator(POT_Agg, Outputs=outs, Children=[flt], Info=AggOpInfo([agg], groups))


def q8_plan(nation="ARGENTINA", region="AMERICA", ptype="ECONOMY BURNISHED TIN"):
    """cases/tpch/query/q8.sql below its final division:  Agg(group by extract(year from o_orderdate); sum(case when nation = X
    then volume else 0 end), sum(volume)) <- lineitem x part[p_type = ..] x supplier x orders[o_orderdate between 1995-01-01 and
    1996-12-31] x customer x nation n1 x region[r_name = ..] x nation n2.  mkt_share = a / b is a DECIMAL quotient above the
    aggregate (host side)."""
    B, V, I, D = K.LType(K.LTID_BOOLEAN), K.VarcharType(), K.IntegerType(), K.DateType()
    cols = {"lineitem": LINEITEM, "orders": ORDERS, "customer": CUSTOMER, "supplier": SUPPLIER, "nation": NATION_R, "region": REGION, "part": Q8_PART}
    oi = {c[0]: i for i, c in enumerate(ORDERS)}
    od = col(0, oi["o_orderdate"], D)
    st = _Stack("lineitem", cols, ["l_orderkey", "l_partkey", "l_suppkey", "l_extendedprice", "l_discount"])
    st.join("part", [("l_partkey", "p_partkey")], [], filters=[func("=", B, col(0, 1, V), const(ptype, V))])
    st.join("supplier", [("l_suppkey", "s_suppkey")], ["s_nationkey"])
    st.join("orders", [("l_orderkey", "o_orderkey")], ["o_custkey", "o_orderdate"],
            filters=[func(">=", B, od, const(days(1995, 1, 1), D)), func("<=", B, od, const(days(1996, 12, 31), D))])
    st.join("customer", [("o_custkey", "c_custkey")], ["c_nationkey"])
    st.join("nation", [("c_nationkey", "n_nationkey")], ["n_regionkey"], alias="n1.")
    st.join("region", [("n1.n_regionkey", "r_regionkey")], [], filters=[func("=", B, col(0, 1, V), const(region, V))])
    st.join("nation", [("s_nationkey", "n_nationkey")], ["n_name"], alias="n2.")
    sum_t, v_t = K.DecimalType(38, 4), K.DecimalType(18, 4)
    vol = _disc_price(st.ref("l_extendedprice"), st.ref("l_discount"))
    mine = func("case", v_t, cast(const(0, I), v_t), func("=", B, st.ref("n2.n_name"), const(nation, V)), vol)
    groups = [func("extract", I, const("year", V), st.ref("o_orderdate"))]
    outs = [col(0, 0, I), col(1, 0, sum_t), col(1, 1, sum_t)]
    return PhysicalOperator(POT_Agg, Outputs=outs, Children=[st.node], Info=AggOpInfo([func("sum", sum_t, mine), func("sum", sum_t, vol)], groups))


Q13_CUSTOMER = [("c_custkey", L.PG_T_INT32, 0, 0, None)]
Q13_ORDERS = [("o_orderkey", L.PG_T_INT64, 0, 0, None), ("o_custkey", L.PG_T_INT32, 0, 0, None), ("o_comment", L.PG_T_VARCHAR, 79, 0, None)]


def q13_plan(pattern="%pending%accounts%", outer=True):
    """cases/tpch/query/q13.sql:  Agg(group by c_count; count(*)) <- Agg(group by c_custkey; count(o_orderkey))
      <- LeftJoin(c_custkey = o_custkey) <- { Scan(customer), Scan(orders; o_comment not like pattern) }.
    The ON-clause predicate on orders alone filters the build side; customers without a surviving order keep one NULL-padded row,
    over which count(o_orderkey) is NULL in the reference (CountOp.Finalize) -- q13.txt's first row.  The GPU runs it as a grouped
    LEFT-join count (join.cu build_left_count).  outer=False: the inner aggregate alone, (c_custkey, c_count) per customer."""
    B, V, I, BI, H = K.LType(K.LTID_BOOLEAN), K.VarcharType(), K.IntegerType(), K.BigintType(), K.HugeintType()
    cust = PhysicalOperator(POT_Scan, Info=ScanOpInfo("customer"))
    orders = PhysicalOperator(POT_Scan, Info=ScanOpInfo("orders"), Filters=[func("not like", B, col(0, 2, V), const(pattern, V))])
    j = PhysicalOperator(POT_Join, Children=[cust, orders], Outputs=[col(0, 0, I), col(1, 0, BI)],
                         Info=JoinOpInfo(JOIN_LEFT, [func("=", B, col(0, 0, I), col(1, 1, I))]))
    per_cust = PhysicalOperator(POT_Agg, Outputs=[col(0, 0, I), col(1, 0, H)], Children=[j], Info=AggOpInfo([func("count", H, col(0, 1, BI))], [col(0, 0, I)]))
    if not outer:
        return per_cust
    return PhysicalOperator(POT_Agg, Outputs=[col(0, 0, H), col(1, 0, H)], Children=[per_cust], Info=AggOpInfo([func("count", H)], [col(0, 1, H)]))


Q10_CUSTOMER = [("c_custkey", L.PG_T_INT32, 0, 0, None), ("c_name", L.PG_T_VARCHAR, 25, 0, None), ("c_acctbal", L.PG_T_DECIMAL64, 15, 2, None),
                ("c_nationkey", L.PG_T_INT32, 0, 0, None), ("c_address", L.PG_T_VARCHAR, 40, 0, None), ("c_phone", L.PG_T_VARCHAR, 15, 0, None),
                ("c_comment", L.PG_T_VARCHAR, 117, 0, None)]


def q10_plan(date_lo=None, date_hi=None, limit=20, agg="sum"):
    """cases/tpch/query/q10.sql:  Limit(20) <- Order(revenue desc) <- Agg(group by c_custkey, c_name, c_acctbal, c_phone, n_name,
    c_address, c_comment; sum(l_extendedprice * (1 - l_discount))) <- lineitem[l_returnflag = 'R'] x orders[o_orderdate in the
    quarter] x customer x nation.  Seven group keys, four of them strings, one a signed DECIMAL.  The GPU runs it as a star join
    grouped by customer rows (every key depends on the customer row; n_name through c_nationkey), with the ORDER BY ... LIMIT
    pre-selected on the device.  limit=None: the bare aggregate.  agg="avg": avg(DECIMAL) = sum.Quo(count), plus count(*)."""
    B, V, D = K.LType(K.LTID_BOOLEAN), K.VarcharType(), K.DateType()
    date_lo = days(1993, 3, 1) if date_lo is None else date_lo
    date_hi = days(1993, 6, 1) if date_hi is None else date_hi
    cols = {"lineitem": LINEITEM, "orders": ORDERS, "customer": Q10_CUSTOMER, "nation": NATION}
    li, oi = {c[0]: i for i, c in enumerate(LINEITEM)}, {c[0]: i for i, c in enumerate(ORDERS)}
    od = col(0, oi["o_orderdate"], D)
    st = _Stack("lineitem", cols, ["l_orderkey", "l_extendedprice", "l_discount"], filters=[func("=", B, col(0, li["l_returnflag"], V), const("R", V))])
    st.join("orders", [("l_orderkey", "o_orderkey")], ["o_custkey"], filters=[func(">=", B, od, const(date_lo, D)), func("<", B, od, const(date_hi, D))])
    st.join("customer", [("o_custkey", "c_custkey")], ["c_custkey", "c_name", "c_acctbal", "c_nationkey", "c_address", "c_phone", "c_comment"])
    st.join("nation", [("c_nationkey", "n_nationkey")], ["n_name"])
    keys = [st.ref(n) for n in ("c_custkey", "c_name", "c_acctbal", "c_phone", "n_name", "c_address", "c_comment")]
    sum_t = K.DecimalType(38, 4)
    aggs = [func(agg, sum_t, _disc_price(st.ref("l_extendedprice"), st.ref("l_discount")))]
    # select list order: c_custkey, c_name, revenue, c_acctbal, n_name, c_address, c_phone, c_comment
    outs = [col(0, 0, keys[0].DataTyp), col(0, 1, V), col(1, 0, sum_t), col(0, 2, keys[2].DataTyp), col(0, 4, V), col(0, 5, V), col(0, 3, V), col(0, 6, V)]
    if agg == "avg":
        aggs.append(func("count", K.HugeintType(), st.ref("l_orderkey")))
        outs.append(col(1, 1, K.HugeintType()))
    node = PhysicalOperator(POT_Agg, Outputs=outs, Children=[st.node], Info=AggOpInfo(aggs, keys))
    if limit is None:
        return node
    order = PhysicalOperator(POT_Order, Outputs=outs, Children=[node], Info=OrderOpInfo([(col(0, 2, sum_t), True)]))
    return PhysicalOperator(POT_Limit, Outputs=outs, Children=[order], Info=LimitOpInfo(limit))
