"""GPU parity on value ranges that dbgen data never produces.

The CUDA path picks its kernel, and the arithmetic that kernel does, from the statistics of the sealed columns:
frame-of-reference narrowing (logical = base + stored at 1, 2 or 4 bytes, table.cu choose_encoding), predicate
bounds moved into the stored domain (scanagg.cu stored_range), narrow / wide / staged / acc32 variants, the
low-cardinality group limit, and four high-cardinality group-by paths.  dbgen columns are non-negative and start
near 0, so with them `base` is 0 and most of that decision tree never runs.  Here SF0.1 columns are transformed
deterministically (shifted, negated, recentred, recoded, forced to the exact width edges), uploaded, and every
query is compared bit for bit with the CPU oracle under each kernel-selection switch, with the kernel variant that
ran asserted from Explain() (scan-aggregates) or the PG_TRACE marks (group-by paths)."""
import ctypes as C
import re

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

I32_MIN, I32_MAX = -2 ** 31, 2 ** 31 - 1
D92 = 8035                      # 1992-01-01
N_SCAN = 200_000                # lineitem rows of the scan-aggregate cases


# ------------------------------------------------------------------ helpers --

def _run(plan, tables):
    from plan_b200 import compute as X
    ex = X.gpuPipelineExec(plan, tables)
    ex.Init()
    chunks = X.drain(ex)
    stats, explain = ex.stats, ex.Explain()
    ex.Close()
    return chunks, stats, explain


def _dec(vec, r):
    x = vec.Data[r]
    return (int(x["coef"]), int(x["scale"]), int(x["neg"]))


def _dec_value(t):
    return (-1 if t[2] else 1) * t[0], t[1]


def _same_decimal(a, b):
    (va, sa), (vb, sb) = _dec_value(a), _dec_value(b)
    s = max(sa, sb)
    return va * 10 ** (s - sa) == vb * 10 ** (s - sb)


def encoding(vmin, vmax, native):
    """Python restatement of choose_encoding (table.cu): the narrowest stored width for [vmin, vmax] and its base."""
    span = vmax - vmin
    pw, base = native, 0
    if span <= 0xff:
        pw, base = 1, (0 if vmin >= 0 and vmax <= 0xff else vmin)
    elif span <= 0xffff:
        pw, base = 2, (0 if vmin >= 0 and vmax <= 0xffff else vmin)
    elif span <= 0xffffffff and native == 8:
        pw = 4
        if I32_MIN <= vmin and vmax <= I32_MAX:
            base = 0
        else:
            base = vmin if span <= I32_MAX else vmin + 2 ** 31
    if pw >= native:
        pw, base = native, 0
    return pw, base


def _upload(name, schema, cols, pack=True):
    from plan_b200 import compute as X
    t = X.DeviceTable.create(name, schema)
    t.append([cols[c[0]] for c in schema])
    if pack:
        t.seal()
    else:
        with pytest.MonkeyPatch.context() as mp:      # PG_NO_PACK is read at seal time
            mp.setenv("PG_NO_PACK", "1")
            t.seal()
    return t


def _check_round_trip(t, host, schema, pack):
    """read_column returns the host array unchanged (pack_kernel / widen_kernel at every width and base), and the
    stored encoding is the one choose_encoding picks (native when packing is off)."""
    from plan_b200 import _lib as L
    for cname, ptype, *_ in schema:
        a = host[cname]
        assert np.array_equal(t.read_column(cname), a), cname
        if ptype in (L.PG_T_INT32, L.PG_T_INT64, L.PG_T_DATE32, L.PG_T_DECIMAL64) and len(a):
            native = 8 if ptype in (L.PG_T_INT64, L.PG_T_DECIMAL64) else 4
            want = encoding(int(a.min()), int(a.max()), native) if pack else (native, 0)
            assert t.column_encoding(cname) == want, cname


# ------------------------------------------------------- scan value classes --
#
# Each class transforms the columns a query reads.  `enc` writes down the stored (width, base) the class must
# produce; `q6` / `q1` the kernel variant the default selection must reach (a substring of Explain()).

STAGED_FIXED = "_staged_kernel<bulk-copy ring, widths compiled in"
STAGED_RT = "_staged_kernel<bulk-copy ring, run-time widths"
SP_STAGED_FIXED, SP_STAGED_RT = "sumprod" + STAGED_FIXED, "sumprod" + STAGED_RT
LC_STAGED_FIXED, LC_STAGED_RT = "lowcard" + STAGED_FIXED, "lowcard" + STAGED_RT
SP_NARROW, SP_WIDE = "sumprod_kernel<narrow", "sumprod_kernel<wide"
LC_NARROW32, LC_WIDE64 = "lowcard_chain_kernel<narrow,acc32", "lowcard_chain_kernel<wide,acc64"
GENERIC = "ScanAgg[generic]"
DATES = ("l_shipdate", "l_commitdate", "l_receiptdate")


def _edge_rows(a, lo, hi, rows=(17, N_SCAN - 5)):
    a[rows[0]] = lo
    a[rows[1]] = hi


def _recode(line, rng, rf_codes, ls_codes, absent=()):
    n = len(line["l_returnflag"])
    rf = np.array(rf_codes, dtype=np.uint8)[rng.integers(0, len(rf_codes), n)]
    ls = np.array(ls_codes, dtype=np.uint8)[rng.integers(0, len(ls_codes), n)]
    for a, b in absent:                      # drop the pair (a, b): move those rows to the first present ls code
        m = (rf == a) & (ls == b)
        ls[m] = [c for c in ls_codes if c != b][0]
    line["l_returnflag"], line["l_linestatus"] = rf, ls


def _t_add(col, k):
    def f(line, rng):
        line[col] = (line[col].astype(np.int64) + k).astype(line[col].dtype)
    return f


def _t_dates(k):
    def f(line, rng):
        for c in DATES:
            line[c] = (line[c] + k).astype(np.int32)
    return f


def _t_price_recentred(line, rng):
    line["l_extendedprice"] = line["l_extendedprice"] + (np.arange(N_SCAN) % 2) * 3_000_000_000


def _t_neg(col):
    def f(line, rng):
        line[col] = -line[col]
    return f


def _t_neg_price_half(line, rng):
    line["l_extendedprice"] = np.where(rng.random(N_SCAN) < 0.5, -line["l_extendedprice"], line["l_extendedprice"])


def _t_edges(col, lo, hi):
    def f(line, rng):
        _edge_rows(line[col], lo, hi)
    return f


# name: (transform, {column: (stored width, base)}, default Q6 variant, default Q1 variant)
SCAN_CLASSES = {
    # base at width 1
    "qty_plus_1000": (_t_add("l_quantity", 1000), {"l_quantity": (1, 1001)}, SP_STAGED_FIXED, LC_STAGED_FIXED),
    "tax_plus_300": (_t_add("l_tax", 300), {"l_tax": (1, 300)}, SP_STAGED_FIXED, LC_STAGED_FIXED),
    # 1 - l_discount < 0: the staged Q1 kernel refuses negative factors
    "disc_plus_500": (_t_add("l_discount", 500), {"l_discount": (1, 500)}, SP_STAGED_FIXED, LC_NARROW32),
    # base at width 2
    "dates_plus_60000": (_t_dates(60000), {"l_shipdate": (2, 68037)}, SP_STAGED_FIXED, LC_STAGED_FIXED),
    "dates_minus_20000": (_t_dates(-20000), {"l_shipdate": (2, -11963)}, SP_STAGED_FIXED, LC_STAGED_FIXED),
    # width 4 with base = vmin: the logical values no longer fit 32 bits
    "price_plus_3e9": (_t_add("l_extendedprice", 3_000_000_000), {"l_extendedprice": (4, 3_000_090_500)}, SP_WIDE, LC_WIDE64),
    # width 4 with span in (2^31, 2^32): stored recentred by 2^31
    "price_recentred": (_t_price_recentred, {"l_extendedprice": (4, 90_500 + 2 ** 31)}, SP_WIDE, LC_WIDE64),
    # negative and mixed-sign values
    "qty_minus_25": (_t_add("l_quantity", -25), {"l_quantity": (1, -24)}, SP_STAGED_FIXED, LC_STAGED_FIXED),
    "neg_discount": (_t_neg("l_discount"), {"l_discount": (1, -10)}, SP_NARROW, LC_STAGED_FIXED),
    "neg_price_half": (_t_neg_price_half, {"l_extendedprice": (4, 0)}, SP_NARROW, LC_NARROW32),
    # exact width edges, vmin = 0 and vmin < 0
    "qty_span255": (_t_edges("l_quantity", 0, 255), {"l_quantity": (1, 0)}, SP_STAGED_FIXED, LC_STAGED_FIXED),
    "qty_span256": (_t_edges("l_quantity", 0, 256), {"l_quantity": (2, 0)}, SP_STAGED_RT, LC_STAGED_RT),
    "qty_span255_neg": (_t_edges("l_quantity", -100, 155), {"l_quantity": (1, -100)}, SP_STAGED_FIXED, LC_STAGED_FIXED),
    "qty_span256_neg": (_t_edges("l_quantity", -100, 156), {"l_quantity": (2, -100)}, SP_STAGED_RT, LC_STAGED_RT),
    "date_span65535": (_t_edges("l_shipdate", 0, 65535), {"l_shipdate": (2, 0)}, SP_STAGED_FIXED, LC_STAGED_FIXED),
    "date_span65536": (_t_edges("l_shipdate", 0, 65536), {"l_shipdate": (4, 0)}, SP_STAGED_RT, LC_STAGED_RT),
    "date_span65535_neg": (_t_edges("l_shipdate", -1000, 64535), {"l_shipdate": (2, -1000)}, SP_STAGED_FIXED, LC_STAGED_FIXED),
    "date_span65536_neg": (_t_edges("l_shipdate", -1000, 64536), {"l_shipdate": (4, 0)}, SP_STAGED_RT, LC_STAGED_RT),
    "price_span2p32m1": (_t_edges("l_extendedprice", 0, 2 ** 32 - 1), {"l_extendedprice": (4, 2 ** 31)}, SP_WIDE, LC_WIDE64),
    "price_span2p32": (_t_edges("l_extendedprice", 0, 2 ** 32), {"l_extendedprice": (8, 0)}, SP_WIDE, LC_WIDE64),
    "price_span2p32m1_neg": (_t_edges("l_extendedprice", -5, 2 ** 32 - 6), {"l_extendedprice": (4, 2 ** 31 - 5)}, SP_WIDE, LC_WIDE64),
    "price_span2p32_neg": (_t_edges("l_extendedprice", -5, 2 ** 32 - 5), {"l_extendedprice": (8, 0)}, SP_WIDE, LC_WIDE64),
    # low-cardinality group counts G = |rf codes| x |ls codes| (LC_MAXG = 8), codes 0x00 and 0xff included
    "groups_1": (lambda l, r: _recode(l, r, [0x00], [0xff]), {}, SP_STAGED_FIXED, LC_STAGED_FIXED),
    "groups_8x1": (lambda l, r: _recode(l, r, [0x00, 0x41, 0x42, 0x4e, 0x52, 0x78, 0x7f, 0xff], [0x46]), {}, SP_STAGED_FIXED,
                   LC_STAGED_FIXED),
    "groups_4x2": (lambda l, r: _recode(l, r, [0x00, 0x41, 0x4e, 0xff], [0x00, 0xff], absent=[(0xff, 0x00), (0x41, 0xff)]), {},
                   SP_STAGED_FIXED, LC_STAGED_FIXED),
    # 3 x 3 = 9 dense groups: too many for the low-cardinality kernels, the generic one must give the same answer
    "groups_3x3": (lambda l, r: _recode(l, r, [0x00, 0x41, 0xff], [0x00, 0x4f, 0xff]), {}, SP_STAGED_FIXED, GENERIC),
}

SWITCHES = {
    "default": {},
    "force_wide": {"PG_FORCE_WIDE": "1"},
    "no_staged": {"PG_NO_STAGED": "1"},
    "lc_no_acc32": {"PG_LC_NO_ACC32": "1"},
    "no_specialised": {"PG_NO_SPECIALISED": "1"},
    "nstage2_qpt1": {"PG_NSTAGE": "2", "PG_QPT": "1"},
    "contig0": {"PG_LOWCARD_CONTIG": "0"},
    "contig1": {"PG_LOWCARD_CONTIG": "1"},
    "force_generic": {"PG_FORCE_GENERIC": "1"},
    "force_vm": {"PG_FORCE_VM": "1"},
    "no_pack": {},                  # a twin table sealed under PG_NO_PACK=1: every column at its native width, base 0
}


def _expect_variant(default, switch, explain):
    """The variant `switch` must select, given the one the default selection takes."""
    if switch == "force_vm":
        assert "ScanAgg[expression programs]" in explain
        return
    if switch == "force_generic" or default == GENERIC:
        assert GENERIC in explain
        return
    sp = default.startswith("sumprod")
    staged = "staged" in default
    if switch == "default":
        assert default in explain
    elif switch == "force_wide":
        assert (SP_WIDE if sp else LC_WIDE64) in explain
    elif switch == "no_staged":
        assert ("sumprod_kernel<" if sp else "lowcard_chain_kernel<") in explain and "staged" not in explain
    elif switch == "lc_no_acc32":
        assert "acc32" not in explain
        if not sp and not staged:
            assert "lowcard_chain_kernel<" in explain and "acc64" in explain
    elif switch == "no_specialised":
        assert (default.replace("widths compiled in", "run-time widths") if staged else default) in explain
    elif switch == "nstage2_qpt1":
        assert default.split("<")[0] in explain
        if staged and not sp:
            assert re.search(r"packed3,[01],1> grid", explain), explain
    elif switch in ("contig0", "contig1") and not sp:
        assert ("tiles=interleaved" if switch == "contig0" else "tiles=contiguous-per-CTA") in explain


@pytest.fixture(scope="module")
def scan_cases(sf01_host):
    """(class, pack) -> (host columns, sealed table); built on first use, freed at the end of the module."""
    from plan_b200 import tpch as T
    cache = {}

    def get(name, pack=True):
        key = (name, pack)
        if key not in cache:
            line = {k: v[:N_SCAN].copy() for k, v in sf01_host["lineitem"].items()}
            SCAN_CLASSES[name][0](line, np.random.default_rng(sum(map(ord, name))))
            cache[key] = (line, _upload("lineitem", T.LINEITEM, line, pack=pack))
        return cache[key]
    yield get
    for _, t in cache.values():
        t.free()


_ORACLE_CACHE = {}


def _oracle(fn, cls, line, *args, **kw):
    key = (fn.__name__, cls, args, tuple(sorted(kw.items())))
    if key not in _ORACLE_CACHE:
        _ORACLE_CACHE[key] = fn(line, *args, **kw)
    return _ORACLE_CACHE[key]


def _q6_cases(line):
    """Q6 parameter sets at the edges of the stored domains of the quantity, date and discount columns."""
    q, d, s = line["l_quantity"], line["l_shipdate"], line["l_discount"]
    qmin, qmax, dmin, dmax, smin, smax = int(q.min()), int(q.max()), int(d.min()), int(d.max()), int(s.min()), int(s.max())
    dmid = int(np.median(d))
    base = dict(date_lo=dmid - 200, date_hi=dmid + 165, disc_lit=round((smin + smax) / 200, 2), disc_eps=0.02,
                qty_lt=int(np.median(q)))
    out = [base]
    for qty_lt in (qmin, qmin + 1, qmax, qmax + 1, I32_MAX):          # empty, only vmin, all but vmax, all, beyond the type
        out.append(dict(base, qty_lt=qty_lt))
    for lo, hi in ((dmin, dmax + 1), (dmin + 1, dmax), (dmax, dmax + 1), (dmin - 1, dmin + 1), (I32_MIN, I32_MAX),
                   (dmin - 70000, dmin), (dmax + 1, dmax + 70000), (dmax, dmin)):
        out.append(dict(base, date_lo=lo, date_hi=hi))
    for lit, eps in ((smin / 100, 0.0), (smax / 100, 0.0), ((smin + smax) / 200, 1000.0)):
        out.append(dict(base, disc_lit=lit, disc_eps=eps))
    return out


def _q1_cases(line):
    d = line["l_shipdate"]
    dmin, dmax = int(d.min()), int(d.max())
    return [dmin - 1, dmin, dmin + 1, int(np.median(d)), dmax - 1, dmax, dmax + 1, dmin + 65536, I32_MAX, I32_MIN]


def _stats_cases(line):
    d, cd, rd, q, s = (line[c] for c in ("l_shipdate", "l_commitdate", "l_receiptdate", "l_quantity", "l_discount"))
    dmin, dmax, qmin, qmax, smin = int(d.min()), int(d.max()), int(q.min()), int(q.max()), int(s.min())
    return [
        (I32_MIN, I32_MAX, I32_MAX, I32_MIN, I32_MIN, I32_MAX, -10 ** 9),                       # everything passes
        (dmin, dmax, int(cd.max()), int(rd.min()), qmin, qmax, smin - 1),                         # bounds at vmin / vmax
        (dmin + 1, dmax - 1, int(cd.max()) - 1, int(rd.min()) + 1, qmin + 1, qmax - 1, smin),    # one step inside
        (dmin - 1, dmin - 1, I32_MAX, I32_MIN, I32_MIN, I32_MAX, -10 ** 9),                      # empty
    ]


def _check_q6(oracle, cls, tables, line, kw):
    from plan_b200 import tpch as T
    chunks, stats, explain = _run(T.q6_plan(**kw), tables)
    ref = _oracle(oracle.q6, cls, line, **kw)
    assert stats.aux[0] == ref["rows_selected"], (kw, explain)
    if not ref["has_row"]:
        assert chunks == []
        return explain
    assert len(chunks) == 1 and chunks[0].Card() == 1
    got = _dec(chunks[0].Data[0], 0)
    assert _dec_value(got)[0] * 10 ** (4 - got[1]) == ref["exact"], (kw, explain)
    assert _same_decimal(got, ref["sum"])
    assert chunks[0].Data[0].GetValue(0).String() == oracle.fmt_decimal(ref["sum"], 4)
    return explain


def _check_q1(oracle, cls, tables, line, ship_le):
    from plan_b200 import tpch as T
    chunks, stats, explain = _run(T.q1_plan(ship_le=ship_le), tables)
    ref = _oracle(oracle.q1, cls, line, ship_le=ship_le)
    assert stats.aux[0] == ref["rows_selected"], (ship_le, explain)
    ngot = sum(c.Card() for c in chunks)
    assert ngot == len(ref["groups"]), (ship_le, explain)
    if ngot == 0:
        return explain
    assert len(chunks) == 1
    c = chunks[0]
    groups = sorted(ref["groups"], key=lambda g: g["first_row"])       # first-insertion order
    for r, g in enumerate(groups):
        assert int(c.Data[0].Data[r]) == ord(g["l_returnflag"]) and int(c.Data[1].Data[r]) == ord(g["l_linestatus"]), (r, explain)
        hq = c.Data[2].Data[r]
        assert (int(hq["upper"]) << 64) + int(hq["lower"]) == g["sum_qty"] == g["x_qty"], explain
        for colidx, key, xkey, sc in ((3, "sum_base_price", "x_base", 2), (4, "sum_disc_price", "x_disc_price", 4),
                                      (5, "sum_charge", "x_charge", 6)):
            got = _dec(c.Data[colidx], r)
            if abs(g[xkey]) < 10 ** 19:      # exact regime: the Decimal holds the exact integer sum
                assert _dec_value(got)[0] * 10 ** (sc - got[1]) == g[xkey], (key, explain)
            assert _same_decimal(got, g[key]), (key, explain)
        assert float(c.Data[6].Data[r]) == g["avg_qty"]
        assert _same_decimal(_dec(c.Data[7], r), g["avg_price"])
        assert _same_decimal(_dec(c.Data[8], r), g["avg_disc"])
        hc = c.Data[9].Data[r]
        assert int(hc["lower"]) == g["count_order"] and int(hc["upper"]) == 0
    # the reference's text rendering, where the group codes are printable characters (a 0x00 / 0xff byte in a
    # VARCHAR has no text form to compare)
    if all(0x20 <= ord(g["l_returnflag"]) < 0x7f and 0x20 <= ord(g["l_linestatus"]) < 0x7f for g in groups):
        got_txt = sorted("\t".join(v.GetValue(r).String() for v in c.Data) for r in range(c.Card()))
        assert got_txt == sorted(oracle.q1_text(ref).strip("\n").split("\n")[1:])
    return explain


def _check_stats(oracle, cls, tables, line, args):
    from plan_b200 import tpch as T
    chunks, stats, explain = _run(T.stats_plan(*args), tables)
    ref = _oracle(oracle.stats, cls, line, *args)
    assert stats.aux[0] == ref["rows_selected"], (args, explain)
    assert sum(c.Card() for c in chunks) == len(ref["groups"])
    if ref["groups"]:
        c = chunks[0]
        for r, g in enumerate(sorted(ref["groups"], key=lambda g: g["first_row"])):
            assert int(c.Data[0].Data[r]) == ord(g["l_returnflag"])
            for colidx, key in ((1, "min_ext"), (2, "max_ext"), (3, "max_disc"), (4, "sum_tax"), (5, "avg_tax"), (6, "sum_taxed")):
                assert _same_decimal(_dec(c.Data[colidx], r), g[key]), (key, args, explain)
            assert int(c.Data[7].Data[r]["lower"]) == g["count"]
    return explain


@pytest.mark.parametrize("switch", list(SWITCHES))
@pytest.mark.parametrize("cls", list(SCAN_CLASSES))
def test_scan_value_classes(pg, oracle, scan_cases, monkeypatch, cls, switch):
    """Q6 / Q1 / stats over one value class under one kernel-selection switch: the oracle's bits at every predicate
    edge, and the kernel variant the switch selects."""
    from plan_b200 import tpch as T
    _, enc, want_q6, want_q1 = SCAN_CLASSES[cls]
    pack = switch != "no_pack"
    line, t = scan_cases(cls, pack)
    if switch in ("default", "no_pack"):
        _check_round_trip(t, line, T.LINEITEM, pack)
        if pack:
            for cname, we in enc.items():
                assert t.column_encoding(cname) == we, cname
    for k, v in SWITCHES[switch].items():
        monkeypatch.setenv(k, v)
    tables = {"lineitem": t}
    sw = "default" if switch == "no_pack" else switch
    for i, kw in enumerate(_q6_cases(line)):
        explain = _check_q6(oracle, cls, tables, line, kw)
        if i == 0 and pack:
            _expect_variant(want_q6, sw, explain)
    for i, ship_le in enumerate(_q1_cases(line)):
        explain = _check_q1(oracle, cls, tables, line, ship_le)
        if i == 3 and pack:
            _expect_variant(want_q1, sw, explain)
    for args in _stats_cases(line):
        explain = _check_stats(oracle, cls, tables, line, args)
        assert ("expression programs" if switch == "force_vm" else GENERIC) in explain


def test_scan_variants_are_all_reached():
    """Every kernel variant named in the selection tree is the default of at least one value class."""
    wanted = {SP_STAGED_FIXED, SP_STAGED_RT, SP_NARROW, SP_WIDE, LC_STAGED_FIXED, LC_STAGED_RT, LC_NARROW32, LC_WIDE64, GENERIC}
    reached = {v for _, _, a, b in SCAN_CLASSES.values() for v in (a, b)}
    assert wanted <= reached


# ---------------------------------------------------------- group-by paths --

N_GROUP = 600_000           # SF0.1 lineitem rows (~150k orders with keys up to ~600k)


def _k_sorted(k, rng):
    return k


def _k_shuffled(k, rng):
    return k


def _k_neg(k, rng):
    return -k - 5_000_000_000


def _k_hot(k, rng):
    return np.where(rng.random(len(k)) < 0.5, np.int64(123_457), k)


def _k_minmax(k, rng):
    k = k.copy()
    k[11], k[len(k) - 7] = int(k.min()) - 1000, int(k.max()) + 1000
    return k


def _k_span(extra):
    def f(k, rng):
        k = k.copy()
        k[len(k) // 2] = int(k.max()) + extra
        return k
    return f


# name: (key transform, shuffle rows, path when nothing is switched off: "sorted" / "dense" / "table")
KEY_CLASSES = {
    "sorted": (_k_sorted, False, "sorted"),
    "shuffled": (_k_shuffled, True, "dense"),                  # dense domain of ~600k keys
    "shuffled_negative": (_k_neg, True, "dense"),              # negative keys, 4-byte storage with a non-zero base
    "hot_key": (_k_hot, True, "dense"),                        # half the rows on one key
    "kmin_kmax": (_k_minmax, True, "dense"),                   # one row each at the ends of the domain
    "span_2p30": (_k_span(2 ** 30), True, "table"),            # domain above 2^28: no dense path; order-preserving table
    "span_2p40": (_k_span(2 ** 40), True, "table"),            # domain above 2^34: hashed table
    # clustered in row order (run aggregation, order-preserving slots by default) but one far outlier: the
    # order-preserving map crowds every other key into a few home slots, so the table must fall back to hashing
    "clustered_outlier": (_k_span(2 ** 30), False, "table"),
}

GROUP_SWITCHES = {
    "default": {},
    "no_sorted_runs": {"PG_NO_SORTED_RUNS": "1"},
    "no_dense_group": {"PG_NO_DENSE_GROUP": "1"},
    "group_generic": {"PG_GROUP_GENERIC": "1"},
    "run_aggregate0": {"PG_RUN_AGGREGATE": "0"},
    "run_aggregate1": {"PG_RUN_AGGREGATE": "1"},
    "order_preserving0": {"PG_ORDER_PRESERVING": "0"},
    "order_preserving1": {"PG_ORDER_PRESERVING": "1"},
    "dense_slice_1mb": {"PG_DENSE_SLICE_MB": "1"},
}

TRACE_MARK = {"sorted": "sorted-run group-by", "dense": "dense group-by passes", "table": "probe+group kernel"}


def _group_path(default, switch):
    if switch == "group_generic":
        return "table"                       # the generic scan_group_kernel over the global table
    if default == "sorted" and switch == "no_sorted_runs":
        return "dense"
    if default == "dense" and switch == "no_dense_group":
        return "table"
    return default


@pytest.fixture(scope="module")
def group_cases(sf01_host):
    """key class -> (host columns, sealed table).  Values carry negative numbers: l_quantity - 25 and
    l_extendedprice negated on a seeded half of the rows."""
    from plan_b200 import tpch as T
    cache = {}

    def get(name):
        if name not in cache:
            fn, shuffle, _ = KEY_CLASSES[name]
            rng = np.random.default_rng(sum(map(ord, name)) + 1)
            line = {k: v[:N_GROUP].copy() for k, v in sf01_host["lineitem"].items()}
            if shuffle:
                perm = rng.permutation(len(line["l_orderkey"]))
                line = {k: v[perm] for k, v in line.items()}
            line["l_orderkey"] = fn(line["l_orderkey"], rng).astype(np.int64)
            line["l_quantity"] = (line["l_quantity"] - 25).astype(np.int32)
            line["l_extendedprice"] = np.where(rng.random(len(line["l_orderkey"])) < 0.5, -line["l_extendedprice"], line["l_extendedprice"])
            cache[name] = (line, _upload("lineitem", T.LINEITEM, line))
        return cache[name]
    yield get
    for _, t in cache.values():
        t.free()


def _group_arrays(chunks, decimal):
    """result chunks -> (keys, sums, counts) sorted by key, every sum exact in int64"""
    ks, ss, ns = [], [], []
    for c in chunks:
        k, s, n = (v.Data for v in c.Data)
        ks.append(np.asarray(k, dtype=np.int64))
        if decimal:
            assert np.all(s["scale"] == 2) and np.all(s["coef"] < 2 ** 63)
            coef = s["coef"].astype(np.int64)
            ss.append(np.where(s["neg"] != 0, -coef, coef))
        else:
            lo = s["lower"].view(np.int64)
            assert np.array_equal(s["upper"], np.where(lo < 0, -1, 0))      # the HUGEINT holds an int64
            ss.append(lo.copy())
        assert np.all(n["upper"] == 0)
        ns.append(n["lower"].astype(np.int64))
    if not ks:
        return np.zeros(0, np.int64), np.zeros(0, np.int64), np.zeros(0, np.int64)
    k, s, n = np.concatenate(ks), np.concatenate(ss), np.concatenate(ns)
    o = np.argsort(k, kind="stable")
    assert len(np.unique(k)) == len(k), "duplicate group emitted"
    return k[o], s[o], n[o]


def _want_arrays(oracle, cls, line, **kw):
    key = ("groupby_arrays", cls, tuple(sorted(kw.items())))
    if key not in _ORACLE_CACHE:
        want = oracle.groupby_sum(line, **kw)
        ks = np.array(sorted(want), dtype=np.int64)
        _ORACLE_CACHE[key] = (ks, np.array([want[k][0] for k in ks], dtype=np.int64), np.array([want[k][1] for k in ks], dtype=np.int64))
    return _ORACLE_CACHE[key]


def _check_groupby(oracle, cls, t, line, capfd, path, **kw):
    from plan_b200 import tpch as T
    capfd.readouterr()
    chunks, stats, _ = _run(T.groupby_plan(**kw), {"lineitem": t})
    err = capfd.readouterr().err
    for p, mark in TRACE_MARK.items():
        assert (mark in err) == (p == path), (kw, path, err[-2000:])
    decimal = kw.get("value") == "l_extendedprice"
    got = _group_arrays(chunks, decimal)
    okw = dict(kw)
    if decimal and "having_gt" in kw:        # the INTEGER literal is cast to DECIMAL(38,2): k is 100 k cents
        okw["having_gt"] = 100 * kw["having_gt"]
    want = _want_arrays(oracle, cls, line, **okw)
    assert len(got[0]) == len(want[0]), kw
    for g, w in zip(got, want):
        assert np.array_equal(g, w), kw
    return stats


def _check_groupby_avg(oracle, cls, t, line, value):
    from plan_b200 import tpch as T
    chunks, _, _ = _run(T.groupby_avg_plan(key="l_orderkey", value=value), {"lineitem": t})
    wk, ws, wn = _want_arrays(oracle, cls, line, key="l_orderkey", value=value)
    ks, avs, ns = [], [], []
    for c in chunks:
        k, a, n = (v.Data for v in c.Data)
        ks.append(np.asarray(k, dtype=np.int64))
        avs.append(a.copy())
        ns.append(n["lower"].astype(np.int64))
    k = np.concatenate(ks)
    o = np.argsort(k, kind="stable")
    a, n = np.concatenate(avs)[o], np.concatenate(ns)[o]
    assert np.array_equal(k[o], wk) and np.array_equal(n, wn)
    if value == "l_quantity":                # avg(INTEGER) = float64(sum) / float64(count)
        assert np.array_equal(a, ws.astype(np.float64) / wn.astype(np.float64))
        return
    L = oracle.lib()                         # avg(DECIMAL) = sum.Quo(count): a seeded sample plus both ends
    idx = np.unique(np.concatenate([[0, len(wk) - 1], np.random.default_rng(5).integers(0, len(wk), 1500)]))
    for i in idx:
        s_, c_ = int(ws[i]), int(wn[i])
        oc, os_, on = C.c_uint64(), C.c_int(), C.c_int()
        assert L.orc_dec_quo(C.c_uint64(abs(s_)), 2, int(s_ < 0), C.c_uint64(c_), 0, 0, C.byref(oc), C.byref(os_), C.byref(on)) == 0
        assert (int(a[i]["coef"]), int(a[i]["scale"]), int(a[i]["neg"])) == (oc.value, os_.value, on.value), int(wk[i])


@pytest.mark.parametrize("switch", list(GROUP_SWITCHES))
@pytest.mark.parametrize("cls", list(KEY_CLASSES))
def test_groupby_paths(pg, oracle, group_cases, monkeypatch, capfd, cls, switch):
    """sum / count / avg grouped by a high-cardinality key, with and without a predicate and a HAVING at an existing
    group's sum, through the path each switch selects (asserted from the PG_TRACE marks)."""
    line, t = group_cases(cls)
    if switch == "default":
        _check_round_trip(t, line, [c for c in t.columns if c[0] in ("l_orderkey", "l_quantity", "l_extendedprice")], True)
    for k, v in GROUP_SWITCHES[switch].items():
        monkeypatch.setenv(k, v)
    monkeypatch.setenv("PG_TRACE", "1")
    path = _group_path(KEY_CLASSES[cls][2], switch)
    for value in ("l_quantity", "l_extendedprice"):
        _check_groupby(oracle, cls, t, line, capfd, path, key="l_orderkey", value=value)
        _check_groupby(oracle, cls, t, line, capfd, path, key="l_orderkey", value=value, ship_le=D92 + 1200)
    # HAVING sum > s on an s some group has: `>` excludes that group, s - 1 keeps it
    _, ws, _ = _want_arrays(oracle, cls, line, key="l_orderkey", value="l_quantity")
    s = int(np.sort(ws)[len(ws) // 2])
    for k in (s, s - 1):
        _check_groupby(oracle, cls, t, line, capfd, path, key="l_orderkey", value="l_quantity", having_gt=k)
    _check_groupby(oracle, cls, t, line, capfd, path, key="l_orderkey", value="l_extendedprice", ship_le=D92 + 1500, having_gt=-1)
    for value in ("l_quantity", "l_extendedprice"):
        _check_groupby_avg(oracle, cls, t, line, value)


def test_dense_group_by_in_several_key_slices(pg, oracle, group_cases, monkeypatch):
    """PG_DENSE_SLICE_MB=1: the ~600k-key dense domain (12 bytes per key) takes 7 passes over the rows, one per key
    slice [key_min + D*ps/npass, key_min + D*(ps+1)/npass); 600k is no multiple of 7, so the slice bounds are uneven.
    The launch count shows the passes ran; the result is the oracle's."""
    from plan_b200 import tpch as T
    line, t = group_cases("shuffled")
    k = line["l_orderkey"]
    D = int(k.max()) - int(k.min()) + 1
    npass = -(-D * 12 // 2 ** 20)
    assert npass == 7 and D % 7 != 0
    plan = dict(key="l_orderkey", value="l_quantity", having_gt=0)
    _, one, _ = _run(T.groupby_plan(**plan), {"lineitem": t})
    monkeypatch.setenv("PG_DENSE_SLICE_MB", "1")
    chunks, sliced, _ = _run(T.groupby_plan(**plan), {"lineitem": t})
    assert sliced.kernel_launches - one.kernel_launches == npass - 1
    got = _group_arrays(chunks, False)
    want = _want_arrays(oracle, "shuffled", line, **plan)
    for g, w in zip(got, want):
        assert np.array_equal(g, w)


@pytest.mark.parametrize("over", [False, True])
def test_group_sum_int64_bound(pg, oracle, sf01_host, over):
    """A value column whose largest magnitude times the row count sits just under 2^63 runs and is exact; just over,
    the plan is refused (PG_EUNSUPPORTED) instead of risking a wrapped 64-bit group sum."""
    from plan_b200 import _lib as L, compute as X, tpch as T
    n = 100_000
    line = {k: v[:n].copy() for k, v in sf01_host["lineitem"].items()}
    big = (2 ** 63) // n + 1 if over else (2 ** 63 - 1) // n
    line["l_extendedprice"][n // 3] = -big
    line["l_extendedprice"][n // 2] = big - 1
    t = _upload("lineitem", T.LINEITEM, line)
    try:
        plan = T.groupby_plan(key="l_orderkey", value="l_extendedprice")
        if over:
            ex = X.gpuPipelineExec(plan, {"lineitem": t})
            with pytest.raises(L.PlanGpuError) as ei:
                ex.Init()
            assert ei.value.status == L.PG_EUNSUPPORTED and "exceed int64" in str(ei.value)
            ex.Close()
        else:
            chunks, _, _ = _run(plan, {"lineitem": t})
            got = _group_arrays(chunks, True)
            want = _want_arrays(oracle, "int64_bound", line, key="l_orderkey", value="l_extendedprice")
            for g, w in zip(got, want):
                assert np.array_equal(g, w)
    finally:
        t.free()


# ------------------------------------------------------ joins on based keys --

ORDERKEY_SHIFT = 2 ** 32 + 12_345
CUSTKEY_SHIFT = -1_000_000

# name: date shift applied to o_orderdate and every lineitem date
JOIN_CLASSES = {"dates_plus_60000": 60000, "dates_minus_20000": -20000}
JOIN_SWITCHES = {
    "default": {},
    "no_bitmap_build": {"PG_JOIN_NO_BITMAP_BUILD": "1"},
    "no_rank_index": {"PG_JOIN_NO_RANK_INDEX": "1"},
    "join_generic": {"PG_JOIN_GENERIC": "1"},
}


@pytest.fixture(scope="module")
def join_cases(sf01_host):
    from plan_b200 import tpch as T
    cache = {}

    def get(name):
        if name not in cache:
            dshift = JOIN_CLASSES[name]
            h = {k: {c: a.copy() for c, a in v.items()} for k, v in sf01_host.items()}
            h["orders"]["o_orderkey"] += ORDERKEY_SHIFT
            h["lineitem"]["l_orderkey"] += ORDERKEY_SHIFT
            h["customer"]["c_custkey"] = (h["customer"]["c_custkey"] + CUSTKEY_SHIFT).astype(np.int32)
            h["orders"]["o_custkey"] = (h["orders"]["o_custkey"] + CUSTKEY_SHIFT).astype(np.int32)
            h["orders"]["o_orderdate"] = (h["orders"]["o_orderdate"] + dshift).astype(np.int32)
            for c in DATES:
                h["lineitem"][c] = (h["lineitem"][c] + dshift).astype(np.int32)
            cache[name] = (h, T.upload_tables(h))
        return cache[name]
    yield get
    for _, ts in cache.values():
        for t in ts.values():
            t.free()


@pytest.mark.parametrize("switch", list(JOIN_SWITCHES))
@pytest.mark.parametrize("cls", list(JOIN_CLASSES))
def test_joins_on_based_keys(pg, oracle, join_cases, monkeypatch, cls, switch):
    """Q3 (grouped and top-k), SEMI / ANTI and EXISTS / NOT EXISTS with o_orderkey = l_orderkey above 2^32, negative
    customer keys and shifted dates: the key bitmap's offset and the date bounds moved into the stored domain."""
    from plan_b200 import compute as X, tpch as T
    h, t = join_cases(cls)
    if switch == "default":
        for name, schema in (("orders", T.ORDERS), ("customer", T.CUSTOMER)):
            _check_round_trip(t[name], h[name], [c for c in schema if c[1] != 10], True)
    for k, v in JOIN_SWITCHES[switch].items():
        monkeypatch.setenv(k, v)
    ds = JOIN_CLASSES[cls]
    o, li = h["orders"]["o_orderdate"], h["lineitem"]["l_shipdate"]
    for kw in (dict(odate_lt=T.days(1995, 3, 29) + ds, ship_gt=T.days(1995, 3, 29) + ds),
               dict(segment="BUILDING", odate_lt=int(o.max()) + 1, ship_gt=int(li.min()) - 1),        # every date passes
               dict(odate_lt=int(o.min()) + 1, ship_gt=int(li.max()) - 1)):                         # vmin / vmax edges
        chunks, stats, _ = _run(T.q3_plan(**kw), t)
        ref = oracle.q3(h["customer"], h["orders"], h["lineitem"], **kw)
        got = {}
        for c in chunks:
            ok, rev, od, sp = (v.Data for v in c.Data)
            for r in range(c.Card()):
                x = rev[r]
                got[(int(ok[r]), int(od[r]), int(sp[r]))] = (-1 if x["neg"] else 1) * int(x["coef"]) * 10 ** (4 - int(x["scale"]))
        want = {(g["l_orderkey"], g["o_orderdate"], g["o_shippriority"]): g["x_revenue"] for g in ref["groups"]}
        assert got == want and len(got) == ref["stats"]["ngroups"], kw
        assert stats.aux[0] == ref["stats"]["n_line_sel"] and stats.aux[1] == ref["stats"]["n_line_joined"]
        assert stats.aux[3] == ref["stats"]["n_cust_sel"] and stats.aux[5] == ref["stats"]["n_orders_joined"]
        chunks, _, _ = _run(T.q3_topk_plan(limit=10, **kw), t)
        rows = [[v.GetValue(r) for v in c.Data] for c in chunks for r in range(c.Card())]
        assert X.rows_text(rows, 4) == oracle.q3_text(ref, 10), kw
    for kw in (dict(odate_lt=T.days(1995, 3, 29) + ds, ship_gt=T.days(1995, 3, 29) + ds),
               dict(odate_lt=int(o.max()) + 1, ship_gt=int(li.max()) - 1),
               dict(odate_lt=int(o.min()), ship_gt=int(li.min()) - 1)):                                # empty probe side
        for anti in (False, True):
            want = oracle.semi_groupby(h["orders"], h["lineitem"], anti=anti, **kw)
            for plan in (T.semi_plan(anti=anti, **kw), T.exists_plan(negated=anti, **kw)):
                chunks, _, _ = _run(plan, t)
                got = {}
                for c in chunks:
                    k, s, n = (v.Data for v in c.Data)
                    for r in range(c.Card()):
                        assert int(k[r]) not in got
                        got[int(k[r])] = ((-1 if s[r]["neg"] else 1) * int(s[r]["coef"]), int(n[r]["lower"]))
                assert got == want, (kw, anti)
