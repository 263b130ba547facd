"""Host-side mirror of the reference's operator interface for the off-loaded path.

Stand-in (Python, because there is no Go toolchain here) for the Go shim described in
INTEGRATION.md.  Names, argument meaning and error behaviour follow the reference:

  OperatorExec{Init,Execute,Close}   /root/reference/pkg/compute/executor_operator.go:52-56
  OperatorResult                     /root/reference/pkg/compute/executor_operator.go:11-18
  PhysicalOperator                   /root/reference/pkg/compute/builder_physical_operator.go:49-66
  Expr / ET_*                        /root/reference/pkg/compute/expr.go:13-60
  AggOpInfo / JoinOpInfo / ScanOpInfo /root/reference/pkg/compute/operator_info.go:10-34
  buildOperatorExec (the seam)       /root/reference/pkg/compute/executor.go:305-350

`gpuPipelineExec` serialises its PhysicalOperator subtree into the flat descriptor of
include/plangpu_desc.h, runs it through the C ABI and re-emits the result as ordinary
<=2048-row Chunks, so parents (Project / Order / Limit) are unchanged.
"""
import ctypes as C
import struct

import numpy as np

from . import _lib as L
from . import chunk as K

# OperatorResult
InvalidOpResult, NeedMoreInput, haveMoreOutput, Done = 0, 1, 2, 3

# POT_* (subset the GPU path understands)
POT_Scan, POT_Filter, POT_Join, POT_Agg, POT_Project, POT_Order, POT_Limit = 1, 2, 3, 4, 5, 6, 7

ET_Column, ET_Func, ET_Const = 0, 5, 7

# join types
JOIN_INNER, JOIN_SEMI, JOIN_ANTI, JOIN_MARK, JOIN_LEFT, JOIN_ANTI_MARK = 1, 2, 3, 4, 5, 6

FUNC_IDS = {"+": 1, "-": 2, "*": 3, "/": 4, "=": 10, "<>": 11, "<": 12, "<=": 13, ">": 14, ">=": 15, "in": 16,
            "like": 17, "not like": 18,      # FuncLike / FuncNotLike (function.go:89-128)
            "extract": 19,                   # extract('year', date) (binStringInt32ExtractOp, function_operator_binary.go:259-265)
            "and": 20, "or": 21, "not": 22, "case": 23,   # case: Children = [ELSE, WHEN1, THEN1, ...] (executeCase, expr_exec.go:144-246)
            "cast": 30}
AGG_IDS = {"sum": 1, "avg": 2, "count": 3, "min": 4, "max": 5}

PG_TK_COL, PG_TK_CONST, PG_TK_STR, PG_TK_FUNC = 1, 2, 3, 4
PG_DESC_MAGIC, PG_DESC_VERSION = 0x31504750, 1


class Expr:
    """pkg/compute/expr.go:49-60.  ColRef = (side, idx): side = child number whose output
    list is indexed (0 for scan filters); for aggregate outputs side 0 = group, 1 = agg."""

    def __init__(self, Typ, DataTyp, Children=None, ColRef=None, ConstValue=None, FunImpl=None):
        self.Typ, self.DataTyp, self.Children = Typ, DataTyp, Children or []
        self.ColRef, self.ConstValue, self.FunImpl = ColRef, ConstValue, FunImpl


def col(side, idx, typ):
    return Expr(ET_Column, typ, ColRef=(side, idx))


def const(value, typ):
    return Expr(ET_Const, typ, ConstValue=value)


def func(name, typ, *children):
    return Expr(ET_Func, typ, Children=list(children), FunImpl=name)


def cast(child, typ):
    return func("cast", typ, child)


class ScanOpInfo:
    def __init__(self, Table, Columns=None):
        self.Table, self.Columns = Table, Columns or []


class JoinOpInfo:
    def __init__(self, JoinTyp, OnConds):
        self.JoinTyp, self.OnConds = JoinTyp, OnConds     # OnConds[i] = func("=", bool, left, right)


class AggOpInfo:
    def __init__(self, Aggs, GroupBys):
        self.Aggs, self.GroupBys = Aggs, GroupBys         # Aggs[i] = func("sum"|..., result type, arg)


class OrderOpInfo:
    def __init__(self, OrderBys):
        self.OrderBys = OrderBys            # [(Expr column ref into the child's outputs, descending)]


class LimitOpInfo:
    def __init__(self, Limit):
        self.Limit = Limit


class PhysicalOperator:
    def __init__(self, Typ, Outputs=None, Filters=None, Children=None, Info=None):
        self.Typ, self.Outputs, self.Filters = Typ, Outputs or [], Filters or []
        self.Children, self.Info = Children or [], Info


# ------------------------------------------------------------ serialisation --

def _ltype_words(t):
    return [t.Id, t.Width, t.Scale]


def _expr_tokens(e, out):
    if e.Typ == ET_Column:
        out.append([PG_TK_COL, e.ColRef[0], e.ColRef[1]] + _ltype_words(e.DataTyp))
    elif e.Typ == ET_Const:
        t = e.DataTyp
        if e.ConstValue is None:            # NULL constant (a CASE without ELSE): ltype 0
            out.append([PG_TK_CONST, 0, 0, 0, 0])
        elif t.Id == K.LTID_VARCHAR:
            b = e.ConstValue.encode()
            words = [int.from_bytes(b[i:i + 8].ljust(8, b"\0"), "little", signed=True) for i in range(0, len(b), 8)]
            out.append([PG_TK_STR, len(b)] + words)
        elif t.Id in (K.LTID_FLOAT, K.LTID_DOUBLE):
            bits = struct.unpack("<q", struct.pack("<d", float(e.ConstValue)))[0]
            out.append([PG_TK_CONST] + _ltype_words(t) + [bits])
        else:
            out.append([PG_TK_CONST] + _ltype_words(t) + [int(e.ConstValue)])
    elif e.Typ == ET_Func:
        for c in e.Children:
            _expr_tokens(c, out)
        out.append([PG_TK_FUNC, FUNC_IDS[e.FunImpl], len(e.Children)] + _ltype_words(e.DataTyp))
    else:
        raise ValueError("expression type %r cannot be off-loaded" % e.Typ)


def _expr_words(e):
    toks = []
    _expr_tokens(e, toks)
    w = [len(toks)]
    for t in toks:
        w += t
    return w


def _node_words(op, slots):
    if op.Typ == POT_Limit and op.Children[0].Typ == POT_Order and op.Children[0].Children[0].Typ == POT_Agg:
        # Limit <- Order <- Agg with ORDER BY on plain output columns fuses into PG_OP_TOPK
        order = op.Children[0]
        w = [5, len(order.Info.OrderBys)]
        for e, desc in order.Info.OrderBys:
            w += [e.ColRef[1], 1 if desc else 0]
        w.append(op.Info.Limit)
        return w + _node_words(order.Children[0], slots)
    if op.Typ == POT_Order and op.Children[0].Typ == POT_Agg:
        w = [5, len(op.Info.OrderBys)]
        for e, desc in op.Info.OrderBys:
            w += [e.ColRef[1], 1 if desc else 0]
        w.append(-1)
        return w + _node_words(op.Children[0], slots)
    if op.Typ == POT_Scan:
        if op.Info.Table not in slots:
            slots[op.Info.Table] = len(slots)
        w = [1, slots[op.Info.Table], len(op.Filters)]
        for f in op.Filters:
            w += _expr_words(f)
        return w
    if op.Typ == POT_Project:
        # row-emitting pipelines: Project <- [Filter]* <- (Scan | Join); Outputs are the projection expressions
        w = [6, len(op.Outputs)]
        for e in op.Outputs:
            w += _expr_words(e)
        return w + _node_words(op.Children[0], slots)
    if op.Typ == POT_Filter:
        w = [2, len(op.Filters)]
        for f in op.Filters:
            w += _expr_words(f)
        return w + _node_words(op.Children[0], slots)
    if op.Typ == POT_Join:
        w = [3, op.Info.JoinTyp, len(op.Info.OnConds)]
        for c in op.Info.OnConds:
            w += _expr_words(c.Children[0]) + _expr_words(c.Children[1])
        w.append(len(op.Outputs))
        for o in op.Outputs:
            w += [o.ColRef[0], o.ColRef[1]]
        return w + _node_words(op.Children[0], slots) + _node_words(op.Children[1], slots)
    if op.Typ == POT_Agg:
        w = [4, len(op.Info.GroupBys)]
        for g in op.Info.GroupBys:
            w += _expr_words(g)
        w.append(len(op.Info.Aggs))
        for a in op.Info.Aggs:
            w += [AGG_IDS[a.FunImpl]] + _ltype_words(a.DataTyp)
            w += _expr_words(a.Children[0]) if a.Children else [0]
        w.append(len(op.Filters))                    # HAVING
        for f in op.Filters:
            w += _expr_words(f)
        w.append(len(op.Outputs))
        for o in op.Outputs:
            w += [o.ColRef[0], o.ColRef[1]]
        return w + _node_words(op.Children[0], slots)
    raise ValueError("operator type %r cannot be off-loaded" % op.Typ)


def serialize_plan(op):
    """PhysicalOperator subtree -> (int64 descriptor, {table name: slot})."""
    slots = {}
    words = [PG_DESC_MAGIC, PG_DESC_VERSION] + _node_words(op, slots)
    return np.array(words, dtype=np.int64), slots


# ------------------------------------------------------------------ tables --

class DeviceTable:
    """A sealed pg_table plus its schema (the device-resident column cache entry)."""

    def __init__(self, name, handle, columns):
        self.name, self.handle, self.columns = name, handle, columns   # columns: [(name, pg_type, width, scale, dict)]

    @classmethod
    def create(cls, name, columns):
        lib = L.lib()
        n = len(columns)
        descs = (L.ColDesc * n)()
        keep = []
        for i, (cname, t, w, s, d) in enumerate(columns):
            descs[i].name = cname.encode()
            descs[i].type, descs[i].width, descs[i].scale = t, w, s
            if d:
                arr = (C.c_char_p * len(d))(*[x.encode() for x in d])
                keep.append(arr)
                descs[i].dict = arr
                descs[i].dict_len = len(d)
        h = C.c_void_p()
        L.check(lib.pg_table_create(name.encode(), n, descs, C.byref(h)))
        return cls(name, h, columns)

    def append(self, arrays, valid=None):
        """arrays: one contiguous numpy array (or raw pointer int) per column, host memory.  A VARCHAR column is a list / array of
        bytes or str, or a (blob uint8 array, offsets int64 array of n + 1) pair: row r is blob[offsets[r]:offsets[r + 1]]."""
        lib = L.lib()
        n = len(self.columns)
        ptrs = (C.c_void_p * n)()
        nrows = None
        for i, a in enumerate(arrays):
            if self.columns[i][1] == L.PG_T_VARCHAR and isinstance(a, tuple) and len(a) == 2 and all(isinstance(x, np.ndarray) for x in a):
                blob, off = np.ascontiguousarray(a[0], dtype=np.uint8), np.asarray(a[1], dtype=np.int64)
                if off.ndim != 1 or len(off) < 1 or (len(off) > 1 and (off[0] < 0 or off[-1] > len(blob) or (np.diff(off) < 0).any())):
                    raise ValueError("VARCHAR column %s: offsets must be n + 1 non-decreasing positions inside the blob" % self.columns[i][0])
                if len(blob) == 0:
                    blob = np.zeros(1, np.uint8)          # a valid address for empty strings
                sv = np.empty(len(off) - 1, dtype=K.PG_STRING)
                sv["len"] = np.diff(off)
                sv["data"] = blob.ctypes.data + off[:-1].astype(np.uint64)
                arrays[i] = (sv, blob)
                ptrs[i] = sv.ctypes.data
                nrows = len(sv) if nrows is None else nrows
                assert len(sv) == nrows
                continue
            if self.columns[i][1] == L.PG_T_VARCHAR:
                # list / array of bytes|str -> one pg_string per row over a single contiguous buffer
                raw = [x.encode() if isinstance(x, str) else bytes(x) for x in a]
                lens = np.fromiter((len(x) for x in raw), dtype=np.int64, count=len(raw))
                blob = np.frombuffer(b"".join(raw) + b"\0", dtype=np.uint8)
                sv = np.empty(len(raw), dtype=K.PG_STRING)
                sv["len"] = lens
                sv["data"] = blob.ctypes.data + np.concatenate([[0], np.cumsum(lens)[:-1]]).astype(np.uint64) if len(raw) else 0
                arrays[i] = (sv, blob)
                ptrs[i] = sv.ctypes.data
                nrows = len(raw) if nrows is None else nrows
                assert len(raw) == nrows
                continue
            if isinstance(a, np.ndarray):
                a = np.ascontiguousarray(a, dtype=K.native_dtype(self.columns[i][1]))
                arrays[i] = a
                ptrs[i] = a.ctypes.data
                nrows = len(a) if nrows is None else nrows
                assert len(a) == nrows
            else:
                ptrs[i] = a[0]
                nrows = a[1] if nrows is None else nrows
        vptrs = None
        if valid is not None:
            vptrs = (C.c_void_p * n)()
            for i, v in enumerate(valid):
                vptrs[i] = None if v is None else v.ctypes.data
        L.check(lib.pg_table_append(self.handle, nrows, ptrs, vptrs))

    def append_cols(self, bufs, nrows):
        """bufs: one (host pointer int, width, base) per column -- narrow host buffers with a frame of reference
        (pg_table_append_cols); width 0 = the column's native width."""
        n = len(self.columns)
        cb = (L.ColBuf * n)()
        for i, (ptr, w, base) in enumerate(bufs):
            cb[i].data, cb[i].width, cb[i].reserved, cb[i].base, cb[i].valid = ptr, w, 0, base, None
        L.check(L.lib().pg_table_append_cols(self.handle, nrows, cb))

    def column_encoding(self, col):
        if isinstance(col, str):
            col = [c[0] for c in self.columns].index(col)
        w, b = C.c_int32(), C.c_int64()
        L.check(L.lib().pg_table_column_encoding(self.handle, col, C.byref(w), C.byref(b)))
        return w.value, b.value

    def seal(self, global_row_offset=0):
        L.check(L.lib().pg_table_seal(self.handle, global_row_offset))
        return self

    def set_replicated(self, replicated=True):
        L.check(L.lib().pg_table_set_distribution(self.handle, L.PG_DIST_REPLICATED if replicated else L.PG_DIST_SHARDED))
        return self

    def rows(self):
        n = C.c_int64()
        L.check(L.lib().pg_table_rows(self.handle, C.byref(n)))
        return n.value

    def read_column(self, col, row=0, nrows=None):
        if isinstance(col, str):
            col = [c[0] for c in self.columns].index(col)
        if nrows is None:
            nrows = self.rows() - row
        out = np.empty(nrows, dtype=K.native_dtype(self.columns[col][1]))
        L.check(L.lib().pg_table_read_column(self.handle, col, row, nrows, out.ctypes.data))
        return out

    def free(self):
        if self.handle:
            L.lib().pg_table_free(self.handle)
            self.handle = None


# --------------------------------------------------------------- executor --

class OperatorExec:
    def Init(self): raise NotImplementedError
    def Execute(self, input, output): raise NotImplementedError
    def Close(self): raise NotImplementedError


class gpuPipelineExec(OperatorExec):
    """OperatorExec for a fusable subtree (Agg <- Scan, Agg <- Join...), selected where
    buildOperatorExec switches on op.Typ.  Raises PlanGpuError(PG_EUNSUPPORTED) from Init
    when the shape has no GPU pipeline: the caller then builds the stock executors."""

    def __init__(self, op, tables):
        self.op, self.tables = op, tables      # tables: {name: DeviceTable}
        self.plan = self.result = None
        self.slots = {}
        self.stats = None

    def Init(self):
        lib = L.lib()
        desc, self.slots = serialize_plan(self.op)
        self.desc = desc
        plan = C.c_void_p()
        L.check(lib.pg_plan_compile(desc.ctypes.data_as(C.POINTER(C.c_int64)), len(desc), C.byref(plan)))
        self.plan = plan
        for name, slot in self.slots.items():
            L.check(lib.pg_plan_bind(plan, slot, self.tables[name].handle))
        L.check(lib.pg_plan_prepare(plan))      # PG_EUNSUPPORTED -> caller builds the stock executors
        return None

    def Reset(self):
        """Forget the last result so the next Execute runs the pipeline again."""
        if self.result:
            L.lib().pg_result_free(self.result)
            self.result = None

    def Explain(self):
        return L.lib().pg_plan_explain(self.plan).decode()

    def _run(self):
        lib = L.lib()
        res = C.c_void_p()
        L.check(lib.pg_plan_execute(self.plan, C.byref(res)))
        self.result = res
        st = L.Stats()
        L.check(lib.pg_result_stats(res, C.byref(st)))
        self.stats = st
        nc = C.c_int()
        L.check(lib.pg_result_num_columns(res, C.byref(nc)))
        self.ncols = nc.value
        self.coltypes = []
        for i in range(self.ncols):
            t, w, s = C.c_int32(), C.c_int32(), C.c_int32()
            L.check(lib.pg_result_column_type(res, i, C.byref(t), C.byref(w), C.byref(s)))
            self.coltypes.append((t.value, w.value, s.value))

    def Execute(self, input, output):
        lib = L.lib()
        if self.result is None:
            self._run()
        n = C.c_int64()
        cols = (C.c_void_p * self.ncols)()
        valids = (C.c_void_p * self.ncols)()
        L.check(lib.pg_result_next(self.result, K.DEFAULT_VECTOR_SIZE, C.byref(n), cols, valids))
        if n.value == 0:
            output.Data, output.Count = [], 0
            return Done, None
        vecs = []
        agg = self._agg_op()
        for i, (t, w, s) in enumerate(self.coltypes):
            dt = np.dtype(K.native_dtype(t))
            buf = (C.c_char * (dt.itemsize * n.value)).from_address(cols[i])
            data = np.frombuffer(buf, dtype=dt, count=n.value).copy()
            if t == L.PG_T_VARCHAR:      # pg_string rows -> python strings (the result owns the bytes until Close)
                data = np.array([C.string_at(int(r["data"]), int(r["len"])) for r in data], dtype=object)
            typ = agg.Outputs[i].DataTyp if i < len(agg.Outputs) else K.LType(0)
            d = None
            if t == L.PG_T_DICT8:
                nd, ents = C.c_int32(), C.POINTER(C.c_char_p)()
                L.check(lib.pg_result_column_dict(self.result, i, C.byref(nd), C.byref(ents)))
                d = [ents[k].decode() for k in range(nd.value)] if nd.value else self._dict_for_output(i)
            mask = None
            if valids[i]:       # packed validity bits, 1 = valid (pkg/util/bitmap.go)
                nb = (n.value + 7) // 8
                mask = np.frombuffer((C.c_char * nb).from_address(valids[i]), dtype=np.uint8, count=nb).copy()
            vecs.append(K.Vector(typ, data, mask=mask, dictionary=d))
        output.Data, output.Count = vecs, n.value
        return haveMoreOutput, None

    def _agg_op(self):
        """The operator whose Outputs type the result columns: the aggregate, or the root of a row-emitting pipeline
        (a Filter's outputs are its child's)."""
        op = self.op
        while op.Typ in (POT_Limit, POT_Order) or (op.Typ == POT_Filter and not op.Outputs):
            op = op.Children[0]
        return op

    def _dict_for_output(self, i):
        # a DICT8 group key is a scan column reached through joins: follow the output references down to its dictionary
        agg = self._agg_op()
        o = agg.Outputs[i]
        if agg.Typ != POT_Agg or o.ColRef[0] != 0:
            return None
        g = agg.Info.GroupBys[o.ColRef[1]]
        if g.Typ != ET_Column:
            return None
        node, idx = agg.Children[0], g.ColRef[1]
        while node.Typ != POT_Scan:
            if node.Typ == POT_Join:
                ref = node.Outputs[idx].ColRef
                node, idx = node.Children[ref[0]], ref[1]
            else:
                node = node.Children[0]
        return self.tables[node.Info.Table].columns[idx][4]

    def Close(self):
        lib = L.lib()
        if self.result:
            lib.pg_result_free(self.result)
            self.result = None
        if self.plan:
            lib.pg_plan_free(self.plan)
            self.plan = None
        return None


def drain(exec_):
    """Pull an OperatorExec to completion the way execOps does (executor.go:151-188)."""
    chunks = []
    while True:
        out = K.Chunk()
        res, err = exec_.Execute(None, out)
        if err is not None:
            raise err
        if res == Done:
            break
        if out.Card() > 0:
            chunks.append(out)
    return chunks


class _Descending:
    """sort key wrapper that inverts the order of values without a unary minus (VARCHAR keys of ORDER BY ... DESC)"""
    __slots__ = ("v",)

    def __init__(self, v):
        self.v = v

    def __lt__(self, other):
        return other.v < self.v

    def __eq__(self, other):
        return self.v == other.v


def order_limit(chunks, order_by, limit=None):
    """Host stand-in for the parents that stay in Go: Order (normalized keys,
    /root/reference/pkg/compute/sort_encoder.go:65-81: a DECIMAL key is Int64(2), i.e. rounded
    to two fractional digits; DESC inverts) and Limit (executor_limit.go:120-137).
    order_by: [(column index, descending)] ; returns a list of rows of Values."""
    rows = []
    for c in chunks:
        for r in range(c.Card()):
            rows.append([v.GetValue(r) for v in c.Data])

    def key(row):
        k = []
        for idx, desc in order_by:
            v = row[idx]
            if v.Typ.Id == K.LTID_DECIMAL:
                coef, scale, neg = K.new_from_int64(v.I64, v.I64_1, v.Typ.Scale) if not v.Str else (None, None, None)
                w, f = K.decimal_int64(coef, scale, neg, 2)
                part = (w, f)
            elif v.Typ.Id in (K.LTID_DOUBLE, K.LTID_FLOAT):
                part = (v.F64,)
            elif v.Typ.Id == K.LTID_VARCHAR:
                part = (v.Str,)
            elif v.Typ.Id == K.LTID_HUGEINT:
                part = ((v.I64 << 64) + (v.I64_1 & 0xFFFFFFFFFFFFFFFF),)
            else:
                part = (v.I64,)
            if desc:
                part = tuple(_Descending(x) if isinstance(x, str) else -x for x in part)
            k.append(part)
        return k
    rows.sort(key=key)
    return rows if limit is None else rows[:limit]


def rows_text(rows, ncols):
    """Chunk.SaveToFile text of a row list, with the reference's '#' headline."""
    return "#" + "\t" * (ncols - 1) + "\n" + "".join("\t".join(v.String() for v in r) + "\n" for r in rows)
