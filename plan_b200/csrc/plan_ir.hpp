// plan_ir.hpp -- plan descriptor parser and lowering to kernel-level forms.
//
// The descriptor (plangpu_desc.h) is the serialised PhysicalOperator subtree of the
// reference (/root/reference/pkg/compute/builder_physical_operator.go:49-66).  Lowering
// restates, once at plan time, what the reference re-evaluates per row:
//   * conjunctive filters (execSelectAnd, expr_exec.go:444-480) of `column <cmp> constant`
//     become inclusive integer ranges on the column's native encoding.  The reference
//     compares DECIMAL columns with FLOAT literals in float32
//     (tryCastDecimalToFloat32, function_cast.go:349-354); that cast is monotone, so the
//     exact integer thresholds are found by bisection over the column's value range with
//     the same float32 arithmetic -- bit-identical row selection, no fp in the kernel;
//   * aggregate arguments built from DECIMAL +,-,* (function_operator_binary.go:134-191)
//     become products of affine factors (c + s*column) on unscaled int64 values; the value
//     scale is the sum of the factor scales (govalues Mul), Add/Sub align to the max scale.
#pragma once
#include <math.h>
#include <string.h>

#include <string>
#include <vector>

#include "common.cuh"

namespace pg {

struct Expr {
    int kind = 0;                 // PG_TK_*
    int side = 0, idx = 0;        // COL
    int ltype = 0, width = 0, scale = 0;
    i64 v0 = 0;                   // CONST
    std::string str;              // STR
    int fn = 0;                   // FUNC
    std::vector<Expr> args;
};

struct AggExpr {
    int fn = 0;
    int ltype = 0, width = 0, scale = 0;   // result type
    bool star = false;
    Expr arg;
};

struct Node {
    int op = 0;
    int slot = -1;                                   // SCAN
    std::vector<Expr> filters;                       // SCAN / FILTER
    int jointype = 0;                                // JOIN
    std::vector<std::pair<Expr, Expr>> conds;        // JOIN (probe expr, build expr)
    std::vector<std::pair<int, int>> outs;           // JOIN (side idx) / AGG (kind idx)
    std::vector<Expr> exprs;                         // PROJECT
    std::vector<Expr> groups;                        // AGG
    std::vector<AggExpr> aggs;
    std::vector<Expr> having;
    std::vector<std::pair<int, int>> order;          // TOPK (output index, descending)
    i64 limit = -1;                                  // TOPK
    std::vector<Node> children;
};

class DescReader {
public:
    DescReader(const int64_t *w, size_t n) : w_(w), n_(n) {}
    bool ok() const { return ok_; }
    size_t pos() const { return pos_; }
    i64 next()
    {
        if (pos_ >= n_) { ok_ = false; return 0; }
        return w_[pos_++];
    }
    bool expr(Expr *out)
    {
        i64 nt = next();
        if (!ok_ || nt < 0 || nt > 4096) return ok_ = false;
        std::vector<Expr> stack;
        for (i64 i = 0; i < nt && ok_; i++) {
            Expr e;
            e.kind = (int)next();
            switch (e.kind) {
            case PG_TK_COL:
                e.side = (int)next(); e.idx = (int)next();
                e.ltype = (int)next(); e.width = (int)next(); e.scale = (int)next();
                break;
            case PG_TK_CONST:
                e.ltype = (int)next(); e.width = (int)next(); e.scale = (int)next(); e.v0 = next();
                break;
            case PG_TK_STR: {
                i64 nb = next();
                if (!ok_ || nb < 0 || nb > 65536) return ok_ = false;
                e.ltype = PG_LT_VARCHAR;
                e.str.resize((size_t)nb);
                for (i64 k = 0; k < (nb + 7) / 8; k++) {
                    i64 word = next();
                    for (int b = 0; b < 8 && k * 8 + b < nb; b++) e.str[(size_t)(k * 8 + b)] = (char)((word >> (8 * b)) & 0xff);
                }
                break;
            }
            case PG_TK_FUNC: {
                e.fn = (int)next();
                int nargs = (int)next();
                e.ltype = (int)next(); e.width = (int)next(); e.scale = (int)next();
                if (!ok_ || nargs < 0 || (size_t)nargs > stack.size()) return ok_ = false;
                e.args.assign(stack.end() - nargs, stack.end());
                stack.resize(stack.size() - (size_t)nargs);
                break;
            }
            default: return ok_ = false;
            }
            stack.push_back(e);
        }
        if (!ok_) return false;
        if (nt == 0) { *out = Expr(); return true; }
        if (stack.size() != 1) return ok_ = false;
        *out = stack[0];
        return true;
    }
    bool node(Node *out, int depth = 0)
    {
        if (depth > 16) return ok_ = false;
        out->op = (int)next();
        switch (out->op) {
        case PG_OP_TOPK: {
            if (depth != 0) return ok_ = false;
            i64 nk = next();
            if (!ok_ || nk < 0 || nk > 16) return ok_ = false;
            out->order.resize((size_t)nk);
            for (auto &o : out->order) { o.first = (int)next(); o.second = (int)next(); }
            out->limit = next();
            out->children.resize(1);
            return node(&out->children[0], depth + 1);
        }
        case PG_OP_SCAN: {
            out->slot = (int)next();
            i64 nf = next();
            if (!ok_ || nf < 0 || nf > 256) return ok_ = false;
            out->filters.resize((size_t)nf);
            for (auto &e : out->filters) if (!expr(&e)) return false;
            return ok_;
        }
        case PG_OP_PROJECT: {
            if (depth != 0) return ok_ = false;
            i64 ne = next();
            if (!ok_ || ne < 1 || ne > 256) return ok_ = false;
            out->exprs.resize((size_t)ne);
            for (auto &e : out->exprs) if (!expr(&e)) return false;
            out->children.resize(1);
            return node(&out->children[0], depth + 1);
        }
        case PG_OP_FILTER: {
            i64 nf = next();
            if (!ok_ || nf < 0 || nf > 256) return ok_ = false;
            out->filters.resize((size_t)nf);
            for (auto &e : out->filters) if (!expr(&e)) return false;
            out->children.resize(1);
            return node(&out->children[0], depth + 1);
        }
        case PG_OP_JOIN: {
            out->jointype = (int)next();
            i64 nc = next();
            if (!ok_ || nc < 0 || nc > 16) return ok_ = false;
            out->conds.resize((size_t)nc);
            for (auto &c : out->conds) if (!expr(&c.first) || !expr(&c.second)) return false;
            i64 no = next();
            if (!ok_ || no < 0 || no > 256) return ok_ = false;
            out->outs.resize((size_t)no);
            for (auto &o : out->outs) { o.first = (int)next(); o.second = (int)next(); }
            out->children.resize(2);
            return node(&out->children[0], depth + 1) && node(&out->children[1], depth + 1);
        }
        case PG_OP_AGG: {
            i64 ng = next();
            if (!ok_ || ng < 0 || ng > 64) return ok_ = false;
            out->groups.resize((size_t)ng);
            for (auto &e : out->groups) if (!expr(&e)) return false;
            i64 na = next();
            if (!ok_ || na < 0 || na > 64) return ok_ = false;
            out->aggs.resize((size_t)na);
            for (auto &a : out->aggs) {
                a.fn = (int)next(); a.ltype = (int)next(); a.width = (int)next(); a.scale = (int)next();
                if (!expr(&a.arg)) return false;
                a.star = a.arg.kind == 0;
            }
            i64 nh = next();
            if (!ok_ || nh < 0 || nh > 64) return ok_ = false;
            out->having.resize((size_t)nh);
            for (auto &e : out->having) if (!expr(&e)) return false;
            i64 no = next();
            if (!ok_ || no < 0 || no > 256) return ok_ = false;
            out->outs.resize((size_t)no);
            for (auto &o : out->outs) { o.first = (int)next(); o.second = (int)next(); }
            out->children.resize(1);
            return node(&out->children[0], depth + 1);
        }
        default: return ok_ = false;
        }
    }

private:
    const int64_t *w_;
    size_t n_, pos_ = 0;
    bool ok_ = true;
};

// ------------------------------------------------------------------ lowering --

struct Range {
    int col = -1;
    i64 lo = INT64_MIN, hi = INT64_MAX;   // inclusive; lo > hi selects nothing
    // byte-coded columns (VARCHAR(1) / dictionary): `<>`, IN lists and ORs of equalities are code SETS
    bool is_set = false;
    uint32_t set[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    // PG_T_VARCHAR columns: 1 LIKE, 2 NOT LIKE (pattern with % and _), 3 =, 4 <> (byte equality) against `pat`
    int like = 0;
    std::string pat;
};

// `%lit%` with 1..8 wildcard-free bytes: the device takes a word-at-a-time substring search for these
inline bool like_is_contains(const std::string &pat, std::string *lit)
{
    if (pat.size() < 3 || pat.size() > 10 || pat.front() != '%' || pat.back() != '%') return false;
    const std::string mid = pat.substr(1, pat.size() - 2);
    if (mid.find('%') != std::string::npos || mid.find('_') != std::string::npos) return false;
    *lit = mid;
    return true;
}

// `%s1%s2%...%sk%`: a leading and a trailing '%', runs of '%' taken as one, 1 <= k <= LIKE_MAXSEG segments of 1..8 bytes
// without '_'.  Such a pattern matches exactly when the segments occur in order without overlapping, and the leftmost
// occurrence of each segment after the end of the previous one decides: the device searches one segment at a time
// with the word-at-a-time search (kinds GEN_LIKE_WORDS / GEN_NOTLIKE_WORDS, leftcount.cuh).
constexpr int LIKE_MAXSEG = 4;
inline bool like_segments(const std::string &pat, std::vector<std::string> *segs)
{
    segs->clear();
    if (pat.size() < 3 || pat.front() != '%' || pat.back() != '%') return false;
    std::vector<std::string> out;
    std::string cur;
    for (char ch : pat) {
        if (ch == '_') return false;
        if (ch != '%') { cur += ch; continue; }
        if (cur.empty()) continue;
        if (cur.size() > 8 || (int)out.size() == LIKE_MAXSEG) return false;
        out.push_back(cur);
        cur.clear();
    }
    if (out.empty()) return false;
    segs->swap(out);
    return true;
}

// The reference's LIKE matcher restated (wildcardMatch, function_operator_boolean.go:336-377): byte-wise,
// '%' matches any run (greedy with backtracking to the last '%'), '_' any single byte.
inline bool wildcard_match(const char *pat, size_t plen, const char *tgt, size_t tlen)
{
    size_t p = 0, t = 0;
    long star_p = -1, star_t = -1;
    while (t < tlen) {
        if (p < plen && pat[p] == '%') {
            p++;
            star_p = (long)p;
            if (p >= plen) return true;
            star_t = (long)t;
        } else if (p < plen && (pat[p] == '_' || pat[p] == tgt[t])) {
            p++;
            t++;
        } else {
            if (star_p == -1 || star_t == -1) return false;
            p = (size_t)star_p;
            star_t++;
            t = (size_t)star_t;
        }
    }
    while (p < plen && pat[p] == '%') p++;
    return p >= plen;
}

struct Factor {
    int col = -1;      // -1: pure constant
    i64 c = 0;         // value = c + s * column   (at the column's scale)
    int s = 1;
    int scale = 0;
    bool operator==(const Factor &o) const { return col == o.col && c == o.c && s == o.s && scale == o.scale; }
};

struct AffProd {
    std::vector<Factor> f;
    int vscale() const { int s = 0; for (auto &x : f) s += x.scale; return s; }
};

inline bool is_int_family(int t) { return t == PG_T_INT32 || t == PG_T_INT64 || t == PG_T_DATE32 || t == PG_T_DECIMAL64; }
inline bool is_byte_family(int t) { return t == PG_T_CHAR1 || t == PG_T_DICT8; }

inline bool is_cmp(int fn) { return fn >= PG_FN_EQ && fn <= PG_FN_GE; }
inline int flip_cmp(int fn)
{
    switch (fn) {
    case PG_FN_LT: return PG_FN_GT;
    case PG_FN_LE: return PG_FN_GE;
    case PG_FN_GT: return PG_FN_LT;
    case PG_FN_GE: return PG_FN_LE;
    default: return fn;
    }
}

inline void range_and(Range &r, i64 lo, i64 hi)
{
    if (lo > r.lo) r.lo = lo;
    if (hi < r.hi) r.hi = hi;
}

// fold range bounds into the code set of a byte column (so that ranges and sets on one column intersect)
inline void range_to_set(Range &r)
{
    if (r.is_set) return;
    r.is_set = true;
    for (int c = 0; c < 256; c++)
        if ((i64)c >= r.lo && (i64)c <= r.hi) r.set[c >> 5] |= 1u << (c & 31);
}

// float32(Float64(decimal c * 10^-scale)) exactly as the reference casts a DECIMAL to FLOAT
// (function_cast.go:349-354: strconv.ParseFloat of the decimal string, then float32()).
// For |c| < 2^53 the correctly rounded parse equals the IEEE division c / 10^scale.
inline float dec_to_f32_exact(i64 c, int scale)
{
    static const double P10[20] = {1e0, 1e1, 1e2, 1e3, 1e4, 1e5, 1e6, 1e7, 1e8, 1e9, 1e10, 1e11, 1e12,
                                   1e13, 1e14, 1e15, 1e16, 1e17, 1e18, 1e19};   // all exact in binary64
    double d = (double)c / P10[scale < 0 ? 0 : scale > 19 ? 19 : scale];   // pg_table_create admits 0..19 only
    return (float)d;
}

// Translate `cast(col AS FLOAT) <op> k` into an integer range on col over [vmin, vmax].
inline void float_cmp_to_range(int op, float k, int scale, i64 vmin, i64 vmax, i64 *lo, i64 *hi)
{
    auto first_true = [&](auto pred) {   // smallest c in [vmin, vmax+1] with pred(c) (pred monotone false->true)
        i64 a = vmin, b = vmax + 1;
        while (a < b) {
            i64 m = a + (b - a) / 2;
            if (pred(m)) b = m; else a = m + 1;
        }
        return a;
    };
    i64 ge = first_true([&](i64 c) { return dec_to_f32_exact(c, scale) >= k; });   // first c with f >= k
    i64 gt = first_true([&](i64 c) { return dec_to_f32_exact(c, scale) > k; });    // first c with f >  k
    switch (op) {
    case PG_FN_GE: *lo = ge; *hi = vmax; break;
    case PG_FN_GT: *lo = gt; *hi = vmax; break;
    case PG_FN_LE: *lo = vmin; *hi = gt - 1; break;
    case PG_FN_LT: *lo = vmin; *hi = ge - 1; break;
    default: /* EQ */ *lo = ge; *hi = gt - 1; break;
    }
}

struct LowerCtx {
    const pg_table *table = nullptr;
    bool allow_nulls = false;   // the consumer handles validity bitmaps (generic scan-aggregate kernel)
    bool saw_nulls = false;     // some referenced column actually holds NULLs
    std::string why;   // reason of the last failure
};

inline bool fail(LowerCtx &cx, const std::string &s) { cx.why = s; return false; }

inline const Expr *strip_value_preserving_casts(const Expr *e)
{
    // DECIMAL(w,s) -> DECIMAL(w',s') widening casts keep the value (tryCastDecimalToDecimal,
    // function_cast.go:380-404); INTEGER/BIGINT widening likewise.
    while (e->kind == PG_TK_FUNC && e->fn == PG_FN_CAST && e->args.size() == 1) {
        const Expr &a = e->args[0];
        bool dec2dec = e->ltype == PG_LT_DECIMAL && a.ltype == PG_LT_DECIMAL && e->scale >= a.scale;
        bool int2int = (e->ltype == PG_LT_BIGINT || e->ltype == PG_LT_INTEGER || e->ltype == PG_LT_HUGEINT) &&
                       (a.ltype == PG_LT_INTEGER || a.ltype == PG_LT_BIGINT);   // incl. tryCastInt32ToHugeint (function_cast.go:321-325)
        bool int2dec = e->ltype == PG_LT_DECIMAL && (a.ltype == PG_LT_INTEGER || a.ltype == PG_LT_BIGINT) && a.kind == PG_TK_CONST;
        if (!(dec2dec || int2int || int2dec)) break;
        e = &a;
    }
    return e;
}

inline i64 byte_code(const Column &col, const std::string &s)
{
    if (col.type == PG_T_CHAR1) return s.size() == 1 ? (i64)(uint8_t)s[0] : -1;
    for (size_t i = 0; i < col.dict.size(); i++) if (col.dict[i] == s) return (i64)i;
    return -1;
}

inline bool lower_compare(LowerCtx &cx, const Expr &e, std::vector<Range> &ranges);

// `col IN (...)` and `a = x OR a = y OR ...` on ONE byte-coded column -> a code set
inline bool lower_byte_set(LowerCtx &cx, const Expr &e, std::vector<Range> &ranges)
{
    Range acc;
    acc.is_set = true;
    std::vector<const Expr *> todo{&e};
    while (!todo.empty()) {
        const Expr *x = todo.back();
        todo.pop_back();
        if (x->kind == PG_TK_FUNC && x->fn == PG_FN_OR) { for (auto &a : x->args) todo.push_back(&a); continue; }
        std::vector<Range> one;
        if (x->kind == PG_TK_FUNC && x->fn == PG_FN_IN && x->args.size() >= 2) {
            const Expr *c = strip_value_preserving_casts(&x->args[0]);
            if (c->kind != PG_TK_COL || c->idx < 0 || c->idx >= (int)cx.table->cols.size()) return fail(cx, "IN over a non-column");
            const Column &col = cx.table->cols[(size_t)c->idx];
            if (!is_byte_family(col.type)) return fail(cx, "IN is supported on dictionary/char columns only");
            if (col.any_nulls()) { if (!cx.allow_nulls) return fail(cx, "nullable column in predicate"); cx.saw_nulls = true; }
            Range r;
            r.col = c->idx;
            r.is_set = true;
            for (size_t i = 1; i < x->args.size(); i++) {
                const Expr *k = strip_value_preserving_casts(&x->args[i]);
                if (k->kind != PG_TK_STR) return fail(cx, "IN list element is not a string literal");
                i64 code = byte_code(col, k->str);
                if (code >= 0) r.set[code >> 5] |= 1u << (code & 31);
            }
            one.push_back(r);
        } else if (!lower_compare(cx, *x, one) || one.size() != 1) {
            return fail(cx, "OR branch is not a single comparison");
        }
        Range &r = one[0];
        if (!is_byte_family(cx.table->cols[(size_t)r.col].type)) return fail(cx, "OR / IN is supported on dictionary/char columns only");
        if (acc.col >= 0 && acc.col != r.col) return fail(cx, "OR over different columns");
        acc.col = r.col;
        range_to_set(r);
        for (int w = 0; w < 8; w++) acc.set[w] |= r.set[w];
    }
    if (acc.col < 0) return fail(cx, "empty OR");
    ranges.push_back(acc);
    return true;
}

// One conjunct `col <cmp> const` (either order) -> range on a table column.
inline bool lower_compare(LowerCtx &cx, const Expr &e, std::vector<Range> &ranges)
{
    if (e.kind != PG_TK_FUNC) return fail(cx, "filter is not a function call");
    if (e.fn == PG_FN_AND) {
        for (auto &a : e.args) if (!lower_compare(cx, a, ranges)) return false;
        return true;
    }
    if (e.fn == PG_FN_OR || e.fn == PG_FN_IN) return lower_byte_set(cx, e, ranges);
    if ((e.fn == PG_FN_LIKE || e.fn == PG_FN_NOT_LIKE) && e.args.size() == 2) {
        const Expr *c = strip_value_preserving_casts(&e.args[0]), *k = strip_value_preserving_casts(&e.args[1]);
        if (c->kind != PG_TK_COL || c->idx < 0 || c->idx >= (int)cx.table->cols.size() || k->kind != PG_TK_STR)
            return fail(cx, "LIKE needs a column and a string literal");
        const Column &col = cx.table->cols[(size_t)c->idx];
        if (col.any_nulls()) { if (!cx.allow_nulls) return fail(cx, "nullable column in predicate"); cx.saw_nulls = true; }
        Range rg;
        rg.col = c->idx;
        if (is_byte_family(col.type)) {          // dictionary / char column: match every code's string once, on the host
            rg.is_set = true;
            for (int code = 0; code < 256; code++) {
                std::string sv;
                if (col.type == PG_T_CHAR1) sv = std::string(1, (char)code);
                else if (code < (int)col.dict.size()) sv = col.dict[(size_t)code];
                else continue;
                bool m = wildcard_match(k->str.data(), k->str.size(), sv.data(), sv.size());
                if (m == (e.fn == PG_FN_LIKE)) rg.set[code >> 5] |= 1u << (code & 31);
            }
        } else if (col.type == PG_T_VARCHAR) {
            rg.like = e.fn == PG_FN_LIKE ? 1 : 2;
            rg.pat = k->str;
        } else {
            return fail(cx, "LIKE on a non-string column");
        }
        ranges.push_back(rg);
        return true;
    }
    if (!is_cmp(e.fn) || e.args.size() != 2) return fail(cx, "filter is not a comparison/AND");
    const Expr *l = &e.args[0], *r = &e.args[1];
    int op = e.fn;
    auto is_const = [](const Expr *x) {
        const Expr *y = strip_value_preserving_casts(x);
        return y->kind == PG_TK_CONST || y->kind == PG_TK_STR;
    };
    if (is_const(l) && !is_const(r)) { std::swap(l, r); op = flip_cmp(op); }
    if (!is_const(r)) return fail(cx, "comparison without a constant side");
    const Expr *k = strip_value_preserving_casts(r);
    // column side: COL or CAST(COL AS FLOAT/DOUBLE)
    bool float_cast = false;
    const Expr *c = l;
    if (c->kind == PG_TK_FUNC && c->fn == PG_FN_CAST && c->args.size() == 1 &&
        (c->ltype == PG_LT_FLOAT) && c->args[0].kind == PG_TK_COL) {
        float_cast = true;
        c = &c->args[0];
    } else {
        c = strip_value_preserving_casts(c);
    }
    if (c->kind != PG_TK_COL) return fail(cx, "comparison left side is not a column");
    if (c->idx < 0 || c->idx >= (int)cx.table->cols.size()) return fail(cx, "column index out of range");
    const Column &col = cx.table->cols[(size_t)c->idx];
    if (col.any_nulls()) {
        if (!cx.allow_nulls) return fail(cx, "nullable column in predicate");
        cx.saw_nulls = true;
    }
    Range rg;
    rg.col = c->idx;
    if (float_cast) {
        // cast(DECIMAL col AS FLOAT) cmp FLOAT const  (Q6 BETWEEN, builder_binder.go:517-580)
        if (col.type != PG_T_DECIMAL64 || k->kind != PG_TK_CONST || k->ltype != PG_LT_FLOAT)
            return fail(cx, "float cast comparison of unsupported types");
        if (op == PG_FN_NE) return fail(cx, "<> on float cast");
        if (col.gmax() >= ((i64)1 << 53) || col.gmin() <= -((i64)1 << 53)) return fail(cx, "decimal too wide for exact float cast");
        double kd;
        memcpy(&kd, &k->v0, 8);
        float kf = (float)kd;   // constants are stored as float32(val.F64) (chunk/vector.go:205-207)
        float_cmp_to_range(op, kf, col.scale, col.gmin(), col.gmax(), &rg.lo, &rg.hi);
        ranges.push_back(rg);
        return true;
    }
    if (is_byte_family(col.type)) {
        if (k->kind != PG_TK_STR) return fail(cx, "byte column compared with non-string");
        if (op != PG_FN_EQ && op != PG_FN_NE) return fail(cx, "only = and <> are supported on dictionary/char columns");
        i64 code = byte_code(col, k->str);
        if (op == PG_FN_EQ) {
            if (code < 0) { rg.lo = 1; rg.hi = 0; } else { rg.lo = rg.hi = code; }
        } else {                       // <> : every code but this one (equalStrOp negated, function_operator_boolean.go:99-104)
            rg.is_set = true;
            for (int c = 0; c < 256; c++) if (c != code) rg.set[c >> 5] |= 1u << (c & 31);
        }
        ranges.push_back(rg);
        return true;
    }
    if (col.type == PG_T_VARCHAR) {                  // equalStrOp / its negation: byte equality (function_operator_boolean.go:99-104)
        if (k->kind != PG_TK_STR) return fail(cx, "VARCHAR column compared with non-string");
        if (op != PG_FN_EQ && op != PG_FN_NE) return fail(cx, "only =, <>, LIKE and NOT LIKE are supported on VARCHAR columns");
        rg.like = op == PG_FN_EQ ? 3 : 4;
        rg.pat = k->str;
        ranges.push_back(rg);
        return true;
    }
    if (!is_int_family(col.type)) return fail(cx, "unsupported column type in predicate");
    if (k->kind != PG_TK_CONST) return fail(cx, "integer column compared with non-numeric constant");
    i64 kv = k->v0;
    if (col.type == PG_T_DECIMAL64) {
        // only `>` has a DECIMAL overload in the reference (function_scalar.go:1296-1303)
        if (k->ltype != PG_LT_DECIMAL || op != PG_FN_GT) return fail(cx, "DECIMAL comparison other than > DECIMAL");
        if (k->scale > col.scale) return fail(cx, "DECIMAL constant finer than column scale");
        for (int i = k->scale; i < col.scale; i++) kv *= 10;
    } else {
        if (k->ltype != PG_LT_INTEGER && k->ltype != PG_LT_BIGINT && k->ltype != PG_LT_DATE)
            return fail(cx, "integer/date column compared with non-integer constant");
    }
    switch (op) {
    case PG_FN_EQ: rg.lo = rg.hi = kv; break;
    case PG_FN_LT: if (kv == INT64_MIN) { rg.lo = 1; rg.hi = 0; } else rg.hi = kv - 1; break;
    case PG_FN_LE: rg.hi = kv; break;
    case PG_FN_GT: if (kv == INT64_MAX) { rg.lo = 1; rg.hi = 0; } else rg.lo = kv + 1; break;
    case PG_FN_GE: rg.lo = kv; break;
    default: return fail(cx, "<> is not a range");
    }
    ranges.push_back(rg);
    return true;
}

inline bool lower_filters(LowerCtx &cx, const std::vector<Expr> &filters, std::vector<Range> &out)
{
    std::vector<Range> raw;
    for (auto &f : filters) if (!lower_compare(cx, f, raw)) return false;
    for (auto &r : raw) {
        bool merged = false;
        for (auto &o : out) if (o.col == r.col && !o.like && !r.like) {
            if (o.is_set || r.is_set) {          // intersect as code sets
                Range rr = r;
                range_to_set(o);
                range_to_set(rr);
                for (int w = 0; w < 8; w++) o.set[w] &= rr.set[w];
            } else {
                range_and(o, r.lo, r.hi);
            }
            merged = true;
        }
        if (!merged) out.push_back(r);
    }
    return true;
}

// constant -> unscaled integer at `scale`
inline bool const_at_scale(const Expr *k, int scale, i64 *out)
{
    if (k->kind != PG_TK_CONST) return false;
    int ks = 0;
    if (k->ltype == PG_LT_DECIMAL) ks = k->scale;
    else if (k->ltype != PG_LT_INTEGER && k->ltype != PG_LT_BIGINT) return false;
    if (ks > scale) return false;
    i128 v = k->v0;
    for (int i = ks; i < scale; i++) v *= 10;
    if (v > INT64_MAX || v < INT64_MIN) return false;
    *out = (i64)v;
    return true;
}

// expression -> product of affine factors over table columns
inline bool lower_affprod(LowerCtx &cx, const Expr &e0, AffProd &out)
{
    const Expr *e = strip_value_preserving_casts(&e0);
    auto col_factor = [&](const Expr *c, Factor *f) {
        if (c->kind != PG_TK_COL) return false;
        if (c->idx < 0 || c->idx >= (int)cx.table->cols.size()) return false;
        const Column &col = cx.table->cols[(size_t)c->idx];
        if (!is_int_family(col.type) || col.type == PG_T_DATE32) return false;
        if (col.any_nulls()) {
            if (!cx.allow_nulls) return false;
            cx.saw_nulls = true;
        }
        f->col = c->idx;
        f->c = 0;
        f->s = 1;
        f->scale = col.type == PG_T_DECIMAL64 ? col.scale : 0;
        return true;
    };
    if (e->kind == PG_TK_COL) {
        Factor f;
        if (!col_factor(e, &f)) return fail(cx, "aggregate argument column unsupported");
        out.f.push_back(f);
        return true;
    }
    if (e->kind != PG_TK_FUNC || e->args.size() != 2) return fail(cx, "aggregate argument is not +,-,* of columns/constants");
    if (e->fn == PG_FN_MUL) return lower_affprod(cx, e->args[0], out) && lower_affprod(cx, e->args[1], out);
    if (e->fn == PG_FN_ADD || e->fn == PG_FN_SUB) {
        const Expr *l = strip_value_preserving_casts(&e->args[0]), *r = strip_value_preserving_casts(&e->args[1]);
        Factor f;
        i64 k;
        if (col_factor(r, &f) && const_at_scale(l, f.scale, &k)) {          // k +/- col
            f.c = k;
            f.s = e->fn == PG_FN_ADD ? 1 : -1;
        } else if (col_factor(l, &f) && const_at_scale(r, f.scale, &k)) {   // col +/- k
            f.c = e->fn == PG_FN_ADD ? k : -k;
            f.s = 1;
        } else {
            return fail(cx, "affine factor is not (constant +/- column)");
        }
        out.f.push_back(f);
        return true;
    }
    return fail(cx, "unsupported function in aggregate argument");
}

}  // namespace pg
