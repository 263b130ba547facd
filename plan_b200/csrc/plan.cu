// plan.cu -- pg_plan / pg_result: compile a plan descriptor, pick fused kernels, run,
// finalise in exact arithmetic, hand results back as native columns.
//
// Plays the role of the reference's executor tree for the off-loaded subtree
// (/root/reference/pkg/compute/executor.go:305-350 buildOperatorExec,
//  executor_aggr.go:106-262 aggExecutor.Execute): HAS_INIT drains the child completely,
// HAS_SCAN emits groups in first-insertion order (aggregate_hash.go:424-438).
#include <algorithm>
#include <chrono>
#include <memory>

#include "common.cuh"
#include "hostdec.hpp"
#include "pipeline.hpp"
#include "plan_ir.hpp"

namespace pg {

Pipeline::~Pipeline() {}

int build_scan_agg(pg_plan *plan, const Node &agg, const Node &scan, std::unique_ptr<Pipeline> *out);
int build_join_agg(pg_plan *plan, const Node &agg, const Node &join, std::unique_ptr<Pipeline> *out, bool nested = false);
int build_rows(pg_plan *plan, std::unique_ptr<Pipeline> *out, const Node *aggn = nullptr);      // rows.cu: row-emitting Scan / Filter / Project / Join; aggn: aggregate over the joined rows
int build_left_count(pg_plan *plan, const Node &root, std::unique_ptr<Pipeline> *out);            // join.cu: per-row counts of a LEFT join [+ Agg over them]

static const Node *skip_filters(const Node *n, std::vector<Expr> *extra)
{
    while (n->op == PG_OP_FILTER) {
        for (auto &f : n->filters) extra->push_back(f);
        n = &n->children[0];
    }
    return n;
}

// ORDER BY + LIMIT over a (small) result: the reference's Order operator compares normalized keys
// (sort_encoder.go:65-81): a DECIMAL key is Int64(2) -- the value rounded half-even to two
// fractional digits -- integers/dates by value, DESC inverts; ties keep an arbitrary order.
static i128 order_key(const ResCol &c, i64 row)
{
    const uint8_t *p = c.data.data() + (size_t)row * (size_t)type_size(c.type);
    switch (c.type) {
    case PG_T_INT32: case PG_T_DATE32: { int32_t v; memcpy(&v, p, 4); return v; }
    case PG_T_INT64: case PG_T_DECIMAL64: { i64 v; memcpy(&v, p, 8); return v; }
    case PG_T_CHAR1: case PG_T_DICT8: return *p;
    case PG_T_HUGEINT: { pg_hugeint h; memcpy(&h, p, 16); return (i128)(((u128)(u64)h.upper << 64) | h.lower); }
    case PG_T_DECIMAL128: {
        pg_decimal d;
        memcpy(&d, p, 16);
        u128 m = d.coef;
        if (d.scale > 2) m = hd_shift_right_even(m, d.scale - 2);
        else m *= hd_pow10(2 - d.scale);
        return d.neg ? -(i128)m : (i128)m;
    }
    default: return 0;
    }
}

static int sort_result(pg_result *r, const std::vector<std::pair<int, int>> &order, i64 limit)
{
    for (auto &o : order)
        if (o.first < 0 || o.first >= (int)r->cols.size()) PG_FAIL(PG_EINVAL, "ORDER BY column %d out of range", o.first);
    std::vector<i64> idx((size_t)r->nrows);
    for (i64 i = 0; i < r->nrows; i++) idx[(size_t)i] = i;
    auto less = [&](i64 a, i64 b) {
        for (auto &o : order) {
            const ResCol &c = r->cols[(size_t)o.first];
            if (c.type == PG_T_FLOAT64) {
                double x, y;
                memcpy(&x, c.data.data() + (size_t)a * 8, 8);
                memcpy(&y, c.data.data() + (size_t)b * 8, 8);
                if (x != y) return o.second ? x > y : x < y;
                continue;
            }
            if (c.type == PG_T_DICT8 && !c.dict.empty()) {       // VARCHAR key: byte order of the strings, not of the codes
                const std::string &x = c.dict[c.data[(size_t)a]], &y = c.dict[c.data[(size_t)b]];
                if (x != y) return o.second ? x > y : x < y;
                continue;
            }
            i128 x = order_key(c, a), y = order_key(c, b);
            if (x != y) return o.second ? x > y : x < y;
        }
        return false;
    };
    std::stable_sort(idx.begin(), idx.end(), less);
    i64 n = limit >= 0 && limit < r->nrows ? limit : r->nrows;
    for (ResCol &c : r->cols) {
        size_t w = (size_t)type_size(c.type);
        std::vector<uint8_t> out((size_t)n * w);
        for (i64 i = 0; i < n; i++) memcpy(out.data() + (size_t)i * w, c.data.data() + (size_t)idx[(size_t)i] * w, w);
        c.data.swap(out);
        if (!c.valid.empty()) {
            std::vector<uint8_t> v((size_t)n);
            for (i64 i = 0; i < n; i++) v[(size_t)i] = c.valid[(size_t)idx[(size_t)i]];
            c.valid.swap(v);
        }
    }
    r->nrows = n;
    return PG_OK;
}

// Statistics of a SHARDED table over all ranks' shards (Column::g_*): one all-gather of 64 bytes per column when a
// plan over the table is prepared.  Every choice that shapes a collective reads the agreed values, so all ranks
// build the same pipeline with the same buffer sizes (a rank whose shard happens to hold NULLs, wider values or
// other years than its peers no longer diverges).  Collective: every rank prepares its plans in the same order.
int agree_table_stats(pg_table *t)
{
    Context &c = ctx();
    const bool shared = c.world > 1 && t->dist == PG_DIST_SHARDED;
    if (t->g_version == t->version && t->g_world == c.world) return PG_OK;
    if (!shared) {
        for (Column &col : t->cols) col.g_ok = false;
        t->g_max_rows = t->g_total_rows = t->nrows;
        t->g_version = t->version;
        t->g_world = c.world;
        return PG_OK;
    }
    struct Rec { i64 vmin, vmax; uint32_t present[8]; i64 has_nulls, nrows; };
    static_assert(sizeof(Rec) == 64, "statistics record is exchanged as 64 bytes");
    const size_t ncol = t->cols.size();
    std::vector<Rec> mine(ncol), all(ncol * (size_t)c.world);
    for (size_t i = 0; i < ncol; i++) {
        const Column &col = t->cols[i];
        mine[i].vmin = col.vmin;
        mine[i].vmax = col.vmax;
        memcpy(mine[i].present, col.present, 32);
        mine[i].has_nulls = col.has_nulls ? 1 : 0;
        mine[i].nrows = t->nrows;
    }
    DevBuf ds, dr;
    PG_TRY(ds.alloc(ncol * 64));
    PG_TRY(dr.alloc(ncol * 64 * (size_t)c.world));
    PG_CUDA(cudaMemcpyAsync(ds.p, mine.data(), ncol * 64, cudaMemcpyHostToDevice, c.stream));
    PG_TRY(comm_allgather(ds.p, dr.p, ncol * 64, c.stream));
    PG_CUDA(cudaMemcpyAsync(all.data(), dr.p, ncol * 64 * (size_t)c.world, cudaMemcpyDeviceToHost, c.stream));
    PG_CUDA(cudaStreamSynchronize(c.stream));
    t->g_max_rows = t->g_total_rows = 0;
    for (int r = 0; r < c.world; r++) {
        const i64 n = all[(size_t)r * ncol].nrows;
        t->g_max_rows = std::max(t->g_max_rows, n);
        t->g_total_rows += n;
    }
    for (size_t i = 0; i < ncol; i++) {
        Column &col = t->cols[i];
        bool any = false;
        col.g_has_nulls = false;
        memset(col.g_present, 0, 32);
        col.g_vmin = col.g_vmax = 0;
        for (int r = 0; r < c.world; r++) {
            const Rec &x = all[(size_t)r * ncol + i];
            if (x.nrows == 0) continue;                  // an empty shard has no statistics
            col.g_vmin = any ? std::min(col.g_vmin, x.vmin) : x.vmin;
            col.g_vmax = any ? std::max(col.g_vmax, x.vmax) : x.vmax;
            any = true;
            col.g_has_nulls = col.g_has_nulls || x.has_nulls != 0;
            for (int w = 0; w < 8; w++) col.g_present[w] |= x.present[w];
        }
        col.g_ok = true;
    }
    t->g_version = t->version;
    t->g_world = c.world;
    return PG_OK;
}

static int build_pipeline(pg_plan *plan)
{
    const Node &root = plan->agg_root();
    if (root.op != PG_OP_AGG) {
        if (plan->topk) PG_FAIL(PG_EUNSUPPORTED, "ORDER BY / LIMIT is fused over aggregates only");
        return build_rows(plan, &plan->pipe);       // a Project / Filter / Join / Scan that returns rows
    }
    std::vector<Expr> extra;
    const Node *child = skip_filters(&root.children[0], &extra);
    if (child->op == PG_OP_SCAN) {
        Node scan = *child;
        for (auto &f : extra) scan.filters.push_back(f);
        // byte-coded (or no) group keys -> the shared-memory scan-aggregate kernels; integer keys of
        // arbitrary cardinality -> the global open-addressing group table (same machinery as the joins)
        bool int_keys = !root.groups.empty();
        for (auto &g : root.groups) {
            const Expr *e = strip_value_preserving_casts(&g);
            const pg_table *t = plan->slots[(size_t)scan.slot];
            if (e->kind != PG_TK_COL || e->idx < 0 || e->idx >= (int)t->cols.size() || !is_int_family(t->cols[(size_t)e->idx].type)) int_keys = false;
        }
        if (int_keys) {
            plan->scan_copy = scan;
            return build_join_agg(plan, root, plan->scan_copy, &plan->pipe);
        }
        return build_scan_agg(plan, root, scan, &plan->pipe);
    }
    if (child->op == PG_OP_JOIN && (child->jointype == PG_JOIN_MARK || child->jointype == PG_JOIN_ANTI_MARK)) {
        // EXISTS / NOT EXISTS: the reference plans a MARK join -- every probe row plus a boolean "found a match"
        // column, NULL for a NULL key (constructMarkJoinResult, join_scan.go:132-165) -- under Filter(mark = true | false)
        // (makeMarkCondFunc, builder_plan.go:380-400).  When the mark column is only filtered this is a SEMI join
        // (mark = true) or an ANTI join (mark = false; the probe key must be NULL-free, a NULL mark selects nothing).
        if (extra.size() != 1 || child->outs.empty() || child->outs.back().first != 2)
            PG_FAIL(PG_EUNSUPPORTED, "MARK join: expected exactly Filter(mark = constant) above it and the mark column last");
        for (size_t i = 0; i + 1 < child->outs.size(); i++)
            if (child->outs[i].first == 2) PG_FAIL(PG_EUNSUPPORTED, "MARK join: the mark column is projected more than once");
        const Expr &f = extra[0];
        if (f.kind != PG_TK_FUNC || (f.fn != PG_FN_EQ && f.fn != PG_FN_NE) || f.args.size() != 2) PG_FAIL(PG_EUNSUPPORTED, "MARK join: filter is not mark = constant");
        const Expr *c = strip_value_preserving_casts(&f.args[0]), *k = strip_value_preserving_casts(&f.args[1]);
        if (c->kind != PG_TK_COL) std::swap(c, k);
        if (c->kind != PG_TK_COL || c->idx != (int)child->outs.size() - 1 || k->kind != PG_TK_CONST || k->ltype != PG_LT_BOOLEAN)
            PG_FAIL(PG_EUNSUPPORTED, "MARK join: filter is not mark = constant");
        const bool want_match = (k->v0 != 0) == (f.fn == PG_FN_EQ);
        plan->mark_copy = *child;
        plan->mark_copy.jointype = want_match ? PG_JOIN_SEMI : PG_JOIN_ANTI;
        plan->mark_copy.outs.pop_back();
        if (!want_match) {
            // ANTI keeps probe rows with a NULL key, `mark = false` does not: only equivalent without NULL keys
            const Node *src = &plan->mark_copy.children[0];
            while (src->op == PG_OP_FILTER) src = &src->children[0];
            const Expr *pe = plan->mark_copy.conds.size() == 1 ? strip_value_preserving_casts(&plan->mark_copy.conds[0].first) : nullptr;
            if (!pe || pe->kind != PG_TK_COL || src->op != PG_OP_SCAN || pe->idx < 0 || pe->idx >= (int)plan->slots[(size_t)src->slot]->cols.size() ||
                plan->slots[(size_t)src->slot]->cols[(size_t)pe->idx].any_nulls())
                PG_FAIL(PG_EUNSUPPORTED, "MARK join filtered with mark = false over a nullable (or non-scan) probe key");
        }
        {
            const int s = build_join_agg(plan, root, plan->mark_copy, &plan->pipe);
            if (s != PG_EUNSUPPORTED || child->jointype != PG_JOIN_MARK) return s;
            // e.g. a build side filtered by a column-to-column comparison (TPC-H Q4's `l_commitdate < l_receiptdate`): the
            // MARK join as it stands, its mark filter and the aggregate run as row programs over the joined rows (rows.cu)
            const std::string why = get_error();
            plan->pipe.reset();
            const int s2 = build_rows(plan, &plan->pipe, &root);
            if (s2 == PG_EUNSUPPORTED) PG_FAIL(PG_EUNSUPPORTED, "%s; expression-driven join aggregate: %s", why.c_str(), std::string(get_error()).c_str());
            return s2;
        }
    }
    if (child->op == PG_OP_JOIN) {
        int s = PG_EUNSUPPORTED;
        std::string why = "filter between aggregate and join";
        if (extra.empty()) {
            s = build_join_agg(plan, root, *child, &plan->pipe);
            if (s != PG_EUNSUPPORTED) return s;
            why = get_error();
        }
        // not a shape of the affine-product join pipelines (CASE / OR / IN in the aggregates, a filter above the join,
        // a LEFT join ...): one join of two scans can still run as row programs over the joined rows (rows.cu)
        plan->pipe.reset();
        s = build_rows(plan, &plan->pipe, &root);
        if (s != PG_EUNSUPPORTED) return s;
        const std::string why2 = get_error();
        // a LEFT join counted per preserved row (TPC-H Q13's inner aggregate)
        plan->pipe.reset();
        s = build_left_count(plan, root, &plan->pipe);
        if (s == PG_EUNSUPPORTED)
            PG_FAIL(PG_EUNSUPPORTED, "%s; expression-driven join aggregate: %s; left-join count: %s", why.c_str(), why2.c_str(), std::string(get_error()).c_str());
        return s;
    }
    if (child->op == PG_OP_AGG) {
        // an aggregate over an aggregate: only the distribution of per-row LEFT-join counts (TPC-H Q13)
        const int s = build_left_count(plan, root, &plan->pipe);
        if (s == PG_EUNSUPPORTED) PG_FAIL(PG_EUNSUPPORTED, "unsupported aggregate input (op %d); left-join count: %s", child->op, std::string(get_error()).c_str());
        return s;
    }
    PG_FAIL(PG_EUNSUPPORTED, "unsupported aggregate input (op %d)", child->op);
}

}  // namespace pg

using namespace pg;

extern "C" {

int pg_plan_compile(const int64_t *desc, size_t nwords, pg_plan **out)
{
    if (!desc || !out || nwords < 3) PG_FAIL(PG_EINVAL, "pg_plan_compile: bad arguments");
    if (desc[0] != PG_DESC_MAGIC || desc[1] != PG_DESC_VERSION)
        PG_FAIL(PG_EINVAL, "pg_plan_compile: bad magic/version (%lld, %lld)", (long long)desc[0], (long long)desc[1]);
    DescReader rd(desc + 2, nwords - 2);
    std::unique_ptr<pg_plan> p(new pg_plan());
    if (!rd.node(&p->root) || !rd.ok()) PG_FAIL(PG_EINVAL, "pg_plan_compile: malformed descriptor near word %zu", rd.pos() + 2);
    if (rd.pos() != nwords - 2) PG_FAIL(PG_EINVAL, "pg_plan_compile: %zu trailing words", nwords - 2 - rd.pos());
    // number of table slots = max scan slot + 1
    int nslots = 0;
    std::vector<const Node *> todo{&p->root};
    while (!todo.empty()) {
        const Node *n = todo.back();
        todo.pop_back();
        if (n->op == PG_OP_SCAN) {
            if (n->slot < 0 || n->slot > 63) PG_FAIL(PG_EINVAL, "pg_plan_compile: scan slot %d out of range", n->slot);
            nslots = std::max(nslots, n->slot + 1);
        }
        for (auto &c : n->children) todo.push_back(&c);
    }
    p->slots.assign((size_t)nslots, nullptr);
    // structural check now, kernel selection when the tables are bound
    if (p->root.op == PG_OP_TOPK) {
        p->topk = &p->root;
        for (auto &o : p->root.order)
            if (o.first < 0 || o.first >= (int)p->root.children[0].outs.size()) PG_FAIL(PG_EINVAL, "pg_plan_compile: ORDER BY refers to output %d", o.first);
    }
    {
        const int op = p->agg_root().op;
        if (op != PG_OP_AGG && (p->topk || (op != PG_OP_PROJECT && op != PG_OP_FILTER && op != PG_OP_JOIN && op != PG_OP_SCAN)))
            PG_FAIL(PG_EUNSUPPORTED, "pg_plan_compile: the root must be an aggregate (optionally under ORDER BY / LIMIT) or a row-emitting Project / Filter / Join / Scan");
    }
    *out = p.release();
    return PG_OK;
}

int pg_plan_bind(pg_plan *p, int slot, pg_table *t)
{
    if (!p || !t || slot < 0 || slot >= (int)p->slots.size()) PG_FAIL(PG_EINVAL, "pg_plan_bind: bad arguments");
    if (!t->sealed) PG_FAIL(PG_ESTATE, "pg_plan_bind: table %s is not sealed", t->name.c_str());
    p->slots[(size_t)slot] = t;
    p->pipe.reset();
    return PG_OK;
}

static int ensure_pipeline(pg_plan *p)
{
    for (size_t i = 0; i < p->slots.size(); i++)
        if (!p->slots[i]) PG_FAIL(PG_ESTATE, "plan slot %zu is not bound", i);
    bool stale = !p->pipe;
    if (p->pipe) {
        for (size_t i = 0; i < p->slots.size(); i++)
            if (p->bound_versions[i] != p->slots[i]->version) stale = true;
        if (p->pipe_world != ctx().world) stale = true;
    }
    if (!stale) return PG_OK;
    p->pipe.reset();
    PG_CUDA(cudaSetDevice(ctx().device));
    for (size_t i = 0; i < p->slots.size(); i++) PG_TRY(agree_table_stats(p->slots[i]));
    PG_TRY(build_pipeline(p));
    p->bound_versions.resize(p->slots.size());
    for (size_t i = 0; i < p->slots.size(); i++) p->bound_versions[i] = p->slots[i]->version;
    p->pipe_world = ctx().world;
    return PG_OK;
}

int pg_plan_prepare(pg_plan *p)
{
    if (!p) PG_FAIL(PG_EINVAL, "pg_plan_prepare: null plan");
    if (!ctx().ready) PG_FAIL(PG_ESTATE, "pg_plan_prepare: call pg_init first");
    return ensure_pipeline(p);
}

const char *pg_plan_explain(pg_plan *p)
{
    if (!p) return "";
    if (ensure_pipeline(p) != PG_OK) return get_error();
    return p->pipe->explain.c_str();
}

int pg_plan_execute(pg_plan *p, pg_result **out)
{
    if (!p || !out) PG_FAIL(PG_EINVAL, "pg_plan_execute: bad arguments");
    if (!ctx().ready) PG_FAIL(PG_ESTATE, "pg_plan_execute: call pg_init first");
    PG_TRY(ensure_pipeline(p));
    PG_CUDA(cudaSetDevice(ctx().device));
    std::unique_ptr<pg_result> r(new pg_result());
    auto t0 = std::chrono::steady_clock::now();
    PG_TRY(p->pipe->run(r.get()));
    if (p->topk) PG_TRY(sort_result(r.get(), p->topk->order, p->topk->limit));   // pipelines pre-select candidates on the device
    auto t1 = std::chrono::steady_clock::now();
    r->stats.exec_ms = std::chrono::duration<double, std::milli>(t1 - t0).count();
    *out = r.release();
    return PG_OK;
}

void pg_plan_free(pg_plan *p)
{
    if (!p) return;
    if (ctx().ready) cudaSetDevice(ctx().device);
    delete p;
}

int pg_result_num_columns(const pg_result *r, int *ncol)
{
    if (!r || !ncol) PG_FAIL(PG_EINVAL, "pg_result_num_columns: bad arguments");
    *ncol = (int)r->cols.size();
    return PG_OK;
}

int pg_result_column_type(const pg_result *r, int col, int32_t *type, int32_t *width, int32_t *scale)
{
    if (!r || col < 0 || col >= (int)r->cols.size()) PG_FAIL(PG_EINVAL, "pg_result_column_type: bad arguments");
    if (type) *type = r->cols[(size_t)col].type;
    if (width) *width = r->cols[(size_t)col].width;
    if (scale) *scale = r->cols[(size_t)col].scale;
    return PG_OK;
}

int pg_result_column_dict(const pg_result *r, int col, int32_t *nentries, const char *const **entries)
{
    if (!r || col < 0 || col >= (int)r->cols.size() || !nentries || !entries) PG_FAIL(PG_EINVAL, "pg_result_column_dict: bad arguments");
    pg_result *w = const_cast<pg_result *>(r);
    if ((size_t)col >= w->dict_ptrs.size()) w->dict_ptrs.resize(r->cols.size());
    std::vector<const char *> &ptrs = w->dict_ptrs[(size_t)col];
    ptrs.clear();
    for (auto &e : r->cols[(size_t)col].dict) ptrs.push_back(e.c_str());
    *nentries = (int32_t)ptrs.size();
    *entries = ptrs.empty() ? nullptr : ptrs.data();
    return PG_OK;
}

int pg_result_rows(const pg_result *r, int64_t *nrows)
{
    if (!r || !nrows) PG_FAIL(PG_EINVAL, "pg_result_rows: bad arguments");
    *nrows = r->nrows;
    return PG_OK;
}

int pg_result_next(pg_result *r, int64_t max_rows, int64_t *nrows, const void **cols, const uint8_t **valid)
{
    if (!r || !nrows || max_rows <= 0) PG_FAIL(PG_EINVAL, "pg_result_next: bad arguments");
    i64 n = std::min<i64>(max_rows, r->nrows - r->cursor);
    if (n < 0) n = 0;
    for (size_t i = 0; i < r->cols.size(); i++) {
        ResCol &c = r->cols[i];
        if (cols) cols[i] = n > 0 ? (const void *)(c.data.data() + (size_t)r->cursor * (size_t)type_size(c.type)) : nullptr;
        if (valid) {
            valid[i] = nullptr;
            bool any_null = false;
            for (i64 k = 0; k < n && !c.valid.empty(); k++) any_null = any_null || !c.valid[(size_t)(r->cursor + k)];
            if (any_null) {      // packed bits, 1 = valid, LSB first (pkg/util/bitmap.go); owned by the result
                r->valid_scratch.emplace_back((size_t)(n + 7) / 8, 0);
                std::vector<uint8_t> &bm = r->valid_scratch.back();
                for (i64 k = 0; k < n; k++) if (c.valid[(size_t)(r->cursor + k)]) bm[(size_t)k >> 3] |= (uint8_t)(1u << (k & 7));
                valid[i] = bm.data();
            }
        }
    }
    *nrows = n;
    r->cursor += n;
    return PG_OK;
}

int pg_result_rewind(pg_result *r)
{
    if (!r) PG_FAIL(PG_EINVAL, "pg_result_rewind: null");
    r->cursor = 0;
    return PG_OK;
}

int pg_result_stats(const pg_result *r, pg_stats *out)
{
    if (!r || !out) PG_FAIL(PG_EINVAL, "pg_result_stats: bad arguments");
    *out = r->stats;
    return PG_OK;
}

void pg_result_free(pg_result *r) { delete r; }

}  // extern "C"
