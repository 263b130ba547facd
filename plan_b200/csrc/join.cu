// join.cu -- `Agg <- Join(...)` pipelines: hash-table builds, probe, high-cardinality group-by.
//
// Reference operators replaced (SURVEY.md 3.3): joinExecutor.hashJoinExec
// (/root/reference/pkg/compute/executor_join.go:62-123) with the build side always
// Children[1] (:237-264), HashJoin.Build / JoinHashTable.Finalize (join_types.go:100,
// join_table.go:85-288), Scan.Next probe (join_scan.go:182-299), and the aggExecutor on
// top (executor_aggr.go:106-262) whose group table is GroupedAggrHashTable.
//
// Supported tree (covers TPC-H Q3): the aggregate's input is an INNER equi-join whose
// probe side is a filtered scan and whose build side is a filtered scan or, recursively,
// such a join; every column needed above a join comes from that join's probe-side source
// table (late gather by row id).  Pipelines, bottom-up (classic pipeline breakers):
//   build(customer) -> build(orders probing customer) -> lineitem probing orders -> group-by
#include <algorithm>

#include <cub/device/device_scan.cuh>

#include "hostdec.hpp"
#include "join.cuh"
#include "exchange.cuh"
#include "leftcount.cuh"
#include "pipeline.hpp"

namespace pg {

namespace {

struct BaseCol { int slot = -1, col = -1; };

// one pipeline: source scan + predicates [+ probe] -> sink
struct Stage {
    int src_slot = -1;
    std::vector<Range> ranges;
    bool has_probe = false;
    int probe_mode = 0;              // 0 INNER, 1 SEMI, 2 ANTI -- how this stage's own probe filters its source rows
    bool existence_only = false;     // the join consuming this build side is SEMI/ANTI: only key existence matters
    int probe_key_col = -1;          // on the source table
    int probe_stage = -1;            // which earlier stage built the probed table
    int ins_key_col = -1;            // SINK_INSERT: key column on the source table
    // device state of the table this stage builds
    DevBuf d_slots, d_bitmap, d_rank_prefix, d_rank_payload, d_keys_tmp, d_scan_tmp, d_bm_all;
    size_t bitmap_words = 0;
    JoinTable jt{};
    bool rank_index = false;         // unique keys + bitmap: the table is bitmap + rank prefix + payload (join.cuh jt_rank)
    // further existence tests on this stage's source rows (pushed-down SEMI / ANTI joins, INNER joins
    // against unique keys): {mode 0 INNER / 1 SEMI / 2 ANTI, key column on the source table, probed stage}
    struct Extra { int mode, key_col, stage; };
    std::vector<Extra> extras;
    // build side that is itself an aggregate (`key IN (select k from t group by k having ...)`): its
    // group keys are computed on the device by a nested pipeline and become an existence bitmap
    std::unique_ptr<Pipeline> sub;
    Node sub_scan;
    int ins_key_col2 = -1;           // two-column build key (k << 32 | k2): hash table, no bitmap
    i64 capacity_rows = 0;
    i64 built_rows = 0;
    bool payload_needed = false;     // some column of this build side is read above the join
    bool unique_key = false;         // build key is strictly increasing in row order (statistics) => unique
    bool no_table = false;           // unique + payload-free + no probe of its own: the exact bitmap IS the build side
    i64 dup_keys = 0;                // duplicates seen while building (bitmap builds only)
    bool bitmap_only() const { return jt.bitmap && !payload_needed && (dup_keys == 0 || existence_only); }
};

static u64 next_pow2(u64 x)
{
    u64 p = 1;
    while (p < x) p <<= 1;
    return p;
}

static TypedCol typed(const pg_table *t, int col)
{
    TypedCol c;
    c.p = t->cols[(size_t)col].d_data;
    c.width = t->cols[(size_t)col].phys_width();
    c.base = t->cols[(size_t)col].base;
    c.valid = t->cols[(size_t)col].has_nulls ? t->cols[(size_t)col].d_valid : nullptr;
    return c;
}

}  // namespace

struct JoinAggPipeline : Pipeline {
    pg_plan *plan = nullptr;
    std::vector<std::unique_ptr<Stage>> stages;   // build stages in execution order
    // final stage: probe source
    int src_slot = -1;
    std::vector<Range> ranges;
    int probe_key_col = -1;
    GroupSpec gs{};
    int nparts = 0;
    BaseCol part_col[GT_MAXKEYPARTS];
    int part_type[GT_MAXKEYPARTS] = {0, 0, 0};
    std::vector<AggExpr> aggs;
    std::vector<int> agg_scale;
    std::vector<int> agg_plane;                  // accumulator plane of each aggregate (count(*) = the row-count plane)
    bool no_join = false;                        // Agg <- Scan on high-cardinality keys: no probe at all
    int top_probe_mode = 0;                      // INNER / SEMI / ANTI of the top join
    int hav_plane = -1;                          // HAVING <aggregate> in [hav_lo, hav_hi]
    i64 hav_lo = INT64_MIN, hav_hi = INT64_MAX;
    i64 group_hint = 0;                          // expected number of groups (no-join case)
    i64 key_min = 0;                             // statistics of the first group key (no-join case)
    u64 key_domain = 0;
    bool key_sorted = false;                     // first group key never descends in row order (no-join case)
    bool device_only = false;                    // nested use: stop after the group list is on the device
    i64 dev_ngroups = 0;
    std::vector<Stage::Extra> extras;            // existence tests on the top probe's source rows
    // Group keys functionally dependent on the top join's unique build key (TPC-H Q18 groups by five
    // columns of one orders row): the group table is keyed by the build ROW ID alone and the key columns
    // are fetched once per output group.  kind 0: column of the top build table at that row; kind 1: the
    // row's `via_key_col` looked up in the table (rank index or hash table) of the deeper unique build side `via_stage`.
    // In a star join (`star && fd_mode`) the groups are the rows of lookup `star_anchor - 1` (hits_star_rows_kernel).
    bool fd_mode = false;
    struct FdOut { int kind, slot, col, via_key_col, via_stage; };
    std::vector<FdOut> fd;
    int fd_stage = -1;                           // the build stage whose row ids the groups are
    int star_anchor = -1;
    // Star joins (see hits_star_kernel): `main_stage` is the existence join the filter pass tests, `lookups`
    // are all INNER joins of the fact-table spine bottom-up; origin 0 = the fact table, j = lookup j-1's table
    bool star = false;
    int main_stage = -1;
    struct HRef { int origin = 0, col = -1; };
    struct HLookup { int nkey = 1; HRef key[2]; int stage = -1; };
    struct HPart { HRef v; int fn = 0; i64 lo = 0; int n = 1; int type = 0; };
    struct HTerm { int nfac = 0; HRef fac[3]; i64 fc[3] = {0, 0, 0}; int fs[3] = {1, 1, 1}; i64 mul = 1; };
    std::vector<HLookup> lookups;
    std::vector<int> origin_slot;
    std::vector<HPart> sparts;
    std::vector<HTerm> sterms;
    int star_ngroups = 0, star_scale = 0;
    i128 star_worst = 0;                         // largest |value| one joined row can add to a group sum
    // Exchange lookup (exchange.cuh): the ONE join of the star whose build side is sharded on another key than the
    // fact table.  Both sides are hash-partitioned by the join key and shipped to the owner rank, which joins and sums.
    int xl = -1;                                 // index into `lookups`, -1: every join is local
    std::vector<int> xcols;                      // build-table columns carried to the owner (read by deferred factors)
    int x_term_mask[STAR_MAXTERM] = {0, 0};      // bit f: factor f of the term reads the exchanged build side
    int x_fac_col[STAR_MAXTERM][3] = {{0, 0, 0}, {0, 0, 0}};   // ... and which carried column it reads
    DevBuf d_xb_rec, d_xb_dest, d_xb_send, d_xb_recv, d_xp_rec, d_xp_dest, d_xp_send, d_xp_recv;
    i64 xb_recv_rows = 0;
    EventPair ev_xb, ev_xp;
    i64 x_sent_rows = 0, x_sent_bytes = 0;
    DevBuf d_star, d_star_all;
    PinBuf h_star;
    Stage &top_stage_ref() { return *stages[(size_t)(main_stage >= 0 ? main_stage : (int)stages.size() - 1)]; }
    DevBuf d_edges, d_dense;
    int dense_passes = 0;
    std::vector<std::pair<int, int>> outs;
    std::vector<int> group_out_type;             // pg_type of each group key
    i64 algorithmic_bytes = 0, main_bytes = 0;
    // device scratch
    DevBuf d_counters, d_gt, d_overflow, d_out_klo, d_out_khi, d_out_acc;
    u64 gt_cap = 0;
    i64 out_cap = 0;
    EventPair ev_all, ev_main;
    bool shuffle = false;          // local groups of different ranks may collide: hash-partition + all-to-all + merge
    bool gather_ranks = false;     // probe side is sharded: every rank ends with the union of all groups
    DevBuf d_g_klo, d_g_khi, d_g_acc, d_g_cnt;
    PinBuf h_out;                  // pinned landing zone of the group lists: [klo | khi | acc planes]
    static constexpr int SG_CAP = 256;   // rows per rank in the single-message gather of top-k candidates
    DevBuf d_sg;
    PinBuf h_sg;
    // fused ORDER BY ... LIMIT k: device pre-selection on the primary key
    bool has_topk = false;
    TopkKey topk_key{};
    i64 topk_limit = -1;
    DevBuf d_hist, d_cand_klo, d_cand_khi, d_cand_acc, d_tstate;
    PinBuf h_hist;
    i64 cand_cap = 0;

    // replace the compacted group list (d_out_*, n groups) by the candidates for the first k rows
    int topk_preselect(i64 *ngroups, pg_result *res)
    {
        cudaStream_t st = ctx().stream;
        i64 n = *ngroups, k = topk_limit;
        if (k < 0 || n <= k) return PG_OK;
        if (k == 0) { *ngroups = 0; return PG_OK; }
        const int planes = gs.nacc + 1 + (int)fd.size();       // dependent keys too: the fast path falls back here after their gather
        constexpr int NB = 1 << TOPK_DIGIT_BITS;
        // hist buffer: [256 bins][min, max as two u64]
        if (!d_hist.p) { PG_TRY(d_hist.alloc(NB * 4 + 16)); PG_TRY(h_hist.alloc(NB * 4 + 16)); }
        int grid = (int)std::max<i64>(std::min<i64>((n + 255) / 256, (i64)ctx().prop.multiProcessorCount * 4), 1);
        u64 prefix = 0;
        i64 remaining = k;       // we look for the remaining-th smallest key among those matching the prefix
        const unsigned *hist = h_hist.as<unsigned>();
        unsigned long long *d_minmax = (unsigned long long *)(d_hist.as<unsigned>() + NB);
        const unsigned long long *h_minmax = (const unsigned long long *)(hist + NB);
        i64 n_equal = n;
        // The passes stop as soon as the bin holding the k-th key is small (the host orders the few
        // candidates anyway), and the first pass also yields min/max so that digits common to every key
        // are skipped: a revenue column uses ~26 of its 64 key bits -> 3 passes instead of 8.
        const i64 stop_at = std::max<i64>(128 - k, 16);
        const int npass = 64 / TOPK_DIGIT_BITS;
        int pass = 0;
        while (pass < npass && (pass == 0 || n_equal > stop_at)) {
            PG_CUDA(cudaMemsetAsync(d_hist.p, 0, NB * 4, st));
            if (pass == 0) {
                PG_CUDA(cudaMemsetAsync(d_minmax, 0xff, 8, st));
                PG_CUDA(cudaMemsetAsync(d_minmax + 1, 0, 8, st));
                topk_hist_kernel<true><<<grid, 256, 0, st>>>(topk_key, d_out_klo.as<i64>(), d_out_khi.as<i64>(), d_out_acc.as<i64>(), out_cap, n,
                                                             prefix, 0, d_hist.as<unsigned>(), d_minmax);
            } else {
                topk_hist_kernel<false><<<grid, 256, 0, st>>>(topk_key, d_out_klo.as<i64>(), d_out_khi.as<i64>(), d_out_acc.as<i64>(), out_cap, n,
                                                              prefix, pass * TOPK_DIGIT_BITS, d_hist.as<unsigned>(), d_minmax);
            }
            PG_CUDA(cudaGetLastError());
            PG_CUDA(cudaMemcpyAsync(h_hist.p, d_hist.p, NB * 4 + 16, cudaMemcpyDeviceToHost, st));
            PG_CUDA(cudaStreamSynchronize(st));
            int d = 0;
            for (; d < NB; d++) {
                if ((i64)hist[d] >= remaining) break;
                remaining -= (i64)hist[d];
            }
            if (d == NB) PG_FAIL(PG_ECUDA, "internal: top-k radix select ran off the histogram");
            prefix = (prefix << TOPK_DIGIT_BITS) | (u64)d;
            n_equal = (i64)hist[d];
            res->stats.kernel_launches += 1;
            pass++;
            if (pass == 1) {
                // digits shared by every key: jump over them (all n keys carry that prefix, none is smaller)
                const u64 diff = (u64)h_minmax[0] ^ (u64)h_minmax[1];
                int common = 64;
                if (diff) { common = 0; while (!((diff << common) >> 63)) common++; }
                const int skip_to = std::min(common / TOPK_DIGIT_BITS, npass);
                if (skip_to > pass) {
                    pass = skip_to;
                    prefix = pass == npass ? (u64)h_minmax[0] : (u64)h_minmax[0] >> (64 - pass * TOPK_DIGIT_BITS);
                    remaining = k;
                    n_equal = n;
                }
            }
        }
        // keys <= threshold are the candidates: the prefix, widened by the digits that were not examined
        const int rest_bits = 64 - pass * TOPK_DIGIT_BITS;
        if (rest_bits > 0) prefix = (prefix << rest_bits) | ((((u64)1) << rest_bits) - 1);
        i64 ncand = (k - remaining) + n_equal;      // strictly smaller keys + every tie of the k-th key
        if (ncand > cand_cap) {
            PG_TRY(d_cand_klo.alloc((size_t)ncand * 8));
            PG_TRY(d_cand_khi.alloc((size_t)ncand * 8));
            PG_TRY(d_cand_acc.alloc((size_t)ncand * 8 * (size_t)planes));
            cand_cap = ncand;
        }
        PG_CUDA(cudaMemsetAsync(d_counters.p, 0, 32, st));
        topk_collect_kernel<<<grid, 256, 0, st>>>(topk_key, d_out_klo.as<i64>(), d_out_khi.as<i64>(), d_out_acc.as<i64>(), out_cap, n, planes,
                                                  prefix, d_cand_klo.as<i64>(), d_cand_khi.as<i64>(), d_cand_acc.as<i64>(), cand_cap,
                                                  d_counters.as<unsigned long long>());
        PG_CUDA(cudaGetLastError());
        res->stats.kernel_launches += 1;
        // the candidate arrays become the output arrays
        std::swap(d_out_klo.p, d_cand_klo.p); std::swap(d_out_klo.bytes, d_cand_klo.bytes);
        std::swap(d_out_khi.p, d_cand_khi.p); std::swap(d_out_khi.bytes, d_cand_khi.bytes);
        std::swap(d_out_acc.p, d_cand_acc.p); std::swap(d_out_acc.bytes, d_cand_acc.bytes);
        std::swap(out_cap, cand_cap);
        *ngroups = ncand;
        return PG_OK;
    }

    const pg_table *tab(int slot) const { return plan->slots[(size_t)slot]; }

    int fill_preds(PipeParams &pp, const std::vector<Range> &all, int slot)
    {
        std::vector<Range> rs;
        pp.nlike = 0;
        for (auto &r : all) {
            if (!r.like) { rs.push_back(r); continue; }
            // string predicate on a VARCHAR column: evaluated by pipeline_kernel (the two-phase filter does not take them)
            const Column &col = tab(slot)->cols[(size_t)r.col];
            if (pp.nlike >= GEN_MAXLIKE || r.pat.size() > GEN_PATMAX || !col.d_off) PG_FAIL(PG_EUNSUPPORTED, "string predicate not off-loadable in a join pipeline");
            GenLike &l = pp.like[pp.nlike++];
            l.bytes = col.d_bytes;
            l.off = (const i64 *)col.d_off;
            l.kind = r.like;
            l.plen = (int)r.pat.size();
            memcpy(l.pat, r.pat.data(), r.pat.size());
            std::string lit;
            if (r.like <= 2 && like_is_contains(r.pat, &lit)) {      // '%lit%': word-at-a-time search
                l.kind = r.like == 1 ? 5 : 6;
                l.plen = (int)lit.size();
                memcpy(l.pat, lit.data(), lit.size());
            }
        }
        if (rs.size() > PIPE_MAXPRED) PG_FAIL(PG_EUNSUPPORTED, "more than %d predicate columns on one scan", PIPE_MAXPRED);
        pp.npred = (int)rs.size();
        for (size_t i = 0; i < rs.size(); i++) {
            pp.pred[i].col = typed(tab(slot), rs[i].col);
            pp.pred[i].lo = rs[i].lo;
            pp.pred[i].hi = rs[i].hi;
            pp.pred[i].is_set = rs[i].is_set ? 1 : 0;          // code sets live on 1-byte columns: never taken by the 32-bit filter pass
            memcpy(pp.pred[i].mask, rs[i].set, sizeof pp.pred[i].mask);
        }
        return PG_OK;
    }

    int fill_extras(PipeParams &pp, const std::vector<Stage::Extra> &ex, int slot)
    {
        if (ex.size() > PIPE_MAXEXTRA) PG_FAIL(PG_EUNSUPPORTED, "more than %d existence joins on one scan", PIPE_MAXEXTRA);
        pp.nextra = (int)ex.size();
        for (size_t i = 0; i < ex.size(); i++) {
            const Stage &b = *stages[(size_t)ex[i].stage];
            if (!b.jt.bitmap) PG_FAIL(PG_EUNSUPPORTED, "existence join against a key domain too wide for a bitmap");
            if (ex[i].mode == 0 && b.dup_keys != 0 && !b.unique_key) PG_FAIL(PG_EUNSUPPORTED, "INNER join pushed to an existence test found duplicate build keys");
            pp.extra[i].key = typed(tab(slot), ex[i].key_col);
            pp.extra[i].bitmap = b.jt.bitmap;
            pp.extra[i].bm_min = b.jt.bm_min;
            pp.extra[i].domain = b.jt.domain;
            pp.extra[i].anti = ex[i].mode == 2 ? 1 : 0;
        }
        return PG_OK;
    }

    // d_counters: words 0..3 are the running stage's counters; words 4..7 keep {rows passing, rows built} of the first two
    // build stages whose own read-back was skipped -- they ride along with whichever read comes next
    pg_result *cur_res = nullptr;
    unsigned deferred_stats = 0;
    int read_counters(unsigned long long *out2)
    {
        unsigned long long h[8];
        PG_CUDA(cudaMemcpyAsync(h, d_counters.p, 64, cudaMemcpyDeviceToHost, ctx().stream));
        PG_CUDA(cudaStreamSynchronize(ctx().stream));
        memcpy(out2, h, 32);
        for (int idx = 0; idx < 2; idx++)
            if (((deferred_stats >> idx) & 1u) && cur_res) {
                cur_res->stats.aux[2 + 2 * idx] = (i64)h[4 + 2 * idx];
                cur_res->stats.aux[3 + 2 * idx] = (i64)h[5 + 2 * idx];
            }
        return PG_OK;
    }

    static int grid_rows(i64 nrows)
    {
        i64 g = (nrows + 255) / 256;
        i64 cap = (i64)ctx().prop.multiProcessorCount * 8;
        if (g > cap) g = cap;
        return (int)std::max<i64>(g, 1);
    }

    // scratch of the two-phase path: hit list (row ids) and its device-side cursor
    DevBuf d_hits, d_hit_count;
    static constexpr i64 HIT_CHUNK = (i64)1 << 30;     // rows screened per filter launch: row-id scratch of at most 4 GB
                                                       // (180 GB of HBM3e; SF100 lineitem needs 2.4 GB and ONE launch)

    static bool two_phase_ok(const PipeParams &pp, const pg_table *t, bool ins_sink)
    {
        bool any_valid = pp.probe_key.valid != nullptr || (ins_sink && pp.ins_key.valid != nullptr);
        for (int k = 0; k < pp.npred; k++) any_valid = any_valid || pp.pred[k].col.valid != nullptr;
        // (a build stage without a probe of its own also qualifies: the filter pass then lists every row that
        //  passes the predicate -- pp.probe_key must name the key column so the vector loads have a source)
        return (pp.has_probe ? pp.probe.bitmap != nullptr : ins_sink) && pp.nlike == 0 && pp.npred <= 1 && (pp.npred == 0 || !pp.pred[0].is_set) && !any_valid && t->nrows < ((i64)1 << 32) &&
               !getenv("PG_JOIN_GENERIC");
    }

    // phase 1 over rows [lo, hi): fills d_hits / d_hit_count (cursor reset first)
    int launch_filter(PipeParams &pp, i64 lo, i64 hi)
    {
        cudaStream_t st = ctx().stream;
        if (!d_hit_count.p) PG_TRY(d_hit_count.alloc(8));
        size_t need = (size_t)std::max<i64>(hi - lo, 1) * 4;
        if (d_hits.bytes < need) PG_TRY(d_hits.alloc(need));
        PG_CUDA(cudaMemsetAsync(d_hit_count.p, 0, 8, st));
        pp.row_begin = lo;
        pp.row_end = hi;
        pp.hits = d_hits.as<unsigned>();
        pp.hit_count = d_hit_count.as<unsigned long long>();
        if (try_staged_filter(pp, lo, hi) == PG_OK) return PG_OK;
        i64 ntiles = (hi - lo + SA_TILE - 1) / SA_TILE;
        int grid = (int)std::max<i64>(std::min<i64>(ntiles, (i64)ctx().prop.multiProcessorCount * 8), 1);
        // (two tiles per step were measured slower: 90 registers cost more occupancy than the extra loads in flight bring)
        if (pp.npred == 1) filter_hits_kernel<true, 1><<<grid, SA_THREADS, 0, st>>>(pp);
        else filter_hits_kernel<false, 1><<<grid, SA_THREADS, 0, st>>>(pp);
        PG_CUDA(cudaGetLastError());
        return PG_OK;
    }

    // The bulk-copy staged filter (join.cuh) when predicate and key are stored in <= 4 bytes and the 32-bit
    // domain test is provably exact.  Returns PG_OK when it was launched, PG_EUNSUPPORTED to use the kernel above.
    bool staged_filter_used = false;
    int try_staged_filter(const PipeParams &pp, i64 lo, i64 hi)
    {
        if (getenv("PG_NO_STAGED") && atoi(getenv("PG_NO_STAGED"))) return PG_EUNSUPPORTED;
        if (hi <= lo || (lo & 15) != 0 || pp.npred > 1) return PG_EUNSUPPORTED;
        const TypedCol &kc = pp.probe_key;
        if (!kc.p || kc.width > 4 || kc.valid) return PG_EUNSUPPORTED;
        FilterSParams fp{};
        fp.bitmap = pp.has_probe ? pp.probe.bitmap : nullptr;
        if (pp.has_probe && !fp.bitmap) return PG_EUNSUPPORTED;
        fp.anti = pp.probe_mode == 2 ? 1 : 0;
        auto stored_span = [](const TypedCol &c, i64 *tmin, i64 *tmax) {
            if (c.width == 4) { *tmin = INT32_MIN; *tmax = INT32_MAX; }
            else { *tmin = 0; *tmax = c.width == 2 ? 0xffff : 0xff; }
        };
        if (fp.bitmap) {
            // off = logical - bm_min = stored + (base - bm_min); every stored value the type can hold must land, mod 2^32,
            // outside [0, dom) unless its true offset is inside
            if (pp.probe.domain > 0xffffffffULL) return PG_EUNSUPPORTED;
            i64 tmin, tmax;
            stored_span(kc, &tmin, &tmax);
            const i128 delta = (i128)kc.base - (i128)pp.probe.bm_min;
            const i128 omin = (i128)tmin + delta, omax = (i128)tmax + delta;
            if (omax >= ((i128)1 << 32) || omin <= (i128)pp.probe.domain - ((i128)1 << 32)) return PG_EUNSUPPORTED;
            fp.kdelta = (unsigned)(u64)(i64)delta;
            fp.dom = (unsigned)pp.probe.domain;
        }
        fp.p_lo = 0; fp.p_span = 0xffffffffu;
        fp.st.ncol = 0;
        fp.rpw[0] = 0; fp.roff[0] = 0;
        int pi = -1;
        if (pp.npred == 1) {
            const TypedCol &pc = pp.pred[0].col;
            if (pp.pred[0].is_set || pc.width > 4 || pc.valid) return PG_EUNSUPPORTED;
            i64 tmin, tmax;
            stored_span(pc, &tmin, &tmax);
            i128 a = (i128)pp.pred[0].lo - pc.base, b = (i128)pp.pred[0].hi - pc.base;
            if (a < tmin) a = tmin;
            if (b > tmax) b = tmax;
            if (pp.pred[0].lo > pp.pred[0].hi || a > b) return PG_EUNSUPPORTED;      // empty range: the plain kernel
            fp.p_lo = (unsigned)(int32_t)(i64)a;
            fp.p_span = (unsigned)(u64)(i64)(b - a);
            pi = fp.st.ncol;
            fp.st.src[pi] = (const char *)pc.p + lo * pc.width;
            fp.st.pw[pi] = pc.width;
            fp.st.ncol++;
        }
        int ki = -1;
        if (pi >= 0 && fp.st.src[pi] == (const char *)kc.p + lo * kc.width) ki = pi;
        else {
            ki = fp.st.ncol;
            fp.st.src[ki] = (const char *)kc.p + lo * kc.width;
            fp.st.pw[ki] = kc.width;
            fp.st.ncol++;
        }
        const int qpt = 2;
        const int tile_rows = ST_CONS_WARPS * 128 * qpt;
        stage_layout(&fp.st, tile_rows);
        if (pi >= 0) { fp.rpw[0] = fp.st.pw[pi]; fp.roff[0] = fp.st.off[pi]; }
        fp.rpw[1] = fp.st.pw[ki]; fp.roff[1] = fp.st.off[ki];
        fp.st.nstage = getenv("PG_NSTAGE") ? atoi(getenv("PG_NSTAGE")) : 4;
        fp.row_begin = lo;
        fp.nloc = hi - lo;
        fp.hits = pp.hits;
        fp.hit_count = pp.hit_count;
        fp.counters = pp.counters;
        typedef void (*FK)(const FilterSParams);
        FK k;
        if (const char *m = getenv("PG_STAGED_FILTER_MASK")) {     // diagnosis: which width classes may use the staged filter
            const int cls = (fp.rpw[0] == 2 && fp.rpw[1] == 4) ? 1 : (fp.rpw[0] == 0 && fp.rpw[1] == 4) ? 2 : fp.rpw[0] == 0 ? 4 : 8;
            if (!(atoi(m) & cls)) return PG_EUNSUPPORTED;
        }
        if (fp.rpw[0] == 2 && fp.rpw[1] == 4) k = filter_hits_staged_kernel<2, 4, 2>;
        else if (fp.rpw[0] == 0 && fp.rpw[1] == 4) k = filter_hits_staged_kernel<0, 4, 2>;
        else if (fp.rpw[0] == 0) k = filter_hits_staged_kernel<0, -1, 2>;
        else k = filter_hits_staged_kernel<-1, -1, 2>;
        const size_t smem = (size_t)ST_HDR + (size_t)fp.st.nstage * fp.st.stage_bytes;
        PG_CUDA(cudaFuncSetAttribute((const void *)k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        int per_sm = 1;
        cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, (const void *)k, ST_THREADS, smem);
        const i64 ntiles = (fp.nloc + tile_rows - 1) / tile_rows;
        const int grid = (int)std::max<i64>(1, std::min<i64>(ntiles, (i64)ctx().prop.multiProcessorCount * std::max(per_sm, 1)));
        k<<<grid, ST_THREADS, smem, ctx().stream>>>(fp);
        PG_CUDA(cudaGetLastError());
        staged_filter_used = true;
        return PG_OK;
    }

    template <int SINK>
    int launch_sink(const PipeParams &pp)
    {
        hits_sink_kernel<SINK><<<ctx().prop.multiProcessorCount * 8, 256, 0, ctx().stream>>>(pp);
        PG_CUDA(cudaGetLastError());
        return PG_OK;
    }

    // one-kernel path (no exact bitmap on the probed table, NULLs, wide predicates ...)
    template <int SINK>
    int launch_pipe(const PipeParams &pp, const pg_table *t)
    {
        pipeline_kernel<SINK><<<grid_rows(pp.pipe_hi > 0 ? pp.pipe_hi - pp.pipe_lo : t->nrows), 256, 0, ctx().stream>>>(pp);
        PG_CUDA(cudaGetLastError());
        return PG_OK;
    }

    // size + (re)initialise the join table a stage builds
    int prepare_table(Stage &s, i64 nbuild, const Column &keycol)
    {
        cudaStream_t st = ctx().stream;
        u64 nb = next_pow2((u64)std::max<i64>((nbuild * 2 + HT_BUCKET - 1) / HT_BUCKET, 16));
        if (nbuild > s.capacity_rows || !s.d_slots.p) {
            PG_TRY(s.d_slots.alloc(nb * HT_BUCKET * sizeof(longlong2)));
            s.capacity_rows = (i64)(nb * HT_BUCKET / 2);
        } else {
            nb = next_pow2((u64)std::max<i64>((nbuild * 2 + HT_BUCKET - 1) / HT_BUCKET, 16));   // fits: capacity only grows
        }
        PG_CUDA(cudaMemsetAsync(s.d_slots.p, 0x80, nb * HT_BUCKET * sizeof(longlong2), st));
        s.jt.slots = s.d_slots.as<longlong2>();
        s.jt.bucket_mask = nb - 1;
        {   // ascending build key (>= 99% of adjacent rows increase): order-preserving buckets
            i128 dom = (i128)keycol.vmax - (i128)keycol.vmin + 1;
            int lg = 0;
            while (((u64)1 << lg) < nb) lg++;
            bool asc = keycol.stats_ok && keycol.adjacent_descents * 100 <= std::max<i64>(nbuild, 1) && dom > 0 && dom <= ((i128)1 << 34) && lg <= 29;
            if (getenv("PG_JOIN_ORDER_PRESERVING")) asc = asc && atoi(getenv("PG_JOIN_ORDER_PRESERVING")) != 0;
            if (s.ins_key_col2 >= 0) asc = false;            // composite keys: hashed buckets
            s.jt.order_preserving = asc ? 1 : 0;
            s.jt.log2buckets = lg;
            s.jt.domain = dom > 0 ? (u64)dom : 1;
        }
        s.jt.rank_prefix = nullptr;
        s.jt.rank_payload = nullptr;
        s.jt.rank_identity = 0;
        s.rank_index = false;
        // exact key-domain bitmap when the build column's value range is small enough
        s.jt.bitmap = nullptr;
        s.jt.bm_min = keycol.vmin;
        s.jt.bm_max = keycol.vmax;
        i128 domain = (i128)keycol.vmax - (i128)keycol.vmin + 1;
        if (keycol.stats_ok && domain > 0 && domain <= ((i128)1 << 32) && s.ins_key_col2 < 0) {
            size_t words = ((size_t)((domain + 31) / 32) + 7) / 8 * 8;      // whole 256-bit blocks (rank index)
            if (s.d_bitmap.bytes < words * 4 + 32) PG_TRY(s.d_bitmap.alloc(words * 4 + 32));   // + a 32-byte tail: counters of a split build
            PG_CUDA(cudaMemsetAsync(s.d_bitmap.p, 0, words * 4 + 32, st));
            s.jt.bitmap = s.d_bitmap.as<unsigned>();
            s.bitmap_words = words;
        }
        return PG_OK;
    }

    // Unique build keys inside a bitmap-able domain: no hash table.  The hit list of the stage's filter
    // pass becomes bitmap + per-block rank prefix + payload[rank] (three streaming-friendly passes without
    // CAS, probing or 64-byte buckets).  *done = 0 when the keys turn out not to be unique: the caller
    // falls back to the hash build over the same hit list.
    int build_rank_index(Stage &s, PipeParams &pp, const pg_table *t, i64 nh, pg_result *res, int *done)
    {
        cudaStream_t st = ctx().stream;
        *done = 0;
        const Column &keycol = t->cols[(size_t)s.ins_key_col];
        PG_TRY(prepare_table(s, 0, keycol));
        if (!s.jt.bitmap) return PG_OK;
        const int grid = ctx().prop.multiProcessorCount * 8;
        if (s.d_keys_tmp.bytes < (size_t)std::max<i64>(nh, 1) * 8) PG_TRY(s.d_keys_tmp.alloc((size_t)std::max<i64>(nh, 1) * 8));
        pp.ins_key = typed(t, s.ins_key_col);
        if (s.ins_key_col2 >= 0) pp.ins_key2 = typed(t, s.ins_key_col2);
        s.jt.dups = d_counters.as<unsigned long long>() + 2;
        pp.ins = s.jt;
        PG_CUDA(cudaMemsetAsync(d_counters.p, 0, 32, st));
        if (s.unique_key) {
            rank_mark_kernel<false><<<grid, 256, 0, st>>>(pp, s.d_keys_tmp.as<i64>());
            s.dup_keys = 0;
        } else {
            rank_mark_kernel<true><<<grid, 256, 0, st>>>(pp, s.d_keys_tmp.as<i64>());
            unsigned long long c2[4];
            PG_TRY(read_counters(c2));
            s.dup_keys = (i64)c2[2];
        }
        PG_CUDA(cudaGetLastError());
        res->stats.kernel_launches += 1;
        if (s.dup_keys != 0) return PG_OK;            // not unique: hash table (prepare_table resets the bitmap)
        if (!s.payload_needed) { *done = 1; return PG_OK; }      // the exact bitmap alone answers every probe
        const u64 nblocks = (s.jt.domain + 255) / 256;
        if (s.d_rank_prefix.bytes < nblocks * 4) PG_TRY(s.d_rank_prefix.alloc(nblocks * 4));
        if (s.d_rank_payload.bytes < (size_t)std::max<i64>(nh, 1) * 4) PG_TRY(s.d_rank_payload.alloc((size_t)std::max<i64>(nh, 1) * 4));
        unsigned *prefix = s.d_rank_prefix.as<unsigned>();
        rank_count_kernel<<<(int)std::min<u64>((nblocks + 255) / 256, (u64)grid), 256, 0, st>>>(s.jt.bitmap, nblocks, prefix);
        PG_CUDA(cudaGetLastError());
        size_t tmp_bytes = 0;
        PG_CUDA(cub::DeviceScan::ExclusiveSum(nullptr, tmp_bytes, prefix, prefix, (int)nblocks, st));
        if (s.d_scan_tmp.bytes < tmp_bytes) PG_TRY(s.d_scan_tmp.alloc(tmp_bytes));
        PG_CUDA(cub::DeviceScan::ExclusiveSum(s.d_scan_tmp.p, tmp_bytes, prefix, prefix, (int)nblocks, st));
        s.jt.rank_prefix = prefix;
        s.jt.rank_payload = s.d_rank_payload.as<unsigned>();
        pp.ins = s.jt;
        rank_fill_kernel<<<grid, 256, 0, st>>>(pp, s.d_keys_tmp.as<i64>(), s.d_rank_payload.as<unsigned>());
        PG_CUDA(cudaGetLastError());
        res->stats.kernel_launches += 3;
        s.rank_index = true;
        *done = 1;
        return PG_OK;
    }

    int run_build_stage(Stage &s, pg_result *res, int idx)
    {
        cudaStream_t st = ctx().stream;
        const pg_table *t = tab(s.src_slot);
        if (s.sub) {
            // the build side is a sub-aggregate: run it on the device, turn its group keys into the bitmap
            JoinAggPipeline *sp = static_cast<JoinAggPipeline *>(s.sub.get());
            const i64 launches = res->stats.kernel_launches;
            const pg_stats keep = res->stats;
            PG_TRY(sp->run(res));
            const i64 sub_launches = res->stats.kernel_launches;
            res->stats = keep;
            res->stats.kernel_launches = launches + sub_launches + 1;
            PG_TRY(prepare_table(s, 0, t->cols[(size_t)s.ins_key_col]));
            if (!s.jt.bitmap) PG_FAIL(PG_EUNSUPPORTED, "sub-aggregate build side: key domain too wide for a bitmap");
            const i64 nk = sp->dev_ngroups;
            if (nk > 0) {
                keys_bitmap_kernel<<<(int)std::max<i64>(std::min<i64>((nk + 255) / 256, (i64)ctx().prop.multiProcessorCount * 8), 1), 256, 0, st>>>(
                    sp->d_out_klo.as<i64>(), nk, s.jt);
                PG_CUDA(cudaGetLastError());
            }
            s.no_table = true;
            s.dup_keys = 0;
            s.built_rows = nk;
            if (idx < 2) { res->stats.aux[2 + 2 * idx] = sp->tab(sp->src_slot)->nrows; res->stats.aux[3 + 2 * idx] = nk; }
            return PG_OK;
        }
        PipeParams pp{};
        pp.nrows = t->nrows;
        PG_TRY(fill_preds(pp, s.ranges, s.src_slot));
        PG_TRY(fill_extras(pp, s.extras, s.src_slot));
        pp.has_probe = s.has_probe ? 1 : 0;
        if (s.has_probe) {
            pp.probe_key = typed(t, s.probe_key_col);
            pp.probe = stages[(size_t)s.probe_stage]->jt;
            pp.probe_bitmap_only = stages[(size_t)s.probe_stage]->bitmap_only() ? 1 : 0;
            pp.probe_mode = s.probe_mode;
        } else {
            pp.probe_key = typed(t, s.ins_key_col);      // the filter pass streams the key column itself
        }
        pp.counters = d_counters.as<unsigned long long>();
        s.no_table = false;
        if ((s.existence_only || (s.unique_key && !s.has_probe)) && !s.payload_needed && !getenv("PG_JOIN_NO_BITMAP_BUILD")) {
            // (a stage with a probe of its own, SEMI/ANTI-consumed, also lands here: pipeline_kernel probes + applies extras)
            // unique keys, nothing but existence is needed: one pass that sets key bits, no hash table at all
            PG_TRY(prepare_table(s, 0, t->cols[(size_t)s.ins_key_col]));
            if (s.jt.bitmap) {
                pp.ins_key = typed(t, s.ins_key_col);
        if (s.ins_key_col2 >= 0) pp.ins_key2 = typed(t, s.ins_key_col2);
                pp.ins = s.jt;
                PG_CUDA(cudaMemsetAsync(d_counters.p, 0, 32, st));
                // A REPLICATED build side is the same on every rank: instead of W identical scans, every rank marks the keys
                // of its 1/W of the rows and the partial bitmaps are all-gathered and OR-ed (2 MB for SF100's customer).
                const int W = ctx().world;
                // Worth it only when the scan is expensive: measured at 8 GPUs on SF100's 15 M customers, the vectorised
                // bitmap_build_kernel scans the whole table in 0.075 ms per rank while 1/8 of it + a 2 MB all-gather + the
                // OR-merge takes 0.119 ms -- so plain range / code-set builds split only from 64 M rows per rank up, builds
                // with a string predicate evaluated per row (Q9's p_name LIKE: 0.65 ms for 20 M parts) from 64 K rows up.
                const i64 split_min = getenv("PG_SPLIT_MIN_ROWS") ? atoll(getenv("PG_SPLIT_MIN_ROWS")) : (pp.nlike > 0 ? (i64)65536 : (i64)64 << 20);
                const bool split = W > 1 && t->dist == PG_DIST_REPLICATED && !s.has_probe && s.extras.empty() && t->nrows >= (i64)W * split_min &&
                                   !getenv("PG_NO_SPLIT_BUILD");
                if (split) {
                    pp.pipe_lo = (t->nrows * ctx().rank / W) & ~(i64)3;
                    pp.pipe_hi = ctx().rank + 1 == W ? t->nrows : ((t->nrows * (ctx().rank + 1) / W) & ~(i64)3);
                    if (pp.pipe_hi <= 0) pp.pipe_hi = pp.pipe_lo = 0;       // (an empty slice: pipe_hi == 0 would mean "every row")
                }
                bool any_valid = pp.ins_key.valid != nullptr;
                for (int k = 0; k < pp.npred; k++) any_valid = any_valid || pp.pred[k].col.valid != nullptr;
                if (!s.has_probe && pp.nextra == 0 && pp.nlike == 0 && pp.npred <= 1 && !any_valid && s.ins_key_col2 < 0 && !getenv("PG_JOIN_GENERIC")) {
                    const i64 lo = split ? pp.pipe_lo : 0, hi = split ? pp.pipe_hi : t->nrows;
                    const int grid = (int)std::max<i64>(std::min<i64>((hi - lo + 1023) / 1024, (i64)ctx().prop.multiProcessorCount * 8), 1);
                    if (hi > lo) {
                        if (pp.npred == 1) bitmap_build_kernel<true><<<grid, 256, 0, st>>>(pp, lo, hi);
                        else bitmap_build_kernel<false><<<grid, 256, 0, st>>>(pp, lo, hi);
                        PG_CUDA(cudaGetLastError());
                    }
                } else if (!split || pp.pipe_hi > pp.pipe_lo) {
                    PG_TRY(launch_pipe<SINK_BITMAP>(pp, t));
                }
                if (split) {
                    const size_t part = s.bitmap_words * 4 + 32;
                    if (s.d_bm_all.bytes < part * (size_t)W) PG_TRY(s.d_bm_all.alloc(part * (size_t)W));
                    PG_CUDA(cudaMemcpyAsync((char *)s.d_bitmap.p + s.bitmap_words * 4, d_counters.p, 32, cudaMemcpyDeviceToDevice, st));
                    PG_TRY(comm_allgather(s.d_bitmap.p, s.d_bm_all.p, part, st));
                    bitmap_or_kernel<<<(int)std::min<u64>((s.bitmap_words + 255) / 256, (u64)ctx().prop.multiProcessorCount * 4), 256, 0, st>>>(
                        s.d_bm_all.as<unsigned>(), W, (u64)s.bitmap_words, s.jt.bitmap, d_counters.as<unsigned long long>());
                    PG_CUDA(cudaGetLastError());
                    res->stats.kernel_launches += 1;
                }
                s.no_table = true;
                s.dup_keys = 0;
                res->stats.kernel_launches += 1;
                const bool need_rows = !star && &s == stages.back().get();      // sizes the group table of the final probe
                if (need_rows) {
                    unsigned long long c0[4];
                    PG_TRY(read_counters(c0));
                    s.built_rows = (i64)c0[1];
                    if (idx < 2) { res->stats.aux[2 + 2 * idx] = (i64)c0[0]; res->stats.aux[3 + 2 * idx] = (i64)c0[1]; }
                } else if (idx < 2) {
                    // no host round trip for a statistic: park the two counters, the next read-back carries them
                    PG_CUDA(cudaMemcpyAsync(d_counters.as<unsigned long long>() + 4 + 2 * idx, d_counters.p, 16, cudaMemcpyDeviceToDevice, st));
                    deferred_stats |= 1u << idx;
                    s.built_rows = t->nrows;                                    // upper bound (only statistics read it)
                }
                return PG_OK;
            }
        }
        if (!s.has_probe && s.unique_key && s.payload_needed && pp.npred == 0 && pp.nlike == 0 && pp.nextra == 0 && s.ins_key_col2 < 0 &&
            !getenv("PG_JOIN_NO_RANK_INDEX")) {
            // Every row of a strictly ascending key column is built: the rank of a key IS its row id, so the index is the
            // bitmap plus its block prefix -- no hit list, no payload array (Q9: the 150 M unfiltered orders).
            PG_TRY(prepare_table(s, 0, t->cols[(size_t)s.ins_key_col]));
            if (s.jt.bitmap) {
                pp.ins_key = typed(t, s.ins_key_col);
                pp.ins = s.jt;
                PG_CUDA(cudaMemsetAsync(d_counters.p, 0, 32, st));
                PG_TRY(launch_pipe<SINK_BITMAP>(pp, t));
                const u64 nblocks = (s.jt.domain + 255) / 256;
                if (s.d_rank_prefix.bytes < nblocks * 4) PG_TRY(s.d_rank_prefix.alloc(nblocks * 4));
                unsigned *prefix = s.d_rank_prefix.as<unsigned>();
                const int grid = ctx().prop.multiProcessorCount * 8;
                rank_count_kernel<<<(int)std::min<u64>((nblocks + 255) / 256, (u64)grid), 256, 0, st>>>(s.jt.bitmap, nblocks, prefix);
                PG_CUDA(cudaGetLastError());
                size_t tmp_bytes = 0;
                PG_CUDA(cub::DeviceScan::ExclusiveSum(nullptr, tmp_bytes, prefix, prefix, (int)nblocks, st));
                if (s.d_scan_tmp.bytes < tmp_bytes) PG_TRY(s.d_scan_tmp.alloc(tmp_bytes));
                PG_CUDA(cub::DeviceScan::ExclusiveSum(s.d_scan_tmp.p, tmp_bytes, prefix, prefix, (int)nblocks, st));
                s.jt.rank_prefix = prefix;
                s.jt.rank_identity = 1;
                s.rank_index = true;
                s.dup_keys = 0;
                s.built_rows = t->nrows;
                res->stats.kernel_launches += 3;
                if (idx < 2) { res->stats.aux[2 + 2 * idx] = t->nrows; res->stats.aux[3 + 2 * idx] = t->nrows; }
                return PG_OK;
            }
        }
        if (two_phase_ok(pp, t, true) && (s.has_probe || (s.unique_key && s.payload_needed))) {
            // phase 1 screens the whole source once: the hit list doubles as the sizing pass
            PG_CUDA(cudaMemsetAsync(d_counters.p, 0, 32, st));
            PG_TRY(launch_filter(pp, 0, t->nrows));
            const bool exact = !pp.has_probe || pp.probe_bitmap_only || pp.probe_mode != 0;      // at most one sink row per hit
            if (!exact) PG_TRY(launch_sink<SINK_COUNT>(pp));
            unsigned long long cnt[4], nh = 0;
            PG_CUDA(cudaMemcpyAsync(&nh, d_hit_count.p, 8, cudaMemcpyDeviceToHost, st));
            PG_TRY(read_counters(cnt));
            s.built_rows = exact ? (i64)nh : (i64)cnt[1];
            if (exact && !getenv("PG_JOIN_NO_RANK_INDEX")) {
                int done = 0;
                PG_TRY(build_rank_index(s, pp, t, (i64)nh, res, &done));
                if (done) {
                    res->stats.kernel_launches += 1;
                    if (idx < 2) { res->stats.aux[2 + 2 * idx] = (i64)cnt[0]; res->stats.aux[3 + 2 * idx] = s.built_rows; }
                    return PG_OK;
                }
            }
            PG_TRY(prepare_table(s, s.built_rows, t->cols[(size_t)s.ins_key_col]));
            pp.ins_key = typed(t, s.ins_key_col);
        if (s.ins_key_col2 >= 0) pp.ins_key2 = typed(t, s.ins_key_col2);
            s.jt.dups = d_counters.as<unsigned long long>() + 2;
            pp.ins = s.jt;
            PG_CUDA(cudaMemsetAsync(d_counters.p, 0, 32, st));
            PG_TRY(launch_sink<SINK_INSERT>(pp));
            s.dup_keys = 1;
            if (!s.payload_needed && s.jt.bitmap) {
                unsigned long long c2[4];
                PG_TRY(read_counters(c2));
                s.dup_keys = (i64)c2[2];
            }
            res->stats.kernel_launches += exact ? 2 : 3;
            if (idx < 2) { res->stats.aux[2 + 2 * idx] = (i64)cnt[0]; res->stats.aux[3 + 2 * idx] = s.built_rows; }
            return PG_OK;
        }
        // sizing pass: how many rows reach the sink
        PG_CUDA(cudaMemsetAsync(d_counters.p, 0, 32, st));
        PG_TRY(launch_pipe<SINK_COUNT>(pp, t));
        unsigned long long cnt[4];
        PG_TRY(read_counters(cnt));
        s.built_rows = (i64)cnt[1];
        PG_TRY(prepare_table(s, s.built_rows, t->cols[(size_t)s.ins_key_col]));
        pp.ins_key = typed(t, s.ins_key_col);
        if (s.ins_key_col2 >= 0) pp.ins_key2 = typed(t, s.ins_key_col2);
        s.jt.dups = d_counters.as<unsigned long long>() + 2;
        pp.ins = s.jt;
        PG_CUDA(cudaMemsetAsync(d_counters.p, 0, 32, st));
        PG_TRY(launch_pipe<SINK_INSERT>(pp, t));
        s.dup_keys = 1;                          // unknown: assume duplicates...
        if (!s.payload_needed && s.jt.bitmap) {  // ...unless it decides whether the bitmap alone can answer probes
            unsigned long long c2[4];
            PG_TRY(read_counters(c2));
            s.dup_keys = (i64)c2[2];
        }
        res->stats.kernel_launches += 2;
        if (idx < 2) { res->stats.aux[2 + 2 * idx] = (i64)cnt[0]; res->stats.aux[3 + 2 * idx] = (i64)cnt[1]; }
        return PG_OK;
    }

    int ensure_group_table(u64 cap)
    {
        if (cap <= gt_cap) return PG_OK;
        PG_TRY(d_gt.alloc(cap * 8 * (size_t)gt_slot_words(gs.nacc)));
        gt_cap = cap;
        return PG_OK;
    }

    // ---- all-to-all hash-partitioned exchange of the local group lists (SURVEY.md 8e) ----
    // rows are packed AoS: [klo, khi, plane 0 .. plane nacc] (W = 3 + nacc words); destination rank =
    // mix64(klo ^ rot(khi)) % world.  Counts travel with an all-gather, rows with grouped
    // ncclSend/ncclRecv over NVLink, then every rank merges what it owns into its (reset) table.
    DevBuf d_sx_send, d_sx_recv, d_sx_cnt, d_sx_cursor, d_sx_allcnt;
    size_t sx_send_rows = 0, sx_recv_rows = 0;

    int shuffle_groups(i64 *ngroups, PipeParams &pp, pg_result *res)
    {
        Context &c = ctx();
        cudaStream_t st = c.stream;
        const int W = c.world, planes = gs.nacc + 1, RW = 2 + planes;
        i64 n = *ngroups;
        if (!d_sx_cnt.p) {
            PG_TRY(d_sx_cnt.alloc(8 * (size_t)W));
            PG_TRY(d_sx_cursor.alloc(8 * (size_t)W));
            PG_TRY(d_sx_allcnt.alloc(8 * (size_t)W * (size_t)W));
        }
        if ((size_t)n > sx_send_rows) { PG_TRY(d_sx_send.alloc((size_t)std::max<i64>(n, 1) * RW * 8)); sx_send_rows = (size_t)n; }
        int grid = (int)std::max<i64>(std::min<i64>((n + 255) / 256, (i64)c.prop.multiProcessorCount * 4), 1);
        // 1. count rows per destination
        PG_CUDA(cudaMemsetAsync(d_sx_cnt.p, 0, 8 * (size_t)W, st));
        shuffle_count_kernel<<<grid, 256, 0, st>>>(d_out_klo.as<i64>(), d_out_khi.as<i64>(), n, W, d_sx_cnt.as<unsigned long long>());
        PG_CUDA(cudaGetLastError());
        // 2. everybody learns the whole count matrix
        PG_TRY(comm_allgather(d_sx_cnt.p, d_sx_allcnt.p, 8 * (size_t)W, st));
        std::vector<i64> all((size_t)W * (size_t)W);
        PG_CUDA(cudaMemcpyAsync(all.data(), d_sx_allcnt.p, 8 * (size_t)W * (size_t)W, cudaMemcpyDeviceToHost, st));
        PG_CUDA(cudaStreamSynchronize(st));
        std::vector<i64> send_cnt((size_t)W), send_off((size_t)W), recv_cnt((size_t)W), recv_off((size_t)W);
        i64 so = 0, ro = 0;
        for (int r = 0; r < W; r++) {
            send_cnt[(size_t)r] = all[(size_t)c.rank * W + r]; send_off[(size_t)r] = so; so += send_cnt[(size_t)r];
            recv_cnt[(size_t)r] = all[(size_t)r * W + c.rank]; recv_off[(size_t)r] = ro; ro += recv_cnt[(size_t)r];
        }
        if ((size_t)ro > sx_recv_rows) { PG_TRY(d_sx_recv.alloc((size_t)std::max<i64>(ro, 1) * RW * 8)); sx_recv_rows = (size_t)ro; }
        // 3. scatter rows into destination order
        PG_CUDA(cudaMemcpyAsync(d_sx_cursor.p, send_off.data(), 8 * (size_t)W, cudaMemcpyHostToDevice, st));
        shuffle_scatter_kernel<<<grid, 256, 0, st>>>(d_out_klo.as<i64>(), d_out_khi.as<i64>(), d_out_acc.as<i64>(), out_cap, n, planes, W,
                                                     d_sx_cursor.as<unsigned long long>(), d_sx_send.as<i64>());
        PG_CUDA(cudaGetLastError());
        // 4. the exchange
        PG_TRY(comm_alltoallv(d_sx_send.p, send_cnt.data(), send_off.data(), d_sx_recv.p, recv_cnt.data(), recv_off.data(), (size_t)RW * 8, st));
        // 5. merge what this rank owns
        PG_CUDA(cudaMemsetAsync(d_gt.p, 0x80, gt_cap * 8 * (size_t)gt_slot_words(gs.nacc), st));
        PG_CUDA(cudaMemsetAsync(d_overflow.p, 0, 4, st));
        int g2 = (int)std::max<i64>(std::min<i64>((ro + 255) / 256, (i64)c.prop.multiProcessorCount * 4), 1);
        shuffle_merge_kernel<<<g2, 256, 0, st>>>(pp.gt, d_sx_recv.as<i64>(), ro, planes);
        PG_CUDA(cudaGetLastError());
        int ovf = 0;
        PG_CUDA(cudaMemcpyAsync(&ovf, d_overflow.p, 4, cudaMemcpyDeviceToHost, st));
        PG_CUDA(cudaStreamSynchronize(st));
        if (ovf) PG_FAIL(PG_ENOMEM, "group table overflow while merging shuffled groups");
        // 6. compact again (HAVING applies to the merged totals)
        if (ro > out_cap) {
            PG_TRY(d_out_klo.alloc((size_t)ro * 8));
            PG_TRY(d_out_khi.alloc((size_t)ro * 8));
            PG_TRY(d_out_acc.alloc((size_t)ro * 8 * (size_t)planes));
            out_cap = ro;
        }
        PG_CUDA(cudaMemsetAsync(d_counters.p, 0, 32, st));
        gt_compact_kernel<<<(int)std::min<u64>((gt_cap + 255) / 256, (u64)c.prop.multiProcessorCount * 8), 256, 0, st>>>(
            pp.gt, d_out_klo.as<i64>(), d_out_khi.as<i64>(), d_out_acc.as<i64>(), out_cap, d_counters.as<unsigned long long>(),
            hav_plane, hav_lo, hav_hi);
        PG_CUDA(cudaGetLastError());
        unsigned long long ng2[4];
        PG_TRY(read_counters(ng2));
        *ngroups = (i64)ng2[0];
        res->stats.kernel_launches += 4;
        res->stats.aux[7] = so;        // rows this rank sent
        return PG_OK;
    }

    // ---- all-to-all hash-partitioned exchange of JOIN ROWS (exchange.cuh; SURVEY.md 8e, BASELINE config 5) ----
    // `d_rec` holds *d_n records of RW words with a destination byte each (X_DROP = not sent) and d_sx_cnt their
    // per-destination counts, all made by one kernel.  Counts travel with an all-gather, records are moved into
    // destination order and exchanged with grouped ncclSend/ncclRecv over NVLink.  Collective: every rank calls it.
    int x_counts_reset()
    {
        const int W = ctx().world;
        if (W > X_MAXWORLD) PG_FAIL(PG_EUNSUPPORTED, "row exchange: more than %d ranks", X_MAXWORLD);
        if (!d_sx_cnt.p) {
            PG_TRY(d_sx_cnt.alloc(8 * (size_t)W));
            PG_TRY(d_sx_cursor.alloc(8 * (size_t)W));
            PG_TRY(d_sx_allcnt.alloc(8 * (size_t)W * (size_t)W));
        }
        PG_CUDA(cudaMemsetAsync(d_sx_cnt.p, 0, 8 * (size_t)W, ctx().stream));
        return PG_OK;
    }
    int exchange_rows(const i64 *d_rec, const unsigned char *d_dest, const unsigned long long *d_n, i64 n_host, int RW, DevBuf &send, DevBuf &recv,
                      EventPair &ev, i64 *recv_rows)
    {
        Context &c = ctx();
        cudaStream_t st = c.stream;
        const int W = c.world;
        PG_TRY(comm_allgather(d_sx_cnt.p, d_sx_allcnt.p, 8 * (size_t)W, st));
        std::vector<i64> all((size_t)W * (size_t)W);
        PG_CUDA(cudaMemcpyAsync(all.data(), d_sx_allcnt.p, 8 * (size_t)W * (size_t)W, cudaMemcpyDeviceToHost, st));
        PG_CUDA(cudaStreamSynchronize(st));
        std::vector<i64> send_cnt((size_t)W), send_off((size_t)W), recv_cnt((size_t)W), recv_off((size_t)W);
        i64 so = 0, ro = 0;
        for (int r = 0; r < W; r++) {
            send_cnt[(size_t)r] = all[(size_t)c.rank * W + r]; send_off[(size_t)r] = so; so += send_cnt[(size_t)r];
            recv_cnt[(size_t)r] = all[(size_t)r * W + c.rank]; recv_off[(size_t)r] = ro; ro += recv_cnt[(size_t)r];
        }
        if (send.bytes < (size_t)std::max<i64>(so, 1) * RW * 8) PG_TRY(send.alloc((size_t)std::max<i64>(so, 1) * RW * 8));
        if (recv.bytes < (size_t)std::max<i64>(ro, 1) * RW * 8) PG_TRY(recv.alloc((size_t)std::max<i64>(ro, 1) * RW * 8));
        PG_CUDA(cudaMemcpyAsync(d_sx_cursor.p, send_off.data(), 8 * (size_t)W, cudaMemcpyHostToDevice, st));
        if (n_host > 0) {
            x_scatter_kernel<<<grid_rows(n_host), 256, 0, st>>>(d_rec, d_dest, d_n, RW, d_sx_cursor.as<unsigned long long>(), send.as<i64>());
            PG_CUDA(cudaGetLastError());
        }
        PG_TRY(ev.init());
        PG_CUDA(cudaEventRecord(ev.a, st));
        PG_TRY(comm_alltoallv(send.p, send_cnt.data(), send_off.data(), recv.p, recv_cnt.data(), recv_off.data(), (size_t)RW * 8, st));
        PG_CUDA(cudaEventRecord(ev.b, st));
        x_sent_rows += so - send_cnt[(size_t)c.rank];
        x_sent_bytes += (so - send_cnt[(size_t)c.rank]) * RW * 8;
        *recv_rows = ro;
        return PG_OK;
    }

    // Build side of the exchange lookup: the local shard's rows that pass its filters travel to the owners of their
    // keys; what arrives is inserted into a bucketized table whose payload indexes the receive buffer.
    int run_exchange_build(Stage &s, pg_result *res)
    {
        cudaStream_t st = ctx().stream;
        const pg_table *t = tab(s.src_slot);
        PipeParams pp{};
        pp.nrows = t->nrows;
        PG_TRY(fill_preds(pp, s.ranges, s.src_slot));
        pp.has_probe = s.has_probe ? 1 : 0;
        if (s.has_probe) {
            pp.probe_key = typed(t, s.probe_key_col);
            pp.probe = stages[(size_t)s.probe_stage]->jt;
            pp.probe_bitmap_only = 1;
            pp.probe_mode = s.probe_mode;
        } else {
            pp.probe_key = typed(t, s.ins_key_col);
        }
        pp.ins_key = typed(t, s.ins_key_col);
        pp.counters = d_counters.as<unsigned long long>();
        if (!two_phase_ok(pp, t, true)) PG_FAIL(PG_EUNSUPPORTED, "row exchange: the build-side scan does not fit the filter pass");
        PG_CUDA(cudaMemsetAsync(d_counters.p, 0, 32, st));
        PG_TRY(launch_filter(pp, 0, t->nrows));
        unsigned long long nh = 0;
        PG_CUDA(cudaMemcpyAsync(&nh, d_hit_count.p, 8, cudaMemcpyDeviceToHost, st));
        PG_CUDA(cudaStreamSynchronize(st));
        const int RW = 1 + (int)xcols.size();
        if (d_xb_rec.bytes < (size_t)std::max<u64>(nh, 1) * RW * 8) PG_TRY(d_xb_rec.alloc((size_t)std::max<u64>(nh, 1) * RW * 8));
        if (d_xb_dest.bytes < (size_t)std::max<u64>(nh, 1)) PG_TRY(d_xb_dest.alloc((size_t)std::max<u64>(nh, 1)));
        PG_TRY(x_counts_reset());
        XBuildParams bp{};
        bp.hits = d_hits.as<unsigned>();
        bp.hit_count = d_hit_count.as<unsigned long long>();
        bp.nkey = s.ins_key_col2 >= 0 ? 2 : 1;
        bp.key[0] = typed(t, s.ins_key_col);
        if (s.ins_key_col2 >= 0) bp.key[1] = typed(t, s.ins_key_col2);
        bp.nx = (int)xcols.size();
        for (size_t i = 0; i < xcols.size(); i++) bp.x[i] = typed(t, xcols[i]);
        bp.world = ctx().world;
        bp.rec = d_xb_rec.as<i64>();
        bp.dest = d_xb_dest.as<unsigned char>();
        bp.cnt = d_sx_cnt.as<unsigned long long>();
        if (nh > 0) {
            x_build_rows_kernel<<<grid_rows((i64)nh), 256, 0, st>>>(bp);
            PG_CUDA(cudaGetLastError());
        }
        PG_TRY(exchange_rows(d_xb_rec.as<i64>(), d_xb_dest.as<unsigned char>(), d_hit_count.as<unsigned long long>(), (i64)nh, RW, d_xb_send, d_xb_recv,
                             ev_xb, &xb_recv_rows));
        // owner side: hashed buckets, no bitmap (the key domain is the whole table's, not this shard's)
        u64 nb = next_pow2((u64)std::max<i64>((xb_recv_rows * 2 + HT_BUCKET - 1) / HT_BUCKET, 16));
        if (s.d_slots.bytes < nb * HT_BUCKET * sizeof(longlong2)) PG_TRY(s.d_slots.alloc(nb * HT_BUCKET * sizeof(longlong2)));
        PG_CUDA(cudaMemsetAsync(s.d_slots.p, 0x80, nb * HT_BUCKET * sizeof(longlong2), st));
        s.jt = JoinTable{};
        s.jt.slots = s.d_slots.as<longlong2>();
        s.jt.bucket_mask = nb - 1;
        s.jt.domain = 1;
        if (xb_recv_rows > 0) {
            x_insert_kernel<<<grid_rows(xb_recv_rows), 256, 0, st>>>(s.jt, d_xb_recv.as<i64>(), xb_recv_rows, RW);
            PG_CUDA(cudaGetLastError());
        }
        s.built_rows = xb_recv_rows;
        s.dup_keys = 1;
        s.no_table = false;
        res->stats.kernel_launches += 4;
        return PG_OK;
    }

    // Probe side: every other join of the star, the group id and the local factors are evaluated where the fact row
    // lives (star_pre_kernel); the records travel to the key's owner, which finishes the join (star_post_kernel).
    int run_star_exchange(const StarParams &sp, pg_result *res, Trace &tr)
    {
        Context &c = ctx();
        cudaStream_t st = c.stream;
        unsigned long long nh = 0;
        PG_CUDA(cudaMemcpyAsync(&nh, d_hit_count.p, 8, cudaMemcpyDeviceToHost, st));
        PG_CUDA(cudaStreamSynchronize(st));
        const int RW = 2 + sp.nterm;
        if (d_xp_rec.bytes < (size_t)std::max<u64>(nh, 1) * RW * 8) PG_TRY(d_xp_rec.alloc((size_t)std::max<u64>(nh, 1) * RW * 8));
        if (d_xp_dest.bytes < (size_t)std::max<u64>(nh, 1)) PG_TRY(d_xp_dest.alloc((size_t)std::max<u64>(nh, 1)));
        PG_TRY(x_counts_reset());
        XPreParams xp{};
        xp.xl = xl;
        xp.world = c.world;
        for (int t = 0; t < STAR_MAXTERM; t++) xp.term_x[t] = x_term_mask[t];
        xp.rec = d_xp_rec.as<i64>();
        xp.dest = d_xp_dest.as<unsigned char>();
        xp.cnt = d_sx_cnt.as<unsigned long long>();
        if (nh > 0) {
            star_pre_kernel<<<c.prop.multiProcessorCount * 8, 256, 0, st>>>(sp, xp);
            PG_CUDA(cudaGetLastError());
        }
        tr.mark("star pre-join (local lookups)");
        i64 np = 0;
        PG_TRY(exchange_rows(d_xp_rec.as<i64>(), d_xp_dest.as<unsigned char>(), d_hit_count.as<unsigned long long>(), (i64)nh, RW, d_xp_send, d_xp_recv,
                             ev_xp, &np));
        tr.mark("star row exchange");
        const Stage &X = *stages[(size_t)lookups[(size_t)xl].stage];
        XPostParams pp{};
        pp.prow = d_xp_recv.as<i64>();
        pp.np = np;
        pp.brow = d_xb_recv.as<i64>();
        pp.nx = (int)xcols.size();
        pp.jt = X.jt;
        pp.nterm = sp.nterm;
        for (int t = 0; t < sp.nterm; t++) {
            int k = 0;
            for (int f = 0; f < sp.term[t].nfac; f++) {
                if (!((x_term_mask[t] >> f) & 1)) continue;
                pp.xcol[t][k] = x_fac_col[t][f];
                pp.xfc[t][k] = sp.term[t].fc[f];
                pp.xfs[t][k] = sp.term[t].fs[f];
                k++;
            }
            pp.nxf[t] = k;
        }
        pp.ngroups = sp.ngroups;
        pp.gsum = sp.gsum;
        pp.gsum_hi = sp.gsum_hi;
        pp.gcnt = sp.gcnt;
        pp.counters = sp.counters;
        if ((size_t)star_ngroups * 16 > 48 * 1024)
            PG_CUDA(cudaFuncSetAttribute(star_post_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, star_ngroups * 16));
        if (np > 0) {
            star_post_kernel<<<c.prop.multiProcessorCount * 8, 256, (size_t)star_ngroups * 16, st>>>(pp);
            PG_CUDA(cudaGetLastError());
        }
        res->stats.kernel_launches += 3;
        return PG_OK;
    }

    // Sink of a star join grouped by the rows of one lookup: per-row sums in d_dense, compacted into the group list that
    // finish_groups() takes over (top-k, dependent-key gather, result columns).  A count-only aggregate has no terms: its
    // sum plane holds zeros that no output reads.
    int run_star_rows(const StarParams &sp, pg_result *res, Trace &tr)
    {
        Context &c = ctx();
        cudaStream_t st = c.stream;
        const u64 D = (u64)std::max<i64>(tab(origin_slot[(size_t)star_anchor])->nrows, 1);
        if (d_dense.bytes < D * 12 + 64) PG_TRY(d_dense.alloc(D * 12 + 64));
        unsigned long long *dsum = d_dense.as<unsigned long long>();
        unsigned *dcnt = (unsigned *)(dsum + D);
        PG_CUDA(cudaMemsetAsync(d_dense.p, 0, D * 12, st));
        hits_star_rows_kernel<<<c.prop.multiProcessorCount * 8, 256, 0, st>>>(sp, star_anchor, dsum, dcnt);
        PG_CUDA(cudaGetLastError());
        PG_CUDA(cudaEventRecord(ev_main.b, st));
        res->stats.kernel_launches += 2;
        unsigned long long cnt[4];
        PG_TRY(read_counters(cnt));
        tr.mark("star sink (per-row sums)");
        if (cnt[2] != 0) PG_FAIL(PG_EUNSUPPORTED, "star join: a lookup matched more than one build row (duplicate build keys)");
        const i64 want = (i64)std::min<u64>(D, std::max<u64>(cnt[1], 1));
        if (want > out_cap) {
            PG_TRY(d_out_klo.alloc((size_t)want * 8));
            PG_TRY(d_out_khi.alloc((size_t)want * 8));
            PG_TRY(d_out_acc.alloc((size_t)want * 8 * (size_t)(gs.nacc + 1 + (int)fd.size())));    // dependent key columns ride as extra planes
            out_cap = want;
        }
        PG_CUDA(cudaMemsetAsync(d_counters.p, 0, 32, st));
        dense_compact_kernel<<<(int)std::min<u64>((D + 255) / 256, (u64)c.prop.multiProcessorCount * 8), 256, 0, st>>>(
            dsum, dcnt, D, 0, d_out_klo.as<i64>(), d_out_khi.as<i64>(), d_out_acc.as<i64>(), out_cap, d_counters.as<unsigned long long>(), -1, 0, 0);
        PG_CUDA(cudaGetLastError());
        res->stats.kernel_launches += 1;
        unsigned long long ng[4];
        PG_TRY(read_counters(ng));
        return finish_groups((i64)ng[0], cnt, res, tr);
    }

    // fact-table pipeline of a star join: existence filter pass, then hits_star_kernel (lookups + dense group sums)
    int run_star(pg_result *res, Trace &tr)
    {
        Context &c = ctx();
        cudaStream_t st = c.stream;
        const pg_table *t = tab(src_slot);
        PipeParams pp{};
        pp.nrows = t->nrows;
        PG_TRY(fill_preds(pp, ranges, src_slot));
        Stage &M = top_stage_ref();
        pp.has_probe = 1;
        pp.probe_key = typed(t, probe_key_col);
        pp.probe = M.jt;
        pp.probe_bitmap_only = 1;
        pp.probe_mode = 0;
        pp.counters = d_counters.as<unsigned long long>();
        if (!two_phase_ok(pp, t, false) || t->nrows > HIT_CHUNK) PG_FAIL(PG_EUNSUPPORTED, "star join: the fact-table scan does not fit the filter pass (one 32-bit range predicate, bitmap-able main join)");
        PG_CUDA(cudaMemsetAsync(d_counters.p, 0, 32, st));
        PG_CUDA(cudaEventRecord(ev_main.a, st));
        PG_TRY(launch_filter(pp, 0, t->nrows));
        tr.mark("star filter");
        StarParams sp{};
        sp.hits = d_hits.as<unsigned>();
        sp.hit_count = d_hit_count.as<unsigned long long>();
        auto href = [&](const HRef &h) { ValRef v; v.col = typed(tab(origin_slot[(size_t)h.origin]), h.col); v.from_build = h.origin; return v; };
        sp.nlookup = (int)lookups.size();
        for (size_t l = 0; l < lookups.size(); l++) {
            const Stage &b = *stages[(size_t)lookups[l].stage];
            sp.lk[l].nkey = lookups[l].nkey;
            for (int k = 0; k < lookups[l].nkey; k++) sp.lk[l].key[k] = href(lookups[l].key[k]);
            sp.lk[l].jt = b.jt;
            sp.lk[l].existence = b.bitmap_only() ? 1 : 0;
            if (!sp.lk[l].existence && b.no_table) PG_FAIL(PG_ECUDA, "internal: star lookup needs a payload but its build side kept none");
        }
        sp.nparts = (int)sparts.size();
        sp.ngroups = star_ngroups;
        for (size_t k = 0; k < sparts.size(); k++) { sp.part[k].v = href(sparts[k].v); sp.part[k].fn = sparts[k].fn; sp.part[k].lo = sparts[k].lo; sp.part[k].n = sparts[k].n; }
        sp.nterm = (int)sterms.size();
        for (size_t i = 0; i < sterms.size(); i++) {
            sp.term[i].nfac = sterms[i].nfac;
            sp.term[i].mul = sterms[i].mul;
            for (int f = 0; f < sterms[i].nfac; f++) { sp.term[i].fac[f] = href(sterms[i].fac[f]); sp.term[i].fc[f] = sterms[i].fc[f]; sp.term[i].fs[f] = sterms[i].fs[f]; }
        }
        sp.counters = d_counters.as<unsigned long long>();
        if (fd_mode) return run_star_rows(sp, res, tr);
        const size_t gbytes = (size_t)star_ngroups * 24;      // sum low word, sum high word, row count
        const int W = (t->dist != PG_DIST_REPLICATED && c.world > 1) ? c.world : 1;
        if (!d_star.p) { PG_TRY(d_star.alloc(gbytes)); PG_TRY(d_star_all.alloc(gbytes * (size_t)c.world)); PG_TRY(h_star.alloc(gbytes * (size_t)c.world)); }
        PG_CUDA(cudaMemsetAsync(d_star.p, 0, gbytes, st));
        sp.gsum = d_star.as<unsigned long long>();
        sp.gsum_hi = sp.gsum + star_ngroups;
        sp.gcnt = sp.gsum + 2 * star_ngroups;
        if ((size_t)star_ngroups * 16 > 48 * 1024)      // above the default dynamic shared memory limit (up to 64 KB at STAR_MAXGROUPS)
            PG_CUDA(cudaFuncSetAttribute(hits_star_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, star_ngroups * 16));
        if (xl >= 0) {
            PG_TRY(run_star_exchange(sp, res, tr));
        } else {
            hits_star_kernel<<<c.prop.multiProcessorCount * 8, 256, (size_t)star_ngroups * 16, st>>>(sp);
            PG_CUDA(cudaGetLastError());
        }
        PG_CUDA(cudaEventRecord(ev_main.b, st));
        res->stats.kernel_launches += 2;
        if (W > 1) {
            PG_TRY(comm_allgather(d_star.p, d_star_all.p, gbytes, st));
            PG_CUDA(cudaMemcpyAsync(h_star.p, d_star_all.p, gbytes * (size_t)W, cudaMemcpyDeviceToHost, st));
        } else {
            PG_CUDA(cudaMemcpyAsync(h_star.p, d_star.p, gbytes, cudaMemcpyDeviceToHost, st));
        }
        unsigned long long cnt[4];
        PG_CUDA(cudaEventRecord(ev_all.b, st));
        PG_TRY(read_counters(cnt));
        tr.mark("star sink + d2h");
        if (cnt[2] != 0) PG_FAIL(PG_EUNSUPPORTED, "star join: a lookup matched more than one build row (duplicate build keys)");
        res->stats.kernel_ms = ev_all.ms();
        if (xl >= 0) {
            res->stats.comm_ms = (double)ev_xb.ms() + (double)ev_xp.ms();     // the two row exchanges (NVLink)
            res->stats.aux[7] = x_sent_rows;                                  // rows / bytes this rank sent to OTHER ranks
            res->stats.aux[5] = x_sent_bytes;
        }
        res->stats.main_kernel_ms = ev_main.ms();
        res->stats.rows_scanned = t->nrows;
        res->stats.algorithmic_bytes = algorithmic_bytes;
        res->stats.main_kernel_bytes = main_bytes;
        res->stats.aux[0] = (i64)cnt[0];
        res->stats.aux[1] = (i64)cnt[1];
        // merge ranks (exact: 128-bit), emit the groups that received rows
        std::vector<i128> sums((size_t)star_ngroups, 0);
        std::vector<i64> cnts((size_t)star_ngroups, 0);
        const i64 *hs = h_star.as<i64>();
        for (int r = 0; r < W; r++)
            for (int g = 0; g < star_ngroups; g++) {
                const i64 *rec = hs + (size_t)r * 3 * (size_t)star_ngroups;
                sums[(size_t)g] += (i128)(((u128)(u64)rec[star_ngroups + g] << 64) | (u128)(u64)rec[g]);
                cnts[(size_t)g] += rec[2 * star_ngroups + g];
            }
        std::vector<int> live;
        for (int g = 0; g < star_ngroups; g++) if (cnts[(size_t)g] > 0) live.push_back(g);
        res->nrows = (i64)live.size();
        res->stats.aux[6] = res->nrows;
        for (auto &o : outs) {
            ResCol col;
            if (o.first == 0) {
                const HPart &hp = sparts[(size_t)o.second];
                i64 stride = 1;
                for (size_t k = (size_t)o.second + 1; k < sparts.size(); k++) stride *= sparts[k].n;
                col.type = hp.type;
                const int w = type_size(col.type);
                col.data.resize(live.size() * (size_t)w);
                if (hp.type == PG_T_DICT8) col.dict = tab(origin_slot[(size_t)hp.v.origin])->cols[(size_t)hp.v.col].dict;
                for (size_t i = 0; i < live.size(); i++) {
                    const i64 v = ((i64)live[i] / stride) % hp.n + hp.lo;
                    if (w == 8) ((i64 *)col.data.data())[i] = v;
                    else if (w == 4) ((int32_t *)col.data.data())[i] = (int32_t)v;
                    else col.data[i] = (uint8_t)v;
                }
            } else {
                const AggExpr &a = aggs[(size_t)o.second];
                col.width = a.width;
                col.scale = a.scale;
                if (a.fn == PG_AGG_AVG && a.ltype == PG_LT_DOUBLE) {             // avg(INT): float64 sum / float64 count
                    col.type = PG_T_FLOAT64;
                    col.data.resize(live.size() * 8);
                    double *d = (double *)col.data.data();
                    for (size_t i = 0; i < live.size(); i++) {
                        const i128 v = sums[(size_t)live[i]];
                        if (v >= ((i128)1 << 53) || v <= -((i128)1 << 53)) PG_FAIL(PG_EOVERFLOW, "avg(INT): sum not exact in float64");
                        d[i] = (double)(i64)v / (double)cnts[(size_t)live[i]];
                    }
                } else if (a.fn == PG_AGG_AVG) {                                 // avg(DECIMAL) = sum.Quo(count)
                    col.type = PG_T_DECIMAL128;
                    col.data.resize(live.size() * sizeof(pg_decimal));
                    pg_decimal *d = (pg_decimal *)col.data.data();
                    for (size_t i = 0; i < live.size(); i++) {
                        HDec sd, nd, qd;
                        if (!hd_from_i128(sums[(size_t)live[i]], star_scale, &sd) || !hd_from_i128((i128)cnts[(size_t)live[i]], 0, &nd) || !hd_quo(sd, nd, &qd))
                            PG_FAIL(PG_EOVERFLOW, "avg: decimal division failed");
                        d[i].coef = qd.coef;
                        d[i].scale = qd.scale;
                        d[i].neg = qd.neg ? 1u : 0u;
                    }
                } else if (a.fn == PG_AGG_COUNT || a.ltype == PG_LT_HUGEINT) {
                    col.type = PG_T_HUGEINT;
                    col.data.resize(live.size() * sizeof(pg_hugeint));
                    pg_hugeint *d = (pg_hugeint *)col.data.data();
                    for (size_t i = 0; i < live.size(); i++) {
                        const i128 v = a.fn == PG_AGG_COUNT ? (i128)cnts[(size_t)live[i]] : sums[(size_t)live[i]];
                        d[i].lower = (u64)v;
                        d[i].upper = (i64)(v >> 64);
                    }
                } else {
                    col.type = PG_T_DECIMAL128;
                    col.data.resize(live.size() * sizeof(pg_decimal));
                    pg_decimal *d = (pg_decimal *)col.data.data();
                    for (size_t i = 0; i < live.size(); i++) {
                        const i128 v = sums[(size_t)live[i]];
                        const u128 m = v < 0 ? (u128)(-v) : (u128)v;
                        if (m >= (u128)10000000000000000000ULL) PG_FAIL(PG_EOVERFLOW, "star join: a group sum needs more than 19 digits");
                        d[i].neg = v < 0;
                        d[i].coef = (u64)m;
                        d[i].scale = star_scale;
                    }
                }
            }
            res->cols.push_back(std::move(col));
        }
        tr.mark("result columns");
        return PG_OK;
    }

    int run(pg_result *res) override
    {
        Context &c = ctx();
        cudaStream_t st = c.stream;
        PG_TRY(ev_all.init());
        PG_TRY(ev_main.init());
        Trace tr("joinagg");
        PG_CUDA(cudaEventRecord(ev_all.a, st));
        res->stats.kernel_launches = 0;
        cur_res = res;
        deferred_stats = 0;
        PG_CUDA(cudaMemsetAsync(d_counters.p, 0, 128, st));
        x_sent_rows = x_sent_bytes = 0;
        for (size_t i = 0; i < stages.size(); i++) {
            if (xl >= 0 && (int)i == lookups[(size_t)xl].stage) { PG_TRY(run_exchange_build(*stages[i], res)); tr.mark("build stage (row exchange)"); continue; }
            PG_TRY(run_build_stage(*stages[i], res, (int)i));
            tr.mark("build stage");
        }
        if (star) return run_star(res, tr);

        const pg_table *t = tab(src_slot);
        PipeParams pp{};
        pp.nrows = t->nrows;
        PG_TRY(fill_preds(pp, ranges, src_slot));
        pp.has_probe = no_join ? 0 : 1;
        if (!no_join) {
            Stage &last = top_stage_ref();
            pp.probe_key = typed(t, probe_key_col);
            pp.probe = last.jt;
            pp.probe_bitmap_only = last.bitmap_only() ? 1 : 0;
            pp.probe_mode = top_probe_mode;
        }
        PG_TRY(fill_extras(pp, extras, src_slot));
        pp.counters = d_counters.as<unsigned long long>();
        pp.gs = gs;
        // group table: start at twice the build-side rows (each joined row matches a build row),
        // grow x2 and rerun if a probe sequence overflows (the reference resizes x2 as well,
        // aggregate_hash.go:538-540)
        u64 cap = next_pow2((u64)std::max<i64>((no_join ? group_hint : stages.back()->built_rows) * 2, 1024));
        unsigned long long cnt[4] = {0, 0, 0, 0};
        // two-phase, whole source in one filter launch: the hit count is known before the group table is
        // sized, so the table (memset + compaction cost) follows the joined rows, not the build side
        const bool two_phase = !no_join && two_phase_ok(pp, t, false);
        const bool single_filter = two_phase && t->nrows <= HIT_CHUNK;
        unsigned long long filter_pass = 0;
        if (single_filter) {
            PG_CUDA(cudaMemsetAsync(d_counters.p, 0, 32, st));
            PG_CUDA(cudaEventRecord(ev_main.a, st));
            PG_TRY(launch_filter(pp, 0, t->nrows));
            unsigned long long c0[4];
            PG_TRY(read_counters(c0));
            filter_pass = c0[0];
            const bool exact = pp.probe_bitmap_only || pp.probe_mode != 0 || stages.back()->dup_keys == 0 || stages.back()->unique_key;   // at most one joined row per hit
            if (exact) cap = next_pow2((u64)std::max<i64>((i64)std::min<unsigned long long>(c0[3], (unsigned long long)cap / 2) * 2, 1024));
            res->stats.kernel_launches += 1;
            tr.mark("probe filter");
        }
        // the shape the vectorised no-join kernels take: 1 key, 1 summed column, <=1 32-bit predicate
        bool one_shape = false;
        if (no_join) {
            bool pred_valid = false;
            for (int k = 0; k < pp.npred; k++) pred_valid = pred_valid || pp.pred[k].col.valid != nullptr;
            one_shape = !pred_valid && gs.nparts == 1 && gs.nacc == 1 && gs.nfac[0] == 1 && pp.npred <= 1 &&
                        (pp.npred == 0 || !pp.pred[0].is_set) && !getenv("PG_GROUP_GENERIC");
        }
        const bool sorted_runs = one_shape && key_sorted && t->nrows > 0 && !(shuffle && c.world > 1) && !getenv("PG_NO_SORTED_RUNS");
        i64 ngroups = 0;
        if (sorted_runs) {
            // key sorted in row order: fused reduce-by-key at scan speed, no table, no compaction
            // one chunk of 128-row tiles per warp
            constexpr int WPB = SA_THREADS / 32;
            const i64 ntiles = (t->nrows + RUN_WTILE - 1) / RUN_WTILE;
            i64 nwarps = std::max<i64>(std::min<i64>(ntiles, (i64)c.prop.multiProcessorCount * 4 * WPB), 1);
            const i64 chunk_tiles = (ntiles + nwarps - 1) / nwarps;
            nwarps = (ntiles + chunk_tiles - 1) / chunk_tiles;
            const i64 grid = (nwarps + WPB - 1) / WPB;
            const i64 nchunks = grid * WPB;
            if (d_edges.bytes < (size_t)nchunks * 2 * sizeof(RunEdge)) PG_TRY(d_edges.alloc((size_t)nchunks * 2 * sizeof(RunEdge)));
            RunEdge *first = d_edges.as<RunEdge>(), *last = first + nchunks;
            // output capacity: a HAVING keeps few groups (the list grows and the pass reruns if not)
            i64 want = hav_plane >= 0 ? std::max<i64>(t->nrows / 64, 1 << 16) : std::min<i64>(t->nrows, group_hint * 4);
            for (int attempt = 0;; attempt++) {
                if (want > out_cap) {
                    PG_TRY(d_out_klo.alloc((size_t)want * 8));
                    PG_TRY(d_out_khi.alloc((size_t)want * 8));
                    PG_TRY(d_out_acc.alloc((size_t)want * 8 * (size_t)(gs.nacc + 1)));
                    out_cap = want;
                }
                PG_CUDA(cudaMemsetAsync(d_counters.p, 0, 32, st));
                RunOut ro{d_out_klo.as<i64>(), d_out_khi.as<i64>(), d_out_acc.as<i64>(), out_cap, d_counters.as<unsigned long long>() + 2,
                          hav_plane, hav_lo, hav_hi};
                PG_CUDA(cudaEventRecord(ev_main.a, st));
                if (pp.npred == 1) run_group_kernel<true><<<(int)grid, SA_THREADS, 0, st>>>(pp, ro, first, last, chunk_tiles);
                else run_group_kernel<false><<<(int)grid, SA_THREADS, 0, st>>>(pp, ro, first, last, chunk_tiles);
                PG_CUDA(cudaGetLastError());
                run_fixup_kernel<<<(int)((nchunks + 255) / 256), 256, 0, st>>>(first, last, (int)nchunks, ro);
                PG_CUDA(cudaGetLastError());
                PG_CUDA(cudaEventRecord(ev_main.b, st));
                res->stats.kernel_launches += 2;
                PG_TRY(read_counters(cnt));
                ngroups = (i64)cnt[2];
                if (ngroups <= out_cap) break;
                if (attempt > 2) PG_FAIL(PG_ECUDA, "internal: sorted-run output keeps overflowing");
                want = ngroups;
            }
            tr.mark("sorted-run group-by");
        }
        // unsorted key with a modest dense domain: direct-addressed accumulators, one pass per L2-sized key slice
        const bool dense_group = !sorted_runs && one_shape && !(shuffle && c.world > 1) && key_domain > 0 && key_domain <= ((u64)1 << 28) &&
                                 t->nrows > 0 && t->nrows < ((i64)1 << 32) && gs.nacc == 1 && !getenv("PG_NO_DENSE_GROUP");
        if (dense_group) {
            const u64 D = key_domain;
            if (d_dense.bytes < D * 12 + 64) PG_TRY(d_dense.alloc(D * 12 + 64));
            unsigned long long *dsum = d_dense.as<unsigned long long>();
            unsigned *dcnt = (unsigned *)(dsum + D);
            PG_CUDA(cudaMemsetAsync(d_dense.p, 0, D * 12, st));
            PG_CUDA(cudaMemsetAsync(d_counters.p, 0, 32, st));
            const u64 slice_bytes = (u64)(getenv("PG_DENSE_SLICE_MB") ? atoll(getenv("PG_DENSE_SLICE_MB")) : 48) << 20;
            const int npass = (int)std::max<u64>((D * 12 + slice_bytes - 1) / slice_bytes, 1);
            const i64 ntiles = (t->nrows + SA_TILE - 1) / SA_TILE;
            const int grid = (int)std::max<i64>(std::min<i64>(ntiles, (i64)c.prop.multiProcessorCount * 8), 1);
            PG_CUDA(cudaEventRecord(ev_main.a, st));
            for (int ps = 0; ps < npass; ps++) {
                const i64 lo = key_min + (i64)(D * (u64)ps / (u64)npass), hi = key_min + (i64)(D * (u64)(ps + 1) / (u64)npass);
                if (pp.npred == 1) group1_dense_kernel<true><<<grid, SA_THREADS, 0, st>>>(pp, dsum, dcnt, key_min, lo, hi, ps == 0);
                else group1_dense_kernel<false><<<grid, SA_THREADS, 0, st>>>(pp, dsum, dcnt, key_min, lo, hi, ps == 0);
                PG_CUDA(cudaGetLastError());
            }
            PG_CUDA(cudaEventRecord(ev_main.b, st));
            res->stats.kernel_launches += npass;
            PG_TRY(read_counters(cnt));
            tr.mark("dense group-by passes");
            const i64 want = (i64)std::min<u64>(D, (u64)std::max<i64>((i64)cnt[0], 1));
            if (want > out_cap) {
                PG_TRY(d_out_klo.alloc((size_t)want * 8));
                PG_TRY(d_out_khi.alloc((size_t)want * 8));
                PG_TRY(d_out_acc.alloc((size_t)want * 8 * (size_t)(gs.nacc + 1)));
                out_cap = want;
            }
            PG_CUDA(cudaMemsetAsync(d_counters.p, 0, 32, st));
            dense_compact_kernel<<<(int)std::min<u64>((D + 255) / 256, (u64)c.prop.multiProcessorCount * 8), 256, 0, st>>>(
                dsum, dcnt, D, key_min, d_out_klo.as<i64>(), d_out_khi.as<i64>(), d_out_acc.as<i64>(), out_cap, d_counters.as<unsigned long long>(),
                hav_plane, hav_lo, hav_hi);
            PG_CUDA(cudaGetLastError());
            res->stats.kernel_launches += 1;
            unsigned long long ng2[4];
            PG_TRY(read_counters(ng2));
            ngroups = (i64)ng2[0];
            dense_passes = npass;
        }
        bool op_crowded = false;         // the order-preserving map overflowed: keys crowd a few home slots
        for (int attempt = 0; !sorted_runs && !dense_group; attempt++) {
            PG_TRY(ensure_group_table(cap));
            cap = gt_cap;
            PG_CUDA(cudaMemsetAsync(d_gt.p, 0x80, cap * 8 * (size_t)gt_slot_words(gs.nacc), st));
            PG_CUDA(cudaMemsetAsync(d_overflow.p, 0, 4, st));
            PG_CUDA(cudaMemsetAsync(d_counters.p, 0, 32, st));
            pp.gt.slots = d_gt.as<i64>();
            pp.gt.mask = cap - 1;
            pp.gt.nacc = gs.nacc;
            pp.gt.rw = gt_slot_words(gs.nacc);
            pp.gt.two_words = gs.nparts > 1 ? 1 : 0;
            pp.gt.order_preserving = 0;
            if (no_join && gs.run_aggregate && key_domain > 0 && key_domain <= ((u64)1 << 34) && !(shuffle && c.world > 1) && !op_crowded) {
                int lg = 0;
                while (((u64)1 << lg) < cap) lg++;
                if (lg <= 29) {      // (key - kmin) << log2cap must fit in 64 bits
                    pp.gt.order_preserving = getenv("PG_ORDER_PRESERVING") ? atoi(getenv("PG_ORDER_PRESERVING")) : 1;
                    pp.gt.kmin = key_min;
                    pp.gt.domain = key_domain;
                    pp.gt.log2cap = lg;
                }
            }
            pp.gt.overflow = d_overflow.as<int>();
            if (!single_filter) PG_CUDA(cudaEventRecord(ev_main.a, st));
            if (single_filter) {
                PG_TRY(launch_sink<SINK_GROUP>(pp));
            } else if (two_phase) {
                // phase 1 at scan speed over chunks of the fact table, phase 2 over each chunk's hit list
                // (no host round trip in between: the sink kernel reads the hit count from device memory)
                for (i64 lo = 0; lo < t->nrows; lo += HIT_CHUNK) {
                    PG_TRY(launch_filter(pp, lo, std::min<i64>(t->nrows, lo + HIT_CHUNK)));
                    PG_TRY(launch_sink<SINK_GROUP>(pp));
                    res->stats.kernel_launches += 2;
                }
                res->stats.kernel_launches -= 1;
            } else if (no_join) {
                // the specialised vectorised kernel when the shape is: 1 key, 1 summed column, <=1 32-bit predicate
                if (one_shape) {
                    i64 ntiles = (t->nrows + SA_TILE - 1) / SA_TILE;
                    int grid = (int)std::max<i64>(std::min<i64>(ntiles, (i64)c.prop.multiProcessorCount * 8), 1);
                    if (pp.npred == 1) group1_kernel<true><<<grid, SA_THREADS, 0, st>>>(pp);
                    else group1_kernel<false><<<grid, SA_THREADS, 0, st>>>(pp);
                } else {
                    scan_group_kernel<<<grid_rows(t->nrows), 256, 0, st>>>(pp);
                }
                PG_CUDA(cudaGetLastError());
            } else {
                PG_TRY(launch_pipe<SINK_GROUP>(pp, t));
            }
            PG_CUDA(cudaEventRecord(ev_main.b, st));
            res->stats.kernel_launches += 1;
            int ovf = 0;
            PG_CUDA(cudaMemcpyAsync(&ovf, d_overflow.p, 4, cudaMemcpyDeviceToHost, st));
            PG_TRY(read_counters(cnt));
            if (single_filter) cnt[0] = filter_pass;
            tr.mark("probe+group kernel");
            if (!ovf) break;
            if (attempt > 8) PG_FAIL(PG_ENOMEM, "group table keeps overflowing");
            // keys spread unevenly over their domain (a few outliers far from the rest) share a handful of home slots
            // under the order-preserving map whatever the capacity: hash them instead
            if (pp.gt.order_preserving) op_crowded = true;
            else cap *= 2;
        }
        // compact
        const bool do_shuffle = shuffle && c.world > 1;
        if (!sorted_runs && !dense_group) {
        i64 max_out = (i64)std::min<u64>(cap, (u64)cnt[1]);
        if (max_out < 1) max_out = 1;
        if (max_out > out_cap) {
            PG_TRY(d_out_klo.alloc((size_t)max_out * 8));
            PG_TRY(d_out_khi.alloc((size_t)max_out * 8));
            PG_TRY(d_out_acc.alloc((size_t)max_out * 8 * (size_t)(gs.nacc + 1 + (int)fd.size())));    // dependent key columns ride as extra planes
            out_cap = max_out;
        }
        PG_CUDA(cudaMemsetAsync(d_counters.p, 0, 32, st));
        gt_compact_kernel<<<(int)std::min<u64>((cap + 255) / 256, (u64)c.prop.multiProcessorCount * 8), 256, 0, st>>>(
            pp.gt, d_out_klo.as<i64>(), d_out_khi.as<i64>(), d_out_acc.as<i64>(), out_cap, d_counters.as<unsigned long long>(),
            do_shuffle ? -1 : hav_plane, hav_lo, hav_hi);
        PG_CUDA(cudaGetLastError());
        res->stats.kernel_launches += 1;
        unsigned long long ng2[4];
        PG_TRY(read_counters(ng2));
        ngroups = (i64)ng2[0];
        }
        if (do_shuffle) { PG_TRY(shuffle_groups(&ngroups, pp, res)); tr.mark("all-to-all shuffle + merge"); }
        return finish_groups(ngroups, cnt, res, tr);
    }

    // The group list is on the device (d_out_*, ngroups entries, planes [nacc sums][row count][dependent keys]): LIMIT
    // pre-selection, dependent-key gather, read-back (all-gathered across ranks when the probe side is sharded) and the
    // result columns.  cnt: the sink's counters {rows passing the filter, joined rows}.
    int finish_groups(i64 ngroups, const unsigned long long *cnt, pg_result *res, Trace &tr)
    {
        Context &c = ctx();
        cudaStream_t st = c.stream;
        const pg_table *t = tab(src_slot);
        res->stats.aux[6] = ngroups;          // groups before any LIMIT
        tr.mark("compact");
        if (device_only) { dev_ngroups = ngroups; return PG_OK; }
        // (FD mode of a plain join has no device top-k: its ORDER BY keys are fetched below and the host orders the groups.
        // A star join grouped by dimension rows orders by an aggregate: the select runs first and the keys are gathered
        // for every group, but VARCHARs are only materialised on the host for the candidates that come back.)
        // LIMIT k with a small k over many groups: the radix select runs with its state on the device and the candidates
        // leave in one fixed-size message (below) -- no host round trip per pass
        const bool topk_fast = has_topk && topk_limit > 0 && topk_limit <= SG_CAP / 2 && ngroups > topk_limit &&
                               !(getenv("PG_TOPK_HOST") && atoi(getenv("PG_TOPK_HOST")));
        if (has_topk && !topk_fast) { PG_TRY(topk_preselect(&ngroups, res)); tr.mark("top-k preselect"); }
        if (fd_mode && ngroups > 0) {
            // dependent key columns are written behind the accumulator planes of the group list, so every
            // read-back / cross-rank gather path below carries them like one more aggregate
            const int grid = (int)std::max<i64>(std::min<i64>((ngroups + 255) / 256, (i64)c.prop.multiProcessorCount * 8), 1);
            const pg_table *bt = tab(stages[(size_t)fd_stage]->src_slot);
            for (size_t f = 0; f < fd.size(); f++) {
                const FdOut &o = fd[f];
                const pg_table *ct = tab(o.slot);
                const bool host_col = ct->cols[(size_t)o.col].type == PG_T_VARCHAR;
                TypedCol none{nullptr, 8, 0, nullptr};
                TypedCol colref = host_col ? none : typed(ct, o.col);
                i64 *dst = d_out_acc.as<i64>() + (size_t)(gs.nacc + 1 + (int)f) * (size_t)out_cap;
                if (o.kind == 0) {
                    fd_gather_kernel<<<grid, 256, 0, st>>>(d_out_klo.as<i64>(), ngroups, colref, 0, none, JoinTable{}, none, host_col ? 1 : 0, dst);
                } else {
                    const Stage &d = *stages[(size_t)o.via_stage];
                    if (!d.unique_key) PG_FAIL(PG_EUNSUPPORTED, "functionally dependent group key: the deeper build side has no unique key");   // rank index or hash table: one row per key
                    fd_gather_kernel<<<grid, 256, 0, st>>>(d_out_klo.as<i64>(), ngroups, none, 1, typed(bt, o.via_key_col), d.jt, colref,
                                                           host_col ? 1 : 0, dst);
                }
                PG_CUDA(cudaGetLastError());
                res->stats.kernel_launches += 1;
            }
            tr.mark("dependent key gather");
        }
        const int planes = gs.nacc + 1 + (int)fd.size();
        i64 *h_klo = nullptr, *h_khi = nullptr, *h_acc = nullptr;
        auto host_arrays = [&](i64 n) -> int {
            size_t need = (size_t)std::max<i64>(n, 1) * 8 * (size_t)(2 + planes);
            if (h_out.bytes < need) PG_TRY(h_out.alloc(need + need / 4));
            h_klo = h_out.as<i64>();
            h_khi = h_klo + n;
            h_acc = h_khi + n;
            return PG_OK;
        };
        bool small_done = false, skip_small = false;
        if (topk_fast) {
            const i64 n = ngroups, k = topk_limit;
            constexpr int NB = 1 << TOPK_DIGIT_BITS;
            constexpr i64 FAST_CAP = 4 * SG_CAP;
            if (!d_hist.p) { PG_TRY(d_hist.alloc(NB * 4 + 16)); PG_TRY(h_hist.alloc(NB * 4 + 16)); }
            if (!d_tstate.p) PG_TRY(d_tstate.alloc(sizeof(TopkState)));
            if (cand_cap < FAST_CAP) {
                PG_TRY(d_cand_klo.alloc((size_t)FAST_CAP * 8));
                PG_TRY(d_cand_khi.alloc((size_t)FAST_CAP * 8));
                PG_TRY(d_cand_acc.alloc((size_t)FAST_CAP * 8 * (size_t)planes));
                cand_cap = FAST_CAP;
            }
            const int grid = (int)std::max<i64>(std::min<i64>((n + 255) / 256, (i64)c.prop.multiProcessorCount * 4), 1);
            unsigned *hist = d_hist.as<unsigned>();
            unsigned long long *minmax = (unsigned long long *)(hist + NB);
            TopkState *ts = d_tstate.as<TopkState>();
            const i64 stop_at = std::max<i64>(128 - k, 16);
            topk_state_init_kernel<<<1, 256, 0, st>>>(ts, k, n, hist, minmax);
            topk_hist_dev_kernel<true><<<grid, 256, 0, st>>>(topk_key, d_out_klo.as<i64>(), d_out_khi.as<i64>(), d_out_acc.as<i64>(), out_cap, n, ts, hist, minmax);
            topk_select_kernel<<<1, 256, 0, st>>>(ts, hist, minmax, k, n, stop_at, 0);
            for (int i = 0; i < TOPK_DEV_MORE; i++) {
                topk_hist_dev_kernel<false><<<grid, 256, 0, st>>>(topk_key, d_out_klo.as<i64>(), d_out_khi.as<i64>(), d_out_acc.as<i64>(), out_cap, n, ts, hist, minmax);
                topk_select_kernel<<<1, 256, 0, st>>>(ts, hist, minmax, k, n, stop_at, i == TOPK_DEV_MORE - 1);
            }
            PG_CUDA(cudaMemsetAsync(d_counters.p, 0, 32, st));
            topk_collect_dev_kernel<<<grid, 256, 0, st>>>(topk_key, d_out_klo.as<i64>(), d_out_khi.as<i64>(), d_out_acc.as<i64>(), out_cap, n, planes, ts,
                                                          d_cand_klo.as<i64>(), d_cand_khi.as<i64>(), d_cand_acc.as<i64>(), cand_cap,
                                                          d_counters.as<unsigned long long>());
            const size_t words = 1 + (size_t)SG_CAP * (size_t)(2 + planes);
            const int W = (gather_ranks && c.world > 1) ? c.world : 1;
            if (!d_sg.p) { PG_TRY(d_sg.alloc(words * 8 * (size_t)(c.world + 1))); PG_TRY(h_sg.alloc(words * 8 * (size_t)c.world)); }
            i64 *send = d_sg.as<i64>();
            topk_pack_kernel<<<4, 256, 0, st>>>(d_cand_klo.as<i64>(), d_cand_khi.as<i64>(), d_cand_acc.as<i64>(), cand_cap, d_counters.as<unsigned long long>(), planes,
                                                SG_CAP, send);
            PG_CUDA(cudaGetLastError());
            res->stats.kernel_launches += 5 + 2 * TOPK_DEV_MORE;
            if (W > 1) {
                PG_TRY(comm_allgather(send, send + words, words * 8, st));
                PG_CUDA(cudaMemcpyAsync(h_sg.p, send + words, words * 8 * (size_t)W, cudaMemcpyDeviceToHost, st));
            } else {
                PG_CUDA(cudaMemcpyAsync(h_sg.p, send, words * 8, cudaMemcpyDeviceToHost, st));
            }
            PG_CUDA(cudaStreamSynchronize(st));
            tr.mark("top-k (device select) + gather");
            const i64 *hs = h_sg.as<i64>();
            i64 total = 0;
            bool ok = true;
            for (int r = 0; r < W; r++) { i64 x = hs[(size_t)r * words]; if (x < 0) ok = false; else total += x; }
            if (ok) {
                PG_TRY(host_arrays(total));
                i64 off = 0;
                for (int r = 0; r < W; r++) {
                    const i64 *rec = hs + (size_t)r * words;
                    i64 nr = rec[0];
                    memcpy(h_klo + off, rec + 1, (size_t)nr * 8);
                    memcpy(h_khi + off, rec + 1 + SG_CAP, (size_t)nr * 8);
                    for (int a = 0; a < planes; a++) memcpy(h_acc + (size_t)a * (size_t)total + (size_t)off, rec + 1 + (size_t)SG_CAP * (size_t)(2 + a), (size_t)nr * 8);
                    off += nr;
                }
                ngroups = total;
                small_done = true;
            } else {
                // more candidates than the message holds on some rank (every rank sees every count, so every rank leaves
                // the single-message path here): the host-driven select, then the general gather below
                PG_TRY(topk_preselect(&ngroups, res));
                skip_small = true;
            }
        }
        if (small_done || skip_small) {
        } else if (gather_ranks && c.world > 1 && has_topk && topk_limit >= 0 && topk_limit <= SG_CAP / 2) {
            // LIMIT k with small k: every rank has at most k (+ties) candidates -> ONE fixed-size all-gather
            // [count | klo[SG_CAP] | khi[SG_CAP] | planes x acc[SG_CAP]] and one read-back.  A rank with more
            // than SG_CAP candidates publishes count = -1 and everybody takes the general path below.
            const size_t words = 1 + (size_t)SG_CAP * (size_t)(2 + planes);
            if (!d_sg.p) { PG_TRY(d_sg.alloc(words * 8 * (size_t)(c.world + 1))); PG_TRY(h_sg.alloc(words * 8 * (size_t)c.world)); }
            i64 *send = d_sg.as<i64>();
            i64 cnt_word = ngroups <= SG_CAP ? ngroups : -1;
            PG_CUDA(cudaMemcpyAsync(send, &cnt_word, 8, cudaMemcpyHostToDevice, st));
            if (cnt_word > 0) {
                PG_CUDA(cudaMemcpyAsync(send + 1, d_out_klo.p, (size_t)ngroups * 8, cudaMemcpyDeviceToDevice, st));
                PG_CUDA(cudaMemcpyAsync(send + 1 + SG_CAP, d_out_khi.p, (size_t)ngroups * 8, cudaMemcpyDeviceToDevice, st));
                for (int a = 0; a < planes; a++)
                    PG_CUDA(cudaMemcpyAsync(send + 1 + (size_t)SG_CAP * (size_t)(2 + a), d_out_acc.as<i64>() + (size_t)a * (size_t)out_cap,
                                            (size_t)ngroups * 8, cudaMemcpyDeviceToDevice, st));
            }
            PG_TRY(comm_allgather(send, send + words, words * 8, st));
            PG_CUDA(cudaMemcpyAsync(h_sg.p, send + words, words * 8 * (size_t)c.world, cudaMemcpyDeviceToHost, st));
            PG_CUDA(cudaStreamSynchronize(st));
            const i64 *hs = h_sg.as<i64>();
            i64 total = 0;
            bool ok = true;
            for (int r = 0; r < c.world; r++) { i64 x = hs[(size_t)r * words]; if (x < 0) ok = false; else total += x; }
            if (ok) {
                PG_TRY(host_arrays(total));
                i64 off = 0;
                for (int r = 0; r < c.world; r++) {
                    const i64 *rec = hs + (size_t)r * words;
                    i64 nr = rec[0];
                    memcpy(h_klo + off, rec + 1, (size_t)nr * 8);
                    memcpy(h_khi + off, rec + 1 + SG_CAP, (size_t)nr * 8);
                    for (int a = 0; a < planes; a++) memcpy(h_acc + (size_t)a * (size_t)total + (size_t)off, rec + 1 + (size_t)SG_CAP * (size_t)(2 + a), (size_t)nr * 8);
                    off += nr;
                }
                ngroups = total;
                small_done = true;
            }
        }
        if (small_done) {
        } else if (gather_ranks && c.world > 1) {
            // shard-local groups are disjoint across ranks (co-partitioned on the join key, checked
            // at plan time): all-gather the per-rank lists over NVLink, every rank ends with the union
            std::vector<i64> counts((size_t)c.world);
            PG_CUDA(cudaMemcpyAsync(d_counters.p, &ngroups, 8, cudaMemcpyHostToDevice, st));
            PG_TRY(d_g_cnt.alloc(8 * (size_t)c.world));
            PG_TRY(comm_allgather(d_counters.p, d_g_cnt.p, 8, st));
            PG_CUDA(cudaMemcpyAsync(counts.data(), d_g_cnt.p, 8 * (size_t)c.world, cudaMemcpyDeviceToHost, st));
            PG_CUDA(cudaStreamSynchronize(st));
            i64 maxn = 1, total = 0;
            for (i64 x : counts) { maxn = std::max(maxn, x); total += x; }
            if (maxn > out_cap) {          // send buffers must hold maxn elements
                DevBuf nk, nh, na;
                PG_TRY(nk.alloc((size_t)maxn * 8));
                PG_TRY(nh.alloc((size_t)maxn * 8));
                PG_TRY(na.alloc((size_t)maxn * 8 * (size_t)planes));
                PG_CUDA(cudaMemcpyAsync(nk.p, d_out_klo.p, (size_t)ngroups * 8, cudaMemcpyDeviceToDevice, st));
                PG_CUDA(cudaMemcpyAsync(nh.p, d_out_khi.p, (size_t)ngroups * 8, cudaMemcpyDeviceToDevice, st));
                for (int a = 0; a < planes; a++)
                    PG_CUDA(cudaMemcpyAsync(na.as<i64>() + (size_t)a * (size_t)maxn, d_out_acc.as<i64>() + (size_t)a * (size_t)out_cap,
                                            (size_t)ngroups * 8, cudaMemcpyDeviceToDevice, st));
                PG_CUDA(cudaStreamSynchronize(st));
                std::swap(d_out_klo.p, nk.p); std::swap(d_out_klo.bytes, nk.bytes);
                std::swap(d_out_khi.p, nh.p); std::swap(d_out_khi.bytes, nh.bytes);
                std::swap(d_out_acc.p, na.p); std::swap(d_out_acc.bytes, na.bytes);
                out_cap = maxn;
            }
            size_t seg = (size_t)maxn * 8;
            if (d_g_klo.bytes < seg * (size_t)c.world) {
                PG_TRY(d_g_klo.alloc(seg * (size_t)c.world));
                PG_TRY(d_g_khi.alloc(seg * (size_t)c.world));
                PG_TRY(d_g_acc.alloc(seg * (size_t)c.world * (size_t)planes));
            }
            PG_TRY(comm_allgather(d_out_klo.p, d_g_klo.p, seg, st));
            PG_TRY(comm_allgather(d_out_khi.p, d_g_khi.p, seg, st));
            for (int a = 0; a < planes; a++)
                PG_TRY(comm_allgather(d_out_acc.as<i64>() + (size_t)a * (size_t)out_cap,
                                      (char *)d_g_acc.p + (size_t)a * seg * (size_t)c.world, seg, st));
            PG_TRY(host_arrays(total));
            i64 off = 0;
            for (int r = 0; r < c.world; r++) {
                size_t n = (size_t)counts[(size_t)r];
                if (n) {
                    PG_CUDA(cudaMemcpyAsync(h_klo + off, (char *)d_g_klo.p + seg * (size_t)r, n * 8, cudaMemcpyDeviceToHost, st));
                    PG_CUDA(cudaMemcpyAsync(h_khi + off, (char *)d_g_khi.p + seg * (size_t)r, n * 8, cudaMemcpyDeviceToHost, st));
                    for (int a = 0; a < planes; a++)
                        PG_CUDA(cudaMemcpyAsync(h_acc + (size_t)a * (size_t)total + (size_t)off,
                                                (char *)d_g_acc.p + (size_t)a * seg * (size_t)c.world + seg * (size_t)r, n * 8,
                                                cudaMemcpyDeviceToHost, st));
                }
                off += (i64)n;
            }
            ngroups = total;
        } else {
            PG_TRY(host_arrays(ngroups));
            if (ngroups > 0) {
                PG_CUDA(cudaMemcpyAsync(h_klo, d_out_klo.p, (size_t)ngroups * 8, cudaMemcpyDeviceToHost, st));
                PG_CUDA(cudaMemcpyAsync(h_khi, d_out_khi.p, (size_t)ngroups * 8, cudaMemcpyDeviceToHost, st));
                for (int a = 0; a < planes; a++)
                    PG_CUDA(cudaMemcpyAsync(h_acc + (size_t)a * (size_t)ngroups, d_out_acc.as<i64>() + (size_t)a * (size_t)out_cap,
                                            (size_t)ngroups * 8, cudaMemcpyDeviceToHost, st));
            }
        }
        PG_CUDA(cudaEventRecord(ev_all.b, st));
        PG_CUDA(cudaStreamSynchronize(st));
        tr.mark("gather+d2h");
        res->stats.kernel_ms = ev_all.ms();
        res->stats.main_kernel_ms = ev_main.ms();
        res->stats.rows_scanned = t->nrows;
        res->stats.algorithmic_bytes = algorithmic_bytes;
        res->stats.main_kernel_bytes = main_bytes + (i64)cnt[1] * 32 * (gs.nparts + 2 * gs.nacc);   // streamed + gathered sectors
        res->stats.aux[0] = (i64)cnt[0];
        res->stats.aux[1] = (i64)cnt[1];

        // result columns (group order is the table's slot order: the reference guarantees no
        // order for a hash aggregate either beyond first insertion, and every BASELINE query
        // sorts above it)
        res->nrows = ngroups;
        for (auto &o : outs) {
            ResCol col;
            if (o.first == 0 && fd_mode) {
                const FdOut &fo = fd[(size_t)o.second];
                const Column &cc = tab(fo.slot)->cols[(size_t)fo.col];
                const i64 *src = h_acc + (size_t)(gs.nacc + 1 + o.second) * (size_t)ngroups;
                col.type = cc.type;
                col.width = cc.width;
                col.scale = cc.scale;
                if (cc.type == PG_T_DICT8) col.dict = cc.dict;
                const int w = type_size(cc.type);
                col.data.resize((size_t)ngroups * (size_t)w);
                if (cc.type == PG_T_VARCHAR) {
                    size_t total = 0;
                    for (i64 i = 0; i < ngroups; i++) {
                        if (src[i] < 0 || src[i] + 1 >= (i64)cc.h_off.size()) PG_FAIL(PG_ECUDA, "internal: dependent key row %lld out of range", (long long)src[i]);
                        total += (size_t)(cc.h_off[(size_t)src[i] + 1] - cc.h_off[(size_t)src[i]]);
                    }
                    col.heap.resize(total + 1);
                    pg_string *d = (pg_string *)col.data.data();
                    size_t at = 0;
                    for (i64 i = 0; i < ngroups; i++) {
                        const size_t b = (size_t)cc.h_off[(size_t)src[i]], n = (size_t)cc.h_off[(size_t)src[i] + 1] - b;
                        memcpy(col.heap.data() + at, cc.h_bytes.data() + b, n);
                        d[i].data = col.heap.data() + at;
                        d[i].len = (int64_t)n;
                        at += n;
                    }
                } else {
                    for (i64 i = 0; i < ngroups; i++) {
                        if (w == 8) ((i64 *)col.data.data())[i] = src[i];
                        else if (w == 4) ((int32_t *)col.data.data())[i] = (int32_t)src[i];
                        else col.data[(size_t)i] = (uint8_t)src[i];
                    }
                }
            } else if (o.first == 0) {
                int k = o.second;
                col.type = group_out_type[(size_t)k];
                const int w = type_size(col.type);
                col.data.resize((size_t)ngroups * (size_t)w);
                if (k == 0 && w == 8) {
                    if (ngroups) memcpy(col.data.data(), h_klo, (size_t)ngroups * 8);
                } else if (k == 0) {
                    int32_t *d = (int32_t *)col.data.data();
                    for (i64 i = 0; i < ngroups; i++) d[i] = (int32_t)h_klo[i];
                } else if (w == 4) {
                    int32_t *d = (int32_t *)col.data.data();
                    if (k == 1) for (i64 i = 0; i < ngroups; i++) d[i] = (int32_t)(h_khi[i] >> 32);
                    else for (i64 i = 0; i < ngroups; i++) d[i] = (int32_t)(h_khi[i] & 0xffffffffLL);
                } else {
                    for (i64 i = 0; i < ngroups; i++) {
                        i64 v = k == 1 ? (h_khi[i] >> 32) : (i64)(int32_t)(h_khi[i] & 0xffffffffLL);
                        if (w == 8) ((i64 *)col.data.data())[i] = v; else col.data[(size_t)i] = (uint8_t)v;
                    }
                }
            } else {
                const AggExpr &a = aggs[(size_t)o.second];
                col.width = a.width;
                col.scale = a.scale;
                const i64 *src = h_acc + (size_t)agg_plane[(size_t)o.second] * (size_t)ngroups;
                const i64 *rows_of = h_acc + (size_t)gs.nacc * (size_t)ngroups;      // the row-count plane
                if (a.fn == PG_AGG_AVG && a.ltype == PG_LT_DOUBLE) {       // avg(INT): float64 sum / float64 count
                    col.type = PG_T_FLOAT64;
                    col.data.resize((size_t)ngroups * 8);
                    double *d = (double *)col.data.data();
                    for (i64 i = 0; i < ngroups; i++) {
                        if (src[i] >= ((i64)1 << 53) || src[i] <= -((i64)1 << 53)) PG_FAIL(PG_EOVERFLOW, "avg(INT): sum not exact in float64");
                        d[i] = (double)src[i] / (double)rows_of[i];
                    }
                } else if (a.fn == PG_AGG_AVG) {                           // avg(DECIMAL) = sum.Quo(count)
                    col.type = PG_T_DECIMAL128;
                    col.data.resize((size_t)ngroups * sizeof(pg_decimal));
                    pg_decimal *d = (pg_decimal *)col.data.data();
                    for (i64 i = 0; i < ngroups; i++) {
                        HDec sd, nd, qd;
                        if (!hd_from_i128((i128)src[i], agg_scale[(size_t)o.second], &sd) || !hd_from_i128((i128)rows_of[i], 0, &nd) || !hd_quo(sd, nd, &qd))
                            PG_FAIL(PG_EOVERFLOW, "avg: decimal division failed");
                        d[i].coef = qd.coef;
                        d[i].scale = qd.scale;
                        d[i].neg = qd.neg ? 1u : 0u;
                    }
                } else if (a.ltype == PG_LT_HUGEINT) {          // sum(INT) / count -> 128-bit integer
                    col.type = PG_T_HUGEINT;
                    col.data.resize((size_t)ngroups * sizeof(pg_hugeint));
                    pg_hugeint *d = (pg_hugeint *)col.data.data();
                    for (i64 i = 0; i < ngroups; i++) { d[i].lower = (u64)src[i]; d[i].upper = src[i] < 0 ? -1 : 0; }
                } else {
                    col.type = PG_T_DECIMAL128;
                    col.data.resize((size_t)ngroups * sizeof(pg_decimal));
                    pg_decimal *d = (pg_decimal *)col.data.data();
                    const int32_t sc = agg_scale[(size_t)o.second];
                    for (i64 i = 0; i < ngroups; i++) {
                        i64 v = src[i];
                        d[i].neg = v < 0;
                        d[i].coef = v < 0 ? (u64)(-(v + 1)) + 1 : (u64)v;
                        d[i].scale = sc;
                    }
                }
            }
            res->cols.push_back(std::move(col));
        }
        tr.mark("result columns");
        return PG_OK;
    }
};

// ------------------------------------------------------------------ building --

namespace {

// resolve output `idx` of node `n` to a base table column
bool resolve(const Node &n, int idx, BaseCol *out)
{
    if (n.op == PG_OP_SCAN) { out->slot = n.slot; out->col = idx; return true; }
    if (n.op == PG_OP_FILTER) return resolve(n.children[0], idx, out);
    if (n.op == PG_OP_JOIN) {
        if (idx < 0 || idx >= (int)n.outs.size()) return false;
        auto o = n.outs[(size_t)idx];
        if (o.first != 0 && o.first != 1) return false;
        return resolve(n.children[(size_t)o.first], o.second, out);
    }
    if (n.op == PG_OP_AGG) {        // an aggregate's group-key output is the grouped column itself
        if (idx < 0 || idx >= (int)n.outs.size()) return false;
        auto o = n.outs[(size_t)idx];
        if (o.first != 0 || o.second < 0 || o.second >= (int)n.groups.size()) return false;
        const Expr *ge = strip_value_preserving_casts(&n.groups[(size_t)o.second]);
        return ge->kind == PG_TK_COL && resolve(n.children[0], ge->idx, out);
    }
    return false;
}

const Node *source_scan(const Node &n)   // probe-side source of a join chain, or the scan itself
{
    const Node *x = &n;
    while (x->op == PG_OP_FILTER) x = &x->children[0];
    if (x->op == PG_OP_SCAN) return x;
    if (x->op == PG_OP_JOIN) return source_scan(x->children[0]);
    return nullptr;
}

}  // namespace

int build_join_agg(pg_plan *plan, const Node &aggn, const Node &join, std::unique_ptr<Pipeline> *out, bool nested);

// build the stage that materialises `n` (a build side) keyed on output `key_idx` of n
static int add_build_stage(JoinAggPipeline *p, const Node &n0, int key_idx, int *stage_out)
{
    const Node *n = &n0;
    std::vector<Expr> extra;
    while (n->op == PG_OP_FILTER) { for (auto &f : n->filters) extra.push_back(f); n = &n->children[0]; }
    std::unique_ptr<Stage> s(new Stage());
    BaseCol key;
    if (!resolve(*n, key_idx, &key)) PG_FAIL(PG_EUNSUPPORTED, "join build key is not a plain column");
    if (n->op == PG_OP_SCAN) {
        s->src_slot = n->slot;
        LowerCtx cx;
        cx.table = p->tab(n->slot);
        cx.allow_nulls = true;
        std::vector<Expr> fl = n->filters;
        for (auto &f : extra) fl.push_back(f);
        if (!lower_filters(cx, fl, s->ranges)) PG_FAIL(PG_EUNSUPPORTED, "build-side filter not off-loadable: %s", cx.why.c_str());
    } else if (n->op == PG_OP_JOIN) {
        if (!extra.empty()) PG_FAIL(PG_EUNSUPPORTED, "filter above a build-side join");
        if (n->jointype != PG_JOIN_INNER && n->jointype != PG_JOIN_SEMI && n->jointype != PG_JOIN_ANTI)
            PG_FAIL(PG_EUNSUPPORTED, "only INNER / SEMI / ANTI joins are off-loaded");
        if (n->conds.size() != 1) PG_FAIL(PG_EUNSUPPORTED, "multi-column join keys are not off-loaded");
        for (auto &o : n->outs) if (n->jointype != PG_JOIN_INNER && o.first != 0) PG_FAIL(PG_EUNSUPPORTED, "SEMI/ANTI join output refers to the build side");
        const Node &probe = n->children[0];
        const Node *src = &probe;
        std::vector<Expr> pf;
        while (src->op == PG_OP_FILTER) { for (auto &f : src->filters) pf.push_back(f); src = &src->children[0]; }
        if (src->op != PG_OP_SCAN) PG_FAIL(PG_EUNSUPPORTED, "probe side of a build-side join must be a scan");
        s->src_slot = src->slot;
        LowerCtx cx;
        cx.table = p->tab(src->slot);
        cx.allow_nulls = true;
        std::vector<Expr> fl = src->filters;
        for (auto &f : pf) fl.push_back(f);
        if (!lower_filters(cx, fl, s->ranges)) PG_FAIL(PG_EUNSUPPORTED, "probe-side filter not off-loadable: %s", cx.why.c_str());
        // the join condition: probe expr on the source scan, build expr on the inner build side
        const Expr *pe = strip_value_preserving_casts(&n->conds[0].first);
        const Expr *be = strip_value_preserving_casts(&n->conds[0].second);
        if (pe->kind != PG_TK_COL || be->kind != PG_TK_COL) PG_FAIL(PG_EUNSUPPORTED, "join condition is not column = column");
        BaseCol pk;
        if (!resolve(probe, pe->idx, &pk) || pk.slot != src->slot) PG_FAIL(PG_EUNSUPPORTED, "probe key is not a column of the probe scan");
        int inner = -1;
        PG_TRY(add_build_stage(p, n->children[1], be->idx, &inner));
        s->has_probe = true;
        s->probe_mode = n->jointype == PG_JOIN_SEMI ? 1 : n->jointype == PG_JOIN_ANTI ? 2 : 0;
        if (s->probe_mode != 0) p->stages[(size_t)inner]->existence_only = true;
        s->probe_key_col = pk.col;
        s->probe_stage = inner;
        if (key.slot != s->src_slot) PG_FAIL(PG_EUNSUPPORTED, "join key of the outer join comes from the inner build side");
    } else if (n->op == PG_OP_AGG) {
        // `key IN (select k from t [where ...] group by k [having ...])`: the group keys of a nested
        // high-cardinality aggregate; only their existence can be consumed (SEMI / ANTI)
        if (!extra.empty()) PG_FAIL(PG_EUNSUPPORTED, "filter above a build-side aggregate");
        if (n->groups.size() != 1 || n->outs.size() != 1 || n->outs[0] != std::make_pair(0, 0))
            PG_FAIL(PG_EUNSUPPORTED, "a build-side aggregate must output exactly its single group key");
        std::vector<Expr> fl;
        const Node *src = &n->children[0];
        while (src->op == PG_OP_FILTER) { for (auto &f : src->filters) fl.push_back(f); src = &src->children[0]; }
        if (src->op != PG_OP_SCAN) PG_FAIL(PG_EUNSUPPORTED, "build-side aggregate over a non-scan input");
        s->sub_scan = *src;
        for (auto &f : fl) s->sub_scan.filters.push_back(f);
        s->src_slot = src->slot;
        PG_TRY(build_join_agg(p->plan, *n, s->sub_scan, &s->sub, true));
        static_cast<JoinAggPipeline *>(s->sub.get())->device_only = true;
        if (ctx().world > 1 && static_cast<JoinAggPipeline *>(s->sub.get())->shuffle)
            PG_FAIL(PG_EUNSUPPORTED, "build-side aggregate whose groups span ranks (needs the shuffled key set on every rank)");
        s->existence_only = true;
    } else {
        PG_FAIL(PG_EUNSUPPORTED, "unsupported build side (op %d)", n->op);
    }
    if (key.slot != s->src_slot) PG_FAIL(PG_EUNSUPPORTED, "build key is not on the build source table");
    const Column &kc = p->tab(key.slot)->cols[(size_t)key.col];
    if (!is_int_family(kc.type)) PG_FAIL(PG_EUNSUPPORTED, "join key must be an integer column");
    if (kc.vmin <= HT_EMPTY && kc.vmax >= HT_EMPTY) PG_FAIL(PG_EUNSUPPORTED, "join key range contains the empty-slot sentinel");
    s->ins_key_col = key.col;
    s->unique_key = s->sub ? true : (kc.stats_ok && kc.adjacent_descents == 0);     // group keys are unique by construction
    p->stages.push_back(std::move(s));
    *stage_out = (int)p->stages.size() - 1;
    return PG_OK;
}

static i64 host_year_of_days(i64 z)
{
    z += 719468;
    const i64 era = (z >= 0 ? z : z - 146096) / 146097;
    const i64 doe = z - era * 146097;
    const i64 yoe = (doe - doe / 1460 + doe / 36524 - doe / 146096) / 365;
    const i64 y = yoe + era * 400;
    const i64 doy = doe - (365 * yoe + yoe / 4 - yoe / 100);
    const i64 mp = (5 * doy + 2) / 153;
    return y + (mp >= 10 ? 1 : 0);
}

// Star join: the aggregate's input is a LEFT-DEEP stack of INNER joins whose leftmost leaf is the fact
// table scan and whose build sides are (filtered) scans -- the shape of TPC-H Q9.  Group keys must map
// to a small dense domain (dictionary / narrow integer columns, EXTRACT(year) of a date) and the single
// SUM argument to a signed sum of products of (constant +/- column) factors over the joined rows.
static int build_star(pg_plan *plan, const Node &aggn, const Node &top, std::unique_ptr<JoinAggPipeline> p, std::unique_ptr<Pipeline> *out)
{
    typedef JoinAggPipeline::HRef HRef;
    p->star = true;
    std::vector<const Node *> spine;
    const Node *x = &top;
    while (x->op == PG_OP_JOIN) {
        if (x->jointype != PG_JOIN_INNER) PG_FAIL(PG_EUNSUPPORTED, "star join: only INNER joins on the fact-table spine");
        spine.push_back(x);
        x = &x->children[0];
    }
    std::vector<Expr> pf;
    while (x->op == PG_OP_FILTER) { for (auto &f : x->filters) pf.push_back(f); x = &x->children[0]; }
    if (x->op != PG_OP_SCAN) PG_FAIL(PG_EUNSUPPORTED, "star join: the leftmost leaf must be a scan");
    if (spine.size() > STAR_MAXLOOKUP) PG_FAIL(PG_EUNSUPPORTED, "star join: more than %d joins", STAR_MAXLOOKUP);
    p->src_slot = x->slot;
    const pg_table *st = p->tab(x->slot);
    {
        LowerCtx cx;
        cx.table = st;
        std::vector<Expr> fl = x->filters;
        for (auto &f : pf) fl.push_back(f);
        if (!lower_filters(cx, fl, p->ranges)) PG_FAIL(PG_EUNSUPPORTED, "fact-table filter not off-loadable: %s", cx.why.c_str());
    }
    p->origin_slot.push_back(p->src_slot);
    // base column -> (origin, column): the fact table or the table of an earlier lookup
    auto locate = [&](const Node &scope, int idx, HRef *h) -> bool {
        BaseCol bc;
        if (!resolve(scope, idx, &bc)) return false;
        for (size_t o = 0; o < p->origin_slot.size(); o++)
            if (p->origin_slot[o] == bc.slot) { h->origin = (int)o; h->col = bc.col; return true; }
        return false;
    };
    auto int_nonnull = [&](const HRef &h) {
        const Column &cc = p->tab(p->origin_slot[(size_t)h.origin])->cols[(size_t)h.col];
        return is_int_family(cc.type) && !cc.any_nulls();
    };
    for (size_t i = spine.size(); i-- > 0;) {          // bottom-up
        const Node &J = *spine[i];
        if (J.conds.empty() || J.conds.size() > 2) PG_FAIL(PG_EUNSUPPORTED, "star join: join keys of 1 or 2 columns only");
        JoinAggPipeline::HLookup lk;
        lk.nkey = (int)J.conds.size();
        const Expr *be0 = strip_value_preserving_casts(&J.conds[0].second);
        if (be0->kind != PG_TK_COL) PG_FAIL(PG_EUNSUPPORTED, "join condition is not column = column");
        PG_TRY(add_build_stage(p.get(), J.children[1], be0->idx, &lk.stage));
        Stage &S = *p->stages[(size_t)lk.stage];
        if (S.has_probe || S.sub) PG_FAIL(PG_EUNSUPPORTED, "star join: build sides must be (filtered) scans");
        for (int k = 0; k < lk.nkey; k++) {
            const Expr *pe = strip_value_preserving_casts(&J.conds[(size_t)k].first);
            if (pe->kind != PG_TK_COL || !locate(J.children[0], pe->idx, &lk.key[k]) || !int_nonnull(lk.key[k]))
                PG_FAIL(PG_EUNSUPPORTED, "star join: probe key %d is not a reachable non-null integer column", k);
        }
        if (lk.nkey == 2) {
            const Expr *be1 = strip_value_preserving_casts(&J.conds[1].second);
            BaseCol b2;
            if (be1->kind != PG_TK_COL || !resolve(J.children[1], be1->idx, &b2) || b2.slot != S.src_slot) PG_FAIL(PG_EUNSUPPORTED, "second build key is not a column of the build scan");
            const pg_table *bt = p->tab(S.src_slot);
            const Column &k1 = bt->cols[(size_t)S.ins_key_col], &k2 = bt->cols[(size_t)b2.col];
            auto fits32 = [](const Column &c) { return is_int_family(c.type) && !c.any_nulls() && c.vmin >= INT32_MIN && c.vmax <= INT32_MAX; };
            if (!fits32(k1) || !fits32(k2)) PG_FAIL(PG_EUNSUPPORTED, "two-column join keys must both fit 32 bits");
            S.ins_key_col2 = b2.col;
            S.unique_key = false;
        }
        p->lookups.push_back(lk);
        p->origin_slot.push_back(S.src_slot);
    }
    // the filter pass: a one-column join on a FACT column, preferably one whose build side is filtered
    int main = -1;
    for (int pass = 0; pass < 2 && main < 0; pass++)
        for (size_t l = 0; l < p->lookups.size(); l++) {
            const auto &lk = p->lookups[l];
            const Stage &S = *p->stages[(size_t)lk.stage];
            const Column &bk = p->tab(S.src_slot)->cols[(size_t)S.ins_key_col];
            const bool bitmapable = bk.stats_ok && (i128)bk.vmax - (i128)bk.vmin + 1 <= ((i128)1 << 32);
            if (lk.nkey == 1 && lk.key[0].origin == 0 && bitmapable && (pass == 1 || !S.ranges.empty())) { main = (int)l; break; }
        }
    if (main < 0) PG_FAIL(PG_EUNSUPPORTED, "star join: no single-column join on a fact-table column to filter with");
    p->main_stage = p->lookups[(size_t)main].stage;
    p->probe_key_col = p->lookups[(size_t)main].key[0].col;
    if (p->ranges.size() > 1) PG_FAIL(PG_EUNSUPPORTED, "star join: at most one range predicate on the fact table");
    // Key equivalence: another join keyed (partly) by the SAME fact column as the filter join can only ever be
    // probed with keys the filter join accepts, so its build side is reduced up front by an existence probe of the
    // filter join's bitmap (Q9: partsupp rows whose ps_partkey is not a '%pink%' part are never inserted).
    for (size_t l = 0; l < p->lookups.size(); l++) {
        if ((int)l == main) continue;
        const auto &lk = p->lookups[l];
        Stage &S = *p->stages[(size_t)lk.stage];
        if (S.has_probe || lk.stage < p->main_stage || p->stages[(size_t)p->main_stage]->ranges.empty()) continue;
        for (int k = 0; k < lk.nkey; k++) {
            if (lk.key[k].origin != 0 || lk.key[k].col != p->probe_key_col) continue;
            S.has_probe = true;
            S.probe_mode = 1;                                   // SEMI: existence only
            S.probe_stage = p->main_stage;
            S.probe_key_col = k == 0 ? S.ins_key_col : S.ins_key_col2;
            break;
        }
    }

    std::vector<bool> used(p->origin_slot.size(), false);
    auto mark = [&](const HRef &h) { used[(size_t)h.origin] = true; };
    for (auto &lk : p->lookups) for (int k = 0; k < lk.nkey; k++) mark(lk.key[k]);

    // group keys -> dense index parts; keys that do not fit a small dense domain may still name the rows of one dimension
    std::string dense_why;
    i64 ng = 1;
    if (aggn.groups.empty() || aggn.groups.size() > STAR_MAXPART) dense_why = "1.." + std::to_string(STAR_MAXPART) + " group keys";
    for (size_t gi = 0; gi < aggn.groups.size() && dense_why.empty(); gi++) {
        const Expr *ge = strip_value_preserving_casts(&aggn.groups[gi]);
        JoinAggPipeline::HPart hp;
        if (ge->kind == PG_TK_FUNC && ge->fn == PG_FN_EXTRACT && ge->args.size() == 2) {
            const Expr *what = strip_value_preserving_casts(&ge->args[0]), *arg = strip_value_preserving_casts(&ge->args[1]);
            if (what->kind != PG_TK_STR || what->str != "year") { dense_why = "only EXTRACT(year ...) is off-loaded"; break; }
            ge = arg;
            hp.fn = 1;
        }
        if (ge->kind != PG_TK_COL || !locate(top, ge->idx, &hp.v)) { dense_why = "group key is not a reachable column"; break; }
        const Column &cc = p->tab(p->origin_slot[(size_t)hp.v.origin])->cols[(size_t)hp.v.col];
        if (cc.any_nulls()) { dense_why = "nullable group key"; break; }
        if (hp.fn == 1) {
            if (cc.type != PG_T_DATE32) { dense_why = "EXTRACT(year) of a non-date column"; break; }
            hp.lo = host_year_of_days(cc.gmin());
            hp.n = (int)(host_year_of_days(cc.gmax()) - hp.lo + 1);
            hp.type = PG_T_INT32;
        } else if (cc.type == PG_T_DICT8 || cc.type == PG_T_CHAR1) {
            hp.lo = 0;
            hp.n = cc.type == PG_T_DICT8 ? std::max<int>((int)cc.dict.size(), 1) : 256;
            hp.type = cc.type;
        } else if (is_int_family(cc.type) && cc.stats_ok && (i128)cc.gmax() - (i128)cc.gmin() + 1 <= STAR_MAXGROUPS) {
            hp.lo = cc.gmin();
            hp.n = (int)(cc.gmax() - cc.gmin() + 1);
            hp.type = cc.type;
        } else {
            dense_why = "group key domain is not small and dense";
            break;
        }
        ng *= hp.n;
        if (ng > STAR_MAXGROUPS) { dense_why = "more than " + std::to_string(STAR_MAXGROUPS) + " dense groups"; break; }
        p->sparts.push_back(hp);
    }
    // Dimension-row groups (TPC-H Q10): every key is a plain column of the build row of one lookup A -- one of them A's unique
    // build key, the anchor -- or of a lookup B keyed by a column of A's row, with a unique key of its own.  A group is then one
    // row of A: hits_star_rows_kernel sums per row and the keys are fetched for the groups that come out (as fd_mode does for
    // plain joins).  Without the anchor, two rows of A could carry equal keys and would have to be merged.
    auto dimension_rows = [&](std::string *why) -> bool {
        if (ctx().world > 1) { *why = "runs on one GPU (with a sharded fact table a group's rows span ranks)"; return false; }
        std::vector<HRef> keys;
        for (size_t k = 0; k < aggn.groups.size(); k++) {
            const Expr *ge = strip_value_preserving_casts(&aggn.groups[k]);
            HRef h;
            if (ge->kind != PG_TK_COL || !locate(top, ge->idx, &h)) { *why = "group key " + std::to_string(k) + " is not a plain column"; return false; }
            if (p->tab(p->origin_slot[(size_t)h.origin])->cols[(size_t)h.col].any_nulls()) { *why = "group key " + std::to_string(k) + " is nullable"; return false; }
            keys.push_back(h);
        }
        int a = -1;
        for (auto &h : keys)
            if (h.origin > 0 && p->lookups[(size_t)h.origin - 1].nkey == 1 && h.col == p->stages[(size_t)p->lookups[(size_t)h.origin - 1].stage]->ins_key_col) { a = h.origin; break; }
        if (a < 0) { *why = "no group key is the build key of a joined table (the anchor whose rows would be the groups)"; return false; }
        const JoinAggPipeline::HLookup &la = p->lookups[(size_t)a - 1];
        const Stage &A = *p->stages[(size_t)la.stage];
        const std::string aname = p->tab(A.src_slot)->name;
        if (!A.unique_key) { *why = "the build key of " + aname + " is not unique"; return false; }
        std::vector<JoinAggPipeline::FdOut> fd;
        for (size_t k = 0; k < keys.size(); k++) {
            const HRef &h = keys[k];
            if (h.origin == a) { fd.push_back({0, A.src_slot, h.col, -1, -1}); continue; }
            const JoinAggPipeline::HLookup *lb = h.origin > 0 ? &p->lookups[(size_t)h.origin - 1] : nullptr;
            if (!lb || lb->key[0].origin != a) { *why = "group key " + std::to_string(k) + " is neither a column of " + aname + " nor of a table joined on one"; return false; }
            const Stage &B = *p->stages[(size_t)lb->stage];
            if (lb->nkey != 1) { *why = "group key " + std::to_string(k) + " comes through a two-column join key"; return false; }
            if (!B.unique_key) { *why = "the build key of " + p->tab(B.src_slot)->name + " is not unique"; return false; }
            fd.push_back({1, B.src_slot, h.col, lb->key[0].col, lb->stage});
            used[(size_t)h.origin] = true;
        }
        used[(size_t)a] = true;
        p->fd_mode = true;
        p->fd = fd;
        p->fd_stage = la.stage;
        p->star_anchor = a;
        p->nparts = p->gs.nparts = 1;
        return true;
    };
    if (dense_why.empty()) {
        for (auto &hp : p->sparts) mark(hp.v);
        p->star_ngroups = (int)ng;
    } else {
        p->sparts.clear();
        std::string rows_why;
        if (!dimension_rows(&rows_why)) PG_FAIL(PG_EUNSUPPORTED, "star join: %s; grouping by dimension rows: %s", dense_why.c_str(), rows_why.c_str());
    }

    // aggregates: one SUM (signed sum of products) and/or COUNT
    p->aggs = aggn.aggs;
    int nsum = 0;
    const AggExpr *sum = nullptr;
    for (auto &ae : aggn.aggs) {
        if (ae.fn == PG_AGG_COUNT) {
            if (p->fd_mode && ae.ltype != PG_LT_HUGEINT) PG_FAIL(PG_EUNSUPPORTED, "star join: count result type");
            continue;
        }
        const bool is_sum = ae.fn == PG_AGG_SUM && (ae.ltype == PG_LT_DECIMAL || ae.ltype == PG_LT_HUGEINT);
        const bool is_avg = ae.fn == PG_AGG_AVG && (ae.ltype == PG_LT_DECIMAL || ae.ltype == PG_LT_DOUBLE);     // sum / row count at result time
        if (!is_sum && !is_avg) PG_FAIL(PG_EUNSUPPORTED, "star join: sum, avg and count only");
        nsum++;
        sum = &ae;
    }
    if (nsum > 1) PG_FAIL(PG_EUNSUPPORTED, "star join: a single sum");
    if (sum) {
        struct Raw { std::vector<const Expr *> leaves; int sign; };
        std::vector<Raw> raw;
        std::vector<std::pair<const Expr *, int>> todo{{&sum->arg, 1}};
        while (!todo.empty()) {
            auto [e0, sg] = todo.back();
            todo.pop_back();
            const Expr *e = strip_value_preserving_casts(e0);
            if (e->kind == PG_TK_FUNC && (e->fn == PG_FN_SUB || e->fn == PG_FN_ADD) && e->args.size() == 2) {
                const Expr *l = strip_value_preserving_casts(&e->args[0]), *r = strip_value_preserving_casts(&e->args[1]);
                const bool affine = (l->kind == PG_TK_CONST && r->kind == PG_TK_COL) || (l->kind == PG_TK_COL && r->kind == PG_TK_CONST);
                if (!affine) { todo.push_back({&e->args[1], e->fn == PG_FN_SUB ? -sg : sg}); todo.push_back({&e->args[0], sg}); continue; }
            }
            Raw rw;
            rw.sign = sg;
            std::vector<const Expr *> prod{e};
            while (!prod.empty()) {
                const Expr *m = strip_value_preserving_casts(prod.back());
                prod.pop_back();
                if (m->kind == PG_TK_FUNC && m->fn == PG_FN_MUL && m->args.size() == 2) { prod.push_back(&m->args[1]); prod.push_back(&m->args[0]); }
                else rw.leaves.push_back(m);
            }
            raw.push_back(rw);
        }
        if (raw.empty() || raw.size() > STAR_MAXTERM) PG_FAIL(PG_EUNSUPPORTED, "star join: the sum has %zu terms (max %d)", raw.size(), STAR_MAXTERM);
        std::vector<int> tscale;
        i128 worst = 0;
        for (auto &rw : raw) {
            if (rw.leaves.empty() || rw.leaves.size() > 3) PG_FAIL(PG_EUNSUPPORTED, "star join: a product of %zu factors", rw.leaves.size());
            JoinAggPipeline::HTerm ht;
            ht.nfac = (int)rw.leaves.size();
            int scale = 0;
            i128 bound = 1;
            for (size_t f = 0; f < rw.leaves.size(); f++) {
                const Expr *e = rw.leaves[f], *ce = nullptr, *ke = nullptr;
                int sgn = 1;
                bool negk = false;
                if (e->kind == PG_TK_COL) ce = e;
                else if (e->kind == PG_TK_FUNC && (e->fn == PG_FN_ADD || e->fn == PG_FN_SUB) && e->args.size() == 2) {
                    const Expr *l = strip_value_preserving_casts(&e->args[0]), *r = strip_value_preserving_casts(&e->args[1]);
                    if (l->kind == PG_TK_CONST && r->kind == PG_TK_COL) { ke = l; ce = r; sgn = e->fn == PG_FN_ADD ? 1 : -1; }
                    else if (l->kind == PG_TK_COL && r->kind == PG_TK_CONST) { ce = l; ke = r; negk = e->fn == PG_FN_SUB; }
                } else if (e->kind == PG_TK_FUNC && e->fn == PG_FN_CAST && e->args.size() == 1) {
                    // INTEGER -> DECIMAL cast of a column keeps the integer value at value scale 0 (tryCastInt32ToDecimal, function_cast.go:337-347)
                    const Expr *a = strip_value_preserving_casts(&e->args[0]);
                    if (a->kind == PG_TK_COL && e->ltype == PG_LT_DECIMAL && (a->ltype == PG_LT_INTEGER || a->ltype == PG_LT_BIGINT)) ce = a;
                }
                if (!ce || !locate(top, ce->idx, &ht.fac[f])) PG_FAIL(PG_EUNSUPPORTED, "star join: factor is not (constant +/- reachable column)");
                const Column &cc = p->tab(p->origin_slot[(size_t)ht.fac[f].origin])->cols[(size_t)ht.fac[f].col];
                if (!is_int_family(cc.type) || cc.type == PG_T_DATE32 || cc.any_nulls()) PG_FAIL(PG_EUNSUPPORTED, "star join: factor column type");
                const int cs = cc.type == PG_T_DECIMAL64 ? cc.scale : 0;
                i64 k = 0;
                if (ke && !const_at_scale(ke, cs, &k)) PG_FAIL(PG_EUNSUPPORTED, "constant does not fit the column scale");
                ht.fc[f] = negk ? -k : k;
                ht.fs[f] = sgn;
                scale += cs;
                i128 lo = (i128)ht.fc[f] + (i128)sgn * cc.gmin(), hi = (i128)ht.fc[f] + (i128)sgn * cc.gmax();
                i128 m = std::max(lo < 0 ? -lo : lo, hi < 0 ? -hi : hi);
                bound *= m > 1 ? m : 1;
                mark(ht.fac[f]);
            }
            ht.mul = rw.sign;
            tscale.push_back(scale);
            p->sterms.push_back(ht);
            worst += bound;
        }
        // Sub/Add of decimals: the result scale is the larger one (govalues Add/Sub); align the coarser terms
        int maxs = 0;
        for (int s : tscale) maxs = std::max(maxs, s);
        i128 scaled_worst = 0;
        for (size_t i = 0; i < p->sterms.size(); i++) {
            i128 m = 1;
            for (int s = tscale[i]; s < maxs; s++) m *= 10;
            p->sterms[i].mul *= (i64)m;
            scaled_worst = std::max(scaled_worst, worst * m);
        }
        if ((sum->ltype == PG_LT_HUGEINT || sum->ltype == PG_LT_DOUBLE) && maxs != 0) PG_FAIL(PG_EUNSUPPORTED, "integer sum over a scaled value");
        p->star_scale = maxs;
        p->star_worst = scaled_worst;
        if (p->fd_mode) {
            // a dimension row's accumulator is int64 and can receive every fact row
            if (scaled_worst * (i128)std::max<i64>(st->nrows, 1) >= ((i128)1 << 63)) PG_FAIL(PG_EUNSUPPORTED, "star join grouped by dimension rows: a group sum could exceed int64");
        } else {
            // a block's shared-memory partial is int64: it receives at most its share of the fact rows (grid-stride over the hits)
            const i64 threads = (i64)ctx().prop.multiProcessorCount * 8 * 256;
            const i64 per_block = ((std::max<i64>(st->nrows, 1) + threads - 1) / threads) * 256;
            if (scaled_worst * (i128)per_block >= ((i128)1 << 63)) PG_FAIL(PG_EUNSUPPORTED, "a block's partial group sum could exceed int64");
        }
    }
    if (p->fd_mode) {
        if (st->nrows >= ((i64)1 << 32)) PG_FAIL(PG_EUNSUPPORTED, "star join grouped by dimension rows: 2^32 fact rows or more (the per-row count is 32-bit)");
        // the group list of finish_groups(): one sum plane (zeros for a count-only aggregate), then the row-count plane
        p->gs.nacc = 1;
        p->agg_plane.assign(aggn.aggs.size(), 1);
        p->agg_scale.assign(aggn.aggs.size(), 0);
        for (size_t i = 0; i < aggn.aggs.size(); i++)
            if (aggn.aggs[i].fn != PG_AGG_COUNT) { p->agg_plane[i] = 0; p->agg_scale[i] = p->star_scale; }
    }
    for (size_t o = 1; o < used.size(); o++) p->stages[(size_t)p->lookups[o - 1].stage]->payload_needed = used[o];
    for (auto &o : aggn.outs) {
        if (o.first == 0 && (o.second < 0 || o.second >= (int)(p->fd_mode ? p->fd.size() : p->sparts.size()))) PG_FAIL(PG_EUNSUPPORTED, "bad group output index");
        if (o.first == 1 && (o.second < 0 || o.second >= (int)aggn.aggs.size())) PG_FAIL(PG_EUNSUPPORTED, "bad aggregate output index");
        if (o.first != 0 && o.first != 1) PG_FAIL(PG_EUNSUPPORTED, "bad output kind");
    }
    p->outs = aggn.outs;
    if (aggn.having.size()) PG_FAIL(PG_EUNSUPPORTED, "star join: HAVING");
    if (p->fd_mode && plan->topk && !plan->topk->order.empty()) {
        // ORDER BY an aggregate ... LIMIT k: device pre-selection on the sum plane, so that only the candidates' keys reach the host
        const auto o = aggn.outs[(size_t)plan->topk->order[0].first];
        if (o.first == 1 && aggn.aggs[(size_t)o.second].fn != PG_AGG_AVG) {
            TopkKey tk{};
            tk.desc = plan->topk->order[0].second ? 1 : 0;
            tk.div = 1;
            tk.src = 3;
            tk.plane = p->agg_plane[(size_t)o.second];
            for (int i = 2; i < p->agg_scale[(size_t)o.second]; i++) tk.div *= 10;     // DECIMAL keys compare at two fractional digits
            p->has_topk = true;
            p->topk_key = tk;
            p->topk_limit = plan->topk->limit;
        }
    }
    // bytes: the filter pass streams the fact key (+ predicate) column; everything else is gathered per hit
    p->main_bytes = st->nrows * st->cols[(size_t)p->probe_key_col].phys_width();
    for (auto &r : p->ranges) p->main_bytes += st->nrows * st->cols[(size_t)r.col].phys_width();
    p->algorithmic_bytes = p->main_bytes;
    for (auto &sp : p->stages) {
        const pg_table *bt = p->tab(sp->src_slot);
        p->algorithmic_bytes += bt->nrows * bt->cols[(size_t)sp->ins_key_col].phys_width();
    }
    // Which joins are local?  With a sharded fact table a build side must be whole on every rank or sharded on the same
    // key ranges (proved from the exchanged ranges); ONE join may instead be keyed differently on its two sides: it
    // becomes the exchange lookup -- both sides are hash-partitioned on the join key and shipped to the owner rank
    // (exchange.cuh).  PG_FORCE_EXCHANGE=1 sends a join through the exchange even where it is not needed (also on one rank).
    const bool force_x = getenv("PG_FORCE_EXCHANGE") && atoi(getenv("PG_FORCE_EXCHANGE")) != 0;
    std::string x_why;
    auto x_candidate = [&](size_t l) -> bool {
        const auto &lk = p->lookups[l];
        const Stage &S = *p->stages[(size_t)lk.stage];
        if ((int)l == main) { x_why = "the filter-pass join cannot be exchanged"; return false; }
        if (S.sub || (S.has_probe && S.probe_stage != p->main_stage)) { x_why = "exchanged build side must be a (filtered) scan"; return false; }
        {   // the exchange's filter pass takes NULL-free key / predicate columns; decided on the statistics agreed across ranks,
            // so that every rank enters (or refuses) the collectives together
            const pg_table *bt = p->tab(S.src_slot);
            bool nulls = bt->cols[(size_t)S.ins_key_col].any_nulls() || (S.ins_key_col2 >= 0 && bt->cols[(size_t)S.ins_key_col2].any_nulls());
            for (auto &r : S.ranges) nulls = nulls || bt->cols[(size_t)r.col].any_nulls();
            if (nulls) { x_why = "exchanged build side has NULLs in its key or predicate columns"; return false; }
            if (S.ranges.size() > 1) { x_why = "exchanged build side has more than one range predicate"; return false; }
            for (auto &r : S.ranges) if (r.like || r.is_set) { x_why = "exchanged build side has a string / code-set predicate"; return false; }
            if (bt->total_rows() >= ((i64)1 << 32)) { x_why = "exchanged build side has 2^32 rows or more"; return false; }
        }
        for (size_t l2 = 0; l2 < p->lookups.size(); l2++)
            for (int k = 0; k < p->lookups[l2].nkey; k++)
                if (p->lookups[l2].key[k].origin == (int)l + 1) { x_why = "another join is keyed by a column of the exchanged build side"; return false; }
        for (auto &hp : p->sparts) if (hp.v.origin == (int)l + 1) { x_why = "a group key comes from the exchanged build side"; return false; }
        std::vector<int> cols;
        for (auto &ht : p->sterms)
            for (int f = 0; f < ht.nfac; f++)
                if (ht.fac[f].origin == (int)l + 1 && std::find(cols.begin(), cols.end(), ht.fac[f].col) == cols.end()) cols.push_back(ht.fac[f].col);
        if (cols.size() > X_MAXCOL) { x_why = "more than 3 columns of the exchanged build side are read"; return false; }
        for (int cidx : cols) if (p->tab(S.src_slot)->cols[(size_t)cidx].any_nulls()) { x_why = "a carried build column holds NULLs"; return false; }
        return true;
    };
    std::vector<size_t> must_x, may_x;
    if (ctx().world > 1 && st->dist != PG_DIST_REPLICATED) {
        for (size_t l = 0; l < p->lookups.size(); l++) {
            const auto &lk = p->lookups[l];
            const Stage &S = *p->stages[(size_t)lk.stage];
            const pg_table *bt = p->tab(S.src_slot);
            if (bt->dist == PG_DIST_REPLICATED) continue;
            bool copart = lk.nkey == 1 && lk.key[0].origin == 0;
            if (copart) {
                const int W = ctx().world;
                const Column &pc = st->cols[(size_t)lk.key[0].col], &bc = bt->cols[(size_t)S.ins_key_col];
                i64 mine[6] = {pc.vmin, pc.vmax, st->nrows, bc.vmin, bc.vmax, bt->nrows};
                DevBuf ds, dr;
                PG_TRY(ds.alloc(sizeof mine));
                PG_TRY(dr.alloc(sizeof mine * (size_t)W));
                PG_CUDA(cudaMemcpyAsync(ds.p, mine, sizeof mine, cudaMemcpyHostToDevice, ctx().stream));
                PG_TRY(comm_allgather(ds.p, dr.p, sizeof mine, ctx().stream));
                std::vector<i64> all(6 * (size_t)W);
                PG_CUDA(cudaMemcpyAsync(all.data(), dr.p, sizeof mine * (size_t)W, cudaMemcpyDeviceToHost, ctx().stream));
                PG_CUDA(cudaStreamSynchronize(ctx().stream));
                for (int r = 0; r < W; r++)
                    for (int q = 0; q < W; q++) {
                        if (r == q || all[(size_t)r * 6 + 2] == 0 || all[(size_t)q * 6 + 5] == 0) continue;
                        if (all[(size_t)r * 6] <= all[(size_t)q * 6 + 4] && all[(size_t)q * 6 + 3] <= all[(size_t)r * 6 + 1]) copart = false;
                    }
            }
            if (!copart) must_x.push_back(l);
            else may_x.push_back(l);
        }
    } else if (ctx().world == 1) {
        for (size_t l = 0; l < p->lookups.size(); l++) may_x.push_back(l);
    }
    if (must_x.size() > 1) PG_FAIL(PG_EUNSUPPORTED, "star join: %zu joins have sides sharded on different keys (one row exchange per star)", must_x.size());
    if (must_x.size() == 1) {
        if (!x_candidate(must_x[0])) PG_FAIL(PG_EUNSUPPORTED, "sharded join sides are not co-partitioned on the key and the row exchange does not apply: %s", x_why.c_str());
        p->xl = (int)must_x[0];
    } else if (force_x && !p->fd_mode) {        // per-row groups are summed where the hit is: never exchanged
        // prefer a join whose build columns the aggregate reads (there is something to carry)
        for (int pass = 0; pass < 2 && p->xl < 0; pass++)
            for (size_t l : may_x)
                if (x_candidate(l) && (pass == 1 || p->stages[(size_t)p->lookups[l].stage]->payload_needed)) { p->xl = (int)l; break; }
    }
    if (p->xl >= 0) {
        const Stage &S = *p->stages[(size_t)p->lookups[(size_t)p->xl].stage];
        const Column &k1 = p->tab(S.src_slot)->cols[(size_t)S.ins_key_col];
        if (p->lookups[(size_t)p->xl].nkey == 1 && k1.gmin() <= HT_EMPTY && k1.gmax() >= HT_EMPTY) PG_FAIL(PG_EUNSUPPORTED, "join key range contains the empty-slot sentinel");
        for (size_t t = 0; t < p->sterms.size(); t++)
            for (int f = 0; f < p->sterms[t].nfac; f++) {
                if (p->sterms[t].fac[f].origin != p->xl + 1) continue;
                auto it = std::find(p->xcols.begin(), p->xcols.end(), p->sterms[t].fac[f].col);
                if (it == p->xcols.end()) { p->xcols.push_back(p->sterms[t].fac[f].col); it = p->xcols.end() - 1; }
                p->x_term_mask[t] |= 1 << f;
                p->x_fac_col[t][f] = (int)(it - p->xcols.begin());
            }
        // the owner's blocks sum rows of every rank's shard: redo the int64 proof with the whole table's row count
        const i64 threads = (i64)ctx().prop.multiProcessorCount * 8 * 256;
        const i64 per_block = ((std::max<i64>(st->total_rows(), 1) + threads - 1) / threads) * 256 * std::max(ctx().world, 1);
        if (p->star_worst * (i128)per_block >= ((i128)1 << 63)) PG_FAIL(PG_EUNSUPPORTED, "a block's partial group sum could exceed int64");
    }
    PG_TRY(p->d_counters.alloc(128));
    PG_TRY(p->d_overflow.alloc(4));
    std::string ex = p->fd_mode ? "StarJoin[existence filter -> per-hit lookups -> per-row global sums] kernel=filter_hits_kernel+hits_star_rows_kernel fact=" + st->name + " joins:"
                                : "StarJoin[existence filter -> per-hit lookups -> dense shared-memory groups] kernel=filter_hits_kernel+hits_star_kernel fact=" + st->name + " joins:";
    for (size_t l = 0; l < p->lookups.size(); l++) {
        const Stage &S = *p->stages[(size_t)p->lookups[l].stage];
        char b[200];
        snprintf(b, sizeof b, " %s(%d-col key%s%s%s)", p->tab(S.src_slot)->name.c_str(), p->lookups[l].nkey, (int)l == main ? ", filter pass" : "",
                 S.payload_needed ? ", payload" : ", existence", (int)l == p->xl ? ", ROW EXCHANGE: both sides hash-partitioned on the key, all-to-all over NVLink, joined on the owner rank" : "");
        ex += b;
    }
    char b[160];
    if (p->fd_mode)
        snprintf(b, sizeof b, " groups=rows of %s (dependent keys fetched per group) terms=%zu%s", p->tab(p->origin_slot[(size_t)p->star_anchor])->name.c_str(),
                 p->sterms.size(), p->has_topk ? " top-k=device" : "");
    else
        snprintf(b, sizeof b, " groups=%d (dense) terms=%zu", p->star_ngroups, p->sterms.size());
    p->explain = ex + b;
    *out = std::move(p);
    return PG_OK;
}

// `join` is the aggregate's input: an INNER join tree, or (high-cardinality group-by straight over a
// table) a SCAN whose filters the caller already merged.
int build_join_agg(pg_plan *plan, const Node &aggn, const Node &top, std::unique_ptr<Pipeline> *out, bool nested)
{
    std::unique_ptr<JoinAggPipeline> p(new JoinAggPipeline());
    p->plan = plan;
    // SEMI / ANTI joins whose probe side is itself a join (`... where k IN (subquery)` above the FROM-list
    // joins, builder_plan.go:234-262) only filter on one base column: they are pushed down to the scan
    // that owns that column as an existence test (a semi join commutes with the inner joins below it).
    // `top` keeps resolving output indices; `join` is the join whose two sides become the pipelines.
    struct Pending { int mode; BaseCol key; int stage; };
    std::vector<Pending> pending;
    const Node *jn = &top;
    while (jn->op == PG_OP_JOIN && (jn->jointype == PG_JOIN_SEMI || jn->jointype == PG_JOIN_ANTI)) {
        const Node *ps = &jn->children[0];
        while (ps->op == PG_OP_FILTER) ps = &ps->children[0];
        if (ps->op != PG_OP_JOIN) break;
        if (jn->children[0].op != PG_OP_JOIN) PG_FAIL(PG_EUNSUPPORTED, "filter between a SEMI/ANTI join and the join below it");
        if (jn->conds.size() != 1) PG_FAIL(PG_EUNSUPPORTED, "multi-column join keys are not off-loaded");
        for (auto &o : jn->outs) if (o.first != 0) PG_FAIL(PG_EUNSUPPORTED, "SEMI/ANTI join output refers to the build side");
        const Expr *pe = strip_value_preserving_casts(&jn->conds[0].first);
        const Expr *be = strip_value_preserving_casts(&jn->conds[0].second);
        if (pe->kind != PG_TK_COL || be->kind != PG_TK_COL) PG_FAIL(PG_EUNSUPPORTED, "join condition is not column = column");
        Pending pd;
        pd.mode = jn->jointype == PG_JOIN_SEMI ? 1 : 2;
        if (!resolve(jn->children[0], pe->idx, &pd.key)) PG_FAIL(PG_EUNSUPPORTED, "SEMI/ANTI probe key is not a base column");
        const Column &kc = plan->slots[(size_t)pd.key.slot]->cols[(size_t)pd.key.col];
        if (!is_int_family(kc.type)) PG_FAIL(PG_EUNSUPPORTED, "probe key must be an integer column");
        PG_TRY(add_build_stage(p.get(), jn->children[1], be->idx, &pd.stage));      // built before the stages that test it
        p->stages[(size_t)pd.stage]->existence_only = true;
        pending.push_back(pd);
        jn = &jn->children[0];
    }
    const Node &join = *jn;
    if (join.op == PG_OP_JOIN && pending.empty() && !nested) {
        const Node *ps = &join.children[0];
        while (ps->op == PG_OP_FILTER) ps = &ps->children[0];
        if (ps->op == PG_OP_JOIN) return build_star(plan, aggn, top, std::move(p), out);      // several joins on the fact-table side
    }
    p->no_join = join.op == PG_OP_SCAN;
    if (!p->no_join) {
        if (join.jointype != PG_JOIN_INNER && join.jointype != PG_JOIN_SEMI && join.jointype != PG_JOIN_ANTI)
            PG_FAIL(PG_EUNSUPPORTED, "only INNER / SEMI / ANTI joins are off-loaded");
        if (join.conds.size() != 1) PG_FAIL(PG_EUNSUPPORTED, "multi-column join keys are not off-loaded");
        p->top_probe_mode = join.jointype == PG_JOIN_SEMI ? 1 : join.jointype == PG_JOIN_ANTI ? 2 : 0;
        for (auto &o : join.outs) if (p->top_probe_mode != 0 && o.first != 0) PG_FAIL(PG_EUNSUPPORTED, "SEMI/ANTI join output refers to the build side");
    }
    if (aggn.having.size() > 1) PG_FAIL(PG_EUNSUPPORTED, "HAVING with more than one conjunct is not off-loaded");
    // probe side: filtered scan
    const Node *src = p->no_join ? &join : &join.children[0];
    std::vector<Expr> pf;
    while (src->op == PG_OP_FILTER) { for (auto &f : src->filters) pf.push_back(f); src = &src->children[0]; }
    if (src->op != PG_OP_SCAN) PG_FAIL(PG_EUNSUPPORTED, "probe side of the top join must be a scan");
    p->src_slot = src->slot;
    const pg_table *st = p->tab(src->slot);
    {
        LowerCtx cx;
        cx.table = st;
        cx.allow_nulls = true;
        std::vector<Expr> fl = src->filters;
        for (auto &f : pf) fl.push_back(f);
        if (!lower_filters(cx, fl, p->ranges)) PG_FAIL(PG_EUNSUPPORTED, "probe-side filter not off-loadable: %s", cx.why.c_str());
    }
    int top_stage = -1;
    const pg_table *bt = nullptr;
    int build_slot = -1;
    if (!p->no_join) {
        const Expr *pe = strip_value_preserving_casts(&join.conds[0].first);
        const Expr *be = strip_value_preserving_casts(&join.conds[0].second);
        if (pe->kind != PG_TK_COL || be->kind != PG_TK_COL) PG_FAIL(PG_EUNSUPPORTED, "join condition is not column = column");
        BaseCol pk;
        if (!resolve(join.children[0], pe->idx, &pk) || pk.slot != src->slot) PG_FAIL(PG_EUNSUPPORTED, "probe key is not a column of the probe scan");
        if (!is_int_family(st->cols[(size_t)pk.col].type)) PG_FAIL(PG_EUNSUPPORTED, "probe key must be an integer column");
        p->probe_key_col = pk.col;
        PG_TRY(add_build_stage(p.get(), join.children[1], be->idx, &top_stage));
        if (p->top_probe_mode != 0) p->stages[(size_t)top_stage]->existence_only = true;
        build_slot = p->stages[(size_t)top_stage]->src_slot;
        bt = p->tab(build_slot);
    }

    // pushed-down SEMI / ANTI joins become existence tests on the stage (or the top probe) that scans the key's table
    for (const auto &pd : pending) {
        if (p->no_join) PG_FAIL(PG_EUNSUPPORTED, "internal: pushed-down join without a join below it");
        Stage::Extra ex{pd.mode, pd.key.col, pd.stage};
        if (pd.key.slot == p->src_slot) { p->extras.push_back(ex); continue; }
        Stage *owner = nullptr;
        for (auto &sp : p->stages) if (!sp->sub && sp->src_slot == pd.key.slot) owner = sp.get();
        if (!owner) PG_FAIL(PG_EUNSUPPORTED, "SEMI/ANTI probe key belongs to no scanned table");
        // Make the (selective) existence test the stage's MAIN probe when its current one is an INNER join
        // against unique keys, i.e. itself only an existence filter for this stage: the filter pass then
        // lists a handful of rows instead of every row that has a matching build key.
        if (owner->has_probe && owner->probe_mode == 0 && p->stages[(size_t)owner->probe_stage]->unique_key) {
            Stage::Extra old_main{0, owner->probe_key_col, owner->probe_stage};
            owner->probe_mode = pd.mode;
            owner->probe_key_col = pd.key.col;
            owner->probe_stage = pd.stage;
            owner->extras.push_back(old_main);
        } else {
            owner->extras.push_back(ex);
        }
    }
    for (auto &sp : p->stages)
        for (auto &ex : sp->extras) {
            const Stage &b = *p->stages[(size_t)ex.stage];
            const Column &bk = p->tab(b.src_slot)->cols[(size_t)b.ins_key_col];
            if ((i128)bk.vmax - (i128)bk.vmin + 1 > ((i128)1 << 32)) PG_FAIL(PG_EUNSUPPORTED, "existence join against a key domain too wide for a bitmap");
            if (ex.mode == 0 && !b.unique_key) PG_FAIL(PG_EUNSUPPORTED, "INNER join as an existence test needs unique build keys");
        }

    // Group keys functionally dependent on the top join's unique build key -> group by the build row id
    // (see JoinAggPipeline::fd).  Used only when the packed key cannot hold the keys: more than three
    // columns, a VARCHAR, or a column of a deeper build side.
    if (!p->no_join && p->top_probe_mode == 0) {
        Stage &T = *p->stages[(size_t)top_stage];
        bool anchor = false, ok = T.unique_key && !T.sub, need = aggn.groups.size() > GT_MAXKEYPARTS;
        std::vector<JoinAggPipeline::FdOut> fd;
        for (size_t k = 0; k < aggn.groups.size() && ok; k++) {
            const Expr *ge = strip_value_preserving_casts(&aggn.groups[k]);
            BaseCol bc;
            if (ge->kind != PG_TK_COL || !resolve(top, ge->idx, &bc)) { ok = false; break; }
            const Column &cc = p->tab(bc.slot)->cols[(size_t)bc.col];
            if (cc.any_nulls()) { ok = false; break; }
            if (cc.type == PG_T_VARCHAR) need = true;
            if (bc.slot == build_slot) {
                if (bc.col == T.ins_key_col) anchor = true;
                fd.push_back({0, bc.slot, bc.col, -1, -1});
            } else if (bc.slot == p->src_slot && bc.col == p->probe_key_col) {
                anchor = true;                                   // equal to the build key by the join condition
                fd.push_back({0, build_slot, T.ins_key_col, -1, -1});
            } else {
                // a column of a build side the top build stage itself joins INNER on unique keys
                int via_stage = -1, via_key = -1;
                if (T.has_probe && T.probe_mode == 0 && p->stages[(size_t)T.probe_stage]->src_slot == bc.slot) { via_stage = T.probe_stage; via_key = T.probe_key_col; }
                for (auto &ex : T.extras)
                    if (ex.mode == 0 && p->stages[(size_t)ex.stage]->src_slot == bc.slot) { via_stage = ex.stage; via_key = ex.key_col; }
                if (via_stage < 0 || !p->stages[(size_t)via_stage]->unique_key || p->stages[(size_t)via_stage]->sub) { ok = false; break; }
                need = true;
                fd.push_back({1, bc.slot, bc.col, via_key, via_stage});
            }
        }
        if (ok && anchor && need) {
            p->fd_mode = true;
            p->fd = fd;
            p->fd_stage = top_stage;
            for (auto &f : fd) if (f.kind == 1) p->stages[(size_t)f.via_stage]->payload_needed = true;
        }
    }

    // a value above the join: output idx of the join -> (source | build) typed column
    auto valref = [&](int join_out, ValRef *vr, const Column **colp) -> bool {
        BaseCol bc;
        if (!resolve(top, join_out, &bc)) return false;
        const pg_table *t = nullptr;
        if (bc.slot == p->src_slot) { vr->from_build = 0; t = st; }
        else if (bc.slot == build_slot) { vr->from_build = 1; t = bt; }
        else return false;
        vr->col = typed(t, bc.col);
        *colp = &t->cols[(size_t)bc.col];
        return !(*colp)->any_nulls();
    };

    // group keys: up to 3 parts packed into two 64-bit words
    if (p->fd_mode) {
        p->nparts = 1;
        p->gs.nparts = 1;
        p->gs.part[0].col = TypedCol{nullptr, 8, 0, nullptr};
        p->gs.part[0].from_build = 2;                  // the build row id is the group key
        p->group_out_type.push_back(PG_T_INT64);
    } else if (aggn.groups.empty() || aggn.groups.size() > GT_MAXKEYPARTS) {
        PG_FAIL(PG_EUNSUPPORTED, "join aggregate needs 1..3 group keys (or keys functionally dependent on a unique build key)");
    } else {
        p->nparts = (int)aggn.groups.size();
        p->gs.nparts = p->nparts;
    }
    for (int k = 0; k < p->nparts && !p->fd_mode; k++) {
        const Expr *ge = strip_value_preserving_casts(&aggn.groups[(size_t)k]);
        const Column *col = nullptr;
        if (ge->kind != PG_TK_COL || !valref(ge->idx, &p->gs.part[k], &col)) PG_FAIL(PG_EUNSUPPORTED, "group key %d is not a reachable non-null column", k);
        if (!is_int_family(col->type)) PG_FAIL(PG_EUNSUPPORTED, "group key %d is not an integer/date/decimal column", k);
        if (k > 0 && type_size(col->type) != 4 && p->nparts == 3) PG_FAIL(PG_EUNSUPPORTED, "second and third group keys must be 32-bit");
        if (k == 1 && p->nparts == 2 && type_size(col->type) != 4) PG_FAIL(PG_EUNSUPPORTED, "second group key must be 32-bit");
        if (k == 0 && col->vmin <= HT_EMPTY && col->vmax >= HT_EMPTY) PG_FAIL(PG_EUNSUPPORTED, "group key range contains the empty-slot sentinel");
        if (k == 1 && col->vmin <= (i64)(int32_t)0x80808080 && col->vmax >= (i64)(int32_t)0x80808080) PG_FAIL(PG_EUNSUPPORTED, "group key range contains the empty-slot sentinel");
        p->group_out_type.push_back(col->type);
    }
    // aggregates: sum of affine products over reachable columns
    if (aggn.aggs.empty() || aggn.aggs.size() > GT_MAXACC) PG_FAIL(PG_EUNSUPPORTED, "high-cardinality aggregate supports 1..%d aggregates", GT_MAXACC);
    p->aggs = aggn.aggs;
    i128 worst = 0;
    int nsum = 0;
    for (auto &ae : aggn.aggs) if (ae.fn != PG_AGG_COUNT) nsum++;
    p->gs.nacc = nsum;
    p->agg_plane.assign(aggn.aggs.size(), nsum);      // count(*) reads the row-count plane (index nacc)
    p->agg_scale.assign(aggn.aggs.size(), 0);
    int next_plane = 0;
    for (size_t ai = 0; ai < aggn.aggs.size(); ai++) {
        const AggExpr &ae = aggn.aggs[ai];
        if (ae.fn == PG_AGG_COUNT) {
            if (ae.ltype != PG_LT_HUGEINT) PG_FAIL(PG_EUNSUPPORTED, "count result type");
            continue;
        }
        const size_t a = (size_t)next_plane;
        p->agg_plane[ai] = next_plane++;
        // sum -> DECIMAL / HUGEINT; avg = the same sum divided by the group's row count at result time
        // (avg(DECIMAL) = sum.Quo(count), avg(INT) -> DOUBLE: function_aggr.go:63-86,881-895)
        const bool is_sum = ae.fn == PG_AGG_SUM && (ae.ltype == PG_LT_DECIMAL || ae.ltype == PG_LT_HUGEINT);
        const bool is_avg = ae.fn == PG_AGG_AVG && (ae.ltype == PG_LT_DECIMAL || ae.ltype == PG_LT_DOUBLE);
        if (!is_sum && !is_avg) PG_FAIL(PG_EUNSUPPORTED, "high-cardinality aggregate supports sum, avg and count only");
        // lower against a virtual table made of the join's outputs: reuse lower_affprod on the
        // probe table for factors, resolving columns by hand
        struct Tmp { std::vector<Factor> f; } tmp;
        std::vector<const Expr *> todo{&ae.arg};
        // flatten the multiplication tree
        std::vector<const Expr *> leaves;
        while (!todo.empty()) {
            const Expr *e = strip_value_preserving_casts(todo.back());
            todo.pop_back();
            if (e->kind == PG_TK_FUNC && e->fn == PG_FN_MUL && e->args.size() == 2) { todo.push_back(&e->args[1]); todo.push_back(&e->args[0]); }
            else leaves.push_back(e);
        }
        if (leaves.empty() || leaves.size() > 3) PG_FAIL(PG_EUNSUPPORTED, "aggregate argument has %zu factors", leaves.size());
        p->gs.nfac[a] = (int)leaves.size();
        int scale = 0;
        i128 bound = 1;
        for (size_t f = 0; f < leaves.size(); f++) {
            const Expr *e = leaves[f];
            const Expr *ce = nullptr, *ke = nullptr;
            int sgn = 1;
            bool negk = false;
            if (e->kind == PG_TK_COL) ce = e;
            else if (e->kind == PG_TK_FUNC && (e->fn == PG_FN_ADD || e->fn == PG_FN_SUB) && e->args.size() == 2) {
                const Expr *l = strip_value_preserving_casts(&e->args[0]), *r = strip_value_preserving_casts(&e->args[1]);
                if (l->kind == PG_TK_CONST && r->kind == PG_TK_COL) { ke = l; ce = r; sgn = e->fn == PG_FN_ADD ? 1 : -1; }
                else if (l->kind == PG_TK_COL && r->kind == PG_TK_CONST) { ce = l; ke = r; negk = e->fn == PG_FN_SUB; }
            }
            const Column *col = nullptr;
            if (!ce || !valref(ce->idx, &p->gs.fac[a][f], &col)) PG_FAIL(PG_EUNSUPPORTED, "aggregate factor is not (constant +/- reachable column)");
            if (!is_int_family(col->type) || col->type == PG_T_DATE32) PG_FAIL(PG_EUNSUPPORTED, "aggregate factor column type");
            int cs = col->type == PG_T_DECIMAL64 ? col->scale : 0;
            i64 k = 0;
            if (ke && !const_at_scale(ke, cs, &k)) PG_FAIL(PG_EUNSUPPORTED, "aggregate constant does not fit the column scale");
            p->gs.fc[a][f] = negk ? -k : k;
            p->gs.fs[a][f] = sgn;
            scale += cs;
            i128 lo = (i128)p->gs.fc[a][f] + (i128)sgn * col->vmin, hi = (i128)p->gs.fc[a][f] + (i128)sgn * col->vmax;
            i128 m = std::max(lo < 0 ? -lo : lo, hi < 0 ? -hi : hi);
            bound *= m > 1 ? m : 1;
        }
        if ((ae.ltype == PG_LT_HUGEINT || ae.ltype == PG_LT_DOUBLE) && scale != 0) PG_FAIL(PG_EUNSUPPORTED, "integer sum over a scaled value");
        p->agg_scale[ai] = scale;
        worst = std::max(worst, bound);
    }
    // HAVING <aggregate> <cmp> <constant>  ->  inclusive range on that accumulator plane
    if (aggn.having.size() == 1) {
        const Expr &h = aggn.having[0];
        if (h.kind != PG_TK_FUNC || !is_cmp(h.fn) || h.args.size() != 2) PG_FAIL(PG_EUNSUPPORTED, "HAVING is not a comparison");
        const Expr *l = strip_value_preserving_casts(&h.args[0]), *r = strip_value_preserving_casts(&h.args[1]);
        int op = h.fn;
        if (l->kind == PG_TK_CONST) { std::swap(l, r); op = flip_cmp(op); }
        if (l->kind != PG_TK_COL || l->side != 1 || r->kind != PG_TK_CONST || l->idx < 0 || l->idx >= (int)aggn.aggs.size())
            PG_FAIL(PG_EUNSUPPORTED, "HAVING must compare an aggregate with a constant");
        i64 k;
        if (!const_at_scale(r, p->agg_scale[(size_t)l->idx], &k)) PG_FAIL(PG_EUNSUPPORTED, "HAVING constant does not fit the aggregate scale");
        if (aggn.aggs[(size_t)l->idx].fn == PG_AGG_AVG) PG_FAIL(PG_EUNSUPPORTED, "HAVING on an average");
        p->hav_plane = p->agg_plane[(size_t)l->idx];
        switch (op) {
        case PG_FN_EQ: p->hav_lo = p->hav_hi = k; break;
        case PG_FN_LT: p->hav_hi = k - 1; break;
        case PG_FN_LE: p->hav_hi = k; break;
        case PG_FN_GT: p->hav_lo = k + 1; break;
        case PG_FN_GE: p->hav_lo = k; break;
        default: PG_FAIL(PG_EUNSUPPORTED, "HAVING <> is not a range");
        }
    }
    // 64-bit accumulators: a group can at most receive every probe row of EVERY rank (the shuffle adds the ranks' partials
    // into the same slots).  (A build side with duplicate keys multiplies the joined rows; that case is detected while
    // the table is built -- dup_keys -- and is bounded by the same product only for unique keys: see DESIGN 9.)
    if (worst * (i128)std::max<i64>(st->total_rows(), 1) >= ((i128)1 << 63)) PG_FAIL(PG_EUNSUPPORTED, "group sums could exceed int64");
    {   // does anything above the top join read a build-side column?
        bool need = false;
        for (int k = 0; k < p->nparts; k++) need = need || p->gs.part[k].from_build != 0;
        for (int a = 0; a < p->gs.nacc; a++) for (int f = 0; f < p->gs.nfac[a]; f++) need = need || p->gs.fac[a][f].from_build;
        if (!p->no_join) p->stages[(size_t)top_stage]->payload_needed = need;
    }
    if (p->no_join) {
        // expected groups: bounded by the rows and by the key domain of the first key
        BaseCol g0;
        const Expr *ge = strip_value_preserving_casts(&aggn.groups[0]);
        resolve(top, ge->idx, &g0);
        const Column &kc = st->cols[(size_t)g0.col];
        i128 domain = (i128)kc.vmax - (i128)kc.vmin + 1;
        p->group_hint = (i64)std::min<i128>(std::max<i128>(domain, 1), (i128)std::max<i64>(st->nrows / 4, 1));   // grows x2 on overflow
        // clustered key (most rows repeat their neighbour's key, e.g. l_orderkey): combine runs in the warp first
        p->key_min = kc.vmin;
        p->key_domain = domain > 0 && domain < ((i128)1 << 62) ? (u64)domain : 0;
        p->gs.run_aggregate = kc.stats_ok && kc.adjacent_equal * 2 >= st->nrows ? 1 : 0;
        p->key_sorted = kc.stats_ok && kc.adjacent_descents == kc.adjacent_equal;
        if (getenv("PG_RUN_AGGREGATE")) p->gs.run_aggregate = atoi(getenv("PG_RUN_AGGREGATE"));
    }
    for (auto &o : aggn.outs) {
        if (o.first == 0 && (o.second < 0 || o.second >= (p->fd_mode ? (int)p->fd.size() : p->nparts))) PG_FAIL(PG_EUNSUPPORTED, "bad group output index");
        if (o.first == 1 && (o.second < 0 || o.second >= (int)aggn.aggs.size())) PG_FAIL(PG_EUNSUPPORTED, "bad aggregate output index");
        if (o.first != 0 && o.first != 1) PG_FAIL(PG_EUNSUPPORTED, "bad output kind");
    }
    p->outs = aggn.outs;

    // algorithmic bytes: every referenced column of every scanned table, read once
    {
        std::vector<std::pair<int, int>> used;   // (slot, col)
        auto use = [&](int slot, int col) { if (std::find(used.begin(), used.end(), std::make_pair(slot, col)) == used.end()) used.push_back({slot, col}); };
        for (auto &r : p->ranges) use(p->src_slot, r.col);
        if (!p->no_join) use(p->src_slot, p->probe_key_col);
        for (auto &sp : p->stages) {
            for (auto &r : sp->ranges) use(sp->src_slot, r.col);
            use(sp->src_slot, sp->ins_key_col);
            if (sp->has_probe) use(sp->src_slot, sp->probe_key_col);
        }
        for (size_t k = 0; k < aggn.groups.size(); k++) {
            BaseCol bc;
            const Expr *ge = strip_value_preserving_casts(&aggn.groups[k]);
            if (resolve(top, ge->idx, &bc) && p->tab(bc.slot)->cols[(size_t)bc.col].type != PG_T_VARCHAR) use(bc.slot, bc.col);
        }
        for (auto &sp : p->stages) for (auto &ex : sp->extras) use(sp->src_slot, ex.key_col);
        for (auto &ex : p->extras) use(p->src_slot, ex.key_col);
        for (size_t a = 0; a < aggn.aggs.size(); a++) {
            std::vector<const Expr *> todo{&aggn.aggs[a].arg};
            while (!todo.empty()) {
                const Expr *e = todo.back();
                todo.pop_back();
                if (e->kind == PG_TK_COL) { BaseCol bc; if (resolve(top, e->idx, &bc)) use(bc.slot, bc.col); }
                for (auto &ch : e->args) todo.push_back(&ch);
            }
        }
        for (auto &u : used) {
            const pg_table *t = p->tab(u.first);
            i64 b = t->nrows * t->cols[(size_t)u.second].phys_width();
            p->algorithmic_bytes += b;      // SURVEY 8d: every referenced column read once
        }
        // the probe kernel itself STREAMS only the predicate and key columns; the other probe-side
        // columns are gathered for matching rows (added per run: 32-byte sector per value)
        for (auto &r : p->ranges) p->main_bytes += st->nrows * st->cols[(size_t)r.col].phys_width();
        bool key_is_pred = p->no_join;
        for (auto &r : p->ranges) key_is_pred = key_is_pred || r.col == p->probe_key_col;
        if (!key_is_pred) p->main_bytes += st->nrows * st->cols[(size_t)p->probe_key_col].phys_width();
        if (p->no_join) p->main_bytes = p->algorithmic_bytes;
    }
    // multi-GPU: which joins are shard-local?  A REPLICATED build side is complete everywhere.  Two
    // SHARDED sides must be co-partitioned on the join key: no rank's probe-key range may touch
    // another rank's build-key range (proved from the column statistics, exchanged once here).
    if (ctx().world > 1) {
        const int W = ctx().world;
        auto copartitioned = [&](const pg_table *pt, int pcol, const pg_table *btab, int bcol, bool *ok) -> int {
            i64 mine[6] = {pt->cols[(size_t)pcol].vmin, pt->cols[(size_t)pcol].vmax, pt->nrows,
                           btab->cols[(size_t)bcol].vmin, btab->cols[(size_t)bcol].vmax, btab->nrows};
            DevBuf ds, dr;
            PG_TRY(ds.alloc(sizeof mine));
            PG_TRY(dr.alloc(sizeof mine * (size_t)W));
            PG_CUDA(cudaMemcpyAsync(ds.p, mine, sizeof mine, cudaMemcpyHostToDevice, ctx().stream));
            PG_TRY(comm_allgather(ds.p, dr.p, sizeof mine, ctx().stream));
            std::vector<i64> all(6 * (size_t)W);
            PG_CUDA(cudaMemcpyAsync(all.data(), dr.p, sizeof mine * (size_t)W, cudaMemcpyDeviceToHost, ctx().stream));
            PG_CUDA(cudaStreamSynchronize(ctx().stream));
            *ok = true;
            for (int r = 0; r < W; r++)
                for (int q = 0; q < W; q++) {
                    if (r == q || all[(size_t)r * 6 + 2] == 0 || all[(size_t)q * 6 + 5] == 0) continue;
                    if (all[(size_t)r * 6] <= all[(size_t)q * 6 + 4] && all[(size_t)q * 6 + 3] <= all[(size_t)r * 6 + 1]) *ok = false;
                }
            return PG_OK;
        };
        // every rank must take the same decisions: they depend only on gathered data and the plan
        // (a) inner build stages probing earlier stages
        for (auto &sp : p->stages) {
            if (!sp->has_probe) continue;
            const Stage &inner = *p->stages[(size_t)sp->probe_stage];
            const pg_table *pt = p->tab(sp->src_slot), *ib = p->tab(inner.src_slot);
            if (ib->dist == PG_DIST_REPLICATED) continue;
            if (pt->dist == PG_DIST_REPLICATED) PG_FAIL(PG_EUNSUPPORTED, "replicated table probing a sharded one");
            bool ok = false;
            PG_TRY(copartitioned(pt, sp->probe_key_col, ib, inner.ins_key_col, &ok));
            if (!ok) PG_FAIL(PG_EUNSUPPORTED, "sharded join sides are not co-partitioned on the key (needs the all-to-all shuffle path)");
        }
        // (b) the top join
        if (!p->no_join && bt->dist != PG_DIST_REPLICATED) {
            if (st->dist == PG_DIST_REPLICATED) PG_FAIL(PG_EUNSUPPORTED, "replicated table probing a sharded one");
            bool ok = false;
            PG_TRY(copartitioned(st, p->probe_key_col, bt, p->stages[(size_t)top_stage]->ins_key_col, &ok));
            if (!ok) PG_FAIL(PG_EUNSUPPORTED, "sharded join sides are not co-partitioned on the key (needs the all-to-all shuffle path)");
        }
        if (st->dist != PG_DIST_REPLICATED) {
            // Are the groups of different ranks disjoint?  Yes when the first group key is a probe-side
            // column whose value ranges do not overlap between ranks (the shard key).  Otherwise the
            // local group lists are hash-partitioned and exchanged (all-to-all over NVLink) and merged.
            BaseCol g0;
            const Expr *ge = strip_value_preserving_casts(&aggn.groups[0]);
            bool ok = resolve(top, ge->idx, &g0) && g0.slot == p->src_slot;
            bool disjoint = false;
            if (ok) PG_TRY(copartitioned(st, g0.col, st, g0.col, &disjoint));
            const char *force = getenv("PG_FORCE_SHUFFLE");
            if (force && atoi(force)) disjoint = false;
            p->gather_ranks = true;
            p->shuffle = !(ok && disjoint);
            if (p->fd_mode) {
                // groups stand for rows of the top build table: rank-local (and disjoint) when that table is sharded
                // with the probe side (co-partitioning was proved above); host-resident key columns must come from
                // replicated tables, whose row ids mean the same on every rank
                if (bt->dist == PG_DIST_REPLICATED) PG_FAIL(PG_EUNSUPPORTED, "dependent group keys over a replicated build table and a sharded probe");
                for (auto &f : p->fd)
                    if (p->tab(f.slot)->cols[(size_t)f.col].type == PG_T_VARCHAR && p->tab(f.slot)->dist != PG_DIST_REPLICATED)
                        PG_FAIL(PG_EUNSUPPORTED, "VARCHAR group key from a sharded table");
                p->shuffle = false;
            }
        }
    }
    if (plan->topk && !plan->topk->order.empty() && !nested && !p->fd_mode) {
        // primary ORDER BY key -> where it lives in the group table
        auto o = aggn.outs[(size_t)plan->topk->order[0].first];
        TopkKey tk{};
        tk.desc = plan->topk->order[0].second ? 1 : 0;
        tk.div = 1;
        if (o.first == 0) {
            tk.src = o.second;            // 0: klo, 1: khi high, 2: khi low
        } else {
            if (aggn.aggs[(size_t)o.second].fn == PG_AGG_AVG) goto no_device_topk;       // ordering by sum/count: left to the host sort
            tk.src = 3;
            tk.plane = p->agg_plane[(size_t)o.second];
            int sc = p->agg_scale[(size_t)o.second];
            for (int i = 2; i < sc; i++) tk.div *= 10;     // DECIMAL keys compare at two fractional digits
        }
        p->has_topk = true;
        p->topk_key = tk;
        p->topk_limit = plan->topk->limit;
    }
no_device_topk:
    PG_TRY(p->d_counters.alloc(128));
    PG_TRY(p->d_overflow.alloc(4));
    std::string ex = "JoinAgg[inner hash join chain -> global group table] stages:";
    for (auto &sp : p->stages) {
        char b[256];
        snprintf(b, sizeof b, " build(%s%s key=%s%s%s)", sp->sub ? "aggregate over " : "", p->tab(sp->src_slot)->name.c_str(),
                 p->tab(sp->src_slot)->cols[(size_t)sp->ins_key_col].name.c_str(), sp->has_probe ? " probing previous" : "",
                 sp->extras.empty() ? "" : " +existence tests");
        ex += b;
    }
    if (p->fd_mode) ex += " group-by=build row id (dependent keys fetched per group)";
    char b[320];
    if (p->no_join)
        snprintf(b, sizeof b, "GroupBy[global open-addressing table] scan(%s) kernel=pipeline_kernel<SINK_GROUP> group_keys=%d sums=%d%s%s%s",
                 st->name.c_str(), p->nparts, p->gs.nacc, p->hav_plane >= 0 ? " having" : "",
                 p->key_sorted ? " sorted-run reduce-by-key when the shape allows (run_group_kernel)"
                               : (p->key_domain > 0 && p->key_domain <= ((u64)1 << 28)) ? " dense direct-addressed accumulators in L2-sized key slices when the shape allows (group1_dense_kernel)" : "",
                 p->shuffle ? " exchange=all-to-all(hash-partitioned)" : "");
    else
        snprintf(b, sizeof b, " probe(%s key=%s) kernel=filter_hits_kernel+hits_sink_kernel<SINK_GROUP> group_keys=%d sums=%d%s", st->name.c_str(),
                 st->cols[(size_t)p->probe_key_col].name.c_str(), p->nparts, p->gs.nacc,
                 p->shuffle ? " exchange=all-to-all(hash-partitioned)" : "");
    if (p->no_join) ex = b; else ex += b;
    p->explain = ex;
    *out = std::move(p);
    return PG_OK;
}

}  // namespace pg

// ------------------------------------------------------------------ grouped LEFT-join count (leftcount.cuh) --
//
// `Agg(group by k; count(x)) <- LeftJoin(k = fk) <- {Scan(preserved), Scan(build)}`, alone or under
// `Agg(group by that count; count(*))` (TPC-H Q13).  A group is one row of the preserved side that passes its filters; its
// key k is the anchor.  The preserved side becomes a key table (the ordinary build stage: rank index, identity rank index
// or hash table; payload = row id), the build side is streamed once into a u32 count per preserved row.
// count(build column) is the number of matched rows whose argument is non-NULL, NULL when that is 0 (CountOp.Finalize over
// the NULL-padded row); count(*) and count(non-null preserved column) are max(matches, 1).

namespace pg {

namespace {

struct LeftCountPipeline : Pipeline {
    JoinAggPipeline jp;                  // plan, tables and stage 0: the preserved side's key table and its build machinery
    int anchor_col = -1;                 // the preserved side's join key
    int build_slot = -1, build_key_col = -1;
    int arg_col = -1;                    // count(build column): its column; -1: every matched row counts
    bool null_if_empty = false;          // count(build column): 0 matches is NULL, otherwise max(matches, 1)
    bool outer = false;                  // Agg(group by count; count(*)) on top
    std::vector<Range> build_ranges;
    std::vector<std::pair<int, int>> outs;
    LcFilter fa{}, fb{};                 // preserved-side (group) and build-side filters
    DevBuf d_counts, d_cnt, d_hist, d_out_key, d_out_cnt;
    i64 big_cap = 0;
    EventPair ev_all, ev_main;
    i64 main_bytes = 0, algorithmic_bytes = 0;

    // range / code-set predicates and string predicates of one scan; desc: what each string predicate runs as
    int fill(LcFilter &f, const std::vector<Range> &rs, int slot, std::vector<std::string> *desc)
    {
        const pg_table *t = jp.tab(slot);
        const bool bytewise = getenv("PG_LIKE_BYTEWISE") && atoi(getenv("PG_LIKE_BYTEWISE")) != 0;
        f.npred = f.nlike = 0;
        for (auto &r : rs) {
            if (!r.like) {
                if (f.npred >= PIPE_MAXPRED) PG_FAIL(PG_EUNSUPPORTED, "more than %d predicate columns on one scan", PIPE_MAXPRED);
                SrcPred &q = f.pred[f.npred++];
                q.col = typed(t, r.col);
                q.lo = r.lo;
                q.hi = r.hi;
                q.is_set = r.is_set ? 1 : 0;
                memcpy(q.mask, r.set, sizeof q.mask);
                continue;
            }
            const Column &col = t->cols[(size_t)r.col];
            if (!col.d_off) PG_FAIL(PG_EUNSUPPORTED, "string predicate on %s without a device copy of the text", col.name.c_str());
            if (f.nlike >= GEN_MAXLIKE) PG_FAIL(PG_EUNSUPPORTED, "more than %d string predicates on one scan", GEN_MAXLIKE);
            GenLike &l = f.like[f.nlike++];
            memset(&l, 0, sizeof l);
            l.bytes = col.d_bytes;
            l.off = (const i64 *)col.d_off;
            std::vector<std::string> segs;
            if (r.like <= 2 && !bytewise && like_segments(r.pat, &segs)) {
                l.kind = r.like == 1 ? GEN_LIKE_WORDS : GEN_NOTLIKE_WORDS;
                l.plen = (int)segs.size();
                for (size_t s = 0; s < segs.size(); s++) {
                    memcpy(l.pat + 8 * s, segs[s].data(), segs[s].size());
                    l.pat[32 + s] = (char)segs[s].size();
                }
                if (desc) desc->push_back(std::to_string(segs.size()) + "-segment word search");
                continue;
            }
            if (r.pat.size() > GEN_PATMAX) PG_FAIL(PG_EUNSUPPORTED, "string pattern longer than %d bytes", GEN_PATMAX);
            l.kind = r.like;
            l.plen = (int)r.pat.size();
            memcpy(l.pat, r.pat.data(), r.pat.size());
            if (desc) desc->push_back(r.like <= 2 ? "byte-wise wildcard match" : "byte equality");
        }
        return PG_OK;
    }

    int run(pg_result *res) override
    {
        Context &c = ctx();
        cudaStream_t st = c.stream;
        PG_TRY(ev_all.init());
        PG_TRY(ev_main.init());
        Trace tr("leftcount");
        PG_CUDA(cudaEventRecord(ev_all.a, st));
        res->stats.kernel_launches = 0;
        jp.cur_res = res;
        jp.deferred_stats = 0;
        PG_CUDA(cudaMemsetAsync(jp.d_counters.p, 0, 128, st));
        Stage &A = *jp.stages[0];
        PG_TRY(jp.run_build_stage(A, res, 0));
        tr.mark("build stage (preserved keys)");
        const pg_table *at = jp.tab(A.src_slot), *bt = jp.tab(build_slot);
        if (!A.unique_key && !A.rank_index) {
            // the statistics do not prove the preserved keys unique: every built row must find itself and nothing else
            PipeParams pp{};
            pp.nrows = at->nrows;
            PG_TRY(jp.fill_preds(pp, A.ranges, A.src_slot));
            pp.has_probe = 1;
            pp.probe_key = typed(at, anchor_col);
            pp.probe = A.jt;
            pp.counters = jp.d_counters.as<unsigned long long>();
            PG_CUDA(cudaMemsetAsync(jp.d_counters.p, 0, 32, st));
            PG_TRY(jp.launch_pipe<SINK_COUNT>(pp, at));
            res->stats.kernel_launches += 1;
            unsigned long long k[4];
            PG_TRY(jp.read_counters(k));
            if (k[1] != k[0]) PG_FAIL(PG_EUNSUPPORTED, "left-join count: the preserved side holds a key more than once (duplicate %s.%s)",
                                      at->name.c_str(), at->cols[(size_t)anchor_col].name.c_str());
            tr.mark("preserved keys unique");
        }
        const i64 D = std::max<i64>(at->nrows, 1);
        if (d_counts.bytes < (size_t)D * 4) PG_TRY(d_counts.alloc((size_t)D * 4));
        if (!d_cnt.p) PG_TRY(d_cnt.alloc(32));
        PG_CUDA(cudaMemsetAsync(d_counts.p, 0, (size_t)D * 4, st));
        PG_CUDA(cudaMemsetAsync(d_cnt.p, 0, 32, st));
        LeftCountParams p{};
        p.nrows = bt->nrows;
        p.f = fb;
        p.key = typed(bt, build_key_col);
        if (arg_col >= 0) p.arg = typed(bt, arg_col);
        p.anchor = A.jt;
        p.counts = d_counts.as<unsigned>();
        p.counters = d_cnt.as<unsigned long long>();
        unsigned long long *cnt = d_cnt.as<unsigned long long>();
        const int grid = c.prop.multiProcessorCount * 8;
        PG_CUDA(cudaEventRecord(ev_main.a, st));
        left_count_kernel<<<grid, 256, 0, st>>>(p);
        PG_CUDA(cudaGetLastError());
        PG_CUDA(cudaEventRecord(ev_main.b, st));
        res->stats.kernel_launches += 1;
        tr.mark("left_count_kernel");
        unsigned long long h_cnt[4];
        auto count_value = [&](u64 m) { return null_if_empty ? m : std::max<u64>(m, 1); };    // 0 = NULL (count(build column) only)
        ResCol kcol, ccol;
        if (outer) {
            const size_t words = (size_t)LC_HBINS + 1 + (size_t)big_cap;
            if (d_hist.bytes < words * 4) PG_TRY(d_hist.alloc(words * 4));
            unsigned *hist = d_hist.as<unsigned>();
            PG_CUDA(cudaMemsetAsync(hist, 0, ((size_t)LC_HBINS + 1) * 4, st));
            count_hist_kernel<<<JoinAggPipeline::grid_rows(at->nrows), 256, 0, st>>>(fa, at->nrows, d_counts.as<unsigned>(), hist, hist + LC_HBINS,
                                                                                     hist + LC_HBINS + 1, (unsigned)big_cap);
            PG_CUDA(cudaGetLastError());
            res->stats.kernel_launches += 1;
            std::vector<unsigned> h((size_t)LC_HBINS + 1);
            PG_CUDA(cudaMemcpyAsync(h.data(), hist, h.size() * 4, cudaMemcpyDeviceToHost, st));
            PG_CUDA(cudaMemcpyAsync(h_cnt, cnt, 32, cudaMemcpyDeviceToHost, st));
            PG_CUDA(cudaEventRecord(ev_all.b, st));
            PG_CUDA(cudaStreamSynchronize(st));
            const u64 nbig = h[LC_HBINS];
            if (nbig > (u64)big_cap) PG_FAIL(PG_ECUDA, "internal: more large counts than counted rows allow");
            std::vector<unsigned> big((size_t)nbig);
            if (nbig) {
                PG_CUDA(cudaMemcpyAsync(big.data(), hist + LC_HBINS + 1, (size_t)nbig * 4, cudaMemcpyDeviceToHost, st));
                PG_CUDA(cudaStreamSynchronize(st));
                std::sort(big.begin(), big.end());
            }
            tr.mark("count_hist_kernel + d2h");
            // (c_count, custdist): the distinct values of the inner count and how many groups have each
            std::vector<std::pair<u64, u64>> dist;
            auto add = [&](u64 v, u64 n) {
                if (!n) return;
                if (!dist.empty() && dist.back().first == v) dist.back().second += n;
                else dist.push_back({v, n});
            };
            for (int b = 0; b < LC_HBINS; b++) add(count_value((u64)b), h[(size_t)b]);
            for (unsigned v : big) add(v, 1);
            res->nrows = (i64)dist.size();
            kcol.type = ccol.type = PG_T_HUGEINT;
            for (auto &d : dist) {
                const size_t i = kcol.data.size() / sizeof(pg_hugeint);
                if (d.first == 0) kcol.push_null(i, sizeof(pg_hugeint));
                else { kcol.push(pg_hugeint{d.first, 0}); kcol.mark_valid(); }
                ccol.push(pg_hugeint{d.second, 0});
            }
        } else {
            if (d_out_key.bytes < (size_t)D * 8) { PG_TRY(d_out_key.alloc((size_t)D * 8)); PG_TRY(d_out_cnt.alloc((size_t)D * 4)); }
            left_compact_kernel<<<JoinAggPipeline::grid_rows(at->nrows), 256, 0, st>>>(fa, at->nrows, typed(at, anchor_col), d_counts.as<unsigned>(),
                                                                                       d_out_key.as<i64>(), d_out_cnt.as<unsigned>(), cnt + 2);
            PG_CUDA(cudaGetLastError());
            res->stats.kernel_launches += 1;
            PG_CUDA(cudaMemcpyAsync(h_cnt, cnt, 32, cudaMemcpyDeviceToHost, st));
            PG_CUDA(cudaStreamSynchronize(st));
            const i64 n = (i64)h_cnt[2];
            std::vector<i64> keys((size_t)n);
            std::vector<unsigned> counts((size_t)n);
            if (n) {
                PG_CUDA(cudaMemcpyAsync(keys.data(), d_out_key.p, (size_t)n * 8, cudaMemcpyDeviceToHost, st));
                PG_CUDA(cudaMemcpyAsync(counts.data(), d_out_cnt.p, (size_t)n * 4, cudaMemcpyDeviceToHost, st));
            }
            PG_CUDA(cudaEventRecord(ev_all.b, st));
            PG_CUDA(cudaStreamSynchronize(st));
            tr.mark("left_compact_kernel + d2h");
            res->nrows = n;
            kcol.type = at->cols[(size_t)anchor_col].type;
            const size_t w = (size_t)type_size(kcol.type);
            kcol.data.resize((size_t)n * w);
            ccol.type = PG_T_HUGEINT;
            ccol.data.resize((size_t)n * sizeof(pg_hugeint));
            pg_hugeint *cv = (pg_hugeint *)ccol.data.data();
            for (i64 i = 0; i < n; i++) {
                if (w == 4) ((int32_t *)kcol.data.data())[i] = (int32_t)keys[(size_t)i];
                else ((i64 *)kcol.data.data())[i] = keys[(size_t)i];
                const u64 v = count_value(counts[(size_t)i]);
                cv[i].lower = v;
                cv[i].upper = 0;
                if (v == 0) {
                    if (ccol.valid.empty()) ccol.valid.assign((size_t)n, 1);
                    ccol.valid[(size_t)i] = 0;
                }
            }
        }
        for (auto &o : outs) res->cols.push_back(o.first == 0 ? kcol : ccol);
        res->stats.aux[0] = (i64)h_cnt[0];
        res->stats.aux[1] = (i64)h_cnt[1];
        res->stats.aux[6] = res->nrows;
        res->stats.rows_scanned = bt->nrows;
        res->stats.kernel_ms = ev_all.ms();
        res->stats.main_kernel_ms = ev_main.ms();
        res->stats.algorithmic_bytes = algorithmic_bytes;
        res->stats.main_kernel_bytes = main_bytes;
        tr.mark("result columns");
        return PG_OK;
    }
};

}  // namespace

// Agg(k; count) <- LeftJoin, optionally under Agg(count; count(*)): `root` is the topmost aggregate.  Tried only where the
// other join-aggregate pipelines refuse; every refusal is PG_EUNSUPPORTED with its reason.
int build_left_count(pg_plan *plan, const Node &root, std::unique_ptr<Pipeline> *out)
{
    std::unique_ptr<LeftCountPipeline> p(new LeftCountPipeline());
    p->jp.plan = plan;
    const Node *inner = &root, *x = &root.children[0];
    bool filtered = false;
    while (x->op == PG_OP_FILTER) { filtered = true; x = &x->children[0]; }
    if (x->op == PG_OP_AGG) {
        if (filtered) PG_FAIL(PG_EUNSUPPORTED, "a filter between the two aggregates (HAVING on the inner one)");
        p->outer = true;
        inner = x;
        x = &inner->children[0];
        while (x->op == PG_OP_FILTER) { filtered = true; x = &x->children[0]; }
        if (root.having.size()) PG_FAIL(PG_EUNSUPPORTED, "HAVING on the outer aggregate");
    }
    if (inner->having.size()) PG_FAIL(PG_EUNSUPPORTED, "HAVING on the per-group count");
    if (x->op != PG_OP_JOIN) PG_FAIL(PG_EUNSUPPORTED, p->outer ? "an aggregate over an aggregate whose input is not a join" : "the aggregate's input is not a join");
    if (filtered) PG_FAIL(PG_EUNSUPPORTED, "a filter between the aggregate and the join");
    const Node &J = *x;
    if (J.jointype != PG_JOIN_LEFT) PG_FAIL(PG_EUNSUPPORTED, "the join is not a LEFT join");
    if (J.conds.size() != 1) PG_FAIL(PG_EUNSUPPORTED, "the join key has more than one column");
    if (ctx().world > 1) PG_FAIL(PG_EUNSUPPORTED, "runs on one GPU (a preserved row's matches span ranks; per-rank counts are not merged)");
    const Node *ps = &J.children[0], *bs = &J.children[1];
    std::vector<Expr> bf;
    while (ps->op == PG_OP_FILTER) ps = &ps->children[0];
    while (bs->op == PG_OP_FILTER) { for (auto &f : bs->filters) bf.push_back(f); bs = &bs->children[0]; }
    if (ps->op != PG_OP_SCAN) PG_FAIL(PG_EUNSUPPORTED, "the preserved side is not a scan");
    if (bs->op != PG_OP_SCAN) PG_FAIL(PG_EUNSUPPORTED, "the build side is not a scan");
    const Expr *pe = strip_value_preserving_casts(&J.conds[0].first), *be = strip_value_preserving_casts(&J.conds[0].second);
    BaseCol pk, bk;
    if (pe->kind != PG_TK_COL || be->kind != PG_TK_COL || !resolve(J.children[0], pe->idx, &pk) || !resolve(J.children[1], be->idx, &bk) ||
        pk.slot != ps->slot || bk.slot != bs->slot)
        PG_FAIL(PG_EUNSUPPORTED, "join condition is not column = column");
    const pg_table *at = p->jp.tab(pk.slot), *bt = p->jp.tab(bk.slot);
    const Column &ac = at->cols[(size_t)pk.col];
    if (ac.type != PG_T_INT32 && ac.type != PG_T_INT64) PG_FAIL(PG_EUNSUPPORTED, "the anchor key %s is not an integer column", ac.name.c_str());
    if (ac.any_nulls()) PG_FAIL(PG_EUNSUPPORTED, "the anchor key %s is nullable", ac.name.c_str());
    if (!is_int_family(bt->cols[(size_t)bk.col].type)) PG_FAIL(PG_EUNSUPPORTED, "the build side's join key is not an integer column");
    // the inner aggregate: group by the anchor, one count
    const Expr *ge = inner->groups.size() == 1 ? strip_value_preserving_casts(&inner->groups[0]) : nullptr;
    BaseCol gk;
    if (!ge || ge->kind != PG_TK_COL || ge->idx < 0 || ge->idx >= (int)J.outs.size() || J.outs[(size_t)ge->idx].first != 0 || !resolve(J, ge->idx, &gk) ||
        gk.slot != pk.slot || gk.col != pk.col)
        PG_FAIL(PG_EUNSUPPORTED, "the group key is not the anchor (the preserved side's join key) alone");
    if (inner->aggs.size() != 1 || inner->aggs[0].fn != PG_AGG_COUNT || inner->aggs[0].ltype != PG_LT_HUGEINT)
        PG_FAIL(PG_EUNSUPPORTED, "the per-group aggregate is not exactly one count");
    if (!inner->aggs[0].star) {
        const Expr *ae = strip_value_preserving_casts(&inner->aggs[0].arg);
        BaseCol ak;
        if (ae->kind != PG_TK_COL || ae->idx < 0 || ae->idx >= (int)J.outs.size() || !resolve(J, ae->idx, &ak))
            PG_FAIL(PG_EUNSUPPORTED, "the count argument is not a column");
        if (J.outs[(size_t)ae->idx].first == 1) {
            p->arg_col = ak.col;
            p->null_if_empty = true;
        } else if (at->cols[(size_t)ak.col].any_nulls()) {
            PG_FAIL(PG_EUNSUPPORTED, "count over a nullable preserved-side column");
        }
    }
    for (auto &o : inner->outs)
        if (o != std::make_pair(0, 0) && o != std::make_pair(1, 0)) PG_FAIL(PG_EUNSUPPORTED, "bad output of the per-group aggregate");
    p->outs = inner->outs;
    if (p->outer) {
        const Expr *oe = root.groups.size() == 1 ? strip_value_preserving_casts(&root.groups[0]) : nullptr;
        if (!oe || oe->kind != PG_TK_COL || oe->idx < 0 || oe->idx >= (int)inner->outs.size() || inner->outs[(size_t)oe->idx] != std::make_pair(1, 0))
            PG_FAIL(PG_EUNSUPPORTED, "the outer aggregate is not grouped by the per-group count alone");
        if (root.aggs.size() != 1 || root.aggs[0].fn != PG_AGG_COUNT || !root.aggs[0].star || root.aggs[0].ltype != PG_LT_HUGEINT)
            PG_FAIL(PG_EUNSUPPORTED, "the outer aggregate is not count(*)");
        for (auto &o : root.outs)
            if (o != std::make_pair(0, 0) && o != std::make_pair(1, 0)) PG_FAIL(PG_EUNSUPPORTED, "bad output of the outer aggregate");
        p->outs = root.outs;
    }
    if (bt->nrows >= ((i64)1 << 32)) PG_FAIL(PG_EUNSUPPORTED, "the build side has 2^32 rows or more (the per-row counts are 32-bit)");
    if (at->nrows >= ((i64)1 << 32)) PG_FAIL(PG_EUNSUPPORTED, "the preserved side has 2^32 rows or more");
    {
        LowerCtx cx;
        cx.table = bt;
        cx.allow_nulls = true;
        std::vector<Expr> fl = bs->filters;
        for (auto &f : bf) fl.push_back(f);
        if (!lower_filters(cx, fl, p->build_ranges)) PG_FAIL(PG_EUNSUPPORTED, "build-side filter not off-loadable: %s", cx.why.c_str());
    }
    int stage = -1;
    PG_TRY(add_build_stage(&p->jp, J.children[0], pe->idx, &stage));
    p->jp.stages[(size_t)stage]->payload_needed = true;
    p->anchor_col = pk.col;
    p->build_slot = bk.slot;
    p->build_key_col = bk.col;
    p->big_cap = bt->nrows / LC_HBINS + 1;
    std::vector<std::string> likes;
    PG_TRY(p->fill(p->fa, p->jp.stages[(size_t)stage]->ranges, pk.slot, nullptr));
    PG_TRY(p->fill(p->fb, p->build_ranges, bk.slot, &likes));
    PG_TRY(p->jp.d_counters.alloc(128));
    // the pass reads the build side's key, count argument, predicate columns and string bytes + offsets once
    auto colbytes = [&](const pg_table *t, int col) -> i64 {
        const Column &cc = t->cols[(size_t)col];
        if (cc.type == PG_T_VARCHAR) return (i64)cc.h_bytes.size() + (t->nrows + 1) * 8;
        return t->nrows * cc.phys_width();
    };
    std::vector<int> read{bk.col};
    if (p->arg_col >= 0) read.push_back(p->arg_col);
    for (auto &r : p->build_ranges) read.push_back(r.col);
    std::sort(read.begin(), read.end());
    read.erase(std::unique(read.begin(), read.end()), read.end());
    for (int col : read) p->main_bytes += colbytes(bt, col);
    p->algorithmic_bytes = p->main_bytes + colbytes(at, pk.col);
    std::string pass;
    if (!p->fb.npred && likes.empty()) pass = " every row";
    if (p->fb.npred) pass += " ranges=" + std::to_string(p->fb.npred);
    for (size_t i = 0; i < likes.size(); i++) pass += (i ? "," : " like=") + likes[i];
    p->explain = "left-join count: groups=rows of " + at->name + "; " + bt->name + " pass" + pass + "; kernel=left_count_kernel+" +
                 (p->outer ? "count_hist_kernel" : "left_compact_kernel");
    *out = std::move(p);
    return PG_OK;
}

}  // namespace pg
