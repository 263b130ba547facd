// join.cuh -- hash join build / probe and high-cardinality group-by kernels (sm_100a).
//
// Reference code replaced:
//   JoinHashTable.Build / Finalize / InsertHashesLoop   pkg/compute/join_table.go:85-288
//     (chained table: bucket heads of nextpow2(2n) pointers, next pointer inside the row)
//   Scan.Next / InnerJoin / resolvePredicates / Match    pkg/compute/join_scan.go:182-299
//   GroupedAggrHashTable.FindOrCreateGroups + UpdateStates  pkg/compute/aggregate_hash.go:201-391,
//                                                          aggregate_exec.go:456
//
// Design for B200 (HBM-bound, random-sector-bound on the table):
//   * BUCKETIZED open addressing: a bucket is one 64-byte line of 8 keys (2 sectors) plus a
//     parallel 64-byte line of 8 payloads read only on a match; duplicates occupy further
//     slots of the probe sequence, an empty slot ends it (no deletes).  Payload = row id of
//     the build-side source row: columns are gathered late, only for matches.
//   * an exact key-domain BITMAP (1 bit per key in [kmin,kmax] of the build column
//     statistics) screens probes before the table is touched.  For dense keys it is a few
//     MB, L2-resident, and TPC-H fact tables are clustered on their join keys so
//     consecutive probes hit the same sectors.
//   * group-by on high-cardinality keys: global open-addressing table in HBM, 64-bit CAS
//     on the key words, 64-bit atomic adds on the accumulators (red.global.add.u64).
#pragma once
#include "common.cuh"
#include "scanagg.cuh"

namespace pg {

constexpr i64 HT_EMPTY = (i64)0x8080808080808080ULL;   // memset(0x80) pattern
constexpr int HT_BUCKET = 4;      // slots per 64-byte bucket line: {key, payload} pairs

__host__ __device__ __forceinline__ u64 mix64(u64 x)
{
    x ^= x >> 33; x *= 0xff51afd7ed558ccdULL; x ^= x >> 33; x *= 0xc4ceb9fe1a85ec53ULL; x ^= x >> 33;
    return x;
}

struct JoinTable {
    longlong2 *slots;   // [nbuckets][4] of {x = key, y = payload}: key and payload share a 32-byte sector,
                        // so an insert or a matching probe touches ONE random sector, not two
    u64 bucket_mask;    // nbuckets - 1 (power of two)
    unsigned *bitmap;   // may be null
    i64 bm_min, bm_max; // key domain covered by the bitmap
    unsigned long long *dups;   // number of inserted keys that were already present (bitmap builds only)
    // Bucket choice: mix64 hash by default; for a build key that ascends in row order (statistics) an
    // ORDER-PRESERVING map of the key domain onto the buckets, so the build writes the table like a
    // stream and a probe side clustered on the same key (TPC-H fact tables) reads it like one.
    int order_preserving;
    int log2buckets;
    u64 domain;                 // bm_max - bm_min + 1
    // RANK INDEX (unique build keys + bitmap): no slots at all.  The r-th set bit of the bitmap owns
    // rank_payload[r]; rank = rank_prefix[256-bit block] + popcount inside the block, and a block is one
    // 32-byte sector, so a lookup is branch-free: bitmap sector + prefix word -> payload word.
    const unsigned *rank_prefix;
    const unsigned *rank_payload;
    int rank_identity;          // every row of a strictly ascending key column was inserted: rank == build row id, no payload array
};

// rank of key offset `off` (its bit must be set): number of set bits before it
__device__ __forceinline__ unsigned jt_rank(const JoinTable &t, u64 off, bool *set)
{
    const uint4 *blk = (const uint4 *)(t.bitmap + ((off >> 8) << 3));
    const uint4 a = __ldg(blk), b = __ldg(blk + 1);
    const unsigned base = __ldg(t.rank_prefix + (off >> 8));
    const unsigned w[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
    const unsigned wi = (unsigned)(off >> 5) & 7u, bit = (unsigned)off & 31u;
    unsigned r = base, word = 0;
#pragma unroll
    for (unsigned i = 0; i < 8; i++) {
        r += i < wi ? __popc(w[i]) : 0;
        word = i == wi ? w[i] : word;
    }
    *set = (word >> bit) & 1u;
    return r + __popc(word & ((1u << bit) - 1u));
}
__device__ __forceinline__ u64 jt_home(const JoinTable &t, i64 key)
{
    if (t.order_preserving) {
        u64 off = (u64)(key - t.bm_min);
        return off < t.domain ? (off << t.log2buckets) / t.domain : (mix64((u64)key) & t.bucket_mask);
    }
    return mix64((u64)key) & t.bucket_mask;
}

__device__ __forceinline__ bool bitmap_test(const JoinTable &t, i64 key)
{
    u64 off = (u64)key - (u64)t.bm_min;          // one unsigned compare covers both ends of the domain
    if (off >= t.domain) return false;
    return (__ldg(t.bitmap + (off >> 5)) >> (off & 31)) & 1u;
}

__device__ __forceinline__ void jt_insert(const JoinTable &t, i64 key, u64 payload)
{
    if (t.bitmap) {
        u64 off = (u64)(key - t.bm_min);
        unsigned bit = 1u << (off & 31);
        if (atomicOr(t.bitmap + (off >> 5), bit) & bit) atomicAdd(t.dups, 1ULL);
    }
    u64 b = jt_home(t, key);
    for (;;) {
        longlong2 *line = t.slots + b * HT_BUCKET;
#pragma unroll
        for (int s = 0; s < HT_BUCKET; s++) {
            if (line[s].x == HT_EMPTY) {
                i64 old = (i64)atomicCAS((unsigned long long *)&line[s].x, (unsigned long long)HT_EMPTY, (unsigned long long)key);
                if (old == HT_EMPTY) { line[s].y = (i64)payload; return; }
            }
        }
        b = (b + 1) & t.bucket_mask;
    }
}

// calls f(payload) for every build row with this key (INNER join emits every pair)
template <typename F>
__device__ __forceinline__ void jt_probe(const JoinTable &t, i64 key, F f)
{
    if (t.rank_prefix) {
        const u64 off = (u64)key - (u64)t.bm_min;
        if (off >= t.domain) return;
        bool set;
        const unsigned r = jt_rank(t, off, &set);
        if (set) f(t.rank_identity ? (u64)r : (u64)__ldg(t.rank_payload + r));
        return;
    }
    u64 b = jt_home(t, key);
    for (;;) {
        const longlong2 *line = t.slots + b * HT_BUCKET;
        longlong2 s0 = __ldg(line), s1 = __ldg(line + 1), s2 = __ldg(line + 2), s3 = __ldg(line + 3);
        if (s0.x == key) f((u64)s0.y);
        if (s1.x == key) f((u64)s1.y);
        if (s2.x == key) f((u64)s2.y);
        if (s3.x == key) f((u64)s3.y);
        if (s0.x == HT_EMPTY || s1.x == HT_EMPTY || s2.x == HT_EMPTY || s3.x == HT_EMPTY) return;
        b = (b + 1) & t.bucket_mask;
    }
}

// a column of a base table in its physical encoding (NCol: logical = base + stored), plus validity
struct TypedCol {
    const void *p;
    int width;             // stored bytes per value: 1, 2, 4 or 8
    i64 base;
    const uint8_t *valid;  // packed validity (1 = not NULL) or null when the column holds no NULLs
};
__device__ __forceinline__ bool typed_valid(const TypedCol &c, i64 row)
{
    return c.valid == nullptr || ((__ldg(c.valid + (row >> 3)) >> (row & 7)) & 1);
}
// LOGICAL value of one row (gathers by row id)
__device__ __forceinline__ i64 load_typed(const TypedCol &c, i64 row)
{
    switch (c.width) {
    case 8: return __ldg((const i64 *)c.p + row);
    case 4: return (i64)__ldg((const int *)c.p + row) + c.base;
    case 2: return (i64)__ldg((const unsigned short *)c.p + row) + c.base;
    default: return (i64)__ldg((const uint8_t *)c.p + row) + c.base;
    }
}
// streaming access to 4 consecutive rows (row a multiple of 4): raw vector load now, LOGICAL values on unpack
__device__ __forceinline__ NCol typed_ncol(const TypedCol &c)
{
    NCol n;
    n.p = c.p; n.pw = c.width; n.pad_ = 0; n.base = c.base;
    return n;
}
__device__ __forceinline__ void ld_typed4(const TypedCol &c, i64 row, Raw4<true> &r) { ld_raw4(typed_ncol(c), row, r); }
__device__ __forceinline__ void unpack_typed4(const TypedCol &c, const Raw4<true> &r, i64 (&v)[4])
{
    unpack4(typed_ncol(c), r, v);
    if (c.width != 8) { v[0] += c.base; v[1] += c.base; v[2] += c.base; v[3] += c.base; }
}
__device__ __forceinline__ void load_typed4(const TypedCol &c, i64 row, i64 (&v)[4])
{
    Raw4<true> r;
    ld_typed4(c, row, r);
    unpack_typed4(c, r, v);
}

struct SrcPred {          // inclusive range on a source column, or (byte-coded columns) a set of codes: IN, <>, OR of =
    TypedCol col;
    i64 lo, hi;
    int is_set;
    unsigned mask[8];
};
__device__ __forceinline__ bool pred_pass(const SrcPred &q, i64 row)
{
    if (!typed_valid(q.col, row)) return false;                 // NULL is never selected
    const i64 v = load_typed(q.col, row);
    return q.is_set ? ((q.mask[(v >> 5) & 7] >> (v & 31)) & 1u) != 0 : (v >= q.lo && v <= q.hi);
}

constexpr int PIPE_MAXPRED = 3;

// A further existence test on a source row besides the pipeline's main probe (a SEMI / ANTI join pushed
// down to the scan that owns its key, or an INNER join against unique keys whose columns are fetched
// late): the exact key bitmap of the probed build side decides.
constexpr int PIPE_MAXEXTRA = 2;
struct ExtraProbe {
    TypedCol key;
    const unsigned *bitmap;
    i64 bm_min;
    u64 domain;
    int anti;              // 1: keep the row when the key is ABSENT (a NULL key is absent)
};

// ---------------------------------------------------------------- pipelines --
// One kernel family: stream a source table, apply range predicates, optionally probe one
// join table with a source key column, and feed a sink:
//   SINK_COUNT   count surviving (joined) rows            -> sizing pass
//   SINK_INSERT  insert (key column, source row id) into a join table  -> build side
//   SINK_GROUP   update the global group table            -> aggregate over the join
enum { SINK_COUNT = 0, SINK_INSERT = 1, SINK_GROUP = 2, SINK_BITMAP = 3 };   // BITMAP: set the key bit only (unique, payload-free build side)

constexpr int GT_MAXACC = 4;
constexpr int GT_MAXKEYPARTS = 3;

// Slots are records {klo, khi, acc[0..nacc-1], count} padded to `rw` = 4 or 8 words, so one group
// update touches ONE 32-byte sector (64 bytes for more than one sum) instead of one sector per
// field.  The whole table is initialised with memset(0x80): key words read HT_EMPTY when free and
// every accumulator starts at HT_EMPTY, which compaction subtracts again (64-bit wrap-around
// arithmetic keeps the sums exact).
struct GroupTable {
    i64 *slots;           // [cap][rw]
    u64 mask;             // cap - 1
    int nacc;
    int rw;               // words per slot (4 or 8)
    int *overflow;        // set when a probe sequence exceeds the limit (table too small)
    // Slot choice.  Default: mix64 hash.  For keys that are CLUSTERED in row order (statistics:
    // most rows repeat their neighbour's key, e.g. l_orderkey) an ORDER-PRESERVING map of the key
    // domain onto the table is used instead: consecutive rows then touch consecutive slots, so the
    // table is written like a stream rather than at random DRAM pages (measured 36 -> ~ms class).
    int two_words;        // keys use both words (more than one key column)
    int order_preserving;
    i64 kmin;
    u64 domain;           // kmax - kmin + 1  (<= 2^34 when order_preserving)
    int log2cap;
};
__device__ __forceinline__ u64 gt_home(const GroupTable &g, i64 klo, i64 khi)
{
    if (g.order_preserving) return (((u64)(klo - g.kmin)) << g.log2cap) / g.domain;
    return mix64((u64)klo * 0x9E3779B97F4A7C15ULL ^ (u64)khi) & g.mask;
}
__host__ __device__ __forceinline__ int gt_slot_words(int nacc) { return nacc <= 1 ? 4 : 8; }

// where a value comes from: the streamed source row or the matched build row
struct ValRef {
    TypedCol col;
    int from_build;       // 0: column at the source row, 1: column at the matched build row (late gather),
                          // 2: the matched build row id itself (group keys functionally dependent on a
                          //    unique build key are fetched once per GROUP after the aggregation)
};

struct GroupSpec {
    // key = up to 3 parts: part 0 -> klo; parts 1,2 -> khi = (p1 << 32) | (p2 & 0xffffffff)
    int nparts;
    ValRef part[GT_MAXKEYPARTS];
    int run_aggregate;   // group keys are clustered in row order: combine runs of equal keys across adjacent
                         // lanes (segmented warp scan) and issue ONE table update per run
    // accumulator a = product over its factors of (c + s * value)
    int nacc;
    int nfac[GT_MAXACC];
    ValRef fac[GT_MAXACC][3];
    i64 fc[GT_MAXACC][3];
    int fs[GT_MAXACC][3];
};

struct PipeParams {
    i64 nrows;
    int npred;
    SrcPred pred[PIPE_MAXPRED];
    int has_probe;
    int probe_mode;          // 0 INNER: every match reaches the sink; 1 SEMI: the row once if any match;
                             // 2 ANTI: the row once if no match (join_scan.go:90-165 NextSemiOrAntiJoin)
    int probe_bitmap_only;   // the exact key bitmap decides alone: unique payload-free INNER build side, or SEMI/ANTI
    TypedCol probe_key;
    JoinTable probe;
    // SINK_INSERT
    TypedCol ins_key;
    TypedCol ins_key2;       // p != null: two-column key, (k << 32) | (k2 & 0xffffffff)
    JoinTable ins;
    // string predicates on VARCHAR columns of the source (build side `p_name like '%pink%'`)
    int nlike;
    GenLike like[GEN_MAXLIKE];
    // SINK_GROUP
    GroupTable gt;
    GroupSpec gs;
    // SINK_COUNT / statistics: [0] rows passing the predicates, [1] joined rows
    unsigned long long *counters;
    int nextra;
    ExtraProbe extra[PIPE_MAXEXTRA];
    // two-phase execution (filter_hits_kernel -> hits_sink_kernel): rows [row_begin, row_end) of the source
    // are screened, the row ids of the hits are appended to `hits` (capacity >= row_end - row_begin),
    // `hit_count` is the device-side cursor
    i64 row_begin, row_end;
    // pipeline_kernel over a slice of the source: rows [pipe_lo, pipe_hi) when pipe_hi > 0 (a REPLICATED build side whose
    // scan is divided among the ranks and whose key bitmaps are OR-merged afterwards), else every row
    i64 pipe_lo, pipe_hi;
    unsigned *hits;
    unsigned long long *hit_count;
};

__device__ __forceinline__ bool extras_pass(const PipeParams &p, i64 row)
{
    for (int e = 0; e < p.nextra; e++) {
        const ExtraProbe &x = p.extra[e];
        bool found = false;
        if (typed_valid(x.key, row)) {
            const u64 off = (u64)load_typed(x.key, row) - (u64)x.bm_min;
            if (off < x.domain) found = (__ldg(x.bitmap + (off >> 5)) >> (off & 31)) & 1u;
        }
        if (found == (x.anti != 0)) return false;
    }
    return true;
}

// add `vals` (nacc sums) and `count` rows to group (klo, khi); claims a free slot with 64-bit CAS
__device__ __forceinline__ void gt_add(const GroupTable &g, i64 klo, i64 khi, const i64 *vals, i64 count)
{
    u64 i = gt_home(g, klo, khi);
    for (u64 n = 0; n <= g.mask && n <= 4096; n++) {
        i64 *slot = g.slots + i * (u64)g.rw;
        i64 cur = slot[0];
        if (cur == HT_EMPTY) cur = (i64)atomicCAS((unsigned long long *)&slot[0], (unsigned long long)HT_EMPTY, (unsigned long long)klo);
        if (cur == HT_EMPTY || cur == klo) {
            i64 h = khi;
            if (g.two_words) {      // single-column keys never touch the second key word
                h = slot[1];
                if (h == HT_EMPTY) h = (i64)atomicCAS((unsigned long long *)&slot[1], (unsigned long long)HT_EMPTY, (unsigned long long)khi);
            }
            if (h == HT_EMPTY || h == khi) {
                for (int a = 0; a < g.nacc; a++) atomicAdd((unsigned long long *)&slot[2 + a], (unsigned long long)vals[a]);
                atomicAdd((unsigned long long *)&slot[2 + g.nacc], (unsigned long long)count);
                return;
            }
        }
        i = (i + 1) & g.mask;
    }
    *g.overflow = 1;
}
__device__ __forceinline__ void gt_update(const GroupTable &g, i64 klo, i64 khi, const i64 *vals) { gt_add(g, klo, khi, vals, 1); }

// Segmented inclusive sum over the warp: lanes with equal (klo, khi) that are ADJACENT form a run;
// the last lane of a run ends up with the run's totals and performs the single table update.
// All 32 lanes must call it; `valid` = this lane has a row.
__device__ __forceinline__ void gt_update_runs(const GroupTable &g, bool valid, i64 klo, i64 khi, i64 *vals)
{
    const unsigned full = 0xffffffffu;
    const int lane = threadIdx.x & 31;
    i64 pk = __shfl_up_sync(full, klo, 1), ph = __shfl_up_sync(full, khi, 1);
    int pv = __shfl_up_sync(full, (int)valid, 1);
    int head = lane == 0 || !valid || !pv || pk != klo || ph != khi;
    int nhead = __shfl_down_sync(full, head, 1);
    bool tail = lane == 31 || nhead;
    i64 cnt = valid ? 1 : 0;
    int f = head;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        int fu = __shfl_up_sync(full, f, o);
        i64 cu = __shfl_up_sync(full, cnt, o);
        i64 vu[GT_MAXACC];
        for (int a = 0; a < g.nacc; a++) vu[a] = __shfl_up_sync(full, vals[a], o);
        if (lane >= o && !f) {
            cnt += cu;
            for (int a = 0; a < g.nacc; a++) vals[a] += vu[a];
            f |= fu;
        }
    }
    if (valid && tail) gt_add(g, klo, khi, vals, cnt);
}

template <int SINK>
__global__ void __launch_bounds__(256)
pipeline_kernel(const PipeParams p)
{
    unsigned long long n_pass = 0, n_join = 0;
    const i64 row_lo = p.pipe_hi > 0 ? p.pipe_lo : 0, row_hi = p.pipe_hi > 0 ? p.pipe_hi : p.nrows;
    for (i64 row = row_lo + (i64)blockIdx.x * blockDim.x + threadIdx.x; row < row_hi; row += (i64)gridDim.x * blockDim.x) {
        bool ok = true;
        for (int k = 0; k < p.npred && ok; k++) {
            ok = pred_pass(p.pred[k], row);
        }
        for (int k = 0; k < p.nlike && ok; k++) ok = gen_like_pass(p.like[k], row);
        if (!ok) continue;
        n_pass++;
        if (p.nextra && !extras_pass(p, row)) continue;
        auto sink = [&](u64 build_row) {
            if ((SINK == SINK_INSERT || SINK == SINK_BITMAP) && !typed_valid(p.ins_key, row)) return;   // NULL keys are not built (join_table.go:152-195)
            n_join++;
            if (SINK == SINK_INSERT) {
                i64 key = load_typed(p.ins_key, row);
                if (p.ins_key2.p) key = (key << 32) | (load_typed(p.ins_key2, row) & 0xffffffffLL);
                jt_insert(p.ins, key, (u64)row);
            } else if (SINK == SINK_BITMAP) {
                u64 off = (u64)(load_typed(p.ins_key, row) - p.ins.bm_min);
                atomicOr(p.ins.bitmap + (off >> 5), 1u << (off & 31));
            } else if (SINK == SINK_GROUP) {
                auto val = [&](const ValRef &r) { return r.from_build == 2 ? (i64)build_row : load_typed(r.col, r.from_build ? (i64)build_row : row); };
                i64 klo = val(p.gs.part[0]);
                i64 khi = 0;
                if (p.gs.nparts > 1) khi = val(p.gs.part[1]) << 32;
                if (p.gs.nparts > 2) khi |= val(p.gs.part[2]) & 0xffffffffLL;
                i64 vals[GT_MAXACC];
                for (int a = 0; a < p.gs.nacc; a++) {
                    i64 x = 1;
                    for (int f = 0; f < p.gs.nfac[a]; f++) x *= p.gs.fc[a][f] + p.gs.fs[a][f] * val(p.gs.fac[a][f]);
                    vals[a] = x;
                }
                gt_update(p.gt, klo, khi, vals);
            }
        };
        if (p.has_probe) {
            i64 key = load_typed(p.probe_key, row);
            if (!typed_valid(p.probe_key, row)) {      // a NULL key matches nothing: only ANTI keeps the row
                if (p.probe_mode == 2) sink(0);
                continue;
            }
            if (p.probe_mode == 0) {
                if (p.probe.bitmap && !bitmap_test(p.probe, key)) continue;
                if (p.probe_bitmap_only) sink(0);
                else jt_probe(p.probe, key, sink);
            } else {
                bool found;
                if (p.probe.bitmap) found = bitmap_test(p.probe, key);       // exact existence
                else { found = false; jt_probe(p.probe, key, [&](u64) { found = true; }); }
                if (found == (p.probe_mode == 1)) sink(0);
            }
        } else {
            sink(0);
        }
    }
    // block-aggregate the two counters
    n_pass = (unsigned long long)warp_sum((i64)n_pass);
    n_join = (unsigned long long)warp_sum((i64)n_join);
    if ((threadIdx.x & 31) == 0) {
        if (n_pass) atomicAdd(&p.counters[0], n_pass);
        if (n_join) atomicAdd(&p.counters[1], n_join);
    }
}

// Group-by straight over a table (no probe): warp-converged loop so that runs of equal keys in
// adjacent lanes can be combined before they reach the table.
__global__ void __launch_bounds__(256)
static scan_group_kernel(const PipeParams p)
{
    unsigned long long n_pass = 0;
    const i64 stride = (i64)gridDim.x * blockDim.x;
    const i64 nround = (p.nrows + stride - 1) / stride;     // same trip count for every thread
    for (i64 it = 0; it < nround; it++) {
        i64 row = it * stride + (i64)blockIdx.x * blockDim.x + threadIdx.x;
        bool ok = row < p.nrows;
        for (int k = 0; k < p.npred && ok; k++) {
            ok = pred_pass(p.pred[k], row);
        }
        i64 klo = 0, khi = 0, vals[GT_MAXACC];
        if (ok) {
            n_pass++;
            klo = load_typed(p.gs.part[0].col, row);
            if (p.gs.nparts > 1) khi = load_typed(p.gs.part[1].col, row) << 32;
            if (p.gs.nparts > 2) khi |= load_typed(p.gs.part[2].col, row) & 0xffffffffLL;
            for (int a = 0; a < p.gs.nacc; a++) {
                i64 x = 1;
                for (int f = 0; f < p.gs.nfac[a]; f++) x *= p.gs.fc[a][f] + p.gs.fs[a][f] * load_typed(p.gs.fac[a][f].col, row);
                vals[a] = x;
            }
        }
        if (p.gs.run_aggregate) gt_update_runs(p.gt, ok, klo, khi, vals);
        else if (ok) gt_add(p.gt, klo, khi, vals, 1);
    }
    n_pass = (unsigned long long)warp_sum((i64)n_pass);
    if ((threadIdx.x & 31) == 0 && n_pass) {
        atomicAdd(&p.counters[0], n_pass);
        atomicAdd(&p.counters[1], n_pass);
    }
}

// Specialised, vectorised group-by for the dominant high-cardinality shape -- ONE integer key,
// ONE summed column (plus the row count), at most one 32-bit range predicate: e.g. TPC-H Q18's
// `group by l_orderkey having sum(l_quantity) > 314`.  16-byte streaming loads (4 rows per thread),
// runs of equal keys are first combined inside the thread's 4 rows, then one compact table update
// per run.  Everything is compile-time except pointers and constants.
template <bool HAS_PRED>
__global__ void __launch_bounds__(SA_THREADS)
group1_kernel(const PipeParams p)
{
    unsigned long long n_pass = 0;
    const i64 ntiles = (p.nrows + SA_TILE - 1) / SA_TILE;
    const i64 plo = p.pred[0].lo, phi = p.pred[0].hi;
    const TypedCol kc = p.gs.part[0].col, vc = p.gs.fac[0][0].col;
    const i64 fc = p.gs.fc[0][0];
    const int fs = p.gs.fs[0][0];
    for (i64 tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
        i64 row = tile * SA_TILE + threadIdx.x * SA_VEC;
        i64 rem = p.nrows - row;
        i64 dv[4] = {0, 0, 0, 0}, k[4], v[4];
        Raw4<true> rd, rk, rv;
        if (HAS_PRED) ld_typed4(p.pred[0].col, row, rd);
        ld_typed4(kc, row, rk);
        ld_typed4(vc, row, rv);
        if (HAS_PRED) unpack_typed4(p.pred[0].col, rd, dv);
        unpack_typed4(kc, rk, k);
        unpack_typed4(vc, rv, v);
        // fold the 4 rows into runs of equal keys
        i64 run_key = 0, run_sum = 0, run_cnt = 0;
#pragma unroll
        for (int j = 0; j < 4; j++) {
            bool ok = j < rem;
            if (HAS_PRED) ok = ok && dv[j] >= plo && dv[j] <= phi;
            if (!ok) continue;
            n_pass++;
            i64 x = fc + fs * v[j];
            if (run_cnt > 0 && k[j] == run_key) { run_sum += x; run_cnt++; continue; }
            if (run_cnt > 0) gt_add(p.gt, run_key, 0, &run_sum, run_cnt);
            run_key = k[j]; run_sum = x; run_cnt = 1;
        }
        if (run_cnt > 0) gt_add(p.gt, run_key, 0, &run_sum, run_cnt);
    }
    n_pass = (unsigned long long)warp_sum((i64)n_pass);
    if ((threadIdx.x & 31) == 0 && n_pass) {
        atomicAdd(&p.counters[0], n_pass);
        atomicAdd(&p.counters[1], n_pass);
    }
}

// ---------------------------------------------------------------- dense, L2-blocked group-by --
// High-cardinality group-by over an UNSORTED integer key with a modest domain (l_partkey: 20 M keys at SF100).  The
// global hash table pays a random 64-byte read-modify-write in HBM per row (47 ms for 600 M rows, 0.02 of the roofline).
// Here the accumulators are direct-addressed arrays sum[key - kmin] (8 B) and count[key - kmin] (4 B), and the table
// is scanned once per KEY SLICE whose accumulators (12 B x slice) fit in the 126 MB L2: every row outside the slice
// is skipped after its key is read, so the atomics of a pass stay in L2 and DRAM only sees the streamed columns.
template <bool HAS_PRED>
__global__ void __launch_bounds__(SA_THREADS)
group1_dense_kernel(const PipeParams p, unsigned long long *__restrict__ dsum, unsigned *__restrict__ dcnt, i64 kmin, i64 klo, i64 khi,
                    int count_rows)
{
    unsigned long long n_pass = 0;
    const i64 ntiles = (p.nrows + SA_TILE - 1) / SA_TILE;
    const i64 plo = p.pred[0].lo, phi = p.pred[0].hi;
    const TypedCol kc = p.gs.part[0].col, vc = p.gs.fac[0][0].col;
    const i64 fc = p.gs.fc[0][0];
    const int fs = p.gs.fs[0][0];
    for (i64 tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
        const i64 row = tile * SA_TILE + threadIdx.x * SA_VEC;
        const i64 rem = p.nrows - row;
        i64 dv[4] = {0, 0, 0, 0}, k[4], v[4];
        Raw4<true> rd, rk, rv;
        if (HAS_PRED) ld_typed4(p.pred[0].col, row, rd);
        ld_typed4(kc, row, rk);
        ld_typed4(vc, row, rv);
        if (HAS_PRED) unpack_typed4(p.pred[0].col, rd, dv);
        unpack_typed4(kc, rk, k);
        unpack_typed4(vc, rv, v);
#pragma unroll
        for (int j = 0; j < 4; j++) {
            bool ok = j < rem;
            if (HAS_PRED) ok = ok && dv[j] >= plo && dv[j] <= phi;
            if (!ok) continue;
            n_pass++;
            if (k[j] < klo || k[j] >= khi) continue;
            const u64 g = (u64)(k[j] - kmin);
            atomicAdd(dsum + g, (unsigned long long)(fc + fs * v[j]));
            atomicAdd(dcnt + g, 1u);
        }
    }
    if (count_rows) {
        n_pass = (unsigned long long)warp_sum((i64)n_pass);
        if ((threadIdx.x & 31) == 0 && n_pass) { atomicAdd(&p.counters[0], n_pass); atomicAdd(&p.counters[1], n_pass); }
    }
}

// dense accumulators -> the compacted group list gt_compact_kernel produces ([klo][khi][sum plane][count plane]), HAVING applied
static __global__ void __launch_bounds__(256)
dense_compact_kernel(const unsigned long long *__restrict__ dsum, const unsigned *__restrict__ dcnt, u64 domain, i64 kmin,
                     i64 *__restrict__ out_klo, i64 *__restrict__ out_khi, i64 *__restrict__ out_acc, i64 max_out,
                     unsigned long long *__restrict__ counter, int hav_plane, i64 hav_lo, i64 hav_hi)
{
    const int lane = threadIdx.x & 31;
    for (u64 i0 = ((u64)blockIdx.x * blockDim.x + threadIdx.x) - lane; i0 < domain; i0 += (u64)gridDim.x * blockDim.x) {
        const u64 i = i0 + lane;
        const unsigned c = i < domain ? dcnt[i] : 0u;
        const i64 sum = c ? (i64)dsum[i] : 0;
        bool keep = c != 0, dropped = false;
        if (keep && hav_plane >= 0) {
            const i64 v = hav_plane == 0 ? sum : (i64)c;
            if (v < hav_lo || v > hav_hi) { keep = false; dropped = true; }
        }
        const unsigned m = __ballot_sync(0xffffffffu, keep), md = __ballot_sync(0xffffffffu, dropped);
        unsigned long long base = 0;
        if (lane == 0) {
            if (m) base = atomicAdd(counter, (unsigned long long)__popc(m));
            if (md) atomicAdd(counter + 1, (unsigned long long)__popc(md));
        }
        base = __shfl_sync(0xffffffffu, base, 0);
        if (keep) {
            const unsigned long long o = base + __popc(m & ((1u << lane) - 1u));
            if ((i64)o < max_out) {
                out_klo[o] = (i64)i + kmin;
                out_khi[o] = 0;
                out_acc[o] = sum;
                out_acc[(u64)max_out + o] = (i64)c;
            }
        }
    }
}

// ---------------------------------------------------------------- sorted-run group-by --
// Group-by over a key column that is SORTED in row order (statistics: no strict descent), e.g.
// l_orderkey: every group is one contiguous run of rows, so no table is needed at all.  A fused
// reduce-by-key at scan speed: each WARP owns a contiguous chunk of 128-row tiles and walks it in order
// (no shared memory, no block barrier -- a block-wide variant with three barriers per tile ran at
// 1.9 TB/s); per tile a lane folds its 4 rows into (leading run | complete interior runs | trailing
// run), a warp segmented scan carries open runs across lanes, the warp carries its open run across
// tiles in registers, closed runs pass HAVING and are appended to the output list with one cursor bump
// per warp tile.  Runs that touch a chunk edge go to first[w] / last[w] and are stitched together by
// run_fixup_kernel (a few thousand records).
struct RunOut {
    i64 *klo, *khi, *acc;             // output list, acc = [2 planes][cap]: sum, row count
    i64 cap;
    unsigned long long *count;        // runs emitted (may exceed cap: the caller grows the list and reruns)
    int hav_plane;                    // -1: none, 0: sum, 1: row count
    i64 hav_lo, hav_hi;
};
struct RunEdge { i64 key, sum, cnt; int valid, spans; };

__device__ __forceinline__ bool run_passes(const RunOut &o, i64 sum, i64 cnt)
{
    if (cnt <= 0) return false;                        // every row of the run failed the predicate: no group
    if (o.hav_plane < 0) return true;
    const i64 v = o.hav_plane == 0 ? sum : cnt;
    return v >= o.hav_lo && v <= o.hav_hi;
}

constexpr int RUN_H = 1, RUN_S = 2;                    // segment head | run touches the start of the warp's chunk
constexpr int RUN_WTILE = 32 * SA_VEC;                 // rows per warp tile
// (register double-buffering and prefetch.global.L2 of later tiles were both measured: no gain, the kernel
//  is issue-bound at ~75 % issue utilisation, not latency-bound)

template <bool HAS_PRED>
__global__ void __launch_bounds__(SA_THREADS, 4)
run_group_kernel(const PipeParams p, const RunOut out, RunEdge *__restrict__ first, RunEdge *__restrict__ last, i64 chunk_tiles)
{
    const unsigned full = 0xffffffffu;
    const int lane = threadIdx.x & 31;
    const i64 gw = (i64)blockIdx.x * (SA_THREADS / 32) + (threadIdx.x >> 5);
    const i64 ntiles = (p.nrows + RUN_WTILE - 1) / RUN_WTILE;
    const i64 tile_begin = gw * chunk_tiles;
    const i64 tile_end = tile_begin + chunk_tiles < ntiles ? tile_begin + chunk_tiles : ntiles;
    if (lane == 0) { first[gw].valid = 0; last[gw].valid = 0; }
    __syncwarp();
    if (tile_begin >= tile_end) return;
    const i64 plo = p.pred[0].lo, phi = p.pred[0].hi;
    const TypedCol kc = p.gs.part[0].col, vc = p.gs.fac[0][0].col;
    const i64 fc = p.gs.fc[0][0], fs = p.gs.fs[0][0];
    const bool plain = fc == 0 && fs == 1;             // sum(column): no multiply
    const i64 tail_key = load_typed(kc, p.nrows - 1);
    // the warp's open run, carried across tiles (warp-uniform); cf == 0: none yet
    int cf = 0;
    i64 ck = 0, cs = 0, cc = 0;
    unsigned n_pass = 0;

    for (i64 tile = tile_begin; tile < tile_end; tile++) {
        const i64 row = tile * RUN_WTILE + lane * SA_VEC;
        const i64 rem = p.nrows - row;
        i64 dv[4] = {0, 0, 0, 0}, k[4], v[4];
        {
            Raw4<true> rd, rk, rv;
            if (HAS_PRED) ld_typed4(p.pred[0].col, row, rd);
            ld_typed4(kc, row, rk);
            ld_typed4(vc, row, rv);
            if (HAS_PRED) unpack_typed4(p.pred[0].col, rd, dv);
            unpack_typed4(kc, rk, k);
            unpack_typed4(vc, rv, v);
        }
        i64 x[4];
        int c[4];
#pragma unroll
        for (int j = 0; j < 4; j++) {
            bool ok = j < rem;
            if (!ok) k[j] = tail_key;                  // pad rows join the table's last run and add nothing
            if (HAS_PRED) ok = ok && dv[j] >= plo && dv[j] <= phi;
            x[j] = ok ? (plain ? v[j] : fc + fs * v[j]) : 0;
            c[j] = ok ? 1 : 0;
            n_pass += ok ? 1u : 0u;
        }
        // lane-local runs, branch-free: prefix sums + the three head flags between the four rows.
        //   leading run  = rows before the first head (may continue the previous lane's run)
        //   trailing run = rows from the last head on (still open)
        //   interior runs (complete): [1, 2 or 3) when h1 and a later head exist; [2, 3) when h2 and h3
        const bool h1 = k[1] != k[0], h2 = k[2] != k[1], h3 = k[3] != k[2];
        const i64 p0 = x[0], p1 = p0 + x[1], p2 = p1 + x[2], p3 = p2 + x[3];
        const int n0 = c[0], n1 = n0 + c[1], n2 = n1 + c[2], n3 = n2 + c[3];
        const bool single = !(h1 || h2 || h3);
        const i64 lead_s = h1 ? p0 : h2 ? p1 : h3 ? p2 : p3;
        const int lead_c = h1 ? n0 : h2 ? n1 : h3 ? n2 : n3;
        const i64 cur_s = p3 - (h3 ? p2 : h2 ? p1 : h1 ? p0 : 0);
        const int cur_c = n3 - (h3 ? n2 : h2 ? n1 : h1 ? n0 : 0);
        // records this lane may close: a = the previous lane's run, b = its leading run, m / n = interior runs
        bool eva = false, evb = false;
        i64 eka = 0, esa = 0, eca = 0, ekb = 0, esb = 0, ecb = 0;
        bool evm = h1 && (h2 || h3), evn = h2 && h3;
        const i64 ekm = k[1], esm = (h2 ? p1 : p2) - p0, ekn = k[2], esn = x[2];
        const int ecm = (h2 ? n1 : n2) - n0, ecn = c[2];
        // element of the warp-wide segmented scan: the run that is still open at the end of this lane
        const i64 kfirst = k[0], klast = k[3];
        i64 pk = __shfl_up_sync(full, klast, 1);
        bool pvalid = true;
        if (lane == 0) { pk = ck; pvalid = cf != 0; }
        const bool chunk_start = tile == tile_begin && lane == 0;
        const bool cont = pvalid && pk == kfirst;      // my leading run continues the previous lane's open run
        // packed scan word: row count of the tile-local partial (<= 128) above the two flag bits
        unsigned w = ((unsigned)cur_c << 2) | ((!single || !cont) ? RUN_H : 0) | ((chunk_start && single) ? RUN_S : 0);
        i64 ss = cur_s;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const unsigned w2 = __shfl_up_sync(full, w, o);
            const i64 s2 = __shfl_up_sync(full, ss, o);
            if (lane >= o && !(w & RUN_H)) { ss += s2; w = (w + (w2 & ~3u)) | (w2 & 3u); }
        }
        int f = (int)(w & 3u);
        i64 sc = (i64)(w >> 2);
        if (!(f & RUN_H)) { ss += cs; sc += cc; f |= cf; }      // reaches back to the warp's carried run
        // the open run as the PREVIOUS lane left it
        int qf = __shfl_up_sync(full, f, 1);
        i64 qs = __shfl_up_sync(full, ss, 1), qc = __shfl_up_sync(full, sc, 1);
        if (lane == 0) { qf = cf; qs = cs; qc = cc; }
        // close runs
        if (pvalid && !cont) {                          // the previous run ended exactly at my first row
            if (qf & RUN_S) { first[gw].key = pk; first[gw].sum = qs; first[gw].cnt = qc; first[gw].spans = 0; first[gw].valid = 1; }
            else if (run_passes(out, qs, qc)) { eka = pk; esa = qs; eca = qc; eva = true; }
        }
        if (!single) {                                  // my leading run ends inside me
            const i64 ts = lead_s + (cont ? qs : 0), tc = (i64)lead_c + (cont ? qc : 0);
            const bool touches = cont ? (qf & RUN_S) != 0 : chunk_start;
            if (touches) { first[gw].key = kfirst; first[gw].sum = ts; first[gw].cnt = tc; first[gw].spans = 0; first[gw].valid = 1; }
            else if (run_passes(out, ts, tc)) { ekb = kfirst; esb = ts; ecb = tc; evb = true; }
        }
        evm = evm && run_passes(out, esm, (i64)ecm);
        evn = evn && run_passes(out, esn, (i64)ecn);
        // carry into the next tile: lane 31's open run
        cf = __shfl_sync(full, f, 31) | RUN_H;
        ck = __shfl_sync(full, klast, 31);
        cs = __shfl_sync(full, ss, 31);
        cc = __shfl_sync(full, sc, 31);
        // append the closed runs: one cursor bump per warp tile
        const int mine = (int)eva + (int)evb + (int)evm + (int)evn;
        if (__any_sync(full, mine != 0)) {
            int incl = mine;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const int t2 = __shfl_up_sync(full, incl, o);
                if (lane >= o) incl += t2;
            }
            const int total = __shfl_sync(full, incl, 31);
            unsigned long long base = 0;
            if (lane == 0) base = atomicAdd(out.count, (unsigned long long)total);
            base = __shfl_sync(full, base, 0);
            unsigned long long pos = base + (unsigned long long)(incl - mine);
            auto put = [&](bool on, i64 key, i64 sum, i64 cnt) {
                if (!on) return;
                if ((i64)pos < out.cap) { out.klo[pos] = key; out.khi[pos] = 0; out.acc[pos] = sum; out.acc[out.cap + (i64)pos] = cnt; }
                pos++;
            };
            put(eva, eka, esa, eca);
            put(evb, ekb, esb, ecb);
            put(evm, ekm, esm, (i64)ecm);
            put(evn, ekn, esn, (i64)ecn);
        }
    }
    if (lane == 0) {     // the run still open at the end of the chunk
        last[gw].key = ck; last[gw].sum = cs; last[gw].cnt = cc; last[gw].spans = (cf & RUN_S) ? 1 : 0; last[gw].valid = 1;
    }
    const unsigned long long np = (unsigned long long)warp_sum((i64)n_pass);
    if (lane == 0 && np) { atomicAdd(&p.counters[0], np); atomicAdd(&p.counters[1], np); }
}

// Stitch the runs that touch chunk edges, one thread per chunk.  Thread b emits first[b] when it does not
// continue the run left open by chunk b-1, and OWNS the run left open at the end of chunk b if that run
// starts in chunk b: it walks forward over chunks the run spans entirely until the chunk that closes it
// (sorted keys: equal keys in neighbouring edge records always mean the same run).
static __global__ void __launch_bounds__(256)
run_fixup_kernel(const RunEdge *__restrict__ first, const RunEdge *__restrict__ last, int nchunks, const RunOut out)
{
    const int b = (int)(blockIdx.x * blockDim.x + threadIdx.x);
    if (b >= nchunks) return;
    auto emit = [&](i64 k, i64 s, i64 c) {
        if (!run_passes(out, s, c)) return;
        unsigned long long pos = atomicAdd(out.count, 1ULL);
        if ((i64)pos < out.cap) { out.klo[pos] = k; out.khi[pos] = 0; out.acc[pos] = s; out.acc[out.cap + (i64)pos] = c; }
    };
    const RunEdge F = first[b], L = last[b];
    bool has_prev = false;
    i64 pkey = 0;
    if (b > 0) { has_prev = last[b - 1].valid != 0; pkey = last[b - 1].key; }
    if (F.valid && !(has_prev && pkey == F.key)) emit(F.key, F.sum, F.cnt);
    if (!L.valid) return;
    if (L.spans && has_prev && pkey == L.key) return;       // a continuation: the thread where the run starts owns it
    i64 s = L.sum, c = L.cnt;
    for (int j = b + 1; j < nchunks; j++) {
        const RunEdge Fj = first[j];
        if (Fj.valid) { if (Fj.key == L.key) { s += Fj.sum; c += Fj.cnt; } break; }
        const RunEdge Lj = last[j];
        if (!(Lj.valid && Lj.spans && Lj.key == L.key)) break;
        s += Lj.sum; c += Lj.cnt;
    }
    emit(L.key, s, c);
}

// ---------------------------------------------------------------- two-phase --
// Phase 1 (streaming, HBM-bound): screen rows [row_begin,row_end) with the range predicate and the exact
// key bitmap of the probed table and append the row ids of the hits to a compact list (one global
// cursor bump per warp step).  Nothing random is touched here, so it runs at scan speed.
// Phase 2 (latency-bound, massively parallel): one thread per hit does the hash-table probe / insert /
// group update.  Splitting the two lets each kernel have the occupancy it needs: measured at SF100, the
// fused warp-queue kernel streamed lineitem at 3.1 TB/s; see profiles/ for the split numbers.
template <bool HAS_PRED, int NT>
__global__ void __launch_bounds__(SA_THREADS)
filter_hits_kernel(const PipeParams p)
{
    const i64 nloc = p.row_end - p.row_begin;
    const i64 ntiles = (nloc + SA_TILE - 1) / SA_TILE;
    const i64 plo = p.pred[0].lo, phi = p.pred[0].hi;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const bool anti = p.probe_mode == 2;
    const unsigned *__restrict__ bm = p.probe.bitmap;
    const u64 bmin = (u64)p.probe.bm_min, dom = p.probe.domain;
    const i64 G = gridDim.x;
    constexpr int WBUF = 512;                        // >= 32 * 4 * NT hits of one step.  (1024 entries = 33 KB per CTA took L1 away from
                                                     //  the bitmap lookups: Q9's filter pass 2.84 ms against 2.33 ms with 512, 2.29 with 256)
    __shared__ unsigned s_buf[SA_THREADS / 32][WBUF];
    int nbuf = 0;                                    // warp-uniform fill level
    unsigned n_pass = 0, n_hits = 0;
    auto flush = [&]() {
        if (nbuf == 0) return;
        unsigned long long base = 0;
        if (lane == 0) base = atomicAdd(p.hit_count, (unsigned long long)nbuf);
        base = __shfl_sync(0xffffffffu, base, 0);
        for (int i = lane; i < nbuf; i += 32) p.hits[base + i] = s_buf[warp][i];
        __syncwarp();
        n_hits += lane == 0 ? (unsigned)nbuf : 0u;
        nbuf = 0;
    };
    // one step = NT tiles (tile0 + u * G); the column buffers carry ROW_PAD rows of slack, so a
    // whole-vector load of a partial tile is in bounds
    auto load = [&](i64 tile0, Raw4<true> (&d)[NT], Raw4<true> (&k)[NT]) {
#pragma unroll
        for (int u = 0; u < NT; u++) {
            const i64 tile = tile0 + u * G;
            if (tile >= ntiles) continue;
            const i64 row = p.row_begin + tile * SA_TILE + threadIdx.x * SA_VEC;
            if (HAS_PRED) ld_typed4(p.pred[0].col, row, d[u]);
            ld_typed4(p.probe_key, row, k[u]);
        }
    };
    auto process = [&](i64 tile0, const Raw4<true> (&d)[NT], const Raw4<true> (&kr)[NT]) {
        bool ok[NT][4];
        unsigned w[NT][4];
        u64 off[NT][4];
        // the bitmap words are fetched with predicated loads issued back to back (no branches)
#pragma unroll
        for (int u = 0; u < NT; u++) {
            const i64 tile = tile0 + u * G;
            const i64 row = p.row_begin + tile * SA_TILE + threadIdx.x * SA_VEC;
            const i64 rem = tile < ntiles ? p.row_end - row : 0;
            i64 dv[4] = {0, 0, 0, 0}, k4[4];
            if (HAS_PRED) unpack_typed4(p.pred[0].col, d[u], dv);
            unpack_typed4(p.probe_key, kr[u], k4);
#pragma unroll
            for (int j = 0; j < 4; j++) {
                ok[u][j] = j < rem;
                if (HAS_PRED) ok[u][j] = ok[u][j] && dv[j] >= plo && dv[j] <= phi;
                off[u][j] = (u64)k4[j] - bmin;            // one unsigned compare covers both ends of the domain
                const bool in = ok[u][j] && bm != nullptr && off[u][j] < dom;
                w[u][j] = in ? __ldg(bm + (unsigned)(off[u][j] >> 5)) : 0u;
            }
        }
        unsigned hitmask = 0;      // bit (4u + j): row j of tile u is a hit
#pragma unroll
        for (int u = 0; u < NT; u++)
#pragma unroll
            for (int j = 0; j < 4; j++) {
                n_pass += ok[u][j] ? 1u : 0u;
                const bool set = bm == nullptr || ((w[u][j] >> ((unsigned)off[u][j] & 31u)) & 1u);   // no probe: every row that passes is a hit
                if (ok[u][j] && set != anti) hitmask |= 1u << (4 * u + j);
            }
        // append to the warp's private staging buffer in shared memory (exclusive scan of the per-lane hit
        // counts); the buffer is flushed to the global list with ONE cursor bump when it is nearly full --
        // a bump per warp step put 2.3 M atomics on one address and cost more than the scan itself
        const int c = __popc(hitmask);
        int incl = c;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            int v = __shfl_up_sync(0xffffffffu, incl, o);
            if (lane >= o) incl += v;
        }
        const int total = __shfl_sync(0xffffffffu, incl, 31);
        if (total == 0) return;
        if (nbuf + total > WBUF) flush();
        int pos = nbuf + incl - c;
#pragma unroll
        for (int u = 0; u < NT; u++) {
            const i64 row = p.row_begin + (tile0 + u * G) * SA_TILE + threadIdx.x * SA_VEC;
#pragma unroll
            for (int j = 0; j < 4; j++)
                if (hitmask & (1u << (4 * u + j))) s_buf[warp][pos++] = (unsigned)(row + j);
        }
        nbuf += total;
        __syncwarp();
    };
    // software pipeline: the next step's vectors are in flight while the current step is screened
    Raw4<true> dA[NT], dB[NT], kA[NT], kB[NT];
#pragma unroll
    for (int u = 0; u < NT; u++) {
        dA[u].a = dA[u].b = dB[u].a = dB[u].b = make_int4(0, 0, 0, 0);
        kA[u].a = kA[u].b = kB[u].a = kB[u].b = make_int4(0, 0, 0, 0);
    }
    i64 tile = blockIdx.x;
    const i64 step = G * NT;
    if (tile < ntiles) load(tile, dA, kA);
    while (tile < ntiles) {
        if (tile + step < ntiles) load(tile + step, dB, kB);
        process(tile, dA, kA);
        tile += step;
        if (tile >= ntiles) break;
        if (tile + step < ntiles) load(tile + step, dA, kA);
        process(tile, dB, kB);
        tile += step;
    }
    flush();
    unsigned long long np = (unsigned long long)warp_sum((i64)n_pass), nh = (unsigned long long)warp_sum((i64)n_hits);
    if (lane == 0 && np) atomicAdd(&p.counters[0], np);
    if (lane == 0 && nh) atomicAdd(&p.counters[3], nh);
}

// Phase 1 over NARROW stored columns (predicate and key in <= 4 bytes, no NULLs): the same screen, fed by the
// bulk-copy tile ring of stage.cuh instead of per-thread vector loads -- at 6 stored bytes per lineitem row the
// register-staged kernel above is issue-bound (r2: 2.0 TB/s).  Predicate and key-domain tests run on the STORED
// 32-bit values:  (v - p_lo) <=u p_span,  off = stored key + kdelta (mod 2^32) < dom  (the host proves the wrap
// cannot alias a key outside the bitmap's domain into it).
struct FilterSParams {
    StageDesc st;
    int roff[2], rpw[2];          // role 0 = predicate column (width 0: none), 1 = probe key
    unsigned p_lo, p_span;
    unsigned kdelta, dom;
    const unsigned *bitmap;       // null: no probe, every row passing the predicate is a hit
    int anti;
    i64 row_begin, nloc;
    unsigned *hits;
    unsigned long long *hit_count;
    unsigned long long *counters;
};

template <int WP, int WK, int QPT, bool MASK>
__device__ __forceinline__ void filter_tile(const FilterSParams &p, const StageRing &ring, StageCursor &cur, int warp, int lane, i64 tile,
                                            unsigned (*s_buf)[512], int &nbuf, unsigned &n_pass, unsigned &n_hits)
{
    constexpr int WBUF = 512;
    const char *stg = stage_acquire(ring, p.st, cur);
    Quad<WP> dv[QPT];
    Quad<WK> kv[QPT];
#pragma unroll
    for (int q = 0; q < QPT; q++) {
        const int qrow = (warp * QPT + q) * 128 + lane * 4;
        dv[q].load(stg + p.roff[0], qrow, p.rpw[0]);
        kv[q].load(stg + p.roff[1], qrow, p.rpw[1]);
    }
    stage_release(ring, p.st, cur);
    const unsigned *__restrict__ bm = p.bitmap;
    const bool anti = p.anti != 0;
    const i64 row0 = tile * p.st.tile_rows;
    const int rows_in_tile = MASK ? (int)(p.nloc - row0) : 0;
    bool ok[QPT][4];
    unsigned w[QPT][4], off[QPT][4];
#pragma unroll
    for (int q = 0; q < QPT; q++) {
        const int rem = rows_in_tile - ((warp * QPT + q) * 128 + lane * 4);
        auto row = [&](auto jc) {
            constexpr int J = decltype(jc)::v;
            ok[q][J] = (!MASK || J < rem) && (WP == 0 || (dv[q].template get<J>() - p.p_lo) <= p.p_span);
            off[q][J] = kv[q].template get<J>() + p.kdelta;
            const bool in = ok[q][J] && bm != nullptr && off[q][J] < p.dom;
            w[q][J] = in ? __ldg(bm + (off[q][J] >> 5)) : 0u;      // predicated loads issued back to back
        };
        PG_FOR4(row);
    }
    unsigned hitmask = 0;
#pragma unroll
    for (int q = 0; q < QPT; q++)
#pragma unroll
        for (int j = 0; j < 4; j++) {
            n_pass += ok[q][j] ? 1u : 0u;
            const bool set = bm == nullptr || ((w[q][j] >> (off[q][j] & 31u)) & 1u);
            if (ok[q][j] && set != anti) hitmask |= 1u << (4 * q + j);
        }
    const int c = __popc(hitmask);
    int incl = c;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        int v = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += v;
    }
    const int total = __shfl_sync(0xffffffffu, incl, 31);
    if (total == 0) return;
    if (nbuf + total > WBUF) {          // flush: ONE cursor bump for the whole buffer
        unsigned long long base = 0;
        if (lane == 0) base = atomicAdd(p.hit_count, (unsigned long long)nbuf);
        base = __shfl_sync(0xffffffffu, base, 0);
        for (int i = lane; i < nbuf; i += 32) p.hits[base + i] = s_buf[warp][i];
        __syncwarp();
        n_hits += lane == 0 ? (unsigned)nbuf : 0u;
        nbuf = 0;
    }
    int pos = nbuf + incl - c;
#pragma unroll
    for (int q = 0; q < QPT; q++) {
        const unsigned rowid = (unsigned)(p.row_begin + row0) + (unsigned)((warp * QPT + q) * 128 + lane * 4);
#pragma unroll
        for (int j = 0; j < 4; j++)
            if (hitmask & (1u << (4 * q + j))) s_buf[warp][pos++] = rowid + j;
    }
    nbuf += total;
    __syncwarp();
}

template <int WP, int WK, int QPT>
__global__ void __launch_bounds__(ST_THREADS)
filter_hits_staged_kernel(const FilterSParams p)
{
    extern __shared__ __align__(128) unsigned char st_smem[];
    __shared__ unsigned s_buf[ST_CONS_WARPS][512];
    const StageDesc &d = p.st;
    const StageRing ring = stage_ring_init(st_smem, d);
    const i64 ntiles = (p.nloc + d.tile_rows - 1) / d.tile_rows;
    const TileSeq seq = tile_seq(ntiles, 0);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (warp == ST_CONS_WARPS) {
        stage_produce(ring, d, seq);
        return;
    }
    StageCursor cur = {0, 0};
    int nbuf = 0;
    unsigned n_pass = 0, n_hits = 0;
    const bool partial = last_tile_is_partial(seq, ntiles, p.nloc, d.tile_rows);
    const int nwhole = (int)seq.count - (partial ? 1 : 0);
    for (int k = 0; k < nwhole; k++)
        filter_tile<WP, WK, QPT, false>(p, ring, cur, warp, lane, seq.first + (i64)k * seq.step, s_buf, nbuf, n_pass, n_hits);
    if (partial) filter_tile<WP, WK, QPT, true>(p, ring, cur, warp, lane, ntiles - 1, s_buf, nbuf, n_pass, n_hits);
    if (nbuf) {
        unsigned long long base = 0;
        if (lane == 0) base = atomicAdd(p.hit_count, (unsigned long long)nbuf);
        base = __shfl_sync(0xffffffffu, base, 0);
        for (int i = lane; i < nbuf; i += 32) p.hits[base + i] = s_buf[warp][i];
        n_hits += lane == 0 ? (unsigned)nbuf : 0u;
    }
    unsigned long long np = (unsigned long long)warp_sum((i64)n_pass), nh = (unsigned long long)warp_sum((i64)n_hits);
    if (lane == 0 && np) atomicAdd(&p.counters[0], np);
    if (lane == 0 && nh) atomicAdd(&p.counters[3], nh);
}

template <int SINK>
__global__ void __launch_bounds__(256)
hits_sink_kernel(const PipeParams p)
{
    const unsigned long long n = *p.hit_count;
    unsigned long long n_join = 0;
    for (unsigned long long i = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (unsigned long long)gridDim.x * blockDim.x) {
        const i64 row = (i64)p.hits[i];
        if (p.nextra && !extras_pass(p, row)) continue;
        auto sink = [&](u64 build_row) {
            n_join++;
            if (SINK == SINK_INSERT) {
                i64 key = load_typed(p.ins_key, row);
                if (p.ins_key2.p) key = (key << 32) | (load_typed(p.ins_key2, row) & 0xffffffffLL);
                jt_insert(p.ins, key, (u64)row);
            } else if (SINK == SINK_BITMAP) {
                u64 off = (u64)(load_typed(p.ins_key, row) - p.ins.bm_min);
                atomicOr(p.ins.bitmap + (off >> 5), 1u << (off & 31));
            } else if (SINK == SINK_GROUP) {
                auto val = [&](const ValRef &r) { return r.from_build == 2 ? (i64)build_row : load_typed(r.col, r.from_build ? (i64)build_row : row); };
                i64 klo = val(p.gs.part[0]);
                i64 khi = 0;
                if (p.gs.nparts > 1) khi = val(p.gs.part[1]) << 32;
                if (p.gs.nparts > 2) khi |= val(p.gs.part[2]) & 0xffffffffLL;
                i64 vals[GT_MAXACC];
                for (int a = 0; a < p.gs.nacc; a++) {
                    i64 x = 1;
                    for (int f = 0; f < p.gs.nfac[a]; f++) x *= p.gs.fc[a][f] + p.gs.fs[a][f] * val(p.gs.fac[a][f]);
                    vals[a] = x;
                }
                gt_update(p.gt, klo, khi, vals);
            }
        };
        if (!p.has_probe || p.probe_bitmap_only || p.probe_mode != 0) sink(0);
        else jt_probe(p.probe, load_typed(p.probe_key, row), sink);
    }
    n_join = (unsigned long long)warp_sum((i64)n_join);
    if ((threadIdx.x & 31) == 0 && n_join) atomicAdd(&p.counters[1], n_join);
}

// ---------------------------------------------------------------- star joins --
// A fact-table pipeline with SEVERAL INNER joins on the way to a low-cardinality group-by (TPC-H Q9:
// lineitem x part x supplier x partsupp x orders x nation, 175 groups).  The most selective existence
// join is the filter pass (filter_hits_kernel); this sink then resolves the other joins for each hit --
// key from the fact row or from an earlier lookup's build row, one or two key columns, rank index or
// hash table -- evaluates sum-of-products terms over the joined rows and adds them to a block-private
// shared-memory table indexed by the dense group id; blocks flush to the global table at the end.
constexpr int STAR_MAXLOOKUP = 5, STAR_MAXTERM = 2, STAR_MAXPART = 2, STAR_MAXGROUPS = 4096;
struct StarLookup {
    int nkey;                 // 1, or 2: key = (k0 << 32) | (k1 & 0xffffffff)
    ValRef key[2];            // from_build: 0 = fact row, j > 0 = build row of lookup j-1
    JoinTable jt;
    int existence;            // payload-free: the exact bitmap answers
};
struct StarPart {             // dense group index part: f(value) - lo in [0, n)
    ValRef v;
    int fn;                   // 0: the value itself, 1: calendar year of a DATE (days since 1970-01-01)
    i64 lo;
    int n;
};
struct StarTerm {             // mul * prod(fc + fs * value)
    int nfac;
    ValRef fac[3];
    i64 fc[3];
    int fs[3];
    i64 mul;
};
struct StarParams {
    const unsigned *hits;
    const unsigned long long *hit_count;
    int nlookup;
    StarLookup lk[STAR_MAXLOOKUP];
    int nparts, ngroups;
    StarPart part[STAR_MAXPART];
    int nterm;
    StarTerm term[STAR_MAXTERM];
    unsigned long long *gsum, *gsum_hi, *gcnt;   // [ngroups] global accumulators: 128-bit sums (two words) and row counts
    unsigned long long *counters;             // [1] joined rows, [2] hits with more than one match in some lookup
};

// civil year of days-since-epoch (proleptic Gregorian; the reference extracts it through time.Time, common/date.go)
__device__ __forceinline__ i64 year_of_days(i64 z)
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

// The joins of hit i: rows[0] = its fact row, rows[l + 1] = the build row lookup l matched (-1 for an existence lookup).
// False when some join finds no build row; a lookup with more than one match counts into n_multi.
__device__ __forceinline__ bool star_lookups(const StarParams &sp, unsigned long long i, i64 (&rows)[STAR_MAXLOOKUP + 1], unsigned long long &n_multi)
{
    rows[0] = (i64)sp.hits[i];
    auto val = [&](const ValRef &r) { return load_typed(r.col, rows[r.from_build]); };
    bool ok = true;
#pragma unroll
    for (int l = 0; l < STAR_MAXLOOKUP; l++) {
        if (l >= sp.nlookup || !ok) continue;
        const StarLookup &L = sp.lk[l];
        i64 key = val(L.key[0]);
        if (L.nkey == 2) key = (key << 32) | (val(L.key[1]) & 0xffffffffLL);
        rows[l + 1] = -1;
        if (L.existence) {
            ok = bitmap_test(L.jt, key);
        } else {
            int matches = 0;
            jt_probe(L.jt, key, [&](u64 r) { rows[l + 1] = (i64)r; matches++; });
            ok = matches > 0;
            n_multi += matches > 1 ? 1 : 0;
        }
    }
    return ok;
}

// the summed value of one joined row: sum over the terms of mul * prod(fc + fs * value)
__device__ __forceinline__ i64 star_amount(const StarParams &sp, const i64 (&rows)[STAR_MAXLOOKUP + 1])
{
    auto val = [&](const ValRef &r) { return load_typed(r.col, rows[r.from_build]); };
    i64 amount = 0;
#pragma unroll
    for (int t = 0; t < STAR_MAXTERM; t++) {
        if (t >= sp.nterm) continue;
        i64 x = sp.term[t].mul;
        for (int f = 0; f < sp.term[t].nfac; f++) x *= sp.term[t].fc[f] + sp.term[t].fs[f] * val(sp.term[t].fac[f]);
        amount += x;
    }
    return amount;
}

static __global__ void __launch_bounds__(256)
hits_star_kernel(const StarParams sp)
{
    extern __shared__ unsigned long long s_star[];      // [ngroups] sums, [ngroups] counts
    unsigned long long *s_sum = s_star, *s_cnt = s_star + sp.ngroups;
    for (int i = threadIdx.x; i < 2 * sp.ngroups; i += blockDim.x) s_star[i] = 0;
    __syncthreads();
    const unsigned long long n = *sp.hit_count;
    unsigned long long n_join = 0, n_multi = 0;
    for (unsigned long long i = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (unsigned long long)gridDim.x * blockDim.x) {
        i64 rows[STAR_MAXLOOKUP + 1];
        if (!star_lookups(sp, i, rows, n_multi)) continue;
        n_join++;
        auto val = [&](const ValRef &r) { return load_typed(r.col, rows[r.from_build]); };
        int g = 0;
#pragma unroll
        for (int k = 0; k < STAR_MAXPART; k++) {
            if (k >= sp.nparts) continue;
            i64 v = val(sp.part[k].v);
            if (sp.part[k].fn == 1) v = year_of_days(v);
            g = g * sp.part[k].n + (int)(v - sp.part[k].lo);
        }
        const i64 amount = star_amount(sp, rows);
        atomicAdd(&s_sum[g], (unsigned long long)amount);
        atomicAdd(&s_cnt[g], 1ULL);
    }
    __syncthreads();
    for (int i = threadIdx.x; i < sp.ngroups; i += blockDim.x) {
        if (s_cnt[i]) {
            // the block's exact int64 partial (the host proved it cannot overflow) goes into a 128-bit total
            const unsigned long long x = s_sum[i];
            const unsigned long long old = atomicAdd(&sp.gsum[i], x);
            const long long hi = (long long)(old + x < old ? 1 : 0) - ((long long)x < 0 ? 1 : 0);
            if (hi) atomicAdd(&sp.gsum_hi[i], (unsigned long long)hi);
            atomicAdd(&sp.gcnt[i], s_cnt[i]);
        }
    }
    n_join = (unsigned long long)warp_sum((i64)n_join);
    n_multi = (unsigned long long)warp_sum((i64)n_multi);
    if ((threadIdx.x & 31) == 0) {
        if (n_join) atomicAdd(&sp.counters[1], n_join);
        if (n_multi) atomicAdd(&sp.counters[2], n_multi);
    }
}

// Star join grouped by the build ROW of one lookup (TPC-H Q10: the customer row; every group key is a column of that row or
// of a unique lookup keyed from it).  Same joins and amount as hits_star_kernel, but the groups are as many as that table's
// rows: the sink adds into global per-row accumulators dsum[row] (u64, the host proved the total fits int64) and
// dcnt[row] (u32, fewer than 2^32 fact rows) -- the layout of group1_dense_kernel, compacted by dense_compact_kernel.
// `anchor` indexes rows[]: 1 + the lookup whose row is the group.
static __global__ void __launch_bounds__(256)
hits_star_rows_kernel(const StarParams sp, int anchor, unsigned long long *__restrict__ dsum, unsigned *__restrict__ dcnt)
{
    const unsigned long long n = *sp.hit_count;
    unsigned long long n_join = 0, n_multi = 0;
    for (unsigned long long i = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (unsigned long long)gridDim.x * blockDim.x) {
        i64 rows[STAR_MAXLOOKUP + 1];
        if (!star_lookups(sp, i, rows, n_multi)) continue;
        n_join++;
        const u64 g = (u64)rows[anchor];
        atomicAdd(dsum + g, (unsigned long long)star_amount(sp, rows));
        atomicAdd(dcnt + g, 1u);
    }
    n_join = (unsigned long long)warp_sum((i64)n_join);
    n_multi = (unsigned long long)warp_sum((i64)n_multi);
    if ((threadIdx.x & 31) == 0) {
        if (n_join) atomicAdd(&sp.counters[1], n_join);
        if (n_multi) atomicAdd(&sp.counters[2], n_multi);
    }
}

// ---------------------------------------------------------------- rank index build --
// pass 1 over the hit list: gather the build key, remember it, set its bit (DETECT: count keys seen twice)
template <bool DETECT>
static __global__ void __launch_bounds__(256)
rank_mark_kernel(const PipeParams p, i64 *__restrict__ keys_tmp)
{
    const unsigned long long n = *p.hit_count;
    const unsigned long long stride = (unsigned long long)gridDim.x * blockDim.x;
    unsigned long long dups = 0;
    for (unsigned long long i = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
        if (p.nextra && !extras_pass(p, (i64)p.hits[i])) { keys_tmp[i] = HT_EMPTY; continue; }   // HT_EMPTY is never a key
        const i64 key = load_typed(p.ins_key, (i64)p.hits[i]);
        keys_tmp[i] = key;
        const u64 off = (u64)key - (u64)p.ins.bm_min;
        const unsigned bit = 1u << (off & 31);
        if (DETECT) dups += (atomicOr(p.ins.bitmap + (off >> 5), bit) & bit) ? 1 : 0;
        else atomicOr(p.ins.bitmap + (off >> 5), bit);      // result unused: a fire-and-forget RED
    }
    if (DETECT) {
        dups = (unsigned long long)warp_sum((i64)dups);
        if ((threadIdx.x & 31) == 0 && dups) atomicAdd(p.ins.dups, dups);
    }
}
// set bits per 256-bit block (exclusive-summed into rank_prefix by the caller)
static __global__ void rank_count_kernel(const unsigned *__restrict__ bitmap, u64 nblocks, unsigned *__restrict__ counts)
{
    for (u64 b = (u64)blockIdx.x * blockDim.x + threadIdx.x; b < nblocks; b += (u64)gridDim.x * blockDim.x) {
        const uint4 x = __ldg((const uint4 *)(bitmap + b * 8)), y = __ldg((const uint4 *)(bitmap + b * 8) + 1);
        counts[b] = __popc(x.x) + __popc(x.y) + __popc(x.z) + __popc(x.w) + __popc(y.x) + __popc(y.y) + __popc(y.z) + __popc(y.w);
    }
}
// pass 2 over the hit list: payload[rank(key)] = build row id
static __global__ void __launch_bounds__(256)
rank_fill_kernel(const PipeParams p, const i64 *__restrict__ keys_tmp, unsigned *__restrict__ payload)
{
    const unsigned long long n = *p.hit_count;
    const unsigned long long stride = (unsigned long long)gridDim.x * blockDim.x;
    for (unsigned long long i = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
        if (keys_tmp[i] == HT_EMPTY) continue;
        bool set;
        const unsigned r = jt_rank(p.ins, (u64)keys_tmp[i] - (u64)p.ins.bm_min, &set);
        payload[r] = p.hits[i];
    }
}

// Key bitmap of a (filtered) build side straight from its columns: 4 consecutive rows per thread with 16-byte vector
// loads, <= 1 range / code-set predicate, no NULLs, no probe.  The row-at-a-time pipeline_kernel needed 146 us for
// SF100's 15 M customers (one dependent load chain per row); this streams the two columns.
template <bool HAS_PRED>
static __global__ void __launch_bounds__(256)
bitmap_build_kernel(const PipeParams p, i64 lo, i64 hi)          // lo a multiple of 4
{
    unsigned long long n_pass = 0;
    for (i64 row = lo + ((i64)blockIdx.x * blockDim.x + threadIdx.x) * 4; row < hi; row += (i64)gridDim.x * blockDim.x * 4) {
        i64 k[4], v[4] = {0, 0, 0, 0};
        load_typed4(p.ins_key, row, k);
        if (HAS_PRED) load_typed4(p.pred[0].col, row, v);
#pragma unroll
        for (int j = 0; j < 4; j++) {
            bool ok = row + j < hi;
            if (HAS_PRED) ok = ok && (p.pred[0].is_set ? ((p.pred[0].mask[(v[j] >> 5) & 7] >> (v[j] & 31)) & 1u) != 0 : (v[j] >= p.pred[0].lo && v[j] <= p.pred[0].hi));
            if (!ok) continue;
            n_pass++;
            const u64 off = (u64)(k[j] - p.ins.bm_min);
            atomicOr(p.ins.bitmap + (off >> 5), 1u << (off & 31));
        }
    }
    n_pass = (unsigned long long)warp_sum((i64)n_pass);
    if ((threadIdx.x & 31) == 0 && n_pass) { atomicAdd(&p.counters[0], n_pass); atomicAdd(&p.counters[1], n_pass); }
}

// OR-merge of the ranks' partial key bitmaps (all-gathered as [world][words + 8]); the 8-word tail of every part
// carries that rank's {rows passing, rows built} counters, which are summed into `counters`
static __global__ void bitmap_or_kernel(const unsigned *__restrict__ parts, int world, u64 words, unsigned *__restrict__ bitmap,
                                        unsigned long long *__restrict__ counters)
{
    const u64 stride = words + 8;
    for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < words; i += (u64)gridDim.x * blockDim.x) {
        unsigned x = 0;
        for (int r = 0; r < world; r++) x |= parts[(u64)r * stride + i];
        bitmap[i] = x;
    }
    if (blockIdx.x == 0 && threadIdx.x < 4) {
        unsigned long long s = 0;
        for (int r = 0; r < world; r++) s += ((const unsigned long long *)(parts + (u64)r * stride + words))[threadIdx.x];
        counters[threadIdx.x] = s;
    }
}

// existence-only build side made of a key LIST (the groups of a sub-aggregate): set the key bits
static __global__ void keys_bitmap_kernel(const i64 *__restrict__ keys, i64 n, JoinTable jt)
{
    for (i64 i = (i64)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (i64)gridDim.x * blockDim.x) {
        const u64 off = (u64)keys[i] - (u64)jt.bm_min;
        if (off < jt.domain) atomicOr(jt.bitmap + (off >> 5), 1u << (off & 31));
    }
}

// Late materialisation of one functionally dependent group key for the n output groups: brow[i] is the
// build row a group stands for.  direct: out = col[brow].  via: key = via_key[brow] is looked up in the
// rank index `dt` of a deeper build side, out = dcol[drow] (or drow itself for host-resident columns).
static __global__ void fd_gather_kernel(const i64 *__restrict__ brow, i64 n, TypedCol direct, int via, TypedCol via_key, JoinTable dt,
                                        TypedCol dcol, int want_rowid, i64 *__restrict__ out)
{
    for (i64 i = (i64)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (i64)gridDim.x * blockDim.x) {
        const i64 b = brow[i];
        if (!via) { out[i] = want_rowid ? b : load_typed(direct, b); continue; }
        i64 drow = -1;
        jt_probe(dt, load_typed(via_key, b), [&](u64 r) { drow = (i64)r; });
        out[i] = drow < 0 ? -1 : (want_rowid ? drow : load_typed(dcol, drow));
    }
}

// (HAVING on one aggregate -- an inclusive range on accumulator plane `hav_plane` -- is applied here)
static __global__ void gt_compact_kernel(const GroupTable g, i64 *__restrict__ out_klo, i64 *__restrict__ out_khi,
                                  i64 *__restrict__ out_acc /* [nacc+1][max_out] */, i64 max_out,
                                  unsigned long long *__restrict__ counter, int hav_plane, i64 hav_lo, i64 hav_hi)
{
    // one output-position atomic per BLOCK step (256 slots), not per surviving slot
    __shared__ unsigned s_warp[8];
    __shared__ unsigned long long s_base;
    const u64 cap = g.mask + 1;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const u64 nstep = (cap + blockDim.x - 1) / blockDim.x;
    for (u64 step = blockIdx.x; step < nstep; step += gridDim.x) {
        u64 i = step * blockDim.x + threadIdx.x;
        const i64 *slot = g.slots + i * (u64)g.rw;
        bool keep = false, dropped = false;
        i64 k = HT_EMPTY;
        if (i < cap) {
            k = slot[0];
            keep = k != HT_EMPTY;
            if (keep && hav_plane >= 0) {
                i64 v = (i64)((u64)slot[2 + hav_plane] - (u64)HT_EMPTY);
                if (v < hav_lo || v > hav_hi) { keep = false; dropped = true; }
            }
        }
        unsigned m = __ballot_sync(0xffffffffu, keep), md = __ballot_sync(0xffffffffu, dropped);
        if (lane == 0) s_warp[warp] = __popc(m) | (__popc(md) << 16);
        __syncthreads();
        if (threadIdx.x == 0) {
            unsigned tot = 0, totd = 0;
            for (int w = 0; w < 8; w++) { unsigned c = s_warp[w] & 0xffff; totd += s_warp[w] >> 16; s_warp[w] = tot; tot += c; }
            s_base = tot ? atomicAdd(counter, (unsigned long long)tot) : 0;
            if (totd) atomicAdd(counter + 1, (unsigned long long)totd);
        }
        __syncthreads();
        if (keep) {
            unsigned long long o = s_base + s_warp[warp] + __popc(m & ((1u << lane) - 1u));
            if ((i64)o < max_out) {
                out_klo[o] = k;
                out_khi[o] = g.two_words ? slot[1] : 0;
                for (int a = 0; a <= g.nacc; a++) out_acc[(u64)a * (u64)max_out + o] = (i64)((u64)slot[2 + a] - (u64)HT_EMPTY);
            }
        }
        __syncthreads();
    }
}

// ------------------------------------------------------------------ top-k --
// Limit <- Order <- Agg fused onto the device (SURVEY.md 8f-1): instead of shipping every group
// to the host to sort, radix-select the k-th smallest PRIMARY sort key over the compacted group
// list (8 histogram passes of 8 bits), collect the groups at or before it (k plus ties) and let
// the host order those few rows with the full key list.  Keys follow sort_encoder.go:65-81:
// a DECIMAL key is the value rounded half-even to two fractional digits.
struct TopkKey {
    int src;        // 0: klo, 1: khi >> 32, 2: low 32 bits of khi (sign extended), 3: accumulator plane
    int plane;
    int desc;
    i64 div;        // DECIMAL: 10^(scale-2) (1 = no rounding)
};

__device__ __forceinline__ u64 topk_u64(const TopkKey &k, const i64 *klo, const i64 *khi, const i64 *acc, i64 stride, i64 i)
{
    i64 v = k.src == 0 ? klo[i] : k.src == 1 ? (khi[i] >> 32) : k.src == 2 ? (i64)(int)(khi[i] & 0xffffffffLL) : acc[(i64)k.plane * stride + i];
    if (k.div > 1) {
        bool neg = v < 0;
        u64 m = neg ? (u64)(-(v + 1)) + 1 : (u64)v, q = m / (u64)k.div, r = m % (u64)k.div;
        if (2 * r > (u64)k.div || (2 * r == (u64)k.div && (q & 1))) q++;
        v = neg ? -(i64)q : (i64)q;
    }
    u64 u = (u64)v ^ 0x8000000000000000ULL;     // order preserving
    return k.desc ? ~u : u;                     // output order = ascending u
}

// one radix-select pass over an 8-bit digit, histogram privatised in shared memory (a 16-bit digit
// with global atomics was tried: 7x slower, the top digits of real keys collide in one bin).
// MINMAX (first pass only): also reduce the smallest / largest key into minmax[0..1], so the host can
// skip every digit the keys have in common.
constexpr int TOPK_DIGIT_BITS = 8;
template <bool MINMAX>
static __global__ void topk_hist_kernel(TopkKey key, const i64 *klo, const i64 *khi, const i64 *acc, i64 stride, i64 n,
                                        u64 prefix, int prefix_bits, unsigned *hist /* [256] */, unsigned long long *minmax)
{
    __shared__ unsigned s_h[256];
    for (int i = threadIdx.x; i < 256; i += blockDim.x) s_h[i] = 0;
    __syncthreads();
    u64 lo = ~0ULL, hi = 0;
    for (i64 i = (i64)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (i64)gridDim.x * blockDim.x) {
        u64 u = topk_u64(key, klo, khi, acc, stride, i);
        if (MINMAX) { lo = u < lo ? u : lo; hi = u > hi ? u : hi; }
        if (prefix_bits == 0 || (u >> (64 - prefix_bits)) == prefix) atomicAdd(&s_h[(u >> (56 - prefix_bits)) & 255], 1u);
    }
    if (MINMAX) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            u64 l2 = __shfl_xor_sync(0xffffffffu, lo, o), h2 = __shfl_xor_sync(0xffffffffu, hi, o);
            lo = l2 < lo ? l2 : lo;
            hi = h2 > hi ? h2 : hi;
        }
        if ((threadIdx.x & 31) == 0) { atomicMin(&minmax[0], lo); atomicMax(&minmax[1], hi); }
    }
    __syncthreads();
    for (int i = threadIdx.x; i < 256; i += blockDim.x)
        if (s_h[i]) atomicAdd(&hist[i], s_h[i]);
}

// (A single-block, single-launch radix select was tried to save the 8 host round trips at small n: one SM
// evaluating every key 8 times took 0.66 ms at 113 k groups against 0.16 ms for the multi-block passes.)
// copy every group whose primary key is <= threshold to the candidate arrays
static __global__ void topk_collect_kernel(TopkKey key, const i64 *klo, const i64 *khi, const i64 *acc, i64 stride, i64 n, int planes,
                                           u64 threshold, i64 *out_klo, i64 *out_khi, i64 *out_acc, i64 out_cap,
                                           unsigned long long *counter)
{
    for (i64 i = (i64)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (i64)gridDim.x * blockDim.x) {
        if (topk_u64(key, klo, khi, acc, stride, i) > threshold) continue;
        unsigned long long o = atomicAdd(counter, 1ULL);
        if ((i64)o >= out_cap) continue;
        out_klo[o] = klo[i];
        out_khi[o] = khi[i];
        for (int a = 0; a < planes; a++) out_acc[(i64)a * out_cap + (i64)o] = acc[(i64)a * stride + i];
    }
}

// ---- the same radix select with its state on the DEVICE: no host round trip between the passes ----
// The host loop above reads every histogram back (3 synchronisations for Q3's revenue key, ~25 us each: more than the
// passes themselves once the shards are small).  Here a one-block kernel takes the host's decision after every pass and
// the next pass reads prefix / shift from device memory; the launch sequence is fixed (first pass, TOPK_DEV_MORE further
// passes that return at once when the selection is finished), the threshold lands in the state for the collect kernel.
constexpr int TOPK_DEV_MORE = 4;
struct TopkState {
    u64 prefix;          // digits chosen so far (high bits of the key)
    u64 threshold;       // valid when done: keys <= threshold are the candidates
    i64 remaining;       // we look for the remaining-th smallest key among those matching the prefix
    i64 n_equal;         // keys matching the prefix
    int pass;            // digits of TOPK_DIGIT_BITS consumed
    int done;
};
static __global__ void topk_state_init_kernel(TopkState *st, i64 k, i64 n, unsigned *hist, unsigned long long *minmax)
{
    if (threadIdx.x == 0) { st->prefix = 0; st->threshold = ~0ULL; st->remaining = k; st->n_equal = n; st->pass = 0; st->done = 0; minmax[0] = ~0ULL; minmax[1] = 0; }
    for (int i = threadIdx.x; i < 256; i += blockDim.x) hist[i] = 0;
}
template <bool MINMAX>
static __global__ void topk_hist_dev_kernel(TopkKey key, const i64 *klo, const i64 *khi, const i64 *acc, i64 stride, i64 n,
                                            const TopkState *st, unsigned *hist, unsigned long long *minmax)
{
    if (st->done) return;
    const u64 prefix = st->prefix;
    const int prefix_bits = st->pass * TOPK_DIGIT_BITS;
    __shared__ unsigned s_h[256];
    for (int i = threadIdx.x; i < 256; i += blockDim.x) s_h[i] = 0;
    __syncthreads();
    u64 lo = ~0ULL, hi = 0;
    for (i64 i = (i64)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (i64)gridDim.x * blockDim.x) {
        u64 u = topk_u64(key, klo, khi, acc, stride, i);
        if (MINMAX) { lo = u < lo ? u : lo; hi = u > hi ? u : hi; }
        if (prefix_bits == 0 || (u >> (64 - prefix_bits)) == prefix) atomicAdd(&s_h[(u >> (56 - prefix_bits)) & 255], 1u);
    }
    if (MINMAX) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            u64 l2 = __shfl_xor_sync(0xffffffffu, lo, o), h2 = __shfl_xor_sync(0xffffffffu, hi, o);
            lo = l2 < lo ? l2 : lo;
            hi = h2 > hi ? h2 : hi;
        }
        if ((threadIdx.x & 31) == 0) { atomicMin(&minmax[0], lo); atomicMax(&minmax[1], hi); }
    }
    __syncthreads();
    for (int i = threadIdx.x; i < 256; i += blockDim.x)
        if (s_h[i]) atomicAdd(&hist[i], s_h[i]);
}
// one block: the host loop's step (choose the digit holding the k-th key, skip digits common to every key after the
// first pass, stop when the bin is small or the digits are used up), then clears the histogram for the next pass
static __global__ void topk_select_kernel(TopkState *st, unsigned *hist, const unsigned long long *minmax, i64 k, i64 n, i64 stop_at, int last)
{
    __shared__ unsigned s_h[256];
    const int npass = 64 / TOPK_DIGIT_BITS;
    if (st->done) return;
    s_h[threadIdx.x] = hist[threadIdx.x];
    hist[threadIdx.x] = 0;
    __syncthreads();
    if (threadIdx.x != 0) return;
    i64 remaining = st->remaining;
    int d = 0;
    for (; d < 256; d++) {
        if ((i64)s_h[d] >= remaining) break;
        remaining -= (i64)s_h[d];
    }
    if (d == 256) d = 255;                       // cannot happen (the bins hold n_equal >= remaining keys)
    u64 prefix = (st->prefix << TOPK_DIGIT_BITS) | (u64)d;
    i64 n_equal = (i64)s_h[d];
    int pass = st->pass + 1;
    if (pass == 1) {
        const u64 diff = minmax[0] ^ minmax[1];
        int common = 64;
        if (diff) { common = 0; while (!((diff << common) >> 63)) common++; }
        int skip_to = common / TOPK_DIGIT_BITS;
        if (skip_to > npass) skip_to = npass;
        if (skip_to > pass) {
            pass = skip_to;
            prefix = pass == npass ? minmax[0] : minmax[0] >> (64 - pass * TOPK_DIGIT_BITS);
            remaining = k;
            n_equal = n;
        }
    }
    st->prefix = prefix;
    st->remaining = remaining;
    st->n_equal = n_equal;
    st->pass = pass;
    if (!(pass < npass && n_equal > stop_at) || last) {
        const int rest_bits = 64 - pass * TOPK_DIGIT_BITS;
        st->threshold = rest_bits > 0 ? (prefix << rest_bits) | ((((u64)1) << rest_bits) - 1) : prefix;
        st->done = 1;
    }
}
static __global__ void topk_collect_dev_kernel(TopkKey key, const i64 *klo, const i64 *khi, const i64 *acc, i64 stride, i64 n, int planes,
                                               const TopkState *st, i64 *out_klo, i64 *out_khi, i64 *out_acc, i64 out_cap,
                                               unsigned long long *counter)
{
    const u64 threshold = st->threshold;
    for (i64 i = (i64)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (i64)gridDim.x * blockDim.x) {
        if (topk_u64(key, klo, khi, acc, stride, i) > threshold) continue;
        unsigned long long o = atomicAdd(counter, 1ULL);
        if ((i64)o >= out_cap) continue;
        out_klo[o] = klo[i];
        out_khi[o] = khi[i];
        for (int a = 0; a < planes; a++) out_acc[(i64)a * out_cap + (i64)o] = acc[(i64)a * stride + i];
    }
}
// candidates -> ONE fixed-size message [count | klo[cap] | khi[cap] | planes x acc[cap]]; count = -1 when they do not fit
static __global__ void topk_pack_kernel(const i64 *klo, const i64 *khi, const i64 *acc, i64 stride, const unsigned long long *counter, int planes,
                                        int cap, i64 *msg)
{
    const i64 n = (i64)*counter;
    if (blockIdx.x == 0 && threadIdx.x == 0) msg[0] = n <= cap ? n : -1;
    if (n > cap) return;
    for (i64 i = (i64)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (i64)gridDim.x * blockDim.x) {
        msg[1 + i] = klo[i];
        msg[1 + cap + i] = khi[i];
        for (int a = 0; a < planes; a++) msg[1 + (i64)cap * (2 + a) + i] = acc[(i64)a * stride + i];
    }
}

// -------------------------------------------------------------- shuffle --
__device__ __forceinline__ int shuffle_dest(i64 klo, i64 khi, int world)
{
    return (int)(mix64((u64)klo ^ ((u64)khi * 0x9E3779B97F4A7C15ULL)) % (u64)world);
}

static __global__ void shuffle_count_kernel(const i64 *klo, const i64 *khi, i64 n, int world, unsigned long long *cnt)
{
    __shared__ unsigned s_c[64];
    if (threadIdx.x < 64) s_c[threadIdx.x] = 0;
    __syncthreads();
    for (i64 i = (i64)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (i64)gridDim.x * blockDim.x)
        atomicAdd(&s_c[shuffle_dest(klo[i], khi[i], world)], 1u);
    __syncthreads();
    if (threadIdx.x < world && s_c[threadIdx.x]) atomicAdd(&cnt[threadIdx.x], (unsigned long long)s_c[threadIdx.x]);
}

// pack rows [klo, khi, planes...] grouped by destination rank (cursor[d] starts at the d-th send offset)
static __global__ void shuffle_scatter_kernel(const i64 *klo, const i64 *khi, const i64 *acc, i64 stride, i64 n, int planes, int world,
                                              unsigned long long *cursor, i64 *send)
{
    const int RW = 2 + planes;
    for (i64 i = (i64)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (i64)gridDim.x * blockDim.x) {
        i64 a = klo[i], b = khi[i];
        unsigned long long pos = atomicAdd(&cursor[shuffle_dest(a, b, world)], 1ULL);
        i64 *row = send + pos * RW;
        row[0] = a;
        row[1] = b;
        for (int p = 0; p < planes; p++) row[2 + p] = acc[(i64)p * stride + i];
    }
}

// add received partial groups (all planes, the last one being the row count) into the group table
static __global__ void shuffle_merge_kernel(const GroupTable g, const i64 *rows, i64 n, int planes)
{
    const int RW = 2 + planes;
    for (i64 r = (i64)blockIdx.x * blockDim.x + threadIdx.x; r < n; r += (i64)gridDim.x * blockDim.x) {
        const i64 *row = rows + r * RW;
        gt_add(g, row[0], row[1], row + 2, row[2 + g.nacc]);
    }
}

}  // namespace pg
