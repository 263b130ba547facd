// leftcount.cuh -- grouped LEFT-join counts (sm_100a): `Agg(group by k; count) <- LeftJoin(k = fk) <- {preserved, build}`,
// optionally under `Agg(group by that count; count(*))` (TPC-H Q13).
//
// A group is one row of the preserved side that passes its filters.  The build side is streamed once: every row that
// passes its predicates and carries a non-NULL key (and count argument) is looked up in the preserved side's key table
// (rank index or hash table, payload = preserved row id) and adds 1 to a u32 count of that row.  The outer aggregate is
// a histogram of those counts; the inner aggregate alone compacts them into (key, count) rows.
#pragma once
#include "join.cuh"

namespace pg {

// String predicates of this pipeline: besides GenLike kinds 1..6 (scanagg.cuh), `%s1%...%sk%` (plan_ir.hpp like_segments) as
// k word-at-a-time searches.  Encoding: plen = k, segment i in pat[8i .. 8i+8) (zero-padded), its length in pat[32 + i].
constexpr int GEN_LIKE_WORDS = 7, GEN_NOTLIKE_WORDS = 8;

// leftmost occurrence of the L-byte literal `lit` (1 <= L <= 8, little-endian) in bytes [b, e): the end of that occurrence,
// or -1.  The search of gen_contains, kept separate so that the kernels using gen_contains compile as before.  The byte
// buffer is 8-byte aligned and padded, so the look-ahead word is always readable.
__device__ __forceinline__ i64 gen_find_word(const char *bytes, i64 b, i64 e, u64 lit, int L)
{
    if (e - b < L) return -1;
    const u64 ONES = 0x0101010101010101ULL, HIGH = 0x8080808080808080ULL;
    const u64 mask = L >= 8 ? ~0ULL : ((1ULL << (8 * L)) - 1);
    const u64 first = ONES * (lit & 0xff);
    const u64 *base = (const u64 *)bytes;
    const i64 wb = b >> 3, we = (e - L) >> 3;             // the last word that can hold a match's first byte
    u64 cur = __ldg(base + wb);
    for (i64 w = wb; w <= we; w++) {
        const u64 nxt = __ldg(base + w + 1);
        const u64 x = cur ^ first;
        u64 t = (x - ONES) & ~x & HIGH;                      // bytes equal to the first literal byte (plus false positives, verified)
        while (t) {
            const int j = (__ffsll((long long)t) - 1) >> 3;
            t &= t - 1;
            const i64 p = (w << 3) + j;
            if (p < b || p + L > e) continue;
            const int sh = j * 8;
            const u64 win = sh == 0 ? cur : (cur >> sh) | (nxt << (64 - sh));
            if ((win & mask) == lit) return p + L;
        }
        cur = nxt;
    }
    return -1;
}

__device__ __forceinline__ bool lc_like_pass(const GenLike &l, i64 row)
{
    if (l.kind != GEN_LIKE_WORDS && l.kind != GEN_NOTLIKE_WORDS) return gen_like_pass(l, row);
    const i64 b = __ldg(l.off + row), e = __ldg(l.off + row + 1);
    i64 pos = b;
    for (int s = 0; s < l.plen && pos >= 0; s++) {
        u64 lit;
        memcpy(&lit, l.pat + 8 * s, 8);
        pos = gen_find_word(l.bytes, pos, e, lit, (int)(unsigned char)l.pat[32 + s]);
    }
    return (pos >= 0) == (l.kind == GEN_LIKE_WORDS);
}

// conjunctive row filter: range / code-set predicates and string predicates
struct LcFilter {
    int npred;
    SrcPred pred[PIPE_MAXPRED];
    int nlike;
    GenLike like[GEN_MAXLIKE];
};
__device__ __forceinline__ bool lc_pass(const LcFilter &f, i64 row)
{
    for (int k = 0; k < f.npred; k++)
        if (!pred_pass(f.pred[k], row)) return false;
    for (int k = 0; k < f.nlike; k++)
        if (!lc_like_pass(f.like[k], row)) return false;
    return true;
}

struct LeftCountParams {
    i64 nrows;                      // build-side rows
    LcFilter f;                     // build-side predicates
    TypedCol key;                   // build-side join key (a NULL key matches nothing)
    TypedCol arg;                   // count(build column): rows whose argument is NULL are not counted (valid == null: count every row)
    JoinTable anchor;               // preserved side's key -> preserved row id
    unsigned *counts;               // [preserved rows]
    unsigned long long *counters;   // [0] build rows passing the predicates, [1] rows counted
};

static __global__ void __launch_bounds__(256) left_count_kernel(const LeftCountParams p)
{
    unsigned long long n_pass = 0, n_match = 0;
    for (i64 row = (i64)blockIdx.x * blockDim.x + threadIdx.x; row < p.nrows; row += (i64)gridDim.x * blockDim.x) {
        if (!lc_pass(p.f, row)) continue;
        n_pass++;
        if (!typed_valid(p.key, row) || !typed_valid(p.arg, row)) continue;
        const i64 key = load_typed(p.key, row);
        if (p.anchor.bitmap && !bitmap_test(p.anchor, key)) continue;
        jt_probe(p.anchor, key, [&](u64 r) {
            atomicAdd(p.counts + r, 1u);
            n_match++;
        });
    }
    n_pass = (unsigned long long)warp_sum((i64)n_pass);
    n_match = (unsigned long long)warp_sum((i64)n_match);
    if ((threadIdx.x & 31) == 0) {
        if (n_pass) atomicAdd(&p.counters[0], n_pass);
        if (n_match) atomicAdd(&p.counters[1], n_match);
    }
}

// Histogram of the counts of the groups (preserved rows passing `g`): counts below LC_HBINS in block-private shared bins,
// larger ones appended to `big` (at most counted rows / LC_HBINS of them, so `big_cap` sized that way never overflows).
constexpr int LC_HBINS = 1024;
static __global__ void __launch_bounds__(256) count_hist_kernel(const LcFilter g, i64 nrows, const unsigned *__restrict__ counts,
                                                                unsigned *__restrict__ hist, unsigned *__restrict__ big_n, unsigned *__restrict__ big,
                                                                unsigned big_cap)
{
    __shared__ unsigned sh[LC_HBINS];
    for (int i = threadIdx.x; i < LC_HBINS; i += blockDim.x) sh[i] = 0;
    __syncthreads();
    for (i64 row = (i64)blockIdx.x * blockDim.x + threadIdx.x; row < nrows; row += (i64)gridDim.x * blockDim.x) {
        if (!lc_pass(g, row)) continue;
        const unsigned c = __ldg(counts + row);
        if (c < LC_HBINS) {
            atomicAdd(&sh[c], 1u);
        } else {
            const unsigned i = atomicAdd(big_n, 1u);
            if (i < big_cap) big[i] = c;
        }
    }
    __syncthreads();
    for (int i = threadIdx.x; i < LC_HBINS; i += blockDim.x)
        if (sh[i]) atomicAdd(hist + i, sh[i]);
}

// The inner aggregate's rows: (preserved key, count) of every group, empty groups included (their count is NULL or 1 on
// the host).  Warp-aggregated output cursor; row order is unspecified.
static __global__ void __launch_bounds__(256) left_compact_kernel(const LcFilter g, i64 nrows, TypedCol key, const unsigned *__restrict__ counts,
                                                                  i64 *__restrict__ out_key, unsigned *__restrict__ out_cnt,
                                                                  unsigned long long *__restrict__ n_out)
{
    const int lane = threadIdx.x & 31;
    for (i64 base = (i64)blockIdx.x * blockDim.x; base < nrows; base += (i64)gridDim.x * blockDim.x) {
        const i64 row = base + threadIdx.x;
        const bool take = row < nrows && lc_pass(g, row);
        const unsigned m = __ballot_sync(0xffffffffu, take);
        unsigned long long at = 0;
        if (lane == 0 && m) at = atomicAdd(n_out, (unsigned long long)__popc(m));
        at = __shfl_sync(0xffffffffu, at, 0);
        if (take) {
            const i64 i = (i64)at + __popc(m & ((1u << lane) - 1u));
            out_key[i] = load_typed(key, row);
            out_cnt[i] = __ldg(counts + row);
        }
    }
}

}  // namespace pg
