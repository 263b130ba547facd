// scanagg_vm.cuh -- expression-driven scan aggregate: the shapes whose filters or aggregate arguments do not lower to
// ranges and affine products (general OR / NOT, IN and <> on integers, CASE WHEN inside sum / avg / min / max,
// column-to-column comparisons).  The predicate and every aggregate argument are rowvm.cuh programs evaluated per row
// with the reference's value semantics (ExprExec, expr_exec.go:85-530; executeCase :144-246); the group tables,
// partials layout, NULL handling (an aggregate skips NULL arguments, function_aggr.go IgnoreNull) and the exact
// 128-bit finalisation are the generic scan aggregate's (generic_scanagg_kernel, GenericPipeline).
// An aggregate accumulates at ONE scale: every value is rescaled to the plane's scale (the static bound of the
// expression's run-time scale), and a value too large for the int64 partial-sum proof raises the overflow status.
#pragma once
#include "rowvm.cuh"

namespace pg {

struct VmAggParams {
    const RvCode *code;
    int *err;
    i64 nrows, row_base;
    int pred0, pred1;
    // rows.cu (aggregate over a join): iterate the (probe row, build row) pairs instead of the table's rows; the filters
    // were applied while the pairs were made
    const i64 *pair0, *pair1;
    int key_side[2];            // which row id indexes key0 / key1 (0: probe / scanned row, 1: build row)
    int nkeys;
    const uint8_t *key0, *key1;
    const uint8_t *luts;
    int n1, ngroups;
    int nacc;
    int kind[GEN_MAXACC], a0[GEN_MAXACC], a1[GEN_MAXACC], ascale[GEN_MAXACC];
    i64 absmax;                 // |value| bound under which a CTA's int64 partial sums are provably exact
};

template <int NT>
__global__ void __launch_bounds__(NT, 512 / NT)       // <= 128 registers: two 256-thread CTAs per SM hide the interpreter's latencies
vm_scanagg_kernel(const VmAggParams p, i64 *__restrict__ partials /* [grid][G*P] */, i64 *__restrict__ first_row /* [G] preset to 0x7f.. */)
{
    extern __shared__ i64 s_acc[];                 // [G*P][NT]
    __shared__ uint8_t s_lut[2][256];
    __shared__ i64 s_first[64];
    const int G = p.ngroups, P = 1 + 2 * p.nacc;
    auto plane_kind = [&](int plane) { return (plane == 0 || plane > p.nacc || p.kind[plane - 1] == GEN_COUNTV) ? (int)GEN_SUM : p.kind[plane - 1]; };
    for (int i = threadIdx.x; i < G * P * NT; i += NT) {
        const int kind = plane_kind((i / NT) % P);
        s_acc[i] = kind == GEN_MIN ? INT64_MAX : kind == GEN_MAX ? INT64_MIN : 0;
    }
    if (p.nkeys > 0) for (int i = threadIdx.x; i < 512; i += NT) s_lut[i >> 8][i & 255] = p.luts[i];
    if (threadIdx.x < 64) s_first[threadIdx.x] = INT64_MAX;
    __syncthreads();
    i64 *my = s_acc + threadIdx.x;
    int err = 0;
    // one selected row -> its group's planes (`it`: position used for the first-row order of the groups)
    auto accumulate = [&](i64 it, i64 row, i64 row1) {
        int g = 0;
        if (p.nkeys > 0) g = s_lut[0][p.key0[p.key_side[0] ? row1 : row]];
        if (p.nkeys > 1) g = g * p.n1 + s_lut[1][p.key1[p.key_side[1] ? row1 : row]];
        i64 *t = my + (i64)g * P * NT;
        // not "the thread's first row of g": the pre-test queue hands a thread its rows out of order
        if (p.row_base + it < s_first[g]) atomicMin((long long *)&s_first[g], (long long)(p.row_base + it));
        t[0] += 1;
        for (int a = 0; a < p.nacc; a++) {
            const RvVal v = rv_eval(*p.code, p.a0[a], p.a1[a], row, row1, &err);
            if (v.null) continue;
            i64 *slot = t + (i64)(a + 1) * NT;
            t[(i64)(p.nacc + 1 + a) * NT] += 1;
            if (p.kind[a] == GEN_COUNTV) { *slot += 1; continue; }
            i128 x = v.v;
            if (v.scale > p.ascale[a]) { err = RV_ERR_OVERFLOW; continue; }
            x *= rv_pow10(p.ascale[a] - v.scale);
            if (x > (i128)p.absmax || x < -(i128)p.absmax) { err = RV_ERR_OVERFLOW; continue; }
            const i64 xv = (i64)x, cur = *slot;
            *slot = p.kind[a] == GEN_SUM ? cur + xv : p.kind[a] == GEN_MIN ? (xv < cur ? xv : cur) : (xv > cur ? xv : cur);
        }
    };
    if (!p.pair0 && rv_has_pre(*p.code, p.pred0, p.pred1)) {
        // Scan with inline pre-tests: a warp would run the interpreter while ANY of its 32 rows survives them, so the
        // survivors of a block are first compacted into a shared-memory queue and interpreted NT at a time, densely.
        // VM_R rows per thread and step: the pre-tests of the VM_R rows are independent (their loads overlap) and the
        // barriers of the append are paid once per VM_R * NT rows.
        constexpr int VM_R = 4;
        __shared__ i64 s_q[(VM_R + 1) * NT];
        __shared__ int s_woff[VM_R][NT / 32];
        __shared__ int s_cnt;
        __shared__ RvPre s_pre[RV_MAXPRE];
        __shared__ RvCol s_cols[RV_MAXCOL];
        __shared__ unsigned s_masks[RV_MAXMASK][8];
        const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
        const int pre0 = p.code->ins[p.pred0].a, pre1 = p.code->ins[p.pred0].b;
        if (threadIdx.x == 0) s_cnt = 0;
        if (threadIdx.x < RV_MAXPRE) s_pre[threadIdx.x] = p.code->pre[threadIdx.x];
        if (threadIdx.x < RV_MAXCOL) s_cols[threadIdx.x] = p.code->cols[threadIdx.x];
        for (int i = threadIdx.x; i < RV_MAXMASK * 8; i += NT) s_masks[i / 8][i % 8] = p.code->masks[i / 8][i % 8];
        __syncthreads();
        for (i64 base = (i64)blockIdx.x * NT * VM_R; base < p.nrows; base += (i64)gridDim.x * NT * VM_R) {      // block-uniform trip count
            bool pass[VM_R];
            unsigned m[VM_R];
#pragma unroll
            for (int k = 0; k < VM_R; k++) {
                const i64 row = base + (i64)k * NT + threadIdx.x;
                pass[k] = row < p.nrows && rv_pre_smem(s_pre, pre0, pre1, s_cols, s_masks, row, -1);
            }
#pragma unroll
            for (int k = 0; k < VM_R; k++) {
                m[k] = __ballot_sync(0xffffffffu, pass[k]);
                if (lane == 0) s_woff[k][warp] = __popc(m[k]);
            }
            __syncthreads();
            if (threadIdx.x == 0) {
                int acc = s_cnt;
                for (int k = 0; k < VM_R; k++)
                    for (int w = 0; w < NT / 32; w++) { const int c = s_woff[k][w]; s_woff[k][w] = acc; acc += c; }
                s_cnt = acc;
            }
            __syncthreads();
#pragma unroll
            for (int k = 0; k < VM_R; k++)
                if (pass[k]) s_q[s_woff[k][warp] + __popc(m[k] & ((1u << lane) - 1u))] = base + (i64)k * NT + threadIdx.x;
            __syncthreads();
            int n = s_cnt;
            while (n >= NT) {                       // block-uniform
                const i64 r = s_q[n - NT + threadIdx.x];
                if (rv_post(*p.code, p.pred0, p.pred1, r, -1, &err)) accumulate(r, r, -1);
                n -= NT;
            }
            __syncthreads();
            if (threadIdx.x == 0) s_cnt = n;
            __syncthreads();
        }
        if ((int)threadIdx.x < s_cnt) {
            const i64 r = s_q[threadIdx.x];
            if (rv_post(*p.code, p.pred0, p.pred1, r, -1, &err)) accumulate(r, r, -1);
        }
    } else {
        for (i64 it = (i64)blockIdx.x * NT + threadIdx.x; it < p.nrows; it += (i64)gridDim.x * NT) {
            const i64 row = p.pair0 ? p.pair0[it] : it, row1 = p.pair0 ? p.pair1[it] : -1;
            if (!rv_true(*p.code, p.pred0, p.pred1, row, row1, &err)) continue;
            accumulate(it, row, row1);
        }
    }
    if (err) *p.err = err;
    __syncthreads();
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    for (int v = warp; v < G * P; v += NT / 32) {
        const int kind = plane_kind(v % P);
        i64 r = kind == GEN_SUM ? 0 : kind == GEN_MIN ? INT64_MAX : INT64_MIN;
        for (int j = 0; j < NT / 32; j++) {
            const i64 x = s_acc[v * NT + lane + 32 * j];
            r = kind == GEN_SUM ? r + x : kind == GEN_MIN ? (x < r ? x : r) : (x > r ? x : r);
        }
        for (int o = 16; o > 0; o >>= 1) {
            const i64 x = __shfl_xor_sync(0xffffffffu, r, o);
            r = kind == GEN_SUM ? r + x : kind == GEN_MIN ? (x < r ? x : r) : (x > r ? x : r);
        }
        if (lane == 0) partials[(i64)blockIdx.x * (G * P) + v] = r;
    }
    if (threadIdx.x < G && s_first[threadIdx.x] != INT64_MAX)
        atomicMin((long long *)&first_row[threadIdx.x], (long long)s_first[threadIdx.x]);
}

}  // namespace pg
