// scan_kernels.cu -- K2..K7: everything that runs over decoded column blocks.
//
//   K3+K7 fused_scan_kernel   predicate terms -> selection bits -> count / sum / min / max (or mask)
//                             replaces apply(::SelectionExecutor) + eval_on_range + the Base folds over
//                             iterate(::DFColumn): /root/reference/src/tables/selection.jl:133-167,
//                             broadcast.jl:96-133, column.jl:102-126, view.jl:192-206 (nrow)
//   K3    vm_mask_kernel      generic typed VM for arbitrary BlockBroadcasting predicates (broadcast.jl:6-17)
//   K4    range_stage_kernel  range / index-vector stages on running survivor ranks (selection.jl:94-111)
//   K2    str_offsets_kernel  unsafe_remake_offsets! (/root/reference/src/FlatStringsVectors.jl:61-70)
//   K5/K6 gather_* kernels    ColProjExec `buffer .= data[name][range]` + append! (projection.jl:130-133,
//                             materialization.jl:27-40) and the FlatStringsVector gather
//                             (FlatStringsVectors.jl:136-157): warp-aggregated prefix-sum compaction
//
// Decoded bodies keep the reference's block-body layouts (src/io/blocks.jl:2-33); every kernel addresses
// rows as (local block, row in block).  All kernels are HBM-bound streaming kernels: algorithmic bytes
// per row are listed in DESIGN.md.
#include <cuda_runtime.h>
#include <math_constants.h>

#include "kernels.cuh"

namespace dfdb {
namespace {

constexpr unsigned FULL = 0xffffffffu;

__device__ __forceinline__ int lane_id() { return threadIdx.x & 31; }
__device__ __forceinline__ int warp_id() { return threadIdx.x >> 5; }

// ---- column access -----------------------------------------------------------------------------------
__device__ __forceinline__ const uint8_t *col_body(const ColView &c, int lb) { return c.base + c.blk_off[lb]; }
__device__ __forceinline__ const uint8_t *col_values(const ColView &c, int lb, int64_t rows_b)
{
    const uint8_t *body = col_body(c, lb);
    return c.nullable ? body + ((rows_b + 63) >> 6) * 8 : body;
}
__device__ __forceinline__ bool col_missing(const ColView &c, int lb, int64_t r)
{
    if (!c.nullable) return false;
    const unsigned long long *w = reinterpret_cast<const unsigned long long *>(col_body(c, lb));
    return (w[r >> 6] >> (r & 63)) & 1ull;
}

// 64-bit payload of a fixed-width value: integers sign/zero extended, floats as double bits, Bool 0/1
__device__ __forceinline__ unsigned long long load_widen(const uint8_t *p, int kind)
{
    switch (kind) {
    case DFDB_I8: return (unsigned long long)(long long)*reinterpret_cast<const int8_t *>(p);
    case DFDB_I16: return (unsigned long long)(long long)*reinterpret_cast<const int16_t *>(p);
    case DFDB_I32: return (unsigned long long)(long long)*reinterpret_cast<const int32_t *>(p);
    case DFDB_U8: case DFDB_BOOL: return *p;
    case DFDB_U16: return *reinterpret_cast<const uint16_t *>(p);
    case DFDB_U32: return *reinterpret_cast<const uint32_t *>(p);
    case DFDB_F32: return (unsigned long long)__double_as_longlong((double)*reinterpret_cast<const float *>(p));
    default: return *reinterpret_cast<const unsigned long long *>(p);   // 8-byte kinds
    }
}

template <bool WIDE>
__device__ __forceinline__ int64_t row_of(int64_t tile0, int k, int tid)
{
    if (WIDE) return tile0 + (k >> 1) * (2 * SCAN_THREADS) + 2 * tid + (k & 1);
    return tile0 + (int64_t)k * SCAN_THREADS + tid;
}

// values of this thread's 8 rows of one tile; `miss` gets bit k set when row k is missing
template <bool WIDE>
__device__ __forceinline__ void load8(const ColView &c, int lb, int64_t rows_b, int64_t tile0, int tid, unsigned long long (&v)[8],
                                      unsigned &miss)
{
    const uint8_t *vals = col_values(c, lb, rows_b);
    if (WIDE) {
#pragma unroll
        for (int s = 0; s < 4; s++) {
            const int64_t r = tile0 + s * (2 * SCAN_THREADS) + 2 * tid;
            if (r + 1 < rows_b) {
                const ulonglong2 x = __ldcs(reinterpret_cast<const ulonglong2 *>(vals + r * 8));
                v[2 * s] = x.x;
                v[2 * s + 1] = x.y;
            } else {
                v[2 * s] = r < rows_b ? __ldcs(reinterpret_cast<const unsigned long long *>(vals + r * 8)) : 0ull;
                v[2 * s + 1] = 0ull;
            }
        }
    } else {
#pragma unroll
        for (int k = 0; k < 8; k++) {
            const int64_t r = tile0 + (int64_t)k * SCAN_THREADS + tid;
            v[k] = r < rows_b ? load_widen(vals + r * c.elsize, c.kind) : 0ull;
        }
    }
    miss = 0;
    if (c.nullable) {
        const unsigned long long *w = reinterpret_cast<const unsigned long long *>(col_body(c, lb));
#pragma unroll
        for (int k = 0; k < 8; k++) {
            const int64_t r = row_of<WIDE>(tile0, k, tid);
            if (r < rows_b) miss |= (unsigned)((__ldg(w + (r >> 6)) >> (r & 63)) & 1ull) << k;
        }
    }
}

__device__ __forceinline__ bool cmp_code(int code, int c3)   // c3: -1,0,1 or 2 = unordered
{
    if (c3 == 2) return code == 1;
    switch (code) {
    case 0: return c3 == 0;
    case 1: return c3 != 0;
    case 2: return c3 < 0;
    case 3: return c3 <= 0;
    case 4: return c3 > 0;
    default: return c3 >= 0;
    }
}

__device__ __forceinline__ unsigned term_bits(const Term &t, const unsigned long long (&v)[8])
{
    unsigned b = 0;
    if (t.cls == VC_INT) {
        const long long c = t.ci;
#pragma unroll
        for (int k = 0; k < 8; k++) {
            const long long x = (long long)v[k];
            b |= (unsigned)cmp_code(t.code, x < c ? -1 : (x > c ? 1 : 0)) << k;
        }
    } else if (t.cls == VC_UINT) {
        const unsigned long long c = (unsigned long long)t.ci;
#pragma unroll
        for (int k = 0; k < 8; k++) {
            const unsigned long long x = v[k];
            b |= (unsigned)cmp_code(t.code, x < c ? -1 : (x > c ? 1 : 0)) << k;
        }
    } else {
        const double c = t.cf;
#pragma unroll
        for (int k = 0; k < 8; k++) {
            const double x = __longlong_as_double((long long)v[k]);
            const int c3 = (x != x || c != c) ? 2 : (x < c ? -1 : (x > c ? 1 : 0));
            b |= (unsigned)cmp_code(t.code, c3) << k;
        }
    }
    return b;
}

// ---- aggregate accumulators ------------------------------------------------------------------------------
__device__ __forceinline__ void two_sum_add(double &hi, double &lo, double x)
{
    const double t = hi + x;
    const double bb = t - hi;
    lo += (hi - (t - bb)) + (x - bb);   // Knuth two-sum: exact error of hi + x
    hi = t;
}
__device__ __forceinline__ double jl_min(double a, double b) { return (a < b || (a == b && signbit(a))) ? a : b; }
__device__ __forceinline__ double jl_max(double a, double b) { return (a > b || (a == b && !signbit(a))) ? a : b; }

__device__ __forceinline__ void agg_init(AggPartial &a)
{
    a.count = 0; a.nmissing = 0; a.sum_i = 0; a.sum_f = 0.0; a.sum_lo = 0.0;
    a.min_i = 0; a.max_i = 0; a.min_f = 0.0; a.max_f = 0.0; a.has_nan = 0; a.has_value = 0;
}

// fixed-order merge (b follows a in row order)
__device__ __forceinline__ void agg_merge(AggPartial &a, const AggPartial &b, int cls)
{
    a.count += b.count;
    a.nmissing += b.nmissing;
    a.sum_i = (long long)((unsigned long long)a.sum_i + (unsigned long long)b.sum_i);
    two_sum_add(a.sum_f, a.sum_lo, b.sum_f);
    a.sum_lo += b.sum_lo;
    a.has_nan |= b.has_nan;
    if (b.has_value) {
        if (!a.has_value) {
            a.min_i = b.min_i; a.max_i = b.max_i; a.min_f = b.min_f; a.max_f = b.max_f;
        } else if (cls == VC_FLT) {
            a.min_f = jl_min(a.min_f, b.min_f);
            a.max_f = jl_max(a.max_f, b.max_f);
        } else if (cls == VC_UINT) {
            if ((unsigned long long)b.min_i < (unsigned long long)a.min_i) a.min_i = b.min_i;
            if ((unsigned long long)b.max_i > (unsigned long long)a.max_i) a.max_i = b.max_i;
        } else {
            if (b.min_i < a.min_i) a.min_i = b.min_i;
            if (b.max_i > a.max_i) a.max_i = b.max_i;
        }
        a.has_value = 1;
    }
}

__device__ __forceinline__ AggPartial agg_shfl_down(const AggPartial &a, int d)
{
    AggPartial b;
    b.count = __shfl_down_sync(FULL, a.count, d);
    b.nmissing = __shfl_down_sync(FULL, a.nmissing, d);
    b.sum_i = __shfl_down_sync(FULL, a.sum_i, d);
    b.sum_f = __shfl_down_sync(FULL, a.sum_f, d);
    b.sum_lo = __shfl_down_sync(FULL, a.sum_lo, d);
    b.min_i = __shfl_down_sync(FULL, a.min_i, d);
    b.max_i = __shfl_down_sync(FULL, a.max_i, d);
    b.min_f = __shfl_down_sync(FULL, a.min_f, d);
    b.max_f = __shfl_down_sync(FULL, a.max_f, d);
    b.has_nan = __shfl_down_sync(FULL, a.has_nan, d);
    b.has_value = __shfl_down_sync(FULL, a.has_value, d);
    return b;
}

// warp-shuffle tree then a sequential fold over the warps of the CTA: the combination order is a fixed
// function of the thread index, so floating-point results are reproducible run to run
__device__ void agg_block_reduce(AggPartial &a, int cls, AggPartial *smem /* [SCAN_THREADS/32] */)
{
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) {
        AggPartial b = agg_shfl_down(a, d);
        if (lane_id() + d < 32) agg_merge(a, b, cls);
    }
    if (lane_id() == 0) smem[warp_id()] = a;
    __syncthreads();
    if (threadIdx.x == 0) {
        AggPartial r = smem[0];
        for (int w = 1; w < SCAN_THREADS / 32; w++) agg_merge(r, smem[w], cls);
        a = r;
    }
    __syncthreads();
}

// ---- K3+K7 fused ---------------------------------------------------------------------------------------
// AGG: 0 = count only, 1 = integer/Bool values, 2 = floating values
template <int AGG, bool WIDE, bool EMIT>
__global__ void __launch_bounds__(SCAN_THREADS) fused_scan_kernel(const FusedArgs A)
{
    __shared__ AggPartial red[SCAN_THREADS / 32];
    const int tid = threadIdx.x;
    const Geometry g = A.g;
    const int nunits = g.nblocks * g.segs_per_block;
    for (int unit = blockIdx.x; unit < nunits; unit += gridDim.x) {
        const int lb = unit / g.segs_per_block;
        const int seg = unit - lb * g.segs_per_block;
        const int64_t rows_b = block_rows(g, lb);
        const int64_t row0 = (int64_t)seg * g.seg_rows;
        int64_t row1 = row0 + g.seg_rows;
        if (row1 > rows_b) row1 = rows_b;
        AggPartial acc;
        agg_init(acc);
        if (g.dead && g.dead[lb]) {
            // ruled out by the zone maps: no row selected, the body was not decoded and is not read
            if (EMIT)
                for (int64_t r0 = row0 + (int64_t)tid * 32; r0 < row1; r0 += (int64_t)SCAN_THREADS * 32) A.mask_out[(int64_t)lb * g.wpb + (r0 >> 5)] = 0u;
            if (tid == 0) A.partials[unit] = acc;
            continue;
        }
        for (int64_t tile0 = row0; tile0 < row1; tile0 += TILE_ROWS) {
            unsigned long long av[8];
            unsigned amiss = 0;
            if (AGG) load8<WIDE>(A.agg_col, lb, rows_b, tile0, tid, av, amiss);
            // valid rows of this thread
            unsigned m = 0;
#pragma unroll
            for (int k = 0; k < 8; k++) m |= (unsigned)(row_of<WIDE>(tile0, k, tid) < row1) << k;
            if (A.const_false) m = 0;
            if (A.mask_in) {
                // non-wide mapping only: row k of this thread is bit `lane` of word (tile0 + k*256 + warp*32) / 32
                unsigned sel = 0;
#pragma unroll
                for (int k = 0; k < 8; k++) {
                    const int64_t r0 = tile0 + (int64_t)k * SCAN_THREADS + warp_id() * 32;
                    if (r0 < rows_b) sel |= ((__ldg(A.mask_in + (int64_t)lb * g.wpb + (r0 >> 5)) >> lane_id()) & 1u) << k;
                }
                m &= sel;
            }
            for (int t = 0; t < A.nterms; t++) {
                const Term &term = A.term[t];
                if (term.constant_result >= 0) continue;   // folded (a false one sets const_false)
                unsigned long long v[8];
                unsigned miss;
                load8<WIDE>(A.term_col[t], lb, rows_b, tile0, tid, v, miss);
                m &= term_bits(term, v) & ~miss;           // missing compares as false under coalesce(..., false)
            }
            if (EMIT) {
#pragma unroll
                for (int k = 0; k < 8; k++) {
                    const unsigned word = __ballot_sync(FULL, (m >> k) & 1u);
                    const int64_t r0 = tile0 + (int64_t)k * SCAN_THREADS + warp_id() * 32;
                    if (lane_id() == 0 && r0 < rows_b) A.mask_out[(int64_t)lb * g.wpb + (r0 >> 5)] = word;
                }
            }
            acc.count += __popc(m);
            if (AGG) {
                acc.nmissing += __popc(m & amiss);
                const unsigned use = m & ~amiss;
#pragma unroll
                for (int k = 0; k < 8; k++) {
                    if ((use >> k) & 1u) {
                        if (AGG == 2) {
                            const double x = __longlong_as_double((long long)av[k]);
                            if (x != x) acc.has_nan = 1;
                            else {
                                two_sum_add(acc.sum_f, acc.sum_lo, x);
                                if (!acc.has_value) { acc.min_f = x; acc.max_f = x; acc.has_value = 1; }
                                else { acc.min_f = jl_min(acc.min_f, x); acc.max_f = jl_max(acc.max_f, x); }
                            }
                        } else {
                            const long long x = (long long)av[k];
                            acc.sum_i = (long long)((unsigned long long)acc.sum_i + (unsigned long long)x);
                            if (!acc.has_value) { acc.min_i = x; acc.max_i = x; acc.has_value = 1; }
                            else if (A.agg_cls == VC_UINT) {
                                if ((unsigned long long)x < (unsigned long long)acc.min_i) acc.min_i = x;
                                if ((unsigned long long)x > (unsigned long long)acc.max_i) acc.max_i = x;
                            } else {
                                if (x < acc.min_i) acc.min_i = x;
                                if (x > acc.max_i) acc.max_i = x;
                            }
                        }
                    }
                }
            }
        }
        agg_block_reduce(acc, AGG == 2 ? VC_FLT : A.agg_cls, red);
        if (tid == 0) A.partials[unit] = acc;
    }
}

// final fold of the per-unit partials: thread t folds units t, t+256, ... in order, then the fixed tree
__global__ void __launch_bounds__(SCAN_THREADS) agg_finalize_kernel(const AggPartial *partials, int nunits, int cls, AggPartial *result)
{
    __shared__ AggPartial red[SCAN_THREADS / 32];
    AggPartial acc;
    agg_init(acc);
    // contiguous chunk per thread keeps row order: thread t owns units [t*per, (t+1)*per)
    const int per = (nunits + SCAN_THREADS - 1) / SCAN_THREADS;
    const int lo = threadIdx.x * per;
    int hi = lo + per;
    if (hi > nunits) hi = nunits;
    for (int u = lo; u < hi; u++) agg_merge(acc, partials[u], cls);
    agg_block_reduce(acc, cls, red);
    if (threadIdx.x == 0) {
        // renormalise the compensated sum; NaN anywhere makes sum / min / max NaN (Julia propagates)
        double s = acc.sum_f + acc.sum_lo;
        acc.sum_lo = (acc.sum_f - s) + acc.sum_lo;
        acc.sum_f = s;
        if (acc.has_nan) { acc.sum_f = CUDART_NAN; acc.sum_lo = 0.0; acc.min_f = CUDART_NAN; acc.max_f = CUDART_NAN; }
        *result = acc;
    }
}

// ---- typed VM ---------------------------------------------------------------------------------------------
struct VmStack {
    unsigned long long v[VM_MAX_STACK];
    int len[VM_MAX_STACK];   // strings: byte length
    unsigned miss;           // bit i = entry i is missing
};

__device__ __forceinline__ int cmp_int_flt(long long a, bool uns, double b)
{
    if (b != b) return 2;
    if (uns) {
        const unsigned long long ua = (unsigned long long)a;
        if (b < 0.0) return 1;
        if (b >= 18446744073709551616.0) return -1;
        const unsigned long long tb = (unsigned long long)b;
        if (ua < tb) return -1;
        if (ua > tb) return 1;
        return (double)tb < b ? -1 : 0;
    }
    if (b >= 9223372036854775808.0) return -1;
    if (b < -9223372036854775808.0) return 1;
    const long long tb = (long long)b;
    if (a < tb) return -1;
    if (a > tb) return 1;
    const double frac = b - (double)tb;
    return frac > 0.0 ? -1 : (frac < 0.0 ? 1 : 0);
}
__device__ __forceinline__ int cmp_u(unsigned long long a, unsigned long long b) { return a < b ? -1 : (a > b ? 1 : 0); }
__device__ __forceinline__ int cmp_s(long long a, long long b) { return a < b ? -1 : (a > b ? 1 : 0); }

__device__ __forceinline__ int cmp3_pair(int cp, unsigned long long a, unsigned long long b)
{
    switch (cp) {
    case CP_II: return cmp_s((long long)a, (long long)b);
    case CP_UU: return cmp_u(a, b);
    case CP_IU: return (long long)a < 0 ? -1 : cmp_u(a, b);
    case CP_UI: return (long long)b < 0 ? 1 : cmp_u(a, b);
    case CP_IF: return cmp_int_flt((long long)a, false, __longlong_as_double((long long)b));
    case CP_UF: return cmp_int_flt((long long)a, true, __longlong_as_double((long long)b));
    case CP_FI: { int c = cmp_int_flt((long long)b, false, __longlong_as_double((long long)a)); return c == 2 ? 2 : -c; }
    case CP_FU: { int c = cmp_int_flt((long long)b, true, __longlong_as_double((long long)a)); return c == 2 ? 2 : -c; }
    default: {
        const double x = __longlong_as_double((long long)a), y = __longlong_as_double((long long)b);
        return (x != x || y != y) ? 2 : (x < y ? -1 : (x > y ? 1 : 0));
    }
    }
}

__device__ __forceinline__ int str_cmp(const uint8_t *a, int la, const uint8_t *b, int lb)
{
    const int m = la < lb ? la : lb;
    for (int i = 0; i < m; i++) {
        const int x = a[i], y = b[i];
        if (x != y) return x < y ? -1 : 1;
    }
    return la < lb ? -1 : (la > lb ? 1 : 0);
}

__device__ __forceinline__ long long wrap_int(long long v, int bytes, bool uns)
{
    if (bytes >= 8) return v;
    const int bits = bytes * 8;
    const unsigned long long m = (1ull << bits) - 1ull;
    unsigned long long u = (unsigned long long)v & m;
    if (!uns && (u >> (bits - 1))) u |= ~m;
    return (long long)u;
}

__device__ __forceinline__ double to_double(unsigned long long v, int cls)
{
    switch (cls) {
    case 3: return __longlong_as_double((long long)v);
    case 2: return (double)v;
    default: return (double)(long long)v;   // signed / Bool
    }
}

// evaluates the program for row r of local block lb; returns payload + missing flag of the result
__device__ void vm_eval(const VmProgram *__restrict__ P, const ColView *slots, const Geometry &g, int lb, int64_t rows_b, int64_t r,
                        unsigned long long &out, bool &out_miss, int *error_flag)
{
    VmStack S;
    S.miss = 0;
    int sp = 0;
    const int n = P->ninstr;
    for (int pc = 0; pc < n; pc++) {
        const VmInstr I = P->instr[pc];
        switch (I.op) {
        case V_LOAD: {
            const ColView &c = slots[I.a];
            S.miss &= ~(1u << sp);
            if (c.cls == VC_STR) {
                const uint8_t *body = col_body(c, lb);
                const int sz = reinterpret_cast<const int32_t *>(body + 4)[r];
                S.v[sp] = (unsigned long long)(uintptr_t)(body + 4 + 4 * rows_b + c.str_off[(int64_t)lb * g.block_size + r]);
                S.len[sp] = sz;
                if (sz < 0) { S.miss |= 1u << sp; S.len[sp] = 0; }
            } else {
                const bool ms = col_missing(c, lb, r);
                S.v[sp] = ms ? 0ull : load_widen(col_values(c, lb, rows_b) + r * c.elsize, c.kind);
                if (ms) S.miss |= 1u << sp;
            }
            sp++;
            break;
        }
        case V_CONST:
            S.v[sp] = (unsigned long long)P->consts[I.imm];
            S.miss &= ~(1u << sp);
            sp++;
            break;
        case V_CONSTSTR:
            S.v[sp] = (unsigned long long)(uintptr_t)(P->strpool + I.imm);
            S.len[sp] = (int)I.a | ((int)I.b << 8);
            S.miss &= ~(1u << sp);
            sp++;
            break;
        case V_CMP: case V_STRCMP: case V_STRNUM: case V_STARTSWITH: case V_ENDSWITH: {
            const int ia = sp - 2, ib = sp - 1;
            const bool ms = ((S.miss >> ia) | (S.miss >> ib)) & 1u;
            bool res = false;
            if (!ms) {
                if (I.op == V_CMP) res = cmp_code(I.a, cmp3_pair(I.b, S.v[ia], S.v[ib]));
                else if (I.op == V_STRNUM) res = I.a == 1;
                else {
                    const uint8_t *pa = reinterpret_cast<const uint8_t *>((uintptr_t)S.v[ia]);
                    const uint8_t *pb = reinterpret_cast<const uint8_t *>((uintptr_t)S.v[ib]);
                    const int la = S.len[ia], lb2 = S.len[ib];
                    if (I.op == V_STRCMP) res = cmp_code(I.a, str_cmp(pa, la, pb, lb2));
                    else if (lb2 > la) res = false;
                    else {
                        const uint8_t *q = I.op == V_STARTSWITH ? pa : pa + (la - lb2);
                        res = true;
                        for (int i = 0; i < lb2; i++) if (q[i] != pb[i]) { res = false; break; }
                    }
                }
            }
            sp--;
            S.v[ia] = res ? 1ull : 0ull;
            S.miss = (S.miss & ~(3u << ia)) | ((unsigned)ms << ia);
            break;
        }
        case V_AND: case V_OR: case V_XOR: {
            const int ia = sp - 2, ib = sp - 1;
            const bool ma = (S.miss >> ia) & 1u, mb = (S.miss >> ib) & 1u;
            const bool va = S.v[ia] != 0, vb = S.v[ib] != 0;
            bool res, ms;
            if (I.op == V_AND) {
                if ((!ma && !va) || (!mb && !vb)) { res = false; ms = false; }
                else if (ma || mb) { res = false; ms = true; }
                else { res = true; ms = false; }
            } else if (I.op == V_OR) {
                if ((!ma && va) || (!mb && vb)) { res = true; ms = false; }
                else if (ma || mb) { res = false; ms = true; }
                else { res = false; ms = false; }
            } else {
                ms = ma || mb;
                res = !ms && (va != vb);
            }
            sp--;
            S.v[ia] = res ? 1ull : 0ull;
            S.miss = (S.miss & ~(3u << ia)) | ((unsigned)ms << ia);
            break;
        }
        case V_NOT: {
            const int ia = sp - 1;
            if (!((S.miss >> ia) & 1u)) S.v[ia] = S.v[ia] ? 0ull : 1ull;
            break;
        }
        case V_ISMISSING: {
            const int ia = sp - 1;
            S.v[ia] = (S.miss >> ia) & 1u;
            S.miss &= ~(1u << ia);
            break;
        }
        case V_COALESCE: {
            const int ia = sp - 2, ib = sp - 1;
            if ((S.miss >> ia) & 1u) { S.v[ia] = S.v[ib]; S.len[ia] = S.len[ib]; }
            sp--;
            S.miss &= ~(3u << ia);
            break;
        }
        case V_IN: {
            const int ia = sp - 1;
            if (!((S.miss >> ia) & 1u)) {
                const int cnt = (int)I.a | ((int)I.b << 8);
                const unsigned long long x = S.v[ia];
                bool hit = false;
                for (int q = 0; q < cnt && !hit; q++) {
                    const long long sv = P->consts[I.imm + q];
                    hit = I.c ? (sv >= 0 && x == (unsigned long long)sv) : ((long long)x == sv);
                }
                S.v[ia] = hit ? 1ull : 0ull;
            }
            break;
        }
        case V_ARITH: {
            const bool unary = I.a == 5;
            const int ia = unary ? sp - 1 : sp - 2, ib = sp - 1;
            const bool ms = unary ? ((S.miss >> ia) & 1u) : (((S.miss >> ia) | (S.miss >> ib)) & 1u);
            const int ca = I.b & 15, cb = I.b >> 4;
            unsigned long long res = 0;
            if (!ms) {
                if (I.c & 0x40) {
                    double x = to_double(S.v[ia], ca), y = unary ? 0.0 : to_double(S.v[ib], cb);
                    const bool f32 = (I.c & 15) == 4;
                    if (f32) { x = (double)(float)x; y = (double)(float)y; }
                    double z;
                    switch (I.a) {
                    case 0: z = x + y; break;
                    case 1: z = x - y; break;
                    case 2: z = x * y; break;
                    case 3: z = x / y; break;
                    case 4: z = fmod(x, y); break;
                    default: z = -x; break;
                    }
                    if (f32) z = (double)(float)z;
                    res = (unsigned long long)__double_as_longlong(z);
                } else {
                    const bool uns = I.c & 0x80;
                    const unsigned long long ux = S.v[ia], uy = unary ? 0ull : S.v[ib];
                    unsigned long long z;
                    switch (I.a) {
                    case 0: z = ux + uy; break;
                    case 1: z = ux - uy; break;
                    case 2: z = ux * uy; break;
                    case 4:
                        if (uy == 0ull) { atomicExch(error_flag, DFDB_ERR_DIVIDE); z = 0ull; }
                        else if (uns) z = ux % uy;
                        else z = ((long long)uy == -1ll) ? 0ull : (unsigned long long)((long long)ux % (long long)uy);
                        break;
                    default: z = 0ull - ux; break;
                    }
                    res = (unsigned long long)wrap_int((long long)z, I.c & 15, uns);
                }
            }
            if (!unary) sp--;
            S.v[ia] = res;
            S.miss = (S.miss & ~((unary ? 1u : 3u) << ia)) | ((unsigned)ms << ia);
            break;
        }
        default: break;
        }
    }
    out = S.v[0];
    out_miss = S.miss & 1u;
}

__global__ void __launch_bounds__(SCAN_THREADS) vm_mask_kernel(const VmArgs A)
{
    const Geometry g = A.g;
    const int tiles_per_block = (int)((g.block_size + TILE_ROWS - 1) / TILE_ROWS);
    const int64_t ntiles = (int64_t)g.nblocks * tiles_per_block;
    for (int64_t tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
        const int lb = (int)(tile / tiles_per_block);
        const int64_t tile0 = (tile - (int64_t)lb * tiles_per_block) * TILE_ROWS;
        const int64_t rows_b = block_rows(g, lb);
#pragma unroll 1
        for (int k = 0; k < ROWS_PER_THREAD; k++) {
            const int64_t r0 = tile0 + (int64_t)k * SCAN_THREADS + warp_id() * 32;
            if (r0 >= rows_b) continue;                                  // warp-uniform
            const int64_t r = r0 + lane_id();
            const int64_t widx = (int64_t)lb * g.wpb + (r0 >> 5);
            bool sel = r < rows_b && !(g.dead && g.dead[lb]);              // (zone maps: the block is not decoded, nothing is evaluated)
            if (A.mask_in) sel = sel && ((A.mask_in[widx] >> lane_id()) & 1u);
            bool res = false;
            if (sel) {
                unsigned long long v;
                bool ms;
                vm_eval(A.prog, A.slot, g, lb, rows_b, r, v, ms, A.error_flag);
                res = !ms && v != 0ull;
            }
            const unsigned word = __ballot_sync(FULL, res);
            if (lane_id() == 0) A.mask_out[widx] = word;
        }
    }
}

// ---- K4: range stages --------------------------------------------------------------------------------------
__device__ __forceinline__ bool stage_member(const RangeArgs &a, int64_t rank1)
{
    if (a.kind == ST_RANGE) {
        if (a.step > 0) return rank1 >= a.start && rank1 <= a.stop && (rank1 - a.start) % a.step == 0;
        return rank1 <= a.start && rank1 >= a.stop && (a.start - rank1) % (-a.step) == 0;
    }
    int64_t lo = 0, hi = a.nidx - 1;
    while (lo <= hi) {
        const int64_t mid = (lo + hi) >> 1;
        const int64_t v = a.idx[mid];
        if (v == rank1) return true;
        if (v < rank1) lo = mid + 1; else hi = mid - 1;
    }
    return false;
}

__global__ void __launch_bounds__(SCAN_THREADS) fill_mask_kernel(const Geometry g, uint32_t *mask)
{
    const int64_t total = (int64_t)g.nblocks * g.wpb;
    for (int64_t w = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; w < total; w += (int64_t)gridDim.x * blockDim.x) {
        const int lb = (int)(w / g.wpb);
        const int64_t r0 = (w - (int64_t)lb * g.wpb) * 32;
        const int64_t rows_b = block_rows(g, lb);
        uint32_t word = 0;
        if (r0 + 32 <= rows_b) word = 0xffffffffu;
        else if (r0 < rows_b) word = (1u << (rows_b - r0)) - 1u;
        mask[w] = word;
    }
}

// one warp per block: sums the popcounts of the block's mask words
__global__ void __launch_bounds__(SCAN_THREADS) block_counts_kernel(const Geometry g, const uint32_t *mask, int64_t *counts)
{
    const int warps = gridDim.x * (SCAN_THREADS / 32);
    for (int lb = blockIdx.x * (SCAN_THREADS / 32) + warp_id(); lb < g.nblocks; lb += warps) {
        const uint32_t *m = mask + (int64_t)lb * g.wpb;
        int c = 0;
        for (int w = lane_id(); w < g.wpb; w += 32) c += __popc(m[w]);
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) c += __shfl_xor_sync(FULL, c, d);
        if (lane_id() == 0) counts[lb] = c;
    }
}

// single CTA exclusive scan of n int64 (n up to a few hundred thousand); out[n] = total
__global__ void __launch_bounds__(1024) exclusive_scan_kernel(const int64_t *in, int64_t *out, int n)
{
    __shared__ int64_t warp_tot[32];
    __shared__ int64_t carry_s;
    const int per = (n + 1023) / 1024;
    const int lo = threadIdx.x * per;
    int hi = lo + per;
    if (hi > n) hi = n;
    int64_t s = 0;
    for (int i = lo; i < hi; i++) s += in[i];
    // block exclusive scan of s
    int64_t incl = s;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const int64_t v = __shfl_up_sync(FULL, incl, d);
        if (lane_id() >= d) incl += v;
    }
    if (lane_id() == 31) warp_tot[warp_id()] = incl;
    __syncthreads();
    if (warp_id() == 0) {
        int64_t t = warp_tot[lane_id()];
        int64_t ti = t;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const int64_t v = __shfl_up_sync(FULL, ti, d);
            if (lane_id() >= d) ti += v;
        }
        warp_tot[lane_id()] = ti - t;
        if (lane_id() == 31) carry_s = ti;
    }
    __syncthreads();
    int64_t run = warp_tot[warp_id()] + incl - s;
    for (int i = lo; i < hi; i++) { const int64_t v = in[i]; out[i] = run; run += v; }
    if (threadIdx.x == 0) out[n] = carry_s;
}

// one warp per block walks the block's mask words in order with a running survivor rank
__global__ void __launch_bounds__(SCAN_THREADS) range_stage_kernel(const RangeArgs A)
{
    const Geometry g = A.g;
    const int warps = gridDim.x * (SCAN_THREADS / 32);
    for (int lb = blockIdx.x * (SCAN_THREADS / 32) + warp_id(); lb < g.nblocks; lb += warps) {
        uint32_t *m = A.mask + (int64_t)lb * g.wpb;
        const int64_t rows_b = block_rows(g, lb);
        int64_t base = A.dense ? (g.blk_lo + lb) * g.block_size : A.blk_base[lb] + A.rank_offset;
        for (int w0 = 0; w0 < g.wpb; w0 += 32) {
            const int w = w0 + lane_id();
            uint32_t word = 0;
            if (w < g.wpb) {
                if (A.dense) {
                    const int64_t r0 = (int64_t)w * 32;
                    word = r0 + 32 <= rows_b ? 0xffffffffu : (r0 < rows_b ? (1u << (rows_b - r0)) - 1u : 0u);
                } else word = m[w];
            }
            // exclusive prefix of popcounts over the 32 words held by the warp
            const int c = __popc(word);
            int incl = c;
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) {
                const int v = __shfl_up_sync(FULL, incl, d);
                if (lane_id() >= d) incl += v;
            }
            int64_t rank = base + (incl - c);
            uint32_t keep = 0, rest = word;
            while (rest) {
                const int bit = __ffs(rest) - 1;
                rest &= rest - 1;
                rank++;
                if (stage_member(A, rank)) keep |= 1u << bit;
            }
            if (w < g.wpb) m[w] = keep;
            base += __shfl_sync(FULL, incl, 31);
        }
    }
}

// ---- K2: string offsets -------------------------------------------------------------------------------------
// one warp per block: exclusive prefix sum of max(size, 0) in row order
// (blocks outside [lo, hi) and blocks flagged in `dead` were not decoded for this scan: their bodies are stale)
// A body whose size table does not describe exactly the bytes that follow it is corrupt (the reference's unsafe_read on the
// block's IOBuffer throws EOFError there, src/io/blocks.jl:62-71): status 5 unless 4 + 4 * rows + datasize == origin and the
// sizes add up to datasize -- no consumer kernel then reads past the decoded slot.
__global__ void __launch_bounds__(SCAN_THREADS) str_offsets_kernel(const Geometry g, const ColView col, int32_t *str_off, int32_t *status,
                                                                  const int32_t *origin, int lo, int hi, const uint8_t *dead)
{
    const int warps = gridDim.x * (SCAN_THREADS / 32);
    for (int lb = lo + blockIdx.x * (SCAN_THREADS / 32) + warp_id(); lb < hi; lb += warps) {
        if (dead && dead[lb]) continue;
        const uint8_t *body = col_body(col, lb);
        const int64_t rows_b = block_rows(g, lb);
        const int32_t datasize = *reinterpret_cast<const int32_t *>(body);
        const int32_t *sizes = reinterpret_cast<const int32_t *>(body + 4);
        int32_t *out = str_off + (int64_t)lb * g.block_size;
        long long run = 0;
        // each lane takes 4 consecutive rows per step (one 16-byte load when aligned is not guaranteed: body+4)
        if (datasize < 0 || 4 + 4 * rows_b + (int64_t)datasize != (int64_t)origin[lb]) {
            if (lane_id() == 0) status[lb] = 5;
            continue;
        }
        for (int64_t r0 = 0; r0 < rows_b; r0 += 128) {
            int s[4];
            long long local = 0;
#pragma unroll
            for (int j = 0; j < 4; j++) {
                const int64_t r = r0 + lane_id() * 4 + j;
                s[j] = r < rows_b ? sizes[r] : 0;
                if (s[j] < 0) s[j] = 0;
                local += s[j];
            }
            long long incl = local;
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) {
                const long long v = __shfl_up_sync(FULL, incl, d);
                if (lane_id() >= d) incl += v;
            }
            long long o = run + (incl - local);
#pragma unroll
            for (int j = 0; j < 4; j++) {
                const int64_t r = r0 + lane_id() * 4 + j;
                if (r < rows_b) out[r] = (int32_t)o;
                o += s[j];
            }
            run += __shfl_sync(FULL, incl, 31);
        }
        if (lane_id() == 0 && run != datasize) status[lb] = 5;   // sizes do not add up to datasize: corrupt body
    }
}

// ---- zone maps: one CTA per block --------------------------------------------------------------------------------
__global__ void __launch_bounds__(SCAN_THREADS) zone_map_kernel(const Geometry g, const ColView col, ZoneOut *out)
{
    __shared__ unsigned long long s_min[SCAN_THREADS / 32], s_max[SCAN_THREADS / 32];
    __shared__ long long s_null[SCAN_THREADS / 32];
    __shared__ int s_flags[SCAN_THREADS / 32];
    for (int lb = blockIdx.x; lb < g.nblocks; lb += gridDim.x) {
        const int64_t rows_b = block_rows(g, lb);
        const uint8_t *vals = col_values(col, lb, rows_b);
        const int cls = col.cls;
        unsigned long long mn = 0, mx = 0;
        long long nulls = 0;
        int flags = 0;
        for (int64_t r = threadIdx.x; r < rows_b; r += SCAN_THREADS) {
            if (col_missing(col, lb, r)) { nulls++; continue; }
            const unsigned long long v = load_widen(vals + r * col.elsize, col.kind);
            if (cls == VC_FLT) {
                const double x = __longlong_as_double((long long)v);
                if (x != x) { flags |= 2; continue; }
                if (!(flags & 1)) { mn = mx = v; flags |= 1; }
                else {
                    if (x < __longlong_as_double((long long)mn)) mn = v;
                    if (x > __longlong_as_double((long long)mx)) mx = v;
                }
            } else if (cls == VC_UINT || cls == VC_BOOL) {
                if (!(flags & 1)) { mn = mx = v; flags |= 1; }
                else { if (v < mn) mn = v; if (v > mx) mx = v; }
            } else {
                if (!(flags & 1)) { mn = mx = v; flags |= 1; }
                else { if ((long long)v < (long long)mn) mn = v; if ((long long)v > (long long)mx) mx = v; }
            }
        }
        auto merge = [&](unsigned long long omn, unsigned long long omx, long long onull, int ofl) {
            nulls += onull;
            if (ofl & 1) {
                if (!(flags & 1)) { mn = omn; mx = omx; }
                else if (cls == VC_FLT) {
                    if (__longlong_as_double((long long)omn) < __longlong_as_double((long long)mn)) mn = omn;
                    if (__longlong_as_double((long long)omx) > __longlong_as_double((long long)mx)) mx = omx;
                } else if (cls == VC_UINT || cls == VC_BOOL) {
                    if (omn < mn) mn = omn;
                    if (omx > mx) mx = omx;
                } else {
                    if ((long long)omn < (long long)mn) mn = omn;
                    if ((long long)omx > (long long)mx) mx = omx;
                }
            }
            flags |= ofl;
        };
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) {
            const unsigned long long omn = __shfl_down_sync(FULL, mn, d), omx = __shfl_down_sync(FULL, mx, d);
            const long long onull = __shfl_down_sync(FULL, nulls, d);
            const int ofl = __shfl_down_sync(FULL, flags, d);
            if (lane_id() + d < 32) merge(omn, omx, onull, ofl);
        }
        if (lane_id() == 0) { s_min[warp_id()] = mn; s_max[warp_id()] = mx; s_null[warp_id()] = nulls; s_flags[warp_id()] = flags; }
        __syncthreads();
        if (threadIdx.x == 0) {
            for (int w = 1; w < SCAN_THREADS / 32; w++) merge(s_min[w], s_max[w], s_null[w], s_flags[w]);
            ZoneOut z;
            z.min_bits = mn; z.max_bits = mx; z.null_count = nulls; z.flags = flags; z.pad = 0;
            out[lb] = z;
        }
        __syncthreads();
    }
}

// ---- group-by reduce -----------------------------------------------------------------------------------------------
// One thread per selected row.  A group is identified by a slot of an open-addressing table that stores a ROW of the group
// (`rep`), not the key: keys are compared by reading the key columns of that row again, which works for any number and
// type of key columns (strings included) without a key store.  Equality is Julia's isequal, the relation RobinDict uses in
// the reference's stub (aggregate.jl:7-27): missing equals missing, NaN equals NaN, -0.0 differs from 0.0.
// Counts, integer sums, minima and maxima are exact and order-independent (atomics on integers); Float64 sums are atomic
// adds in arrival order: reproducible to rounding, not bit for bit (stated in DESIGN.md).
__device__ __forceinline__ unsigned long long gmix(unsigned long long x)
{
    x += 0x9E3779B97F4A7C15ull;
    x = (x ^ (x >> 30)) * 0xBF58476D1CE4E5B9ull;
    x = (x ^ (x >> 27)) * 0x94D049BB133111EBull;
    return x ^ (x >> 31);
}
// isequal image of a fixed-width key: one NaN per float kind, every other value its own bits (-0.0 and 0.0 differ).
// Float16 and Char are read at their own width here; load_widen serves the numeric kinds of the scan paths only.
__device__ __forceinline__ unsigned long long key_bits(int kind, const uint8_t *p)
{
    switch (kind) {
    case DFDB_F16: {
        const unsigned h = *reinterpret_cast<const uint16_t *>(p);
        return ((h & 0x7c00u) == 0x7c00u && (h & 0x3ffu)) ? 0x7e00ull : h;
    }
    case DFDB_CHAR: return *reinterpret_cast<const uint32_t *>(p);
    case DFDB_F32: case DFDB_F64: {
        const unsigned long long v = load_widen(p, kind);
        const double x = __longlong_as_double((long long)v);
        return x != x ? 0x7ff8000000000000ull : v;
    }
    default: return load_widen(p, kind);
    }
}
__device__ unsigned long long group_key_hash(const GroupArgs &A, int lb, int64_t rows_b, int64_t r)
{
    unsigned long long h = 0x243F6A8885A308D3ull;
    for (int k = 0; k < A.nkeys; k++) {
        const ColView &c = A.key[k];
        if (c.cls == VC_STR) {
            const uint8_t *body = col_body(c, lb);
            const int sz = reinterpret_cast<const int32_t *>(body + 4)[r];
            const uint8_t *p = body + 4 + 4 * rows_b + c.str_off[(int64_t)lb * A.g.block_size + r];
            unsigned long long f = 0xCBF29CE484222325ull;
            for (int i = 0; i < sz; i++) f = (f ^ p[i]) * 0x100000001B3ull;
            h = gmix(h ^ f ^ ((unsigned long long)(unsigned)sz << 32));
        } else if (col_missing(c, lb, r)) {
            h = gmix(h ^ 0xA5A5A5A5A5A5A5A5ull);
        } else {
            h = gmix(h ^ key_bits(c.kind, col_values(c, lb, rows_b) + r * c.elsize));
        }
    }
    return h;
}
__device__ bool group_keys_equal(const GroupArgs &A, int lb1, int64_t r1, int lb2, int64_t r2)
{
    const int64_t rows1 = block_rows(A.g, lb1), rows2 = block_rows(A.g, lb2);
    for (int k = 0; k < A.nkeys; k++) {
        const ColView &c = A.key[k];
        if (c.cls == VC_STR) {
            const uint8_t *b1 = col_body(c, lb1), *b2 = col_body(c, lb2);
            const int s1 = reinterpret_cast<const int32_t *>(b1 + 4)[r1], s2 = reinterpret_cast<const int32_t *>(b2 + 4)[r2];
            if (s1 != s2) return false;
            const uint8_t *p1 = b1 + 4 + 4 * rows1 + c.str_off[(int64_t)lb1 * A.g.block_size + r1];
            const uint8_t *p2 = b2 + 4 + 4 * rows2 + c.str_off[(int64_t)lb2 * A.g.block_size + r2];
            for (int i = 0; i < s1; i++) if (p1[i] != p2[i]) return false;
        } else {
            const bool m1 = col_missing(c, lb1, r1), m2 = col_missing(c, lb2, r2);
            if (m1 != m2) return false;
            if (!m1 && key_bits(c.kind, col_values(c, lb1, rows1) + r1 * c.elsize) != key_bits(c.kind, col_values(c, lb2, rows2) + r2 * c.elsize))
                return false;
        }
    }
    return true;
}
// order-preserving integer image of a double (NaN never gets here)
__device__ __forceinline__ long long dbl_order_key(double x)
{
    const long long b = __double_as_longlong(x);
    return b < 0 ? (long long)(0x8000000000000000ull - (unsigned long long)b) : b;      // -0.0 -> 0 - ... below +0.0
}

// The accumulators of a group are hit by every one of its rows: with a handful of groups (the usual GROUP BY) that is a hundred
// million atomics on a few dozen addresses, and they serialise -- in L2, and just the same in shared memory (first version:
// 84 ms for 100M selected rows in 8 groups, IPC 0.22; a per-CTA shared-memory copy of the accumulators alone: 83 ms).  So a
// warp first sorts its 32 rows by group (MATCH.ANY on the table slot) and, when they fall into at most GROUP_WARP_MAX groups,
// reduces every group's rows in registers -- shuffle trees over the member lanes -- and its leader lane issues ONE set of
// atomics; those go to a small direct-mapped cache of groups in the CTA's shared memory (entry = table slot mod GROUP_CACHE,
// claimed by the first group that maps to it), which is merged into the table once, at the end.  Warps whose rows are spread
// over many groups (a query with millions of groups) take the direct path: one set of atomics per row on the table itself,
// where they do not collide.
constexpr int GROUP_CACHE = 64;
constexpr int GROUP_WARP_MAX = 12;

__device__ __forceinline__ void group_acc_neutral(GroupAcc &a, int cls)
{
    a.count = 0; a.nmissing = 0; a.sum_i = 0; a.sum_f = 0.0; a.flags = 0; a.pad = 0;
    if (cls == VC_UINT || cls == VC_BOOL) { a.min_k = -1ll; a.max_k = 0; }
    else { a.min_k = INT64_MAX; a.max_k = INT64_MIN; }
}
// one row's (or one pre-reduced group's) contribution to an accumulator
__device__ __forceinline__ void group_acc_add(GroupAcc *acc, int cls, unsigned long long count, unsigned long long nmissing, long long sum_i, double sum_f,
                                              long long min_k, long long max_k, int flags)
{
    atomicAdd(&acc->count, count);
    if (nmissing) atomicAdd(&acc->nmissing, nmissing);
    if (count == nmissing) return;
    if (cls == VC_FLT) atomicAdd(&acc->sum_f, sum_f);
    else atomicAdd(reinterpret_cast<unsigned long long *>(&acc->sum_i), (unsigned long long)sum_i);
    if (flags & 1) {
        if (cls == VC_UINT || cls == VC_BOOL) {
            atomicMin(reinterpret_cast<unsigned long long *>(&acc->min_k), (unsigned long long)min_k);
            atomicMax(reinterpret_cast<unsigned long long *>(&acc->max_k), (unsigned long long)max_k);
        } else {
            atomicMin(&acc->min_k, min_k);
            atomicMax(&acc->max_k, max_k);
        }
    }
    if (flags) atomicOr(&acc->flags, flags);
}

__global__ void __launch_bounds__(SCAN_THREADS) group_reduce_kernel(const GroupArgs A)
{
    __shared__ unsigned long long ctag[GROUP_CACHE];                    // table slot + 1 of the group the entry holds, 0 = free
    __shared__ unsigned long long chash[GROUP_CACHE];                   // ... the hash of its key
    __shared__ long long crep[GROUP_CACHE];                             // ... a row of the group (the table's representative)
    __shared__ int cready[GROUP_CACHE];                                 // hash and row are published
    __shared__ long long cfirst[GROUP_CACHE];
    __shared__ GroupAcc cacc[GROUP_CACHE * GROUP_MAX_VALS];
    const Geometry g = A.g;
    const unsigned lane = lane_id();
    for (int i = threadIdx.x; i < GROUP_CACHE; i += SCAN_THREADS) { ctag[i] = 0; cready[i] = 0; cfirst[i] = INT64_MAX; }
    for (int i = threadIdx.x; i < GROUP_CACHE * A.nvals; i += SCAN_THREADS) group_acc_neutral(cacc[i], A.val[i % A.nvals].cls);
    __syncthreads();
    const int64_t total_words = (int64_t)g.nblocks * g.wpb;
    for (int64_t w = (int64_t)blockIdx.x * (SCAN_THREADS / 32) + warp_id(); w < total_words; w += (int64_t)gridDim.x * (SCAN_THREADS / 32)) {
        // (the table is full: the host runs again with a larger one.  Looked at once in 64 words: the flag is one address for every warp of the grid)
        if (((w / ((int64_t)gridDim.x * (SCAN_THREADS / 32))) & 63) == 0 && *reinterpret_cast<volatile int *>(A.overflow)) break;
        const int lb = (int)(w / g.wpb);
        const int64_t r = (w - (int64_t)lb * g.wpb) * 32 + lane;
        const int64_t rows_b = block_rows(g, lb);
        const bool active = r < rows_b && ((A.mask[w] >> lane) & 1u);
        const long long row = (long long)lb * g.block_size + r;                 // shard row
        unsigned long long slot = 0;
        bool placed = false, cached = false;
        int e = 0;
        if (active) {
            // The CTA's cache first: entry = hash mod GROUP_CACHE.  A hit is verified against the group's representative row (its key
            // bytes are immutable and come through L1), so the table -- where the few slots of a query with few groups are a hot
            // spot every row of the column would queue up at, in L2 -- is only consulted by the first rows of a group in this CTA.
            const unsigned long long h = group_key_hash(A, lb, rows_b, r);
            e = (int)((h >> 20) & (GROUP_CACHE - 1));
            if (*reinterpret_cast<volatile int *>(&cready[e]) && chash[e] == h) {
                const long long rep = crep[e];
                if (rep == row || group_keys_equal(A, lb, r, (int)(rep / g.block_size), rep % g.block_size)) {
                    slot = ctag[e] - 1;
                    placed = cached = true;
                }
            }
            if (!placed) {
                long long cur = -1;
                slot = h & A.cap_mask;
                for (unsigned long long probe = 0; probe <= A.cap_mask; probe++, slot = (slot + 1) & A.cap_mask) {
                    cur = __ldcg(&A.rep[slot]);                                 // (a slot changes once, from -1 to its group's row)
                    if (cur == -1) {
                        const unsigned long long old = atomicCAS(reinterpret_cast<unsigned long long *>(&A.rep[slot]), (unsigned long long)-1ll, (unsigned long long)row);
                        if (old == (unsigned long long)-1ll) { atomicAdd(A.ngroups, 1ull); cur = row; }
                        else cur = (long long)old;
                    }
                    if (cur == row || group_keys_equal(A, lb, r, (int)(cur / g.block_size), cur % g.block_size)) { placed = true; break; }
                    if (probe > 4096) break;                                    // hopelessly full: grow
                }
                if (!placed) {
                    atomicExch(A.overflow, 1);
                } else {
                    // claim the cache entry for this group if it is free
                    unsigned long long tag = *reinterpret_cast<volatile unsigned long long *>(&ctag[e]);
                    if (tag == 0) {
                        const unsigned long long old = atomicCAS(&ctag[e], 0ull, slot + 1);
                        if (old == 0) {
                            chash[e] = h;
                            crep[e] = cur;
                            __threadfence_block();
                            *reinterpret_cast<volatile int *>(&cready[e]) = 1;
                            tag = slot + 1;
                        } else {
                            tag = old;
                        }
                    }
                    cached = tag == slot + 1;
                }
            }
        }
        __syncwarp();
        const unsigned am = __ballot_sync(FULL, placed);
        if (am == 0) continue;
        unsigned peers = 0;
        if (placed) peers = __match_any_sync(am, slot);                         // the lanes whose rows belong to my group
        const bool leader = placed && (unsigned)(__ffs(peers) - 1) == lane;     // (lowest lane = lowest row of the group in this word)
        const unsigned leaders = __ballot_sync(FULL, leader);
        if (__popc(leaders) > GROUP_WARP_MAX) {
            // ---- many groups in this word: every row goes to the table on its own ----
            if (placed) {
                atomicMin(reinterpret_cast<long long *>(&A.first[slot]), row);
                for (int v = 0; v < A.nvals; v++) {
                    const ColView &c = A.val[v];
                    GroupAcc *acc = A.acc + slot * A.nvals + v;
                    if (col_missing(c, lb, r)) { group_acc_add(acc, c.cls, 1, 1, 0, 0.0, 0, 0, 0); continue; }
                    const unsigned long long bits = load_widen(col_values(c, lb, rows_b) + r * c.elsize, c.kind);
                    if (c.cls == VC_FLT) {
                        const double x = __longlong_as_double((long long)bits);
                        const long long k = x != x ? 0 : dbl_order_key(x);
                        group_acc_add(acc, c.cls, 1, 0, 0, x, k, k, x != x ? 2 : 1);
                    } else {
                        group_acc_add(acc, c.cls, 1, 0, (long long)bits, 0.0, (long long)bits, (long long)bits, 1);
                    }
                }
            }
            continue;
        }
        // ---- few groups: reduce each group's rows in registers, its leader lane adds the result to the CTA's cache ----
        GroupAcc *dst = nullptr;          // leader: where this group's accumulators are (cache entry or table)
        if (leader) {
            atomicMin(cached ? &cfirst[e] : reinterpret_cast<long long *>(&A.first[slot]), row);
            dst = cached ? &cacc[e * A.nvals] : A.acc + slot * A.nvals;
        }
        for (int v = 0; v < A.nvals; v++) {
            const ColView &c = A.val[v];
            const bool uns = c.cls == VC_UINT || c.cls == VC_BOOL;
            bool missing = false, isnan = false;
            unsigned long long bits = 0;
            if (placed) {
                missing = col_missing(c, lb, r);
                if (!missing) bits = load_widen(col_values(c, lb, rows_b) + r * c.elsize, c.kind);
            }
            double x = 0.0;
            long long key = (long long)bits;
            if (c.cls == VC_FLT) {
                x = __longlong_as_double((long long)bits);
                isnan = placed && !missing && x != x;
                key = isnan ? 0 : dbl_order_key(x);
            }
            const bool has = placed && !missing;            // contributes to the sum
            const bool ord = has && !isnan;                 // contributes to min / max
            for (unsigned rest = leaders; rest; rest &= rest - 1) {             // (uniform: one round per group of the word)
                const int l = __ffs(rest) - 1;
                const unsigned mem = __shfl_sync(FULL, peers, l);
                const bool in = (mem >> lane) & 1u;
                const unsigned nmiss = __popc(__ballot_sync(FULL, in && missing));
                const unsigned nnan = __popc(__ballot_sync(FULL, in && isnan));
                const unsigned nord = __popc(__ballot_sync(FULL, in && ord));
                double sf = (in && has) ? x : 0.0;
                unsigned long long si = (in && has) ? bits : 0ull;
                long long mn = (in && ord) ? key : (uns ? -1ll : INT64_MAX), mx = (in && ord) ? key : (uns ? 0ll : INT64_MIN);
#pragma unroll
                for (int d = 16; d > 0; d >>= 1) {
                    if (c.cls == VC_FLT) sf += __shfl_xor_sync(FULL, sf, d);
                    else si += __shfl_xor_sync(FULL, si, d);
                    const long long omn = __shfl_xor_sync(FULL, mn, d), omx = __shfl_xor_sync(FULL, mx, d);
                    if (uns) {
                        if ((unsigned long long)omn < (unsigned long long)mn) mn = omn;
                        if ((unsigned long long)omx > (unsigned long long)mx) mx = omx;
                    } else {
                        if (omn < mn) mn = omn;
                        if (omx > mx) mx = omx;
                    }
                }
                if ((int)lane == l)
                    group_acc_add(dst + v, c.cls, (unsigned long long)__popc(mem), nmiss, (long long)si, sf, mn, mx, (nord ? 1 : 0) | (nnan ? 2 : 0));
            }
        }
    }
    // merge the cache into the table
    __syncthreads();
    for (int e = threadIdx.x; e < GROUP_CACHE; e += SCAN_THREADS)
        if (ctag[e] != 0 && cfirst[e] != INT64_MAX) atomicMin(reinterpret_cast<long long *>(&A.first[ctag[e] - 1]), cfirst[e]);
    for (int i = threadIdx.x; i < GROUP_CACHE * A.nvals; i += SCAN_THREADS) {
        const int e = i / A.nvals, v = i - e * A.nvals;
        if (ctag[e] == 0) continue;
        const GroupAcc &ca = cacc[i];
        if (ca.count == 0) continue;
        group_acc_add(A.acc + (ctag[e] - 1) * A.nvals + v, A.val[v].cls, ca.count, ca.nmissing, ca.sum_i, ca.sum_f, ca.min_k, ca.max_k, ca.flags);
    }
}

// ---- K5/K6: warp-aggregated compaction --------------------------------------------------------------------
// Work unit = (block, warp range of mask words).  Each CTA takes one block at a time; its 8 warps own
// contiguous word ranges; a first pass counts, a second pass walks the words in order so every selected
// row gets its output index = block base + prefix of earlier survivors (row order is preserved).
template <typename F>
__device__ __forceinline__ void compact_block(const Geometry &g, const uint32_t *mask, int lb, int64_t blk_base, int64_t *smem_base, F emit)
{
    const uint32_t *m = mask + (int64_t)lb * g.wpb;
    const int nw = SCAN_THREADS / 32;
    const int per = (g.wpb + nw - 1) / nw;
    const int w_lo = warp_id() * per;
    int w_hi = w_lo + per;
    if (w_hi > g.wpb) w_hi = g.wpb;
    int c = 0;
    for (int w = w_lo + lane_id(); w < w_hi; w += 32) c += __popc(m[w]);
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) c += __shfl_xor_sync(FULL, c, d);
    __syncthreads();
    if (lane_id() == 0) smem_base[warp_id()] = c;
    __syncthreads();
    int64_t base = blk_base;
    for (int i = 0; i < warp_id(); i++) base += smem_base[i];
    for (int w = w_lo; w < w_hi; w++) {
        const uint32_t word = m[w];
        if (word == 0) continue;
        const bool sel = (word >> lane_id()) & 1u;
        const int64_t idx = base + __popc(word & ((1u << lane_id()) - 1u));
        if (sel) emit((int64_t)w * 32 + lane_id(), idx);
        base += __popc(word);
    }
}

__global__ void __launch_bounds__(SCAN_THREADS) gather_fixed_kernel(const GatherArgs A)
{
    __shared__ int64_t sbase[SCAN_THREADS / 32];
    const Geometry g = A.g;
    for (int lb = blockIdx.x; lb < g.nblocks; lb += gridDim.x) {
        const int64_t rows_b = block_rows(g, lb);
        const ColView &c = A.col;
        const uint8_t *vals = col_values(c, lb, rows_b);
        const int es = c.elsize;
        compact_block(g, A.mask, lb, A.blk_base[lb], sbase, [&](int64_t r, int64_t idx) {
            const bool ms = col_missing(c, lb, r);
            if (A.out_missing) A.out_missing[idx] = ms ? 1 : 0;
            uint8_t *o = A.out_values + idx * es;
            const uint8_t *p = vals + r * es;
            switch (es) {
            case 8: *reinterpret_cast<unsigned long long *>(o) = ms ? 0ull : *reinterpret_cast<const unsigned long long *>(p); break;
            case 4: *reinterpret_cast<uint32_t *>(o) = ms ? 0u : *reinterpret_cast<const uint32_t *>(p); break;
            case 2: *reinterpret_cast<uint16_t *>(o) = ms ? (uint16_t)0 : *reinterpret_cast<const uint16_t *>(p); break;
            case 1: *o = ms ? (uint8_t)0 : *p; break;
            default:
                for (int i = 0; i < es; i++) o[i] = ms ? (uint8_t)0 : p[i];
                break;
            }
        });
    }
}

__global__ void __launch_bounds__(SCAN_THREADS) gather_indices_kernel(const GatherArgs A)
{
    __shared__ int64_t sbase[SCAN_THREADS / 32];
    const Geometry g = A.g;
    for (int lb = blockIdx.x; lb < g.nblocks; lb += gridDim.x) {
        const int64_t row_base = (g.blk_lo + lb) * g.block_size + 1;
        compact_block(g, A.mask, lb, A.blk_base[lb], sbase, [&](int64_t r, int64_t idx) { A.out_indices[idx] = row_base + r; });
    }
}

// selected string bytes per block (one warp per block)
// One CTA per block; warp k owns the contiguous chunk of mask words [k*C, (k+1)*C).  Mask words are fetched 32 at a
// time (one coalesced load per lane) and handed round by shuffle, so the per-word loop carries no dependent mask load.
__device__ __forceinline__ void str_chunk_totals(const GatherArgs &A, int lb, int w0, int w1, long long &rows, long long &bytes)
{
    const Geometry &g = A.g;
    const uint32_t *m = A.mask + (int64_t)lb * g.wpb;
    const int32_t *sizes = reinterpret_cast<const int32_t *>(col_body(A.col, lb) + 4);
    rows = 0;
    bytes = 0;
    for (int wb = w0; wb < w1; wb += 32) {
        const uint32_t mine = wb + lane_id() < w1 ? m[wb + lane_id()] : 0u;
        uint32_t nz = __ballot_sync(FULL, mine != 0);
        while (nz) {
            const int j = __ffs(nz) - 1;
            nz &= nz - 1;
            const uint32_t word = __shfl_sync(FULL, mine, j);
            if ((word >> lane_id()) & 1u) {
                const int s = sizes[(int64_t)(wb + j) * 32 + lane_id()];
                rows++;
                if (s > 0) bytes += s;
            }
        }
    }
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) {
        rows += __shfl_xor_sync(FULL, rows, d);
        bytes += __shfl_xor_sync(FULL, bytes, d);
    }
}

__global__ void __launch_bounds__(SCAN_THREADS) str_block_bytes_kernel(const GatherArgs A, int64_t *blk_bytes)
{
    __shared__ long long s_bytes[SCAN_THREADS / 32];
    const Geometry g = A.g;
    const int C = (g.wpb + SCAN_THREADS / 32 - 1) / (SCAN_THREADS / 32);
    for (int lb = blockIdx.x; lb < g.nblocks; lb += gridDim.x) {
        const int w0 = warp_id() * C, w1 = w0 + C < g.wpb ? w0 + C : g.wpb;
        long long rows, bytes;
        str_chunk_totals(A, lb, w0, w1, rows, bytes);
        if (lane_id() == 0) s_bytes[warp_id()] = bytes;
        __syncthreads();
        if (threadIdx.x == 0) {
            long long tot = 0;
            for (int k = 0; k < SCAN_THREADS / 32; k++) tot += s_bytes[k];
            blk_bytes[lb] = tot;
        }
        __syncthreads();
    }
}

// sizes + chars of the selected rows (FlatStringsVector gather, offset-aware, /root/reference/src/FlatStringsVectors.jl:136-157).
// One CTA per block, tiles of 1024 rows (4 consecutive rows per thread).  A CTA-wide scan over (selected rows, selected
// bytes, all bytes) gives every row its output row, its output byte position and -- since a block's chars are the
// concatenation of its rows -- its source position too, so the per-row offsets of K2 are not read here.  The tile's chars
// come in with aligned 16-byte loads, are compacted in shared memory and leave as one contiguous run; only tiles whose
// chars do not fit the staging buffers (very long strings) copy row by row through global memory.
constexpr int STR_TILE = SCAN_THREADS * 4;
constexpr int STR_STAGE = 20480;

__global__ void __launch_bounds__(SCAN_THREADS) gather_strings_kernel(const GatherArgs A)
{
    __shared__ __align__(16) uint8_t s_in[STR_STAGE + 32];
    __shared__ __align__(16) uint8_t s_out[STR_STAGE];
    __shared__ long long s_tot[3][SCAN_THREADS / 32];
    const Geometry g = A.g;
    const int tid = threadIdx.x, lane = lane_id(), wid = warp_id();
    for (int lb = blockIdx.x; lb < g.nblocks; lb += gridDim.x) {
        const uint32_t *m = A.mask + (int64_t)lb * g.wpb;
        const int64_t rows_b = block_rows(g, lb);
        const uint8_t *body = col_body(A.col, lb);
        const int32_t *sizes = reinterpret_cast<const int32_t *>(body + 4);
        const uint8_t *chars = body + 4 + 4 * rows_b;
        if (A.blk_base[lb + 1] == A.blk_base[lb]) continue;   // no selected row in this block (it may not even be decoded)
        int64_t row_pos = A.blk_base[lb];          // output row / output byte / source byte position of the tile (uniform)
        int64_t byte_pos = A.blk_char_base[lb];
        int64_t char_pos = 0;
        for (int64_t tile0 = 0; tile0 < rows_b; tile0 += STR_TILE) {
            const int64_t r0 = tile0 + 4 * tid;
            const uint32_t bits = r0 < rows_b ? (m[r0 >> 5] >> (r0 & 31)) & 15u : 0u;
            int sz[4];
            long long nsel = 0, bsel = 0, ball = 0;
#pragma unroll
            for (int k = 0; k < 4; k++) {
                sz[k] = r0 + k < rows_b ? sizes[r0 + k] : 0;
                const long long nb = sz[k] > 0 ? sz[k] : 0;
                ball += nb;
                if ((bits >> k) & 1u) { nsel++; bsel += nb; }
            }
            // exclusive CTA scan of the three sums
            long long xs = nsel, xb = bsel, xa = ball;
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) {
                const long long a = __shfl_up_sync(FULL, xs, d), b = __shfl_up_sync(FULL, xb, d), c = __shfl_up_sync(FULL, xa, d);
                if (lane >= d) { xs += a; xb += b; xa += c; }
            }
            if (lane == 31) { s_tot[0][wid] = xs; s_tot[1][wid] = xb; s_tot[2][wid] = xa; }
            __syncthreads();
            long long ps = xs - nsel, pb = xb - bsel, pa = xa - ball, ts = 0, tb = 0, ta = 0;
#pragma unroll
            for (int k = 0; k < SCAN_THREADS / 32; k++) {
                const long long a = s_tot[0][k], b = s_tot[1][k], c = s_tot[2][k];
                if (k < wid) { ps += a; pb += b; pa += c; }
                ts += a; tb += b; ta += c;
            }
            if (ts > 0) {
                // sizes of the selected rows
                int q = 0;
#pragma unroll
                for (int k = 0; k < 4; k++)
                    if ((bits >> k) & 1u) { A.out_sizes[row_pos + ps + q] = sz[k]; q++; }
                const uint8_t *src0 = chars + char_pos;
                uint8_t *dst0 = A.out_chars + byte_pos;
                if (ta <= STR_STAGE && tb > 0) {
                    // stage the tile's chars (aligned 16-byte loads; the over-read stays inside the block's slot)
                    const int mis = (int)(reinterpret_cast<uintptr_t>(src0) & 15);
                    const uint4 *src16 = reinterpret_cast<const uint4 *>(src0 - mis);
                    const int nch = (int)((ta + mis + 15) >> 4);
                    for (int c = tid; c < nch; c += SCAN_THREADS) reinterpret_cast<uint4 *>(s_in)[c] = src16[c];
                    __syncthreads();
                    int so = (int)pa + mis, dpos = (int)pb;
#pragma unroll
                    for (int k = 0; k < 4; k++) {
                        const int nb = sz[k] > 0 ? sz[k] : 0;
                        if ((bits >> k) & 1u)
                            for (int i = 0; i < nb; i++) s_out[dpos + i] = s_in[so + i];
                        if ((bits >> k) & 1u) dpos += nb;
                        so += nb;
                    }
                    __syncthreads();
                    // one contiguous run: bytes up to the first 4-byte boundary of the destination, then words
                    const int head = (int)((4 - (reinterpret_cast<uintptr_t>(dst0) & 3)) & 3);
                    const int nhead = head < (int)tb ? head : (int)tb;
                    if (tid < nhead) dst0[tid] = s_out[tid];
                    const int nwords = ((int)tb - nhead) >> 2;
                    uint32_t *dw = reinterpret_cast<uint32_t *>(dst0 + nhead);
                    for (int w = tid; w < nwords; w += SCAN_THREADS) {
                        const uint8_t *b4 = s_out + nhead + 4 * w;
                        dw[w] = (uint32_t)b4[0] | ((uint32_t)b4[1] << 8) | ((uint32_t)b4[2] << 16) | ((uint32_t)b4[3] << 24);
                    }
                    const int done = nhead + 4 * nwords;
                    if (tid < (int)tb - done) dst0[done + tid] = s_out[done + tid];
                } else if (tb > 0) {
                    // long strings: row by row through global memory
                    long long so = pa, dpos = pb;
#pragma unroll
                    for (int k = 0; k < 4; k++) {
                        const int nb = sz[k] > 0 ? sz[k] : 0;
                        if ((bits >> k) & 1u) {
                            for (int i = 0; i < nb; i++) dst0[dpos + i] = src0[so + i];
                            dpos += nb;
                        }
                        so += nb;
                    }
                }
            }
            row_pos += ts;
            byte_pos += tb;
            char_pos += ta;
            __syncthreads();
        }
    }
}

// computed projection column: VM value of every selected row, in row order
__global__ void __launch_bounds__(SCAN_THREADS) proj_vm_kernel(const ProjVmArgs A)
{
    __shared__ int64_t sbase[SCAN_THREADS / 32];
    const Geometry g = A.g;
    for (int lb = blockIdx.x; lb < g.nblocks; lb += gridDim.x) {
        const int64_t rows_b = block_rows(g, lb);
        compact_block(g, A.mask, lb, A.blk_base[lb], sbase, [&](int64_t r, int64_t idx) {
            unsigned long long v;
            bool ms;
            vm_eval(A.prog, A.slot, g, lb, rows_b, r, v, ms, A.error_flag);
            if (A.out_missing) A.out_missing[idx] = ms ? 1 : 0;
            if (ms) v = 0ull;
            uint8_t *o = A.out_values + idx * A.elsize;
            const bool is_f32 = A.prog->result_class == VC_FLT && A.elsize == 4;
            if (is_f32) { const float f = (float)__longlong_as_double((long long)v); *reinterpret_cast<float *>(o) = f; return; }
            switch (A.elsize) {
            case 8: *reinterpret_cast<unsigned long long *>(o) = v; break;
            case 4: *reinterpret_cast<uint32_t *>(o) = (uint32_t)v; break;
            case 2: *reinterpret_cast<uint16_t *>(o) = (uint16_t)v; break;
            default: *o = (uint8_t)v; break;
            }
        });
    }
}

// reductions over a computed column (Base folds over iterate(::DFColumn), /root/reference/src/tables/column.jl:102-126, for
// a column that is a BlockBroadcasting, columnbroadcast.jl:35-62): one CTA per work unit like K3+K7, thread t takes rows
// t, t + 256, ... of a tile in that order, then the fixed block reduction
__global__ void __launch_bounds__(SCAN_THREADS) agg_vm_kernel(const AggVmArgs A)
{
    __shared__ AggPartial red[SCAN_THREADS / 32];
    const Geometry g = A.g;
    const int tid = threadIdx.x, cls = A.cls;
    const int nunits = g.nblocks * g.segs_per_block;
    for (int unit = blockIdx.x; unit < nunits; unit += gridDim.x) {
        const int lb = unit / g.segs_per_block;
        const int seg = unit - lb * g.segs_per_block;
        const int64_t rows_b = block_rows(g, lb);
        const int64_t row0 = (int64_t)seg * g.seg_rows;
        int64_t row1 = row0 + g.seg_rows;
        if (row1 > rows_b) row1 = rows_b;
        AggPartial acc;
        agg_init(acc);
        for (int64_t tile0 = row0; tile0 < row1; tile0 += TILE_ROWS) {
#pragma unroll 1
            for (int k = 0; k < 8; k++) {
                const int64_t r = tile0 + (int64_t)k * SCAN_THREADS + tid;
                if (r >= row1) continue;
                if (!((__ldg(A.mask + (int64_t)lb * g.wpb + (r >> 5)) >> (r & 31)) & 1u)) continue;
                unsigned long long v;
                bool ms;
                vm_eval(A.prog, A.slot, g, lb, rows_b, r, v, ms, A.error_flag);
                acc.count++;
                if (ms) { acc.nmissing++; continue; }
                if (cls == VC_FLT) {
                    const double x = __longlong_as_double((long long)v);
                    if (x != x) acc.has_nan = 1;
                    else {
                        two_sum_add(acc.sum_f, acc.sum_lo, x);
                        if (!acc.has_value) { acc.min_f = x; acc.max_f = x; acc.has_value = 1; }
                        else { acc.min_f = jl_min(acc.min_f, x); acc.max_f = jl_max(acc.max_f, x); }
                    }
                } else {
                    const long long x = (long long)v;
                    acc.sum_i = (long long)((unsigned long long)acc.sum_i + (unsigned long long)x);
                    if (!acc.has_value) { acc.min_i = x; acc.max_i = x; acc.has_value = 1; }
                    else if (cls == VC_UINT) {
                        if ((unsigned long long)x < (unsigned long long)acc.min_i) acc.min_i = x;
                        if ((unsigned long long)x > (unsigned long long)acc.max_i) acc.max_i = x;
                    } else {
                        if (x < acc.min_i) acc.min_i = x;
                        if (x > acc.max_i) acc.max_i = x;
                    }
                }
            }
        }
        agg_block_reduce(acc, cls, red);
        if (tid == 0) A.partials[unit] = acc;
    }
}

// ---- unique ---------------------------------------------------------------------------------------------------------
// Local pass: the group table of the key column holds, per distinct value, its lowest selected row; setting those rows in
// a mask laid out like the selection mask lets the gathers of materialize emit the values in row order, which is the order
// of first appearance.
__global__ void __launch_bounds__(SCAN_THREADS) unique_first_mask_kernel(const long long *first, long long cap, long long sentinel, const Geometry g,
                                                                          uint32_t *mask)
{
    for (long long sl = (long long)blockIdx.x * blockDim.x + threadIdx.x; sl < cap; sl += (long long)gridDim.x * blockDim.x) {
        const long long f = first[sl];
        if (f == sentinel) continue;
        const long long lb = f / g.block_size, r = f - lb * g.block_size;
        atomicOr(mask + lb * g.wpb + (r >> 5), 1u << (r & 31));
    }
}

// Cross-shard merge over the rank-order concatenation of local results (flat arrays, one thread per position): a key tuple's
// slot ends up holding the lowest position with that tuple (the slot's representative only ever moves to an equal tuple, so
// comparisons against it stay valid while it moves), and a position is kept when it is that lowest one.  Hash and equality
// are group_key_hash's and group_keys_equal's over the flat layout.
__device__ unsigned long long merge_hash(const MergeArgs &A, long long i)
{
    unsigned long long h = 0x243F6A8885A308D3ull;
    for (int k = 0; k < A.nkeys; k++) {
        const MergeKey &c = A.key[k];
        if (c.sizes) {
            const int sz = c.sizes[i];
            const uint8_t *p = c.chars + c.char_off[i];
            unsigned long long f = 0xCBF29CE484222325ull;
            for (int b = 0; b < sz; b++) f = (f ^ p[b]) * 0x100000001B3ull;
            h = gmix(h ^ f ^ ((unsigned long long)(unsigned)sz << 32));
        } else if (c.missing && c.missing[i]) {
            h = gmix(h ^ 0xA5A5A5A5A5A5A5A5ull);
        } else {
            h = gmix(h ^ key_bits(c.kind, c.values + i * c.elsize));
        }
    }
    return h;
}
__device__ bool merge_equal(const MergeArgs &A, long long i, long long j)
{
    for (int k = 0; k < A.nkeys; k++) {
        const MergeKey &c = A.key[k];
        if (c.sizes) {
            const int si = c.sizes[i];
            if (si != c.sizes[j]) return false;
            const uint8_t *p = c.chars + c.char_off[i], *q = c.chars + c.char_off[j];
            for (int b = 0; b < si; b++) if (p[b] != q[b]) return false;
        } else {
            const bool mi = c.missing && c.missing[i], mj = c.missing && c.missing[j];
            if (mi != mj) return false;
            if (!mi && key_bits(c.kind, c.values + i * c.elsize) != key_bits(c.kind, c.values + j * c.elsize)) return false;
        }
    }
    return true;
}
__global__ void __launch_bounds__(SCAN_THREADS) merge_insert_kernel(const MergeArgs A)
{
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < A.n; i += (long long)gridDim.x * blockDim.x) {
        unsigned long long slot = merge_hash(A, i) & A.cap_mask;
        for (;;) {                                                      // (the table has at least twice as many slots as positions)
            long long cur = __ldcg(&A.rep[slot]);
            if (cur == -1) {
                cur = (long long)atomicCAS(reinterpret_cast<unsigned long long *>(&A.rep[slot]), (unsigned long long)-1ll, (unsigned long long)i);
                if (cur == -1) break;
            }
            if (merge_equal(A, cur, i)) { atomicMin(&A.rep[slot], i); break; }
            slot = (slot + 1) & A.cap_mask;
        }
        A.slot[i] = (long long)slot;
    }
}
// keep[i] = 1 when position i is its key's first; kept_bytes[i] = its char bytes then (String key columns)
__global__ void __launch_bounds__(SCAN_THREADS) merge_keep_kernel(const MergeArgs A, int64_t *keep)
{
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < A.n; i += (long long)gridDim.x * blockDim.x) {
        const bool k = __ldcg(&A.rep[A.slot[i]]) == i;
        keep[i] = k;
        for (int c = 0; c < A.nkeys; c++)
            if (A.key[c].kept_bytes) A.key[c].kept_bytes[i] = k && A.key[c].sizes[i] > 0 ? A.key[c].sizes[i] : 0;
    }
}
__global__ void __launch_bounds__(SCAN_THREADS) str_lengths_kernel(const int32_t *sizes, long long n, int64_t *out)
{
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) out[i] = sizes[i] > 0 ? sizes[i] : 0;
}
// kept positions to their output slots (keep_pos / kept_bytes: exclusive scans of keep / the kept char bytes)
__global__ void __launch_bounds__(SCAN_THREADS) merge_emit_kernel(const MergeArgs A, const int64_t *keep_pos, const long long *first, long long *out_first)
{
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < A.n; i += (long long)gridDim.x * blockDim.x) {
        const long long o = keep_pos[i];
        if (keep_pos[i + 1] == o) continue;
        if (out_first) out_first[o] = first[i];
        for (int c = 0; c < A.nkeys; c++) {
            const MergeKey &K = A.key[c];
            if (K.sizes) {
                const int sz = K.sizes[i];
                K.out_sizes[o] = sz;
                const uint8_t *p = K.chars + K.char_off[i];
                uint8_t *q = K.out_chars + K.kept_bytes[i];
                for (int b = 0; b < sz; b++) q[b] = p[b];
            } else {
                const bool ms = K.missing && K.missing[i];
                if (K.out_missing) K.out_missing[o] = ms ? 1 : 0;
                const uint8_t *p = K.values + i * K.elsize;
                uint8_t *q = K.out_values + o * K.elsize;
                for (int b = 0; b < K.elsize; b++) q[b] = ms ? (uint8_t)0 : p[b];
            }
        }
    }
}
// group-by: one rank's positions [lo, hi) into their merged groups.  The keys of one part are distinct, so no two threads of
// a launch share a group; one launch per rank in rank order makes every group's fold the rank-order dfdb_agg_fold.
__global__ void __launch_bounds__(SCAN_THREADS) merge_fold_kernel(const MergeArgs A, const int64_t *keep_pos, const dfdb_agg *in, int nvals, long long lo,
                                                                  long long hi, dfdb_agg *out, int *dup)
{
    for (long long i = lo + (long long)blockIdx.x * blockDim.x + threadIdx.x; i < hi; i += (long long)gridDim.x * blockDim.x) {
        const long long r = __ldcg(&A.rep[A.slot[i]]);
        if (r != i && r >= lo) { atomicExch(dup, 1); continue; }                    // the key occurs earlier in this same part
        const long long g = keep_pos[r];
        for (int v = 0; v < nvals; v++) dfdb_agg_fold_step(out[g * nvals + v], in[i * nvals + v]);
    }
}
__global__ void __launch_bounds__(SCAN_THREADS) merge_fold_finish_kernel(dfdb_agg *out, long long n)
{
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) dfdb_agg_fold_finish(out[i]);
}

// Exclusive scan of n int64 in place, in chunks of SCAN_CHUNK: chunk sums, a scan of the sums (exclusive_scan_kernel), then
// every chunk rescanned from its base.  data[n] = total.
constexpr int SCAN_PER_THREAD = 16;
constexpr int SCAN_CHUNK = SCAN_THREADS * SCAN_PER_THREAD;
__device__ __forceinline__ int64_t cta_exclusive_sum(int64_t v, int64_t *s_warp, int64_t *total)
{
    int64_t incl = v;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const int64_t o = __shfl_up_sync(FULL, incl, d);
        if (lane_id() >= d) incl += o;
    }
    if (lane_id() == 31) s_warp[warp_id()] = incl;
    __syncthreads();
    int64_t before = 0, all = 0;
#pragma unroll
    for (int w = 0; w < SCAN_THREADS / 32; w++) {
        if (w < warp_id()) before += s_warp[w];
        all += s_warp[w];
    }
    __syncthreads();
    *total = all;
    return before + incl - v;
}
__global__ void __launch_bounds__(SCAN_THREADS) chunk_sums_kernel(const int64_t *data, long long n, int64_t *sums)
{
    __shared__ int64_t s_warp[SCAN_THREADS / 32];
    const long long nchunks = (n + SCAN_CHUNK - 1) / SCAN_CHUNK;
    for (long long c = blockIdx.x; c < nchunks; c += gridDim.x) {
        const long long lo = c * SCAN_CHUNK + (long long)threadIdx.x * SCAN_PER_THREAD;
        int64_t s = 0;
        for (int k = 0; k < SCAN_PER_THREAD; k++) if (lo + k < n) s += data[lo + k];
        int64_t total;
        cta_exclusive_sum(s, s_warp, &total);
        if (threadIdx.x == 0) sums[c] = total;
    }
}
__global__ void __launch_bounds__(SCAN_THREADS) chunk_rescan_kernel(int64_t *data, long long n, const int64_t *bases)
{
    __shared__ int64_t s_warp[SCAN_THREADS / 32];
    const long long nchunks = (n + SCAN_CHUNK - 1) / SCAN_CHUNK;
    if (blockIdx.x == 0 && threadIdx.x == 0) data[n] = bases[nchunks];
    for (long long c = blockIdx.x; c < nchunks; c += gridDim.x) {
        const long long lo = c * SCAN_CHUNK + (long long)threadIdx.x * SCAN_PER_THREAD;
        int64_t v[SCAN_PER_THREAD], s = 0;
#pragma unroll
        for (int k = 0; k < SCAN_PER_THREAD; k++) { v[k] = lo + k < n ? data[lo + k] : 0; s += v[k]; }
        int64_t total;
        int64_t run = bases[c] + cta_exclusive_sum(s, s_warp, &total);
#pragma unroll
        for (int k = 0; k < SCAN_PER_THREAD; k++) {
            if (lo + k < n) data[lo + k] = run;
            run += v[k];
        }
    }
}

int grid_for(int64_t work, int sm_count, int per_sm)
{
    int64_t g = (int64_t)sm_count * per_sm;
    if (work < g) g = work;
    if (g < 1) g = 1;
    return (int)g;
}
int g_sm_count = 148;

}  // namespace

#define CHECK_LAUNCH() (cudaGetLastError() == cudaSuccess ? 0 : 1)

int launch_fused(const FusedArgs &a, int agg, bool emit_mask, bool wide, int sm_count, cudaStream_t stream)
{
    g_sm_count = sm_count;
    const int nunits = a.g.nblocks * a.g.segs_per_block;
    if (nunits <= 0) return 0;
    const int grid = grid_for(nunits, sm_count, 8);
    if (emit_mask) {
        if (agg == 0) fused_scan_kernel<0, false, true><<<grid, SCAN_THREADS, 0, stream>>>(a);
        else if (agg == 1) fused_scan_kernel<1, false, true><<<grid, SCAN_THREADS, 0, stream>>>(a);
        else fused_scan_kernel<2, false, true><<<grid, SCAN_THREADS, 0, stream>>>(a);
    } else if (wide) {
        if (agg == 0) fused_scan_kernel<0, true, false><<<grid, SCAN_THREADS, 0, stream>>>(a);
        else if (agg == 1) fused_scan_kernel<1, true, false><<<grid, SCAN_THREADS, 0, stream>>>(a);
        else fused_scan_kernel<2, true, false><<<grid, SCAN_THREADS, 0, stream>>>(a);
    } else {
        if (agg == 0) fused_scan_kernel<0, false, false><<<grid, SCAN_THREADS, 0, stream>>>(a);
        else if (agg == 1) fused_scan_kernel<1, false, false><<<grid, SCAN_THREADS, 0, stream>>>(a);
        else fused_scan_kernel<2, false, false><<<grid, SCAN_THREADS, 0, stream>>>(a);
    }
    return CHECK_LAUNCH();
}

int launch_agg_finalize(const AggPartial *partials, int nunits, int cls, AggPartial *result, cudaStream_t stream)
{
    agg_finalize_kernel<<<1, SCAN_THREADS, 0, stream>>>(partials, nunits, cls, result);
    return CHECK_LAUNCH();
}

int launch_vm_mask(const VmArgs &a, int sm_count, cudaStream_t stream)
{
    g_sm_count = sm_count;
    const int tiles_per_block = (int)((a.g.block_size + TILE_ROWS - 1) / TILE_ROWS);
    const int64_t ntiles = (int64_t)a.g.nblocks * tiles_per_block;
    if (ntiles <= 0) return 0;
    vm_mask_kernel<<<grid_for(ntiles, sm_count, 8), SCAN_THREADS, 0, stream>>>(a);
    return CHECK_LAUNCH();
}

int launch_block_counts(const Geometry &g, const uint32_t *mask, int64_t *counts, cudaStream_t stream)
{
    if (g.nblocks <= 0) return 0;
    block_counts_kernel<<<grid_for((g.nblocks + 7) / 8, g_sm_count, 8), SCAN_THREADS, 0, stream>>>(g, mask, counts);
    return CHECK_LAUNCH();
}

int launch_exclusive_scan(const int64_t *in, int64_t *out, int n, cudaStream_t stream)
{
    exclusive_scan_kernel<<<1, 1024, 0, stream>>>(in, out, n);
    return CHECK_LAUNCH();
}

int launch_range_stage(const RangeArgs &a, cudaStream_t stream)
{
    if (a.g.nblocks <= 0) return 0;
    range_stage_kernel<<<grid_for((a.g.nblocks + 7) / 8, g_sm_count, 8), SCAN_THREADS, 0, stream>>>(a);
    return CHECK_LAUNCH();
}

int launch_fill_mask(const Geometry &g, uint32_t *mask, cudaStream_t stream)
{
    const int64_t total = (int64_t)g.nblocks * g.wpb;
    if (total <= 0) return 0;
    fill_mask_kernel<<<grid_for((total + SCAN_THREADS - 1) / SCAN_THREADS, g_sm_count, 8), SCAN_THREADS, 0, stream>>>(g, mask);
    return CHECK_LAUNCH();
}

int launch_str_offsets(const Geometry &g, const ColView &col, int32_t *str_off, int32_t *status, const int32_t *origin, cudaStream_t stream, int lo,
                       int hi, const uint8_t *dead)
{
    if (hi > g.nblocks) hi = g.nblocks;
    if (lo < 0) lo = 0;
    if (hi <= lo) return 0;
    str_offsets_kernel<<<grid_for((hi - lo + 7) / 8, g_sm_count, 8), SCAN_THREADS, 0, stream>>>(g, col, str_off, status, origin, lo, hi, dead);
    return CHECK_LAUNCH();
}

__global__ void group_init_kernel(GroupAcc *acc, long long n, int nvals, int c0, int c1, int c2, int c3)
{
    const int cls[4] = {c0, c1, c2, c3};
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) group_acc_neutral(acc[i], cls[i % nvals]);
}
// the used slots of the table, packed: (first row, accumulators) per group, in no particular order
__global__ void group_compact_kernel(const long long *first, const GroupAcc *acc, long long cap, int nv, long long sentinel, unsigned long long *counter,
                                     long long *out_first, GroupAcc *out_acc)
{
    for (long long sl = (long long)blockIdx.x * blockDim.x + threadIdx.x; sl < cap; sl += (long long)gridDim.x * blockDim.x) {
        const long long f = first[sl];
        if (f == sentinel) continue;
        const unsigned long long i = atomicAdd(counter, 1ull);
        out_first[i] = f;
        for (int v = 0; v < nv; v++) out_acc[i * nv + v] = acc[sl * nv + v];
    }
}
int launch_group_init(GroupAcc *acc, long long n, int nvals, const int *cls, cudaStream_t stream)
{
    if (n <= 0) return 0;
    group_init_kernel<<<grid_for((n + 255) / 256, g_sm_count, 8), 256, 0, stream>>>(acc, n, nvals > 0 ? nvals : 1, cls[0], cls[1], cls[2], cls[3]);
    return CHECK_LAUNCH();
}
int launch_group_compact(const long long *first, const GroupAcc *acc, long long cap, int nv, long long sentinel, unsigned long long *counter,
                         long long *out_first, GroupAcc *out_acc, cudaStream_t stream)
{
    group_compact_kernel<<<grid_for((cap + 255) / 256, g_sm_count, 8), 256, 0, stream>>>(first, acc, cap, nv, sentinel, counter, out_first, out_acc);
    return CHECK_LAUNCH();
}

int launch_group_reduce(const GroupArgs &a, int sm_count, cudaStream_t stream)
{
    const int64_t words = (int64_t)a.g.nblocks * a.g.wpb;
    if (words <= 0) return 0;
    group_reduce_kernel<<<grid_for((words + 7) / 8, sm_count, 8), SCAN_THREADS, 0, stream>>>(a);
    return CHECK_LAUNCH();
}

int launch_unique_first_mask(const long long *first, long long cap, long long sentinel, const Geometry &g, uint32_t *mask, cudaStream_t stream)
{
    unique_first_mask_kernel<<<grid_for((cap + SCAN_THREADS - 1) / SCAN_THREADS, g_sm_count, 8), SCAN_THREADS, 0, stream>>>(first, cap, sentinel, g, mask);
    return CHECK_LAUNCH();
}

int launch_merge_insert(const MergeArgs &a, cudaStream_t stream)
{
    if (a.n <= 0) return 0;
    merge_insert_kernel<<<grid_for((a.n + SCAN_THREADS - 1) / SCAN_THREADS, g_sm_count, 8), SCAN_THREADS, 0, stream>>>(a);
    return CHECK_LAUNCH();
}

int launch_merge_keep(const MergeArgs &a, int64_t *keep, cudaStream_t stream)
{
    if (a.n <= 0) return 0;
    merge_keep_kernel<<<grid_for((a.n + SCAN_THREADS - 1) / SCAN_THREADS, g_sm_count, 8), SCAN_THREADS, 0, stream>>>(a, keep);
    return CHECK_LAUNCH();
}

int launch_str_lengths(const int32_t *sizes, long long n, int64_t *out, cudaStream_t stream)
{
    if (n <= 0) return 0;
    str_lengths_kernel<<<grid_for((n + SCAN_THREADS - 1) / SCAN_THREADS, g_sm_count, 8), SCAN_THREADS, 0, stream>>>(sizes, n, out);
    return CHECK_LAUNCH();
}

int launch_merge_emit(const MergeArgs &a, const int64_t *keep_pos, const long long *first, long long *out_first, cudaStream_t stream)
{
    if (a.n <= 0) return 0;
    merge_emit_kernel<<<grid_for((a.n + SCAN_THREADS - 1) / SCAN_THREADS, g_sm_count, 8), SCAN_THREADS, 0, stream>>>(a, keep_pos, first, out_first);
    return CHECK_LAUNCH();
}

int launch_merge_fold(const MergeArgs &a, const int64_t *keep_pos, const dfdb_agg *in, int nvals, long long lo, long long hi, dfdb_agg *out, int *dup,
                      cudaStream_t stream)
{
    if (hi <= lo || nvals <= 0) return 0;
    merge_fold_kernel<<<grid_for((hi - lo + SCAN_THREADS - 1) / SCAN_THREADS, g_sm_count, 8), SCAN_THREADS, 0, stream>>>(a, keep_pos, in, nvals, lo, hi, out, dup);
    return CHECK_LAUNCH();
}

int launch_merge_fold_finish(dfdb_agg *out, long long n, cudaStream_t stream)
{
    if (n <= 0) return 0;
    merge_fold_finish_kernel<<<grid_for((n + SCAN_THREADS - 1) / SCAN_THREADS, g_sm_count, 8), SCAN_THREADS, 0, stream>>>(out, n);
    return CHECK_LAUNCH();
}

long long scan_i64_tmp_len(long long n) { return 2 * ((n + SCAN_CHUNK - 1) / SCAN_CHUNK + 1); }

int launch_scan_i64(int64_t *data, long long n, int64_t *tmp, cudaStream_t stream)
{
    const long long nchunks = (n + SCAN_CHUNK - 1) / SCAN_CHUNK;
    if (nchunks > 0x7fffffff) return 1;
    int64_t *sums = tmp, *bases = tmp + nchunks + 1;
    if (nchunks > 0) {
        chunk_sums_kernel<<<grid_for(nchunks, g_sm_count, 8), SCAN_THREADS, 0, stream>>>(data, n, sums);
        if (CHECK_LAUNCH()) return 1;
    }
    exclusive_scan_kernel<<<1, 1024, 0, stream>>>(sums, bases, (int)nchunks);
    if (CHECK_LAUNCH()) return 1;
    chunk_rescan_kernel<<<grid_for(nchunks > 0 ? nchunks : 1, g_sm_count, 8), SCAN_THREADS, 0, stream>>>(data, n, bases);
    return CHECK_LAUNCH();
}

int launch_zone_map(const Geometry &g, const ColView &col, ZoneOut *out, cudaStream_t stream)
{
    if (g.nblocks <= 0) return 0;
    zone_map_kernel<<<grid_for(g.nblocks, g_sm_count, 8), SCAN_THREADS, 0, stream>>>(g, col, out);
    return CHECK_LAUNCH();
}

int launch_gather_fixed(const GatherArgs &a, cudaStream_t stream)
{
    if (a.g.nblocks <= 0) return 0;
    gather_fixed_kernel<<<grid_for(a.g.nblocks, g_sm_count, 8), SCAN_THREADS, 0, stream>>>(a);
    return CHECK_LAUNCH();
}

int launch_gather_indices(const GatherArgs &a, cudaStream_t stream)
{
    if (a.g.nblocks <= 0) return 0;
    gather_indices_kernel<<<grid_for(a.g.nblocks, g_sm_count, 8), SCAN_THREADS, 0, stream>>>(a);
    return CHECK_LAUNCH();
}

int launch_str_block_bytes(const GatherArgs &a, int64_t *blk_bytes, cudaStream_t stream)
{
    if (a.g.nblocks <= 0) return 0;
    str_block_bytes_kernel<<<grid_for(a.g.nblocks, g_sm_count, 8), SCAN_THREADS, 0, stream>>>(a, blk_bytes);
    return CHECK_LAUNCH();
}

int launch_gather_strings(const GatherArgs &a, cudaStream_t stream)
{
    if (a.g.nblocks <= 0) return 0;
    gather_strings_kernel<<<grid_for(a.g.nblocks, g_sm_count, 8), SCAN_THREADS, 0, stream>>>(a);
    return CHECK_LAUNCH();
}

int launch_agg_vm(const AggVmArgs &a, int sm_count, cudaStream_t stream)
{
    const int nunits = a.g.nblocks * a.g.segs_per_block;
    if (nunits <= 0) return 0;
    agg_vm_kernel<<<grid_for(nunits, sm_count, 8), SCAN_THREADS, 0, stream>>>(a);
    return CHECK_LAUNCH();
}

int launch_proj_vm(const ProjVmArgs &a, cudaStream_t stream)
{
    if (a.g.nblocks <= 0) return 0;
    proj_vm_kernel<<<grid_for(a.g.nblocks, g_sm_count, 8), SCAN_THREADS, 0, stream>>>(a);
    return CHECK_LAUNCH();
}

}  // namespace dfdb
