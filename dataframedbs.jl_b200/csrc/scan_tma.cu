// scan_tma.cu -- K3+K7 fast path: TMA-staged, persistent, fused predicate + aggregate over 8-byte columns.
//
// Same contract as fused_scan_kernel (scan_kernels.cu): conjunction of `column <cmp> constant` terms ->
// selection bits -> count / sum / min / max of one column, one partial per work unit, fixed combination
// order.  Stands in for apply(::SelectionExecutor) + eval_on_range + the Base folds over iterate(::DFColumn)
// (/root/reference/src/tables/selection.jl:133-167, broadcast.jl:96-133, column.jl:102-126).
//
// Data movement: one elected thread streams 16 KB column tiles HBM -> shared memory with
// cp.async.bulk (SASS UBLKCP) into an N-stage ring, completion tracked by one mbarrier per stage; the
// 256 consumer threads read the tiles with conflict-free 128-bit LDS.  Memory-level parallelism is set
// by the ring depth (up to ~190 KB in flight per SM), not by registers or occupancy.
// The predicate is normalised on the host into one closed interval per column (plus != terms), so the
// inner loop is a subtract + one unsigned compare per integer column, or two DSETP per Float64 column.
//
// Algorithmic bytes: 8 B per row per distinct column touched (+ 1 bit per row per nullable column).
#include <cuda_runtime.h>
#include <math_constants.h>

#include "kernels.cuh"

namespace dfdb {
namespace {

constexpr unsigned FULL = 0xffffffffu;
constexpr int TILE_BYTES = TILE_ROWS * 8;   // 16 KB per column per stage
constexpr int TILE_MASK_BYTES = TILE_ROWS / 8;   // the tile's selection bits (mask-in form)

__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t *bar, uint32_t count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, uint32_t bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t *bar, uint32_t parity)
{
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(smem_u32(bar)), "r"(parity)
        : "memory");
    return ok != 0;
}
__device__ __forceinline__ void bulk_g2s(void *dst_smem, const void *src_gmem, uint32_t bytes, uint64_t *bar)
{
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst_smem)),
                 "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}

struct TileCursor {
    int unit;        // current work unit of this CTA (strided by gridDim.x)
    int lb;          // local block of the unit
    int64_t rows_b;  // rows of that block
    int64_t row1;    // end row of the unit inside the block
    int64_t tile0;   // first row of the current tile
};

__device__ __forceinline__ void cursor_load_unit(TileCursor &c, const Geometry &g)
{
    c.lb = c.unit / g.segs_per_block;
    const int seg = c.unit - c.lb * g.segs_per_block;
    c.rows_b = block_rows(g, c.lb);
    c.tile0 = (int64_t)seg * g.seg_rows;
    c.row1 = c.tile0 + g.seg_rows;
    if (c.row1 > c.rows_b) c.row1 = c.rows_b;
    if (g.dead && g.dead[c.lb]) c.row1 = c.tile0;      // ruled out by the zone maps: the unit is empty (its partial stays zero)
}
// advance to the next non-empty tile; false when the CTA has no more work
__device__ __forceinline__ bool cursor_next(TileCursor &c, const Geometry &g, int nunits, bool first)
{
    if (!first) c.tile0 += TILE_ROWS;
    for (;;) {
        if (c.unit >= nunits) return false;
        if (first) { cursor_load_unit(c, g); first = false; }
        if (c.tile0 < c.row1) return true;
        c.unit += gridDim.x;
        if (c.unit >= nunits) return false;
        cursor_load_unit(c, g);
    }
}

__device__ __forceinline__ void two_sum_add(double &hi, double &lo, double x)
{
    const double t = hi + x;
    const double bb = t - hi;
    lo += (hi - (t - bb)) + (x - bb);
    hi = t;
}

struct Acc {
    long long count, nmissing, sum_i;
    double sum_hi, sum_lo;
    long long min_i, max_i;
    double min_f, max_f;
    int has_nan, neg_zero, pos_zero;
};

template <int AGG>
__device__ __forceinline__ void acc_reset(Acc &a, bool uns)
{
    a.count = 0; a.nmissing = 0; a.sum_i = 0; a.sum_hi = 0.0; a.sum_lo = 0.0;
    a.min_i = uns ? -1ll : 0x7fffffffffffffffll;                 // identity of min (as unsigned: all ones)
    a.max_i = uns ? 0ll : (long long)0x8000000000000000ull;
    a.min_f = CUDART_INF; a.max_f = -CUDART_INF;
    a.has_nan = 0; a.neg_zero = 0; a.pos_zero = 0;
}

__device__ __forceinline__ AggPartial acc_to_partial(const Acc &a, int agg)
{
    AggPartial p;
    p.count = a.count; p.nmissing = a.nmissing; p.sum_i = a.sum_i;
    p.sum_f = a.sum_hi; p.sum_lo = a.sum_lo;
    p.min_i = a.min_i; p.max_i = a.max_i;
    p.min_f = a.min_f; p.max_f = a.max_f;
    // signed zeros: -0.0 orders before 0.0 in Julia's min/max
    if (agg == 2) {
        if (p.min_f == 0.0 && a.neg_zero) p.min_f = -0.0;
        if (p.min_f == 0.0 && !a.neg_zero) p.min_f = 0.0;
        if (p.max_f == 0.0 && a.pos_zero) p.max_f = 0.0;
        if (p.max_f == 0.0 && !a.pos_zero) p.max_f = -0.0;
    }
    p.has_nan = a.has_nan;
    p.has_value = (agg != 0) && (a.count - a.nmissing > 0);
    return p;
}

__device__ __forceinline__ double jl_min(double a, double b) { return (a < b || (a == b && signbit(a))) ? a : b; }
__device__ __forceinline__ double jl_max(double a, double b) { return (a > b || (a == b && !signbit(a))) ? a : b; }

__device__ __forceinline__ void partial_merge(AggPartial &a, const AggPartial &b, int cls)
{
    a.count += b.count;
    a.nmissing += b.nmissing;
    a.sum_i = (long long)((unsigned long long)a.sum_i + (unsigned long long)b.sum_i);
    two_sum_add(a.sum_f, a.sum_lo, b.sum_f);
    a.sum_lo += b.sum_lo;
    a.has_nan |= b.has_nan;
    if (b.has_value) {
        if (!a.has_value) { a.min_i = b.min_i; a.max_i = b.max_i; a.min_f = b.min_f; a.max_f = b.max_f; }
        else if (cls == VC_FLT) { a.min_f = jl_min(a.min_f, b.min_f); a.max_f = jl_max(a.max_f, b.max_f); }
        else if (cls == VC_UINT) {
            if ((unsigned long long)b.min_i < (unsigned long long)a.min_i) a.min_i = b.min_i;
            if ((unsigned long long)b.max_i > (unsigned long long)a.max_i) a.max_i = b.max_i;
        } else {
            if (b.min_i < a.min_i) a.min_i = b.min_i;
            if (b.max_i > a.max_i) a.max_i = b.max_i;
        }
        a.has_value = 1;
    }
}

__device__ AggPartial partial_block_reduce(AggPartial a, int cls, AggPartial *smem)
{
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) {
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
        if (lane + d < 32) partial_merge(a, b, cls);
    }
    if (lane == 0) smem[warp] = a;
    __syncthreads();
    if (threadIdx.x == 0) {
        AggPartial r = smem[0];
        for (int w = 1; w < SCAN_THREADS / 32; w++) partial_merge(r, smem[w], cls);
        a = r;
    }
    __syncthreads();
    return a;
}

// selection bits of this thread's 8 rows of the staged tile for one column test
__device__ __forceinline__ unsigned test_bits(const ColTest &t, const ulonglong2 *tile, int tid)
{
    unsigned bits = 0;
    if (t.cls == VC_FLT) {
#pragma unroll
        for (int s = 0; s < 4; s++) {
            const ulonglong2 x = tile[s * SCAN_THREADS + tid];
            const bool pa = coltest_flt(t, __longlong_as_double((long long)x.x)), pb = coltest_flt(t, __longlong_as_double((long long)x.y));
            bits |= ((unsigned)pa << (2 * s)) | ((unsigned)pb << (2 * s + 1));
        }
    } else {
#pragma unroll
        for (int s = 0; s < 4; s++) {
            const ulonglong2 x = tile[s * SCAN_THREADS + tid];
            bits |= ((unsigned)coltest_int(t, x.x) << (2 * s)) | ((unsigned)coltest_int(t, x.y) << (2 * s + 1));
        }
    }
    return bits;
}

// missing bits of this thread's 8 rows (bit k = row k of the thread is missing)
__device__ __forceinline__ unsigned missing_bits(const ColView &c, int lb, int64_t tile0, int tid)
{
    const unsigned long long *w = reinterpret_cast<const unsigned long long *>(c.base + c.blk_off[lb]);
    unsigned m = 0;
#pragma unroll
    for (int s = 0; s < 4; s++) {
        const int64_t r = tile0 + s * (2 * SCAN_THREADS) + 2 * tid;    // even row: both rows live in the same word
        const unsigned long long word = __ldg(w + (r >> 6));
        m |= (unsigned)((word >> (r & 63)) & 3ull) << (2 * s);
    }
    return m;
}

// MASK: the selection comes from A.mask_in, staged with the tile, instead of the tests (the rows, their order and the folds
// are the same, so the results are bit for bit those of the tests)
template <int AGG, bool MASK>
__global__ void __launch_bounds__(SCAN_THREADS, MASK ? TMA_MASK_CTAS : 2) fused_scan_tma_kernel(const TmaScanArgs A)
{
    extern __shared__ __align__(128) uint8_t smem_raw[];
    __shared__ uint64_t full_bar[TMA_MAX_STAGES];
    __shared__ AggPartial red[SCAN_THREADS / 32];

    const Geometry g = A.g;
    const int tid = threadIdx.x;
    const int nunits = g.nblocks * g.segs_per_block;
    const int ncols = A.ncols, nstages = A.nstages;
    const bool agg_uns = A.agg_cls == VC_UINT || A.agg_cls == VC_BOOL;
    const size_t stage_bytes = (size_t)ncols * TILE_BYTES + (MASK ? TILE_MASK_BYTES : 0);

    if (tid == 0) {
        for (int s = 0; s < nstages; s++) mbar_init(&full_bar[s], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    }
    __syncthreads();

    // producer cursor (thread 0 only) runs up to nstages tiles ahead of the consumer cursor
    TileCursor pc, cc;
    pc.unit = cc.unit = blockIdx.x;
    bool p_more = false;
    auto issue = [&](int stage) {
        // one tile of every staged column into `stage`
        const int64_t nrows = (pc.row1 - pc.tile0 < TILE_ROWS) ? pc.row1 - pc.tile0 : TILE_ROWS;
        const uint32_t bytes = (uint32_t)((nrows * 8 + 15) & ~15ll);
        // (mask-in: whole words, rounded up to 16 bytes -- the block's words are a multiple of four)
        const uint32_t mbytes = MASK ? (uint32_t)((((nrows + 31) >> 5) * 4 + 15) & ~15ll) : 0u;
        mbar_expect_tx(&full_bar[stage], bytes * (uint32_t)ncols + mbytes);
        for (int c = 0; c < ncols; c++) {
            const ColView &cv = A.col[c];
            const uint8_t *vals = cv.base + cv.blk_off[pc.lb] + (cv.nullable ? ((pc.rows_b + 63) >> 6) * 8 : 0);
            bulk_g2s(smem_raw + (size_t)stage * stage_bytes + (size_t)c * TILE_BYTES, vals + pc.tile0 * 8, bytes, &full_bar[stage]);
        }
        if (MASK)
            bulk_g2s(smem_raw + (size_t)stage * stage_bytes + (size_t)ncols * TILE_BYTES, A.mask_in + (int64_t)pc.lb * g.wpb + (pc.tile0 >> 5), mbytes,
                     &full_bar[stage]);
    };
    if (tid == 0) {
        p_more = cursor_next(pc, g, nunits, true);
        for (int s = 0; s < nstages && p_more; s++) {
            issue(s);
            p_more = cursor_next(pc, g, nunits, false);
        }
    }

    Acc acc;
    acc_reset<AGG>(acc, agg_uns);
    bool more = cursor_next(cc, g, nunits, true);
    int stage = 0;
    uint32_t parity = 0;
    while (more) {
        while (!mbar_try_wait(&full_bar[stage], parity)) { }
        const uint8_t *sbase = smem_raw + (size_t)stage * stage_bytes;

        // rows of this thread that exist in the tile: rows 2*tid, 2*tid+1 of four 512-row sub-tiles
        unsigned m = 0xffu;
        if (cc.tile0 + TILE_ROWS > cc.row1) {
            m = 0;
#pragma unroll
            for (int k = 0; k < 8; k++) m |= (unsigned)(cc.tile0 + (k >> 1) * (2 * SCAN_THREADS) + 2 * tid + (k & 1) < cc.row1) << k;
        }
        if (MASK) {
            // row tile0 + 512 s + 2 tid + j is bit (2 tid + j) & 31 of the tile's mask word 16 s + tid / 16
            const uint32_t *mk = reinterpret_cast<const uint32_t *>(sbase + (size_t)ncols * TILE_BYTES);
            unsigned bits = 0;
#pragma unroll
            for (int s = 0; s < 4; s++) bits |= ((mk[16 * s + (tid >> 4)] >> ((2 * tid) & 31)) & 3u) << (2 * s);
            m &= bits;
        }
        for (int t = 0; t < (MASK ? 0 : A.ntests); t++) {
            const ColTest &ct = A.test[t];
            unsigned bits = test_bits(ct, reinterpret_cast<const ulonglong2 *>(sbase + (size_t)ct.col * TILE_BYTES), tid);
            if (A.col[ct.col].nullable) bits &= ~missing_bits(A.col[ct.col], cc.lb, cc.tile0, tid);   // missing -> false
            m &= bits;
        }
        acc.count += __popc(m);
        if (AGG) {
            const ulonglong2 *tile = reinterpret_cast<const ulonglong2 *>(sbase + (size_t)A.agg_col * TILE_BYTES);
            unsigned use = m;
            if (A.col[A.agg_col].nullable) {
                const unsigned ms = missing_bits(A.col[A.agg_col], cc.lb, cc.tile0, tid);
                acc.nmissing += __popc(m & ms);
                use &= ~ms;
            }
            if (AGG == 2) {
                double tsum = 0.0;
#pragma unroll
                for (int s = 0; s < 4; s++) {
                    const ulonglong2 x = tile[s * SCAN_THREADS + tid];
                    const double v[2] = {__longlong_as_double((long long)x.x), __longlong_as_double((long long)x.y)};
#pragma unroll
                    for (int j = 0; j < 2; j++) {
                        if ((use >> (2 * s + j)) & 1u) {
                            const double a = v[j];
                            tsum += a;
                            if (a < acc.min_f) acc.min_f = a;
                            if (a > acc.max_f) acc.max_f = a;
                            if (a != a) acc.has_nan = 1;
                            if (a == 0.0) { if (signbit(a)) acc.neg_zero = 1; else acc.pos_zero = 1; }
                        }
                    }
                }
                two_sum_add(acc.sum_hi, acc.sum_lo, tsum);
            } else {
#pragma unroll
                for (int s = 0; s < 4; s++) {
                    const ulonglong2 x = tile[s * SCAN_THREADS + tid];
                    const unsigned long long v[2] = {x.x, x.y};
#pragma unroll
                    for (int j = 0; j < 2; j++) {
                        if ((use >> (2 * s + j)) & 1u) {
                            const unsigned long long a = v[j];
                            acc.sum_i = (long long)((unsigned long long)acc.sum_i + a);
                            if (agg_uns) {
                                if (a < (unsigned long long)acc.min_i) acc.min_i = (long long)a;
                                if (a > (unsigned long long)acc.max_i) acc.max_i = (long long)a;
                            } else {
                                if ((long long)a < acc.min_i) acc.min_i = (long long)a;
                                if ((long long)a > acc.max_i) acc.max_i = (long long)a;
                            }
                        }
                    }
                }
            }
        }
        // unit finished? fold the CTA's accumulators in a fixed order and emit the unit partial
        const int this_unit = cc.unit;
        const bool unit_done = cc.tile0 + TILE_ROWS >= cc.row1;
        __syncthreads();                                   // every thread is done reading this stage
        if (tid == 0 && p_more) {
            issue(stage);
            p_more = cursor_next(pc, g, nunits, false);
        }
        if (unit_done) {
            AggPartial p = acc_to_partial(acc, AGG);
            p = partial_block_reduce(p, AGG == 2 ? VC_FLT : A.agg_cls, red);
            if (tid == 0) A.partials[this_unit] = p;
            acc_reset<AGG>(acc, agg_uns);
        }
        more = cursor_next(cc, g, nunits, false);
        if (++stage == nstages) { stage = 0; parity ^= 1u; }
    }
}

}  // namespace

int launch_fused_tma(const TmaScanArgs &a, int agg, int sm_count, cudaStream_t stream)
{
    const int nunits = a.g.nblocks * a.g.segs_per_block;
    if (nunits <= 0) return 0;
    const size_t smem = (size_t)a.nstages * ((size_t)a.ncols * TILE_BYTES + (a.mask_in ? TILE_MASK_BYTES : 0));
    static bool configured = false;
    if (!configured) {
        cudaFuncSetAttribute(fused_scan_tma_kernel<0, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 110 * 1024);
        cudaFuncSetAttribute(fused_scan_tma_kernel<1, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 110 * 1024);
        cudaFuncSetAttribute(fused_scan_tma_kernel<2, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 110 * 1024);
        cudaFuncSetAttribute(fused_scan_tma_kernel<1, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 110 * 1024);
        cudaFuncSetAttribute(fused_scan_tma_kernel<2, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 110 * 1024);
        configured = true;
    }
    const int per_sm = a.mask_in ? TMA_MASK_CTAS : 2;
    const int grid = nunits < per_sm * sm_count ? nunits : per_sm * sm_count;   // persistent CTAs
    if (a.mask_in) {
        if (agg == 1) fused_scan_tma_kernel<1, true><<<grid, SCAN_THREADS, smem, stream>>>(a);
        else if (agg == 2) fused_scan_tma_kernel<2, true><<<grid, SCAN_THREADS, smem, stream>>>(a);
        else return 1;   // (mask-in is an aggregate's form: a count stages no column)
    } else if (agg == 0) fused_scan_tma_kernel<0, false><<<grid, SCAN_THREADS, smem, stream>>>(a);
    else if (agg == 1) fused_scan_tma_kernel<1, false><<<grid, SCAN_THREADS, smem, stream>>>(a);
    else fused_scan_tma_kernel<2, false><<<grid, SCAN_THREADS, smem, stream>>>(a);
    return cudaGetLastError() == cudaSuccess ? 0 : 1;
}

}  // namespace dfdb
