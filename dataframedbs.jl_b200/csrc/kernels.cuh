// kernels.cuh -- kernel argument PODs and launch wrappers shared by the .cu translation units.
#pragma once
#include <cuda_runtime.h>

#include "internal.hpp"

namespace dfdb {

// ---- K1: LZ4 block decode ------------------------------------------------------------------------
constexpr int DECODE_MAX_COLS = 16;
struct DecodeCol {
    const uint8_t *comp;        // packed compressed payloads (16-byte aligned, 16-byte padded slots)
    const int64_t *comp_off;    // per local block
    const int32_t *comp_len;
    const int64_t *dec_off;     // per local block: offset of the 256-byte aligned body slot
    const int32_t *origin;
    uint8_t *out;
    int32_t *status;
    const uint8_t *skip;        // per local block, may be null: 1 = stored block whose body is referenced in place
};
struct DecodeArgs {
    DecodeCol col[DECODE_MAX_COLS];
    int ncols;
    int nblocks;   // blocks per column in this launch
    int blk0;      // first local block of the launch (chunked, copy-overlapped decode)
    unsigned long long *stats;   // optional diagnostics counters (null = off), see lz4_decode_v3.cu
    int hot;       // lane decoder only: the columns are word-regular (nearly every token is 0x04 with an offset that is a multiple of 8): hot-step schedule
};
int launch_lz4_decode(const DecodeArgs &args, unsigned int *d_counter, int sm_count, cudaStream_t stream);      // warp per block, one sequence at a time (decode_simple)
constexpr int LZ4_SLOTS_PER_SM = 60;   // column blocks one decoder CTA keeps in flight (NSLOT of the walker / consumer decoder)
int launch_lz4_decode_v3(const DecodeArgs &args, unsigned int *d_counter, int sm_count, cudaStream_t stream, int cta_limit = 0);
int launch_lz4_decode_long(const DecodeArgs &args, unsigned int *d_counter, int sm_count, cudaStream_t stream, int cta_limit = 0);   // warp per block, one sequence at a time, headers parsed out of a shared-memory window of the stream (long-sequence columns)
int launch_lz4_decode_bytes(const DecodeArgs &args, unsigned int *d_counter, int sm_count, cudaStream_t stream, int cta_limit = 0);  // warp per block, bare-match byte streams: verified token positions, byte copies by pointer jumping (lz4_decode_bytes.cu)
int launch_lz4_decode_spec(const DecodeArgs &args, unsigned int *d_counter, int sm_count, cudaStream_t stream, int cta_limit = 0);   // warp per block, plain token runs verified in parallel (word-regular columns)

// ---- write path: raw LZ4 block compression (lz4_compress.cu), one warp per body ---------------------------------------
struct CompressArgs {
    const uint8_t *src;         // bodies, each readable 16 bytes past its end
    const int64_t *src_off, *src_len;
    uint8_t *dst;               // one slot of LZ4_compressBound(len) bytes per body
    const int64_t *dst_off;
    int64_t *dst_len;           // out: compressed size per body
    int nblocks;
};
int launch_lz4_compress(const CompressArgs &a, unsigned int *d_counter, int sm_count, cudaStream_t stream);

// ---- scan geometry -------------------------------------------------------------------------------
constexpr int SCAN_THREADS = 256;
constexpr int ROWS_PER_THREAD = 8;
constexpr int TILE_ROWS = SCAN_THREADS * ROWS_PER_THREAD;   // 2048 rows per CTA iteration

struct Geometry {
    int64_t nrows_total;     // rows of the whole table
    int64_t block_size;      // rows per column block
    int64_t blk_lo;          // first table block of this shard
    int32_t nblocks;         // local blocks
    int32_t wpb;             // mask words (32 rows each) per block
    int32_t segs_per_block;  // work units per block
    int32_t seg_rows;        // rows per work unit (multiple of TILE_ROWS)
    const uint8_t *dead;     // per local block, may be null: 1 = no row of the block can be selected (zone maps); its body is not decoded
};

__host__ __device__ inline int64_t block_rows(const Geometry &g, int lb)
{
    int64_t r = g.nrows_total - (g.blk_lo + lb) * g.block_size;
    return r < g.block_size ? (r < 0 ? 0 : r) : g.block_size;
}

// per-unit aggregate partial (also the final result layout on device)
struct AggPartial {
    long long count, nmissing, sum_i;
    double sum_f, sum_lo;
    long long min_i, max_i;
    double min_f, max_f;
    int has_nan, has_value;
};

// ---- K3/K7 fused: conjunction of terms (or a precomputed mask) -> count / aggregate / mask -----------
struct FusedArgs {
    Geometry g;
    ColView term_col[MAX_TERMS];
    Term term[MAX_TERMS];
    int nterms;
    int const_false;              // some term folded to `false`
    const uint32_t *mask_in;      // selection comes from this mask instead of the terms (may be null)
    uint32_t *mask_out;           // EMIT: write the selection mask (AND with mask_in when given)
    ColView agg_col;              // aggregated column (AGG != 0)
    int agg_cls;                  // VC_INT / VC_UINT / VC_FLT / VC_BOOL
    AggPartial *partials;         // one per unit
};
int launch_fused(const FusedArgs &a, int agg, bool emit_mask, bool wide, int sm_count, cudaStream_t stream);
int launch_agg_finalize(const AggPartial *partials, int nunits, int cls, AggPartial *result, cudaStream_t stream);

// ---- K3+K7 TMA-staged fast path (scan_tma.cu) -----------------------------------------------------------
constexpr int TMA_MAX_STAGES = 12;
constexpr int TMA_MAX_COLS = 4;
// all terms on one column folded into a closed interval [lo, hi] plus up to two != constants
struct ColTest {
    int col;            // index into TmaScanArgs::col
    int cls;            // VC_INT / VC_UINT / VC_FLT
    int n_ne;
    int nan_passes;     // Float64 column with only != terms: NaN rows pass
    long long lo_i, hi_i;
    double lo_f, hi_f;
    long long ne_i[2];
    double ne_f[2];
};
struct TmaScanArgs {
    Geometry g;
    ColView col[TMA_MAX_COLS];   // staged 8-byte columns
    int ncols, nstages;
    ColTest test[TMA_MAX_COLS];
    int ntests;
    int agg_col, agg_cls;
    AggPartial *partials;
};
int launch_fused_tma(const TmaScanArgs &a, int agg, int sm_count, cudaStream_t stream);

// ---- K1 lane-per-block decoder (lz4_decode_lane.cu) ---------------------------------------------------------------
int launch_lz4_decode_lane(const DecodeArgs &args, unsigned int *d_counter, int sm_count, cudaStream_t stream, int cta_limit = 0);

// ---- K3 generic: VM predicate -> mask ------------------------------------------------------------------
struct VmArgs {
    Geometry g;
    ColView slot[MAX_SLOTS];
    const VmProgram *prog;        // device copy
    const uint32_t *mask_in;      // rows to evaluate (null = all rows)
    uint32_t *mask_out;
    int *error_flag;              // DivideError etc.
};
int launch_vm_mask(const VmArgs &a, int sm_count, cudaStream_t stream);

// ---- `in` collections: the hash-set build, and the selection stage in(stored fixed-width column, set) ----------------------
// build: inserts the n canonical keys of `in` (fixed width: the keys; String: off | len << 32 into set.chars) into the table
// of `set`, whose occupancy bits the caller zeroed
struct SetBuildArgs {
    SetDesc set;
    const unsigned long long *in;
    long long n;
};
int launch_inset_build(const SetBuildArgs &a, cudaStream_t stream);
// mask: bits of the rows whose value is in the set, ANDed with mask_in when given
constexpr long long INSET_SMEM_SLOTS = 8192;   // tables of at most this many slots are staged in shared memory (64 KB + occupancy)
struct InSetMaskArgs {
    Geometry g;
    ColView col;
    SetDesc set;
    const uint32_t *mask_in;      // rows to evaluate (null = all rows)
    uint32_t *mask_out;
};
int launch_inset_mask(const InSetMaskArgs &a, int sm_count, cudaStream_t stream);

// ---- K4: range / index-vector stages on running survivor ranks ----------------------------------------
struct RangeArgs {
    Geometry g;
    uint32_t *mask;               // in/out
    int dense;                    // 1: every row of the shard survives so far -> rank = global row number
    const int64_t *blk_base;      // exclusive scan of per-block survivor counts (when !dense)
    int64_t rank_offset;          // survivors before this shard (multi-GPU) -- added to every rank
    int kind;                     // ST_RANGE / ST_INDEXVEC
    int64_t start, step, stop;
    const int64_t *idx;
    int64_t nidx;
};
int launch_block_counts(const Geometry &g, const uint32_t *mask, int64_t *counts, cudaStream_t stream);
int launch_exclusive_scan(const int64_t *in, int64_t *out, int n, cudaStream_t stream);   // out[n] = total
int launch_range_stage(const RangeArgs &a, cudaStream_t stream);
int launch_fill_mask(const Geometry &g, uint32_t *mask, cudaStream_t stream);

// ---- K2: String bodies: per-row char offsets (unsafe_remake_offsets!) --------------------------------
int launch_str_offsets(const Geometry &g, const ColView &col, int32_t *str_off, int32_t *status, const int32_t *origin, cudaStream_t stream, int lo = 0, int hi = 0x7fffffff,
                       const uint8_t *dead = nullptr);   // local blocks [lo, hi) except those flagged in `dead`

// ---- zone maps (SURVEY.md 8f: block index sidecar): per block min / max / null count of a decoded fixed-width column ----
struct ZoneOut { unsigned long long min_bits, max_bits; long long null_count; int flags, pad; };
int launch_zone_map(const Geometry &g, const ColView &col, ZoneOut *out, cudaStream_t stream);

// ---- group-by reduce (SURVEY.md 8f rank 4; the stub at src/tables/aggregate.jl:1-36): hash aggregation of the selected rows -----
struct GroupAcc {                    // per (group, value column)
    unsigned long long count;        // selected rows of the group (missing included)
    unsigned long long nmissing;
    long long sum_i;                 // wrapping integer sum
    double sum_f;
    long long min_k, max_k;          // integers: the values; floats: their order-preserving integer encoding (NaN excluded)
    int flags, pad;                  // 1 = has a non-missing, non-NaN value, 2 = has NaN
};
struct GroupArgs {
    Geometry g;
    const uint32_t *mask;
    int nkeys, nvals;
    ColView key[GROUP_MAX_KEYS];
    ColView val[GROUP_MAX_VALS];
    long long *rep;                  // cap slots: a row of the group (0-based shard row), -1 = empty
    long long *first;                // cap slots: lowest row of the group
    GroupAcc *acc;                   // cap x nvals
    unsigned long long cap_mask;     // cap - 1 (cap is a power of two)
    int *overflow;                   // set when the table filled up: the host doubles it and runs again
    unsigned long long *ngroups;
};
int launch_group_reduce(const GroupArgs &a, int sm_count, cudaStream_t stream);
int launch_group_init(GroupAcc *acc, long long n, int nvals, const int *cls, cudaStream_t stream);     // accumulators at the identities of their order
int launch_group_compact(const long long *first, const GroupAcc *acc, long long cap, int nv, long long sentinel, unsigned long long *counter,
                         long long *out_first, GroupAcc *out_acc, cudaStream_t stream);                // used slots, packed

// dfdb_agg_fold's arithmetic, shared by the host fold and the device fold of merged groups so that the two give the same bits:
// one partial into the running result (which starts all zero), then the final renormalisation of the compensated sum
__host__ __device__ inline bool agg_signbit(double x)
{
    unsigned long long b;
    memcpy(&b, &x, 8);
    return (b >> 63) != 0;
}
__host__ __device__ inline void dfdb_agg_fold_step(dfdb_agg &r, const dfdb_agg &p)
{
    r.count += p.count;
    r.nmissing += p.nmissing;
    r.sum_i64 = (int64_t)((uint64_t)r.sum_i64 + (uint64_t)p.sum_i64);
    {
        // two-sum: the result does not depend on how the rows were split beyond the last bit of the compensated pair
        const double t = r.sum_f64 + p.sum_f64;
        const double bb = t - r.sum_f64;
        r.sum_f64_lo += (r.sum_f64 - (t - bb)) + (p.sum_f64 - bb);
        r.sum_f64_lo += p.sum_f64_lo;
        r.sum_f64 = t;
    }
    r.has_nan |= p.has_nan;
    if (!p.value_class) return;
    if (!r.value_class) {
        r.min_i64 = p.min_i64; r.max_i64 = p.max_i64; r.min_f64 = p.min_f64; r.max_f64 = p.max_f64;
        r.value_class = p.value_class;
    } else if (p.value_class == 3) {
        // Julia's min / max: NaN propagates, -0.0 < 0.0
        const double a = r.min_f64, b = p.min_f64, c = r.max_f64, d = p.max_f64;
        r.min_f64 = (a != a) ? a : (b != b) ? b : ((a < b || (a == b && agg_signbit(a))) ? a : b);
        r.max_f64 = (c != c) ? c : (d != d) ? d : ((c > d || (c == d && !agg_signbit(c))) ? c : d);
    } else if (p.value_class == 2) {
        if ((uint64_t)p.min_i64 < (uint64_t)r.min_i64) r.min_i64 = p.min_i64;
        if ((uint64_t)p.max_i64 > (uint64_t)r.max_i64) r.max_i64 = p.max_i64;
    } else {
        if (p.min_i64 < r.min_i64) r.min_i64 = p.min_i64;
        if (p.max_i64 > r.max_i64) r.max_i64 = p.max_i64;
    }
}
__host__ __device__ inline void dfdb_agg_fold_finish(dfdb_agg &r)
{
    if (!isfinite(r.sum_f64)) { r.sum_f64_lo = 0.0; return; }   // an infinite sum's compensation term is inf - inf = NaN
    const double s = r.sum_f64 + r.sum_f64_lo;
    r.sum_f64_lo = (r.sum_f64 - s) + r.sum_f64_lo;
    r.sum_f64 = s;
}

// ---- unique (Base.unique over iterate(::DFColumn)) -------------------------------------------------------------------
// local pass: the rows where the used slots of a group table (`first`, `sentinel` = unused) first appear, set in `mask`
// (laid out like the selection mask, zeroed by the caller)
int launch_unique_first_mask(const long long *first, long long cap, long long sentinel, const Geometry &g, uint32_t *mask, cudaStream_t stream);
// cross-shard merge over the rank-order concatenation of local results (unique: one column; group-by: the key tuple): keeps
// every position whose key tuple (isequal) does not occur at a lower position
struct MergeKey {
    int kind, elsize;             // fixed width: DFDB_* kind and bytes per value
    const uint8_t *values;        // fixed width: n * elsize bytes
    const uint8_t *missing;       // fixed width: 1 byte per position (1 = missing), may be null
    const int32_t *sizes;         // strings: n sizes (-1 = missing), null for fixed width
    const uint8_t *chars;
    const int64_t *char_off;      // strings: exclusive scan of max(size, 0)
    int64_t *kept_bytes;          // strings: per position, its char bytes when kept (scanned in place -> output char offsets)
    uint8_t *out_values, *out_missing;    // merge_emit: the kept positions' values in materialize's layout
    int32_t *out_sizes;
    uint8_t *out_chars;
};
struct MergeArgs {
    long long n;                  // positions
    int nkeys;
    MergeKey key[GROUP_MAX_KEYS];
    long long *rep;               // cap slots: lowest position with the slot's key, -1 = empty
    unsigned long long cap_mask;  // cap - 1 (cap: power of two >= 2n)
    long long *slot;              // per position: the slot of its key
};
int launch_merge_insert(const MergeArgs &a, cudaStream_t stream);
int launch_merge_keep(const MergeArgs &a, int64_t *keep, cudaStream_t stream);
int launch_str_lengths(const int32_t *sizes, long long n, int64_t *out, cudaStream_t stream);           // max(size, 0)
// kept positions to their output slots (keep_pos: exclusive scan of keep); first / out_first: group-by's first rows, else null
int launch_merge_emit(const MergeArgs &a, const int64_t *keep_pos, const long long *first, long long *out_first, cudaStream_t stream);
// group-by: folds the nvals aggregates of positions [lo, hi) -- one rank's part, whose keys are distinct -- into their merged
// group's slot of `out` (ngroups x nvals, zeroed), with dfdb_agg_fold_step.  A key that occurs twice in the part sets *dup.
// Launched once per rank in rank order; dfdb_agg_fold_finish over every slot last.
int launch_merge_fold(const MergeArgs &a, const int64_t *keep_pos, const dfdb_agg *in, int nvals, long long lo, long long hi, dfdb_agg *out, int *dup,
                      cudaStream_t stream);
int launch_merge_fold_finish(dfdb_agg *out, long long n, cudaStream_t stream);
// exclusive scan of n int64 in place, data[n] = total; tmp holds scan_i64_tmp_len(n) int64
long long scan_i64_tmp_len(long long n);
int launch_scan_i64(int64_t *data, long long n, int64_t *tmp, cudaStream_t stream);

// ---- order statistics (median / quantile): one MSD radix-select round over isless keys ----------------------------------
// key: the column's bits at its width W, mapped so that unsigned order is isless: unsigned / Bool as they are, signed with the
// sign bit flipped, floats XOR (sign ? all ones : sign bit).  A candidate whose prefix key >> hi_shift (0 when hi_shift == 64)
// is one of the open prefixes adds one to its digit (key >> (hi_shift - bits)) & (2^bits - 1) in that prefix's histogram.
constexpr int ORDER_MAX_BINS = 16384;     // nprefix << bits never exceeds this (shared-memory histogram)
struct OrderHistArgs {
    const uint8_t *values;                // gathered values (elsize bytes each) -- or null: candidates are `keys`
    const uint8_t *missing;               // 1 byte per value (1 = missing), may be null
    const unsigned long long *keys;       // compacted candidate keys
    long long n;                          // values or keys
    int kind, elsize;
    const unsigned long long *prefixes;   // nprefix open prefixes, ascending
    int nprefix, hi_shift, bits;
    unsigned long long *counts;           // nprefix << bits, zeroed by the caller
    unsigned long long *out_keys;         // non-null: the keys of every candidate of an open prefix are appended here (any order)
    unsigned long long *out_n;            // their count (zeroed by the caller)
};
int launch_order_hist(const OrderHistArgs &a, cudaStream_t stream);

// ---- K5/K6: stream compaction / gathers ---------------------------------------------------------------
struct GatherArgs {
    Geometry g;
    const uint32_t *mask;
    const int64_t *blk_base;      // exclusive scan of per-block selected counts
    ColView col;
    uint8_t *out_values;          // fixed width
    uint8_t *out_missing;         // 1 byte per row (nullable), may be null
    int32_t *out_sizes;           // strings
    uint8_t *out_chars;
    const int64_t *blk_char_base; // exclusive scan of per-block selected string bytes
    int64_t *out_indices;         // row numbers (1-based, table order) when non-null
};
int launch_gather_fixed(const GatherArgs &a, cudaStream_t stream);
int launch_gather_indices(const GatherArgs &a, cudaStream_t stream);
int launch_str_block_bytes(const GatherArgs &a, int64_t *blk_bytes, cudaStream_t stream);
int launch_gather_strings(const GatherArgs &a, cudaStream_t stream);

// computed projection columns: VM value per selected row
struct ProjVmArgs {
    Geometry g;
    ColView slot[MAX_SLOTS];
    const VmProgram *prog;
    const uint32_t *mask;
    const int64_t *blk_base;
    uint8_t *out_values;
    uint8_t *out_missing;
    int elsize;
    int *error_flag;
};
int launch_proj_vm(const ProjVmArgs &a, cudaStream_t stream);

// aggregates over a computed column (sum(t.a .* t.c), maximum(v.price .* 2) ...): VM value of every selected row folded
// into the per-unit partials of K7 (same units, same fixed combination order, same finalize kernel)
struct AggVmArgs {
    Geometry g;
    ColView slot[MAX_SLOTS];
    const VmProgram *prog;
    const uint32_t *mask;
    AggPartial *partials;
    int cls;                      // VC_* of the program's result
    int *error_flag;
};
int launch_agg_vm(const AggVmArgs &a, int sm_count, cudaStream_t stream);

}  // namespace dfdb
