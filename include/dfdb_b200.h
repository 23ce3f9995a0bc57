/*
 * dfdb_b200.h -- C ABI of libdfdb_b200.so: the B200-native column-scan path of DataFrameDBs.jl.
 *
 * The reference (pure Julia) has no FFI/plugin layer of its own; its only foreign call on this path is
 * liblz4 (src/io/BlockStreams.jl:39,42,110).  The seams this library replaces are the Julia generic
 * functions every consumer pulls from (SURVEY.md section 8b).  Each entry point cites the reference
 * interface it stands in for (paths relative to /root/reference); INTEGRATION.md shows the `ccall`
 * methods a maintainer adds on the Julia side, and dataframedbs.jl_b200/_capi.py is the ctypes
 * binding used by the Python mirror of the same API.
 *
 * Conventions: every function returns an int32 status (0 = ok); the message of the last failure on
 * the calling thread is available from dfdb_last_error().  Plain pointers and sizes only; the caller
 * owns every output buffer; the library owns device memory and the opaque handles.  One in-flight
 * call per handle.  All scans run on CUDA kernels for sm_100a -- there is no CPU fallback: without a
 * usable device every compute entry point returns DFDB_ERR_CUDA.
 */
#ifndef DFDB_B200_H
#define DFDB_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DFDB_API __attribute__((visibility("default")))

/* status codes; the Julia shim maps them to the exception the reference throws */
enum {
    DFDB_OK = 0,
    DFDB_ERR_IO = 1,          /* error("Table ... don't exists") creators.jl:8-9, filesystem.jl:58           */
    DFDB_ERR_FORMAT = 2,      /* check_column_head mismatch filesystem.jl:47-54, unknown typestring          */
    DFDB_ERR_CORRUPT = 3,     /* @assert size == sizes.origin "decompression error" BlockStreams.jl:112      */
    DFDB_ERR_ARGUMENT = 4,    /* ArgumentError: selection.jl:54, empty range selection.jl:73                 */
    DFDB_ERR_UNSUPPORTED = 5, /* expression outside the operator set -> shim raises ArgumentError            */
    DFDB_ERR_KEY = 6,         /* KeyError(column) table.jl:54                                                */
    DFDB_ERR_DIVIDE = 7,      /* DivideError from integer rem by zero inside a broadcast                     */
    DFDB_ERR_CUDA = 8,        /* CUDA runtime failure / no device                                            */
    DFDB_ERR_NOMEM = 9,
    DFDB_ERR_STATE = 10,      /* handle used in the wrong state (e.g. table not loaded)                      */
    DFDB_NEED_EXCHANGE = 11   /* not an error: a sharded scan needs survivor counts of the other shards first */
};

/* column element kinds (src/columntypes/base.jl:97-126,163-168 ; complex.jl) */
enum {
    DFDB_I8 = 1, DFDB_I16, DFDB_I32, DFDB_I64, DFDB_I128, DFDB_U8, DFDB_U16, DFDB_U32, DFDB_U64, DFDB_U128,
    DFDB_F16, DFDB_F32, DFDB_F64, DFDB_BOOL, DFDB_CHAR, DFDB_STRING, DFDB_DATE, DFDB_DATETIME, DFDB_TIME, DFDB_TUPLE
};

/* residency modes for dfdb_table_load */
enum {
    DFDB_LOAD_HOST = 0,     /* compressed blocks in pinned host memory; every scan copies them H2D ("transfer-inclusive") */
    DFDB_LOAD_HBM = 1,      /* compressed blocks resident in HBM; every scan decodes them ("HBM-resident")                */
    DFDB_LOAD_DECODED = 2   /* HBM-resident + decoded bodies cached in HBM after the first scan                          */
};

typedef struct dfdb_table dfdb_table;
typedef struct dfdb_scan dfdb_scan;

/* result of sum/count/min/max over the selected rows of one projected column.
 * Replaces the Base folds over Base.iterate(::DFColumn) (src/tables/column.jl:102-126). */
typedef struct dfdb_agg {
    int64_t count;       /* selected rows, missing included (length(col))                              */
    int64_t nmissing;    /* selected rows that are missing (sum(col) is `missing` when > 0)             */
    int64_t sum_i64;     /* wrapping two's-complement sum of integer / Bool values (Base.add_sum)       */
    double sum_f64;      /* floating sum: fixed-order tree, compensated final fold; hi part             */
    double sum_f64_lo;   /* low part of the compensated sum (hi + lo is the full-precision value)       */
    int64_t min_i64, max_i64;
    double min_f64, max_f64;   /* Julia semantics: NaN propagates, -0.0 < 0.0                           */
    int32_t has_nan;
    int32_t value_class; /* 1 signed int, 2 unsigned int, 3 float, 4 Bool, 0 = no non-missing values    */
} dfdb_agg;

/* caller-allocated output column for dfdb_scan_materialize (mirrors make_materialization +
 * append! in src/tables/materialization.jl:27-40; strings use the FlatStringsVector layout of
 * src/FlatStringsVectors.jl:5-9: Int32 sizes with -1 = missing, plus flat chars). */
typedef struct dfdb_outcol {
    void *values;        /* nrows * elsize bytes (fixed-width columns), else NULL                       */
    uint8_t *missing;    /* nrows bytes, 1 = missing (Union{T,Missing} columns), may be NULL            */
    int32_t *str_sizes;  /* nrows Int32 (String columns), else NULL                                     */
    uint8_t *str_chars;  /* string bytes, size from dfdb_scan_materialize_sizes                         */
} dfdb_outcol;

/* ---- runtime ------------------------------------------------------------------------------ */
DFDB_API int32_t dfdb_init(int32_t device);                 /* one process per GPU: selects the device, creates the stream */
DFDB_API int32_t dfdb_shutdown(void);
DFDB_API const char *dfdb_last_error(void);
DFDB_API int32_t dfdb_set_stream(void *cuda_stream);        /* run on the caller's cudaStream_t (NULL = library stream)     */
DFDB_API int32_t dfdb_synchronize(void);
DFDB_API int64_t dfdb_kernel_launches(void);                /* number of kernels this library has launched so far           */
DFDB_API int32_t dfdb_numa_node(void);                      /* NUMA node dfdb_init bound this process's host memory to (-1: none) */
DFDB_API int32_t dfdb_set_option(const char *name, int64_t value);
/* per-phase device timing (CUDA events on the scan stream): phases "h2d","decode","unpack","select","consume","d2h", and
 * "group_keys" (the key gather of dfdb_scan_groupreduce, part of its "consume" time too);
 * "k1_v1","k1_v3","k1_long","k1_bytes","k1_lane","k1_spec" report the decode launches and algorithmic bytes per K1 kernel (no time);
 * "k1_v1" is the sequential decoder (option "lz4_simple") */
DFDB_API int32_t dfdb_profile_enable(int32_t on);
DFDB_API int32_t dfdb_profile_reset(void);
DFDB_API int32_t dfdb_profile_get(const char *phase, double *total_ms, int64_t *launches, int64_t *bytes);

/* ---- table: open_table (src/tables/creators.jl:7-16), read_table_meta (src/io/table_io.jl:21-33),
 *      check_column_head (src/io/filesystem.jl:47-54); the block index replaces the header walk of
 *      skip_block (src/io/BlockStreams.jl:74-78) ------------------------------------------------ */
DFDB_API int32_t dfdb_table_open(const char *path, dfdb_table **out);
DFDB_API int32_t dfdb_table_close(dfdb_table *t);
DFDB_API int64_t dfdb_table_nrows(const dfdb_table *t);
DFDB_API int64_t dfdb_table_ncols(const dfdb_table *t);
DFDB_API int64_t dfdb_table_block_size(const dfdb_table *t);
DFDB_API int64_t dfdb_table_nblocks(const dfdb_table *t);
DFDB_API int32_t dfdb_table_column(const dfdb_table *t, int32_t index, int64_t *id, char *name, int32_t name_cap,
                                   char *typestring, int32_t ts_cap, int32_t *kind, int32_t *nullable, int32_t *elsize);
DFDB_API int32_t dfdb_table_column_stats(const dfdb_table *t, int64_t col_id, int64_t *compressed, int64_t *uncompressed);
/* loaded column: how many of the shard's blocks are stored (incompressible: one LZ4 literal run, what
 * LZ4_compress_fast emits when nothing matches, src/io/BlockStreams.jl:42-48) and are therefore referenced in
 * place inside the compressed buffer instead of being copied by the decoder; bytes = their body bytes */
DFDB_API int32_t dfdb_table_column_stored(const dfdb_table *t, int64_t col_id, int64_t *blocks, int64_t *bytes);
/* block-range shard of this process: blocks [nblocks*rank/world, nblocks*(rank+1)/world) of every column */
DFDB_API int32_t dfdb_table_set_shard(dfdb_table *t, int32_t rank, int32_t world);
DFDB_API int32_t dfdb_table_shard_range(const dfdb_table *t, int64_t *block_lo, int64_t *block_hi, int64_t *row_lo, int64_t *row_hi);
/* read the shard's compressed blocks of the given columns (all columns when n == 0) */
DFDB_API int32_t dfdb_table_load(dfdb_table *t, const int64_t *col_ids, int32_t n, int32_t mode);
DFDB_API int32_t dfdb_table_drop_decoded(dfdb_table *t);    /* forget cached decoded bodies (mode DFDB_LOAD_DECODED) */

/* ---- block index + zone maps (SURVEY.md section 8f; no reference counterpart: the format has no index -- skip_block walks
 *      the headers, src/io/BlockStreams.jl:74-78 -- and no per-block statistics).  dfdb_table_build_zonemaps decodes the columns
 *      on the device, reduces every block to (min, max, null count) of its non-missing values and writes the optional sidecar
 *      <table>/<id>.zmap beside the untouched column file, together with the block index {file offset, rows, origin,
 *      compressed}.  dfdb_table_open uses a sidecar whose recorded size / mtime still match the column file: the index
 *      replaces the header walk, and predicate stages made of `column <cmp> constant` terms skip (never copy, never decode)
 *      every block whose range rules the predicate out.  Unsharded tables only; fixed-width numeric columns. ------------- */
typedef struct dfdb_zone {
    int64_t rows, null_count;
    int64_t min_i64, max_i64;     /* integer / Bool / Date columns (unsigned columns: the same bits)                 */
    double min_f64, max_f64;      /* Float32 / Float64 columns, NaN excluded                                          */
    int32_t has_value, has_nan;
} dfdb_zone;
DFDB_API int32_t dfdb_table_build_zonemaps(dfdb_table *t, const int64_t *col_ids, int32_t n);   /* n == 0: every eligible column */
DFDB_API int32_t dfdb_table_zonemap(const dfdb_table *t, int64_t col_id, int64_t block, dfdb_zone *out);   /* DFDB_ERR_STATE without a zone map */
/* blocks the zone maps ruled out in the scan's last run, and blocks of the shard */
DFDB_API int32_t dfdb_scan_pruned(const dfdb_scan *s, int64_t *pruned, int64_t *blocks);

/* ---- scan: BlocksIterator(v::DFView) (src/io/blocksiterator.jl:20-66) built from the view's
 *      SelectionQueue (src/tables/selection.jl:4-10) and Projection (src/tables/projection.jl:1-9);
 *      plan wire format in dataframedbs.jl_b200/plan.py ----------------------------------------- */
DFDB_API int32_t dfdb_scan_prepare(dfdb_table *t, const uint8_t *plan, int64_t plan_len, dfdb_scan **out);
DFDB_API int32_t dfdb_scan_free(dfdb_scan *s);
DFDB_API int32_t dfdb_scan_nproj(const dfdb_scan *s);
DFDB_API int32_t dfdb_scan_proj_type(const dfdb_scan *s, int32_t proj_idx, int32_t *kind, int32_t *nullable, int32_t *elsize);
/* nrow(v): src/tables/view.jl:192-206 (BlockRowsIterator blocksiterator.jl:123-145) */
DFDB_API int32_t dfdb_scan_count(dfdb_scan *s, int64_t *n);
/* sum/minimum/maximum/mean/count over a DFColumn: src/tables/column.jl:102-126 */
DFDB_API int32_t dfdb_scan_aggregate(dfdb_scan *s, int32_t proj_idx, dfdb_agg *out);
/* parity hooks: apply(::SelectionExecutor, rows, block) src/tables/selection.jl:161-167 --
 * global bitmask (bit r&63 of word r>>6 set <=> 0-based table row r selected) and 1-based row numbers */
DFDB_API int32_t dfdb_scan_mask(dfdb_scan *s, uint64_t *words, int64_t nwords);
DFDB_API int32_t dfdb_scan_indices(dfdb_scan *s, int64_t *idx, int64_t cap, int64_t *n);
/* materialize(v::DFView) src/tables/materialization.jl:27-40: sizes first (pass 1 = nrow), then fill */
DFDB_API int32_t dfdb_scan_materialize_sizes(dfdb_scan *s, int64_t *nrows, int64_t *str_bytes_per_col);
DFDB_API int32_t dfdb_scan_materialize(dfdb_scan *s, dfdb_outcol *cols, int32_t ncols);

/* ---- group-by reduce (SURVEY.md section 8f rank 4): finishes what the reference stubs in src/tables/aggregate.jl:1-36
 *      (groupreduce(view, by; cols...): a RobinDict from the tuple of key values to a group number in order of first
 *      appearance, "Future plans" docs/src/index.md:597).  Hash aggregation on the device over the selected rows: keys = 1..2
 *      projected stored columns (every type unique takes except Float16 and Char; missing is a key value of its own,
 *      equality is isequal: one NaN, -0.0 and 0.0 differ, strings by bytes and "" is not missing), values = up to 4 projected
 *      numeric columns, each reduced to a dfdb_agg (count / nmissing / sum / min / max) per group.  Counts, integer sums,
 *      minima and maxima are exact; Float64 sums are accumulated in arrival order (reproducible to rounding).
 *      dfdb_scan_groupreduce runs the shard-local pass and returns the number of groups (first rows stay 1-based TABLE rows
 *      on a shard).  The result lives on the handle until the next group-by call on it or dfdb_scan_free; a later
 *      materialize on the same handle is unaffected:
 *      dfdb_scan_group_results copies out, in order of first appearance, the row where each group first appears and
 *      ngroups x nvals aggregates (row-major);
 *      dfdb_scan_group_key_bytes gives the char bytes of each String key column (0 for fixed width) and dfdb_scan_group_keys
 *      copies the key values out, one row per group, in the layout of dfdb_scan_materialize (fixed width = values +
 *      (nullable) one missing byte per value; String = Int32 sizes (-1 = missing) + chars; result-arena buffers take the
 *      queued pinned copy).  Both return DFDB_ERR_STATE before any group-by call on the handle;
 *      dfdb_scan_groupreduce_merge combines per-rank results carried by the host on the device; the merged result
 *      replaces the handle's.  Part r (in rank order) holds part_n[r] groups: keys[r * nkeys + k] is its key column k
 *      (part_str_bytes[r * nkeys + k] chars for a String key, may be NULL without one), and its first rows and its
 *      part_n[r] x nvals aggregates follow those of part r - 1 in `first_rows` and `aggs`.  The key types are those of the
 *      handle's projections key_proj; the handle need not have run a scan.  A group is kept where its key tuple first
 *      occurs, and its aggregates are the parts' folded in rank order with dfdb_agg_fold's arithmetic (the same bits on
 *      every rank, final renormalisation included).  A part that holds one key tuple twice is DFDB_ERR_ARGUMENT;
 *      dfdb_scan_groupreduce_all is the local pass on every rank followed by the merge over the library's communicator
 *      (ncclAllGather of each payload array between device buffers, each rank's status travelling with its sizes): every
 *      rank ends with the same result.  Unsharded without a communicator it is dfdb_scan_groupreduce. ------------------- */
DFDB_API int32_t dfdb_scan_groupreduce(dfdb_scan *s, const int32_t *key_proj, int32_t nkeys, const int32_t *val_proj, int32_t nvals,
                                       int64_t *ngroups);
DFDB_API int32_t dfdb_scan_group_results(dfdb_scan *s, int64_t *first_rows, dfdb_agg *aggs);
DFDB_API int32_t dfdb_scan_group_key_bytes(dfdb_scan *s, int64_t *str_bytes_per_key);
DFDB_API int32_t dfdb_scan_group_keys(dfdb_scan *s, dfdb_outcol *keys, int32_t nkeys);
DFDB_API int32_t dfdb_scan_groupreduce_merge(dfdb_scan *s, const int32_t *key_proj, int32_t nkeys, int32_t nvals, const dfdb_outcol *keys,
                                             const int64_t *first_rows, const dfdb_agg *aggs, const int64_t *part_n, const int64_t *part_str_bytes,
                                             int32_t nparts, int64_t *ngroups);
DFDB_API int32_t dfdb_scan_groupreduce_all(dfdb_scan *s, const int32_t *key_proj, int32_t nkeys, const int32_t *val_proj, int32_t nvals,
                                           int64_t *ngroups);

/* ---- multi-GPU: one process per GPU; each rank scans its shard, the tiny partials are exchanged by
 *      the host (NCCL all-gather) and folded in rank order on every rank ------------------------- */
DFDB_API int32_t dfdb_agg_fold(const dfdb_agg *partials, int32_t n, dfdb_agg *out);
/* Range / index-vector stages that follow a predicate select on the rank among ALL survivors
 * (RangeToProcess.offset runs across blocks, src/tables/selection.jl:94-111), so a shard has to know how many
 * rows of the preceding shards survived up to that stage.  Protocol on a sharded table, for every such stage in
 * turn: every rank calls dfdb_scan_exchange_count -- it runs the selection up to the first stage whose offset is
 * still unknown and returns this shard's survivor count there (*pending = 1), or *pending = 0 when nothing is
 * missing; the host all-gathers the counts (NCCL / gloo) and hands each rank the sum over lower ranks with
 * dfdb_scan_exchange_offset.  Any scan entry point called before the offsets are complete returns
 * DFDB_NEED_EXCHANGE. */
DFDB_API int32_t dfdb_scan_exchange_count(dfdb_scan *s, int64_t *local_survivors, int32_t *pending);
DFDB_API int32_t dfdb_scan_exchange_offset(dfdb_scan *s, int64_t survivors_in_lower_ranks);
/* device-resident copy of the last dfdb_scan_aggregate result (sizeof(dfdb_agg) bytes), for NCCL */
DFDB_API int32_t dfdb_scan_aggregate_device(dfdb_scan *s, int32_t proj_idx, void *device_out);

/* ---- multi-GPU inside the library: one process per GPU, NCCL over NVLink / NVSwitch.  The library opens libnccl.so.2 at
 *      dfdb_comm_init (no NCCL dependency until then).  Rank 0 creates the 128-byte id with dfdb_comm_unique_id, the host
 *      distributes it by whatever means it has (MPI, a file, torch.distributed), every rank calls dfdb_comm_init on the device
 *      it gave dfdb_init.  No reference counterpart: the reference is a single process. ---------------------------------- */
#define DFDB_COMM_ID_BYTES 128
DFDB_API int32_t dfdb_comm_unique_id(uint8_t *id);                                   /* ncclGetUniqueId                    */
DFDB_API int32_t dfdb_comm_init(int32_t rank, int32_t world, const uint8_t *id);     /* ncclCommInitRank                   */
DFDB_API int32_t dfdb_comm_destroy(void);
DFDB_API int32_t dfdb_comm_info(int32_t *rank, int32_t *world);                      /* world = 0: no communicator          */
/* Reductions over a block-range sharded table (Base folds over iterate(::DFColumn), src/tables/column.jl:102-126): every rank
 * aggregates its shard, the 88-byte partials are all-gathered with ncclAllGather on the scan stream and folded in rank order
 * (dfdb_agg_fold) -- every rank returns the same bits.  Survivor-count exchanges that the plan needs (range stage behind a
 * predicate, see dfdb_scan_exchange_count) are resolved over the same communicator first. */
DFDB_API int32_t dfdb_scan_aggregate_all(dfdb_scan *s, int32_t proj_idx, dfdb_agg *out);
/* nrow(v) over all shards (src/tables/view.jl:192-206): all-gather of the per-shard counts */
DFDB_API int32_t dfdb_scan_count_all(dfdb_scan *s, int64_t *n);
/* resolves every pending survivor-count exchange of the scan over the communicator (dfdb_scan_exchange_count / _offset) */
DFDB_API int32_t dfdb_scan_resolve_exchange(dfdb_scan *s);
/* materialize over all shards: *row_offset = selected rows of the lower-ranked shards, *total = selected rows of the whole
 * table; this rank's rows go to [row_offset, row_offset + local) of the result (dfdb_scan_materialize fills the local part) */
DFDB_API int32_t dfdb_scan_row_offset_all(dfdb_scan *s, int64_t *local, int64_t *row_offset, int64_t *total);

/* ---- unique(col) (Base.unique over iterate(::DFColumn), src/tables/column.jl:102-126): the distinct values of one projected
 *      stored column over the selected rows, in order of first appearance.  Equality is isequal: missing is one value, every
 *      NaN is one value (the first NaN row's bits are returned), -0.0 and 0.0 differ, strings compare by bytes and "" is not
 *      missing.  Every stored type except Int128 / UInt128 / Tuple; a computed projection is DFDB_ERR_UNSUPPORTED.  The result
 *      lives on the scan handle (device memory) until the next unique call on it or dfdb_scan_free; a later materialize on
 *      the same handle is unaffected.  Layout of dfdb_scan_materialize: fixed width = values + (nullable) one missing byte per
 *      value; String = Int32 sizes (-1 = missing) + chars.  Sizes first, then the copy:
 *      dfdb_scan_unique runs the shard-local pass and returns the count and the char bytes (0 for fixed width);
 *      dfdb_scan_unique_values copies the handle's result into caller buffers (result-arena buffers take the queued pinned copy);
 *      dfdb_scan_unique_merge combines per-rank results carried by the host (parts[r] holds part_n[r] values -- and
 *      part_str_bytes[r] chars -- of rank r, in rank order) on the device; the merged result replaces the handle's.  The
 *      parts have the column type of the handle's last dfdb_scan_unique, or of projection 0 before any;
 *      dfdb_scan_unique_all is the local pass on every rank followed by the merge over the library's communicator
 *      (ncclAllGather of each payload array between device buffers); every rank ends with the same result.  Unsharded
 *      without a communicator it is dfdb_scan_unique. -------------------------------------------------------------------- */
DFDB_API int32_t dfdb_scan_unique(dfdb_scan *s, int32_t proj_idx, int64_t *n, int64_t *str_bytes);
DFDB_API int32_t dfdb_scan_unique_values(dfdb_scan *s, dfdb_outcol *out);
DFDB_API int32_t dfdb_scan_unique_merge(dfdb_scan *s, const dfdb_outcol *parts, const int64_t *part_n, const int64_t *part_str_bytes, int32_t nparts,
                                        int64_t *n, int64_t *str_bytes);
DFDB_API int32_t dfdb_scan_unique_all(dfdb_scan *s, int32_t proj_idx, int64_t *n, int64_t *str_bytes);

/* ---- result buffers.  materialize(::DFView) allocates its result vectors (`sizehint!` + `append!`,
 *      src/tables/materialization.jl:1-25,29-37); a caller that takes them from here gets page-locked memory, which
 *      dfdb_scan_materialize recognises and fills with one device-to-host copy at full PCIe rate (ordinary pageable
 *      buffers work too, through pinned bounce buffers, at a fraction of that).  Freed buffers are kept for reuse
 *      (option "host_arena_cap_mb", default 24576).  The Julia shim wraps the pointer with unsafe_wrap(Array, ...; own =
 *      false) and a finalizer that calls dfdb_host_free. --------------------------------------------------------- */
DFDB_API int32_t dfdb_host_alloc(int64_t bytes, void **ptr);
DFDB_API int32_t dfdb_host_free(void *ptr);

/* ---- write path (SURVEY.md section 8f rank 2): LZ4 block compression and block framing on the device.
 *      dfdb_write_column_file = make_column_file (src/io/filesystem.jl:22-31) + write_column (src/io/columns.jl:65-84,
 *      one commit_block_write! per block, src/io/BlockStreams.jl:36-60): <table>/<id>.bin = Int64 block_size | typestring |
 *      { Int32 rows | Int64 origin | Int64 compressed | one raw LZ4 block }*, the body of every block laid out as
 *      src/io/blocks.jl:2-33 writes it (bits T; Union{T,Missing}: BitArray chunks + values; String: Int32 datasize | Int32
 *      sizes, -1 = missing | chars).  The bodies are assembled and compressed on the device (lz4_compress.cu), the host only
 *      frames them.  HOST input buffers: `values` nrows * elsize bytes (fixed width), `missing` nrows bytes (1 = missing,
 *      nullable types, else NULL), `str_sizes` / `str_chars` for String columns.  The file must not exist.  The compressed
 *      bytes are not liblz4's (never compared, SURVEY.md 8c); any LZ4_decompress_safe decodes them to the same body.
 *      dfdb_write_table_meta = write_table_meta (src/io/table_io.jl:9-19): creates the directory when needed. ----------- */
DFDB_API int32_t dfdb_write_column_file(const char *table_path, int64_t col_id, const char *typestring, int64_t block_size, int64_t nrows,
                                        const void *values, const uint8_t *missing, const int32_t *str_sizes, const uint8_t *str_chars,
                                        int64_t nchars, int64_t *compressed_total, int64_t *uncompressed_total);
DFDB_API int32_t dfdb_write_table_meta(const char *table_path, int64_t block_size, int32_t ncols, const int64_t *ids,
                                       const char *const *names, const char *const *typestrings);
/* codec hook of the write path: LZ4_compress_fast (src/io/BlockStreams.jl:42-48) for n independent HOST bodies; out slots
 * must hold LZ4_compressBound(len) = len + len / 255 + 16 bytes; comp_len[i] = compressed size */
DFDB_API int32_t dfdb_lz4_compress_blocks(const uint8_t *bodies, const int64_t *body_off, const int64_t *body_len, int32_t n,
                                          uint8_t *out, const int64_t *out_off, int64_t *comp_len);

/* ---- codec hook: read_block (src/io/BlockStreams.jl:101-119) for n independent raw LZ4 blocks.
 *      comp/out are HOST buffers; status[i] = 0 or DFDB_ERR_CORRUPT ------------------------------ */
DFDB_API int32_t dfdb_lz4_decode_blocks(const uint8_t *comp, const int64_t *comp_off, const int64_t *comp_len,
                                        uint8_t *out, const int64_t *out_off, const int64_t *origin, int32_t n,
                                        int32_t *status);

/* which K1 decoder dfdb_table_load would pick for a column whose blocks look like this raw LZ4 block (host memory, no device needed;
 * the choice at load is a vote of the first, middle and last block): 1 = walker / consumer, 2 = verified word runs, 3 = long
 * sequences, 4 = match-only byte streams, -1 = too short to tell, -2 = bad arguments (dfdb_last_error says which) */
DFDB_API int32_t dfdb_lz4_classify_block(const uint8_t *comp, int64_t comp_len, int64_t origin);

#ifdef __cplusplus
}
#endif
#endif /* DFDB_B200_H */
