// internal.hpp -- shared declarations of libdfdb_b200 (host structures + kernel argument PODs).
#pragma once
#include <cstdint>
#include <cstdio>
#include <cstring>
#include <string>
#include <vector>

#include "../../include/dfdb_b200.h"

namespace dfdb {

// ------------------------------------------------------------------------------------------------
// errors
int fail(int code, const char *fmt, ...) __attribute__((format(printf, 2, 3)));
const char *last_error();

// ------------------------------------------------------------------------------------------------
// column types (src/columntypes/base.jl, complex.jl)
struct ColType {
    int kind = 0;
    bool nullable = false;
    int elsize = 0;   // bytes per element in the block body; 0 for String
    int align = 1;
};
int parse_typestring(const char *s, size_t n, ColType *out);

// value classes used by the kernels
enum { VC_NONE = 0, VC_INT = 1, VC_UINT = 2, VC_FLT = 3, VC_BOOL = 4, VC_STR = 5 };
int value_class(int kind);

// ------------------------------------------------------------------------------------------------
// table
struct BlockInfo {
    int64_t file_off;     // offset of the compressed payload in <id>.bin
    int32_t rows;
    int64_t origin;       // uncompressed body bytes
    int64_t compressed;
};

// zone map of one column block (sidecar <id>.zmap): range of the non-missing values as 64-bit payloads of the column's
// value class (signed / unsigned integer bits, or double bits with NaN kept out of the range and flagged)
struct ZoneEntry {
    uint64_t min_bits = 0, max_bits = 0;
    int64_t null_count = 0;
    int32_t flags = 0;        // 1 = has a non-missing, non-NaN value, 2 = has NaN
};

struct Column {
    int64_t id = 0;
    std::string name, typestr;
    ColType type;
    int64_t data_start = 0;
    std::vector<BlockInfo> blocks;
    int64_t total_compressed = 0, total_origin = 0;
    std::vector<ZoneEntry> zones;    // per table block, empty = no (valid) sidecar
    bool index_from_sidecar = false; // the block index came from the sidecar instead of the header walk

    // ---- residency of the current shard (blocks [blk_lo, blk_hi) of the table) ----
    bool loaded = false;
    int mode = 0;
    uint8_t *h_comp = nullptr;       // pinned host copy of the compressed payloads (DFDB_LOAD_HOST keeps it)
    uint8_t *d_comp = nullptr;       // device copy / H2D staging target
    size_t comp_bytes = 0;           // size of the packed compressed buffer
    uint8_t *d_decoded = nullptr;    // decoded bodies, one 256B-aligned slot per block
    size_t decoded_bytes = 0;
    bool decoded_valid = false;
    int dec_lo = 0, dec_hi = 0;      // local block range whose decoded bodies are current (decoded_valid: all of them)
    uint64_t dec_live_gen = 0;       // generation of the survivor counts (dfdb_scan::live_gen) whose live blocks are the ones decoded (skip_cols); 0 = none
    // per local block device arrays
    int64_t *d_comp_off = nullptr;   // offset of payload in (h|d)_comp
    int32_t *d_comp_len = nullptr;
    int64_t *d_dec_off = nullptr;    // offset of body slot in d_decoded
    int32_t *d_origin = nullptr;
    int32_t *d_status = nullptr;     // decode status per block
    uint8_t *d_skip = nullptr;       // 1 = stored block (one literal run): its body is referenced in place inside d_comp
    std::vector<uint8_t> h_skip;
    std::vector<int32_t> h_corrupt;  // per local block: LZ4_decompress_safe's verdict (0 = accepted), decided once at load by the lane-per-block decoder
    int64_t stored_blocks = 0;
    int lz4_general = 1;             // K1 flavour, decided at load from a token sample: 1 = walker / consumer decoder (v3),
                                     // 2 = warp per block with verified runs (spec: nearly every sequence is one aligned word),
                                     // 3 = warp per block, one sequence at a time through a stream window (long sequences),
                                     // 4 = warp per block, bare-match byte streams
    int32_t *d_str_off = nullptr;    // String columns: per-row char offset inside the block's char area
    bool str_off_valid = false;
    std::vector<int64_t> h_dec_off, h_comp_off;
};

}  // namespace dfdb

struct dfdb_table {
    std::string path;
    int64_t format_version = 0, block_size = 0;
    std::vector<dfdb::Column> cols;
    int64_t nrows = 0, nblocks = 0;
    int32_t rank = 0, world = 1;
    uint64_t epoch = 1;                // bumped whenever the shard changes: masks and counts of older epochs are stale
    int64_t blk_lo = 0, blk_hi = 0;    // shard
    dfdb::Column *find(int64_t id)
    {
        for (auto &c : cols) if (c.id == id) return &c;
        return nullptr;
    }
};

namespace dfdb {

int table_open_host(const char *path, dfdb_table **out);   // format.cpp
// runtime of api.cu for the other translation units that launch kernels (write_path.cu)
struct RuntimeView { void *stream; unsigned int *counter; int sm_count; bool inited; };
RuntimeView runtime_view();
void runtime_count_launch();
int zonemap_write(const dfdb_table *t, const Column &c);    // format.cpp: <table>/<id>.zmap from c.blocks + c.zones

// ------------------------------------------------------------------------------------------------
// plan (host): parsed + typed expression programs
enum { ST_RANGE = 1, ST_INDEXVEC = 2, ST_PRED = 3 };
enum { PJ_COL = 1, PJ_EXPR = 2 };

// wire opcodes (dataframedbs.jl_b200/plan.py)
enum {
    W_COL = 0x01, W_I64 = 0x02, W_F64 = 0x03, W_STR = 0x04, W_BOOL = 0x05,
    W_EQ = 0x10, W_NE, W_LT, W_LE, W_GT, W_GE,
    W_AND = 0x20, W_OR, W_XOR, W_NOT,
    W_ADD = 0x30, W_SUB, W_MUL, W_DIV, W_REM, W_NEG,
    W_ISMISSING = 0x40, W_COALESCE,
    W_STARTSWITH = 0x50, W_ENDSWITH,
    W_IN = 0x60
};

// ---- device VM (typed, tag-free): every stack entry is a 64-bit payload + missing bit ----
enum {
    V_LOAD = 1,      // a = slot
    V_CONST = 2,     // imm = index into consts (payload bits)
    V_CONSTSTR = 3,  // imm = offset in string pool, a|b<<8 = length  (payload = pool ref)
    V_CMP = 4,       // a = code (0 EQ,1 NE,2 LT,3 LE,4 GT,5 GE), b = class pair
    V_AND = 5, V_OR = 6, V_XOR = 7, V_NOT = 8,
    V_ARITH = 9,     // a = code (0 ADD,1 SUB,2 MUL,3 DIV,4 REM,5 NEG), b = operand classes (lo nibble lhs, hi nibble rhs), c = result: bits | (uns<<7) for ints, 32/64 for floats
    V_ISMISSING = 10,
    V_COALESCE = 11,
    V_STRCMP = 12,   // a = code ; both operands strings
    V_STARTSWITH = 13, V_ENDSWITH = 14,
    V_IN = 15,       // imm = first const index, a|b<<8 = count, c = uns flag of the value
    V_STRNUM = 16    // String ==/!= non-String: a = code; constant result with missing propagation
};
// class pairs for V_CMP (lhs,rhs): I = signed int (Bool included), U = unsigned, F = double
enum { CP_II = 0, CP_UU, CP_IU, CP_UI, CP_IF, CP_UF, CP_FI, CP_FU, CP_FF };

struct VmInstr { uint8_t op, a, b, c; int32_t imm; };

constexpr int VM_MAX_INSTR = 96;
constexpr int VM_MAX_CONST = 64;
constexpr int VM_STRPOOL = 512;
constexpr int VM_MAX_STACK = 12;
constexpr int MAX_SLOTS = 8;

struct VmProgram {
    int32_t ninstr;
    int32_t result_class;    // VC_*
    int32_t result_nullable;
    int32_t result_bits;     // ints: 8..64 ; floats 32/64
    int32_t result_uns;
    VmInstr instr[VM_MAX_INSTR];
    int64_t consts[VM_MAX_CONST];
    uint8_t strpool[VM_STRPOOL];
};

// fast path: conjunction of (column cmp constant) terms over fixed-width numeric columns
struct Term {
    int32_t slot;
    int32_t cls;        // VC_INT / VC_UINT / VC_FLT
    int32_t code;       // 0 EQ,1 NE,2 LT,3 LE,4 GT,5 GE
    int32_t constant_result;  // -1 = evaluate, 0/1 = term folded to a constant
    int64_t ci;
    double cf;
};
constexpr int MAX_TERMS = 6;

struct Expr {
    std::vector<uint8_t> wire;     // raw postfix bytes (for error messages)
    std::vector<int64_t> col_ids;  // distinct referenced columns, first-use order
    VmProgram prog;                // slots refer to Scan::slots
    bool simple = false;           // matches the fast path
    int nterms = 0;
    Term terms[MAX_TERMS];
};

struct Stage {
    int kind = 0;
    int64_t start = 0, step = 1, stop = 0;   // RANGE
    std::vector<int64_t> idx;                // INDEXVEC, sorted unique
    int64_t first = 0, last = 0;
    Expr e;
    int64_t *d_idx = nullptr;
};

struct Proj {
    int kind = 0;
    int64_t col = 0;
    Expr e;
    ColType type;       // result type
};

// device-visible description of one decoded column of the shard
struct ColView {
    const uint8_t *base;      // decoded bodies
    const int64_t *blk_off;   // per local block: byte offset of the body
    const int32_t *str_off;   // String: per (local block * block_size + row) char offset in the block's char area
    int32_t kind, elsize, nullable, cls;
};

constexpr int GROUP_MAX_KEYS = 2;     // group-by: key columns
constexpr int GROUP_MAX_VALS = 4;     // ... and value columns

// one result column in device memory, in materialize's layout: the result of dfdb_scan_unique / _all / _merge until the next of
// those calls or dfdb_scan_free, and each key column of a group-by result until the next group-by call or dfdb_scan_free
struct UniqueResult {
    int32_t kind = 0, elsize = 0, nullable = 0;   // column type; kind 0 = no result yet
    int64_t n = 0, bytes = 0;                     // distinct values, char bytes (String)
    uint8_t *d_values = nullptr, *d_missing = nullptr, *d_chars = nullptr;
    int32_t *d_sizes = nullptr;
};

}  // namespace dfdb

struct dfdb_scan {
    dfdb_table *tbl = nullptr;
    std::vector<dfdb::Stage> stages;
    std::vector<dfdb::Proj> projs;
    std::vector<int64_t> slots;        // column ids referenced anywhere, slot index = position
    // device scratch owned by the scan
    uint32_t *d_mask = nullptr;        // selection bitmask, wpb words per local block
    int64_t mask_words = 0;
    int64_t *d_blk_counts = nullptr;   // per local block selected-row counts (+1 total)
    int64_t *d_blk_base = nullptr;     // exclusive scan of the above (+1)
    int64_t *d_blk_bytes = nullptr;    // string gather: bytes per block / bases
    void *d_partials = nullptr;        // aggregate partials per unit
    size_t partials_cap = 0;
    void *d_result = nullptr;          // final dfdb_agg (+ scalars) on device
    void *h_result = nullptr;          // pinned host mirror
    bool mask_valid = false;
    uint64_t mask_epoch = 0;           // table epoch the mask was computed in
    uint64_t live_gen = 0;             // generation of blk_live (a new one every time the survivor counts are recomputed)
    int64_t selected = -1;
    std::vector<int64_t> str_bytes;    // per projection
    std::vector<int64_t> blk_live;     // selected rows per local block (host copy of the counts behind d_blk_base), valid with `selected`
    // sharded tables: survivors of lower-ranked shards entering each range stage that follows a predicate
    std::vector<uint8_t> zone_dead;    // per local block: 1 = the zone maps rule out every row for some predicate stage (never decoded)
    uint8_t *d_zone_dead = nullptr;
    int64_t zone_pruned = 0;           // blocks ruled out by the zone maps in the last run
    std::vector<int64_t> group_first;  // group-by: 1-based table row of each group's first appearance, ascending
    std::vector<dfdb_agg> group_aggs;  // ngroups x nvals
    int32_t group_nkeys = 0;           // key columns of the last group-by result, 0 = none yet
    dfdb::UniqueResult group_keys[dfdb::GROUP_MAX_KEYS];   // its key values, one row per group, in group order
    dfdb::UniqueResult uniq;           // unique: distinct values of one column in order of first appearance
    std::vector<int64_t> rank_offsets;
    int64_t exchange_count = -1;       // this shard's count at the first stage whose offset is missing
};

namespace dfdb {
int plan_parse(dfdb_table *t, const uint8_t *bytes, int64_t len, dfdb_scan *s);   // plan.cpp
}
