// api.cu -- C ABI of libdfdb_b200 (include/dfdb_b200.h): runtime, table residency, scan orchestration.
//
// Scan driver: stands in for BlocksIterator{DataReader|SizeReader} (/root/reference/src/io/blocksiterator.jl:
// 20-145).  Where the reference walks one block at a time (read selection columns -> apply -> read
// projection columns -> project), this driver decodes every needed column block of the shard with one
// K1 launch and then runs each selection stage / consumer as one kernel over all blocks.
#include <cuda_runtime.h>
#include <dlfcn.h>
#include <fcntl.h>
#include <sys/syscall.h>
#include <unistd.h>

#include <algorithm>
#include <atomic>
#include <functional>
#include <cmath>
#include <map>
#include <mutex>
#include <optional>
#include <string>
#include <vector>

#include "kernels.cuh"

using namespace dfdb;

namespace {

struct PhaseRec { int phase; cudaEvent_t a, b; int64_t launches, bytes; };
const char *k_phases[] = {"h2d", "decode", "unpack", "select", "consume", "d2h", "group_keys", "order"};
enum { PH_H2D = 0, PH_DECODE, PH_UNPACK, PH_SELECT, PH_CONSUME, PH_D2H, PH_GROUP_KEYS, PH_ORDER, PH_COUNT };

struct Runtime {
    bool inited = false;
    int device = 0;
    int sm_count = 148;
    int numa_node = -1;       // node this process's memory policy prefers (the GPU's), -1 = untouched
    cudaStream_t own_stream = nullptr, stream = nullptr, copy_stream = nullptr;
    cudaStream_t decode_stream = nullptr, decode_stream2 = nullptr;   // above the scan stream's priority: the full rounds and the last round of a
                                                                      // decode that the scan of the earlier rounds runs beside (ensure_decoded)
    unsigned int *d_counter = nullptr;
    int *d_error = nullptr;
    uint64_t next_gen = 1;    // generation of the next survivor counts (select_rows)
    std::atomic<int64_t> launches{0};
    // options
    int64_t lz4_simple = 0;   // every column through K1::Sequential, one sequence at a time (baseline; forced_decoder)
    int64_t no_wide = 0;
    int64_t no_fused = 0;
    int64_t no_tma = 0;
    int64_t pred_bits = 0;      // an aggregate's predicate bits from the decoder: 0 = when the decode is large enough (ensure_decoded), 1 = always, 2 = never (A/B)
    std::optional<K1> lz4_flavour;   // the decoder option lz4_flavour forces on every column (set_lz4_flavour); none = each column's own
    int64_t no_overlap = 0;   // do not run the scan of the decoded part of a shard beside the decode of its last part
    int64_t no_alias = 0;     // copy stored (incompressible) blocks like any other block instead of referencing them in place
    int64_t no_zonemap = 0;   // ignore zone maps (A/B: results must not change)
    int64_t lane_hot = -1;    // K1::Lane: -1 = hot-step schedule for the columns that sampled as K1::Spec, 0 / 1 = force off / on (A/B, tests)
    // profiling
    bool profiling = false;
    std::vector<PhaseRec> recs;
    double acc_ms[PH_COUNT] = {0};
    int64_t acc_launches[PH_COUNT] = {0}, acc_bytes[PH_COUNT] = {0};
    int64_t k1_launches[K1_COUNT] = {0}, k1_bytes[K1_COUNT] = {0};   // decode launches / algorithmic bytes per K1 decoder, indexed by K1 (dfdb_profile_get)
} rt;

#define CUDA_TRY(expr)                                                                                         \
    do {                                                                                                       \
        cudaError_t _e = (expr);                                                                               \
        if (_e != cudaSuccess) return fail(DFDB_ERR_CUDA, "%s failed: %s", #expr, cudaGetErrorString(_e));     \
    } while (0)

#define LAUNCH(expr)                                                                                           \
    do {                                                                                                       \
        if ((expr) != 0) return fail(DFDB_ERR_CUDA, "kernel launch failed: %s (%s)", #expr, cudaGetErrorString(cudaGetLastError())); \
        rt.launches++;                                                                                         \
    } while (0)

int need_init()
{
    if (!rt.inited) return fail(DFDB_ERR_CUDA, "dfdb_init has not been called (or no CUDA device is usable)");
    return DFDB_OK;
}

struct PhaseScope {
    int idx = -1;
    int64_t l0 = 0;
    cudaStream_t st;
    PhaseScope(int phase, int64_t bytes, cudaStream_t stream = nullptr) : st(stream ? stream : rt.stream)
    {
        if (!rt.profiling) return;
        PhaseRec r{phase, nullptr, nullptr, 0, bytes};
        cudaEventCreate(&r.a);
        cudaEventCreate(&r.b);
        cudaEventRecord(r.a, st);
        rt.recs.push_back(r);
        idx = (int)rt.recs.size() - 1;
        l0 = rt.launches.load();
    }
    ~PhaseScope()
    {
        if (idx < 0) return;
        cudaEventRecord(rt.recs[(size_t)idx].b, st);
        rt.recs[(size_t)idx].launches = rt.launches.load() - l0;
    }
};

void profile_collect()
{
    for (auto &r : rt.recs) {
        cudaEventSynchronize(r.b);
        float ms = 0;
        cudaEventElapsedTime(&ms, r.a, r.b);
        rt.acc_ms[r.phase] += ms;
        rt.acc_launches[r.phase] += r.launches;
        rt.acc_bytes[r.phase] += r.bytes;
        cudaEventDestroy(r.a);
        cudaEventDestroy(r.b);
    }
    rt.recs.clear();
}

template <typename T>
int dev_upload(T **dptr, const std::vector<T> &h)
{
    CUDA_TRY(cudaMalloc(reinterpret_cast<void **>(dptr), std::max<size_t>(h.size(), 1) * sizeof(T)));
    if (!h.empty()) CUDA_TRY(cudaMemcpy(*dptr, h.data(), h.size() * sizeof(T), cudaMemcpyHostToDevice));
    return DFDB_OK;
}

// ---- result arena: page-locked host memory handed to the caller for materialized columns (dfdb_host_alloc) ------
// cudaHostAlloc is slow (it pins page by page), so freed buffers are kept and reused: a scan that runs again finds
// its result buffers ready.  `live` lets copy_out recognise a pinned destination and copy straight into it.
struct HostArena {
    std::mutex mu;
    std::map<uintptr_t, size_t> live;                  // base -> capacity of buffers handed out
    std::multimap<size_t, void *> spare;               // capacity -> cached buffer
    size_t spare_bytes = 0;
    size_t cap_bytes = (size_t)24 << 30;               // cache at most this much (option "host_arena_cap_mb")
    bool pinned(const void *p, size_t n)
    {
        std::lock_guard<std::mutex> lk(mu);
        auto it = live.upper_bound(reinterpret_cast<uintptr_t>(p));
        if (it == live.begin()) return false;
        --it;
        return reinterpret_cast<uintptr_t>(p) + n <= it->first + it->second;
    }
    void trim(size_t keep)
    {
        while (spare_bytes > keep && !spare.empty()) {
            auto it = std::prev(spare.end());
            cudaFreeHost(it->second);
            spare_bytes -= it->first;
            spare.erase(it);
        }
    }
} arena;

// Stream-ordered device scratch (gather outputs): the pool keeps its memory between scans.
cudaError_t scratch_alloc(void **p, size_t n)
{
    static bool configured = false;
    if (!configured) {
        cudaMemPool_t pool;
        if (cudaDeviceGetDefaultMemPool(&pool, rt.device) == cudaSuccess) {
            unsigned long long keep = ~0ull;
            cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &keep);
        }
        configured = true;
    }
    return cudaMallocAsync(p, std::max<size_t>(n, 1), rt.stream);
}
void scratch_free(void *p, cudaStream_t stream = nullptr) { if (p) cudaFreeAsync(p, stream ? stream : rt.stream); }
}  // namespace

cudaError_t dfdb::PoolBuf::alloc(size_t n)
{
    reset();
    const cudaError_t e = scratch_alloc(&p, n);
    if (e != cudaSuccess) p = nullptr;
    return e;
}

void dfdb::PoolBuf::free_on(cudaStream_t stream)
{
    scratch_free(p, stream);
    p = nullptr;
}

void dfdb::ResultCol::set_type(const ColType &ty)
{
    kind = ty.kind;
    elsize = ty.kind == DFDB_STRING ? 0 : ty.elsize;
    nullable = ty.kind == DFDB_STRING ? 0 : (ty.nullable ? 1 : 0);
}

int dfdb::ResultCol::alloc(int64_t n_, int64_t bytes_)
{
    release();
    const bool str = kind == DFDB_STRING;
    if (str ? sizes.alloc((size_t)n_ * 4) != cudaSuccess || chars.alloc((size_t)bytes_) != cudaSuccess
            : values.alloc((size_t)n_ * elsize) != cudaSuccess || (nullable && missing.alloc((size_t)n_) != cudaSuccess)) {
        release();
        return fail(DFDB_ERR_NOMEM, "out of device memory for a result of %lld values", (long long)n_);
    }
    n = n_;
    bytes = str ? bytes_ : 0;
    return DFDB_OK;
}

void dfdb::ResultCol::release(cudaStream_t stream)
{
    values.free_on(stream); missing.free_on(stream); sizes.free_on(stream); chars.free_on(stream);
    n = bytes = 0;
}

namespace {
cudaError_t copy_out(void *dst, const void *d_src, size_t n);

// Result column -> caller memory without stalling the scan stream: a destination in the result arena is copied on the
// copy stream (behind an event on the scan stream), so that the gather -- or the decode -- of the next projected column
// runs during the transfer.  Returns true when the copy was queued that way (the caller then frees the scratch on the copy
// stream and synchronises it before returning); anything else is copied synchronously by copy_out.
bool copy_out_queued(void *dst, const void *d_src, size_t n, cudaError_t *err)
{
    *err = cudaSuccess;
    if (n == 0) return false;
    if (!arena.pinned(dst, n)) { *err = copy_out(dst, d_src, n); return false; }
    cudaEvent_t ready;
    if ((*err = cudaEventCreateWithFlags(&ready, cudaEventDisableTiming)) != cudaSuccess) return false;
    cudaEventRecord(ready, rt.stream);
    cudaStreamWaitEvent(rt.copy_stream, ready, 0);
    cudaEventDestroy(ready);
    *err = cudaMemcpyAsync(dst, d_src, n, cudaMemcpyDeviceToHost, rt.copy_stream);
    return *err == cudaSuccess;
}

// Device -> caller memory.  A destination inside the result arena is page-locked: one asynchronous copy at full PCIe
// rate.  Anything else is ordinary (pageable) host memory, which the driver copies at a few GB/s; large results go
// through two pinned bounce buffers instead, the copy of chunk k+1 overlapping the host memcpy of chunk k.  Returns
// after the data is in `dst`.
cudaError_t copy_out(void *dst, const void *d_src, size_t n)
{
    constexpr size_t CHUNK = 32u << 20;
    if (n < (8u << 20) || arena.pinned(dst, n)) {
        cudaError_t e = cudaMemcpyAsync(dst, d_src, n, cudaMemcpyDeviceToHost, rt.stream);
        return e != cudaSuccess ? e : cudaStreamSynchronize(rt.stream);
    }
    static uint8_t *bounce[2] = {nullptr, nullptr};
    static cudaEvent_t done[2];
    if (!bounce[0]) {
        for (int i = 0; i < 2; i++) {
            cudaError_t e = cudaMallocHost(reinterpret_cast<void **>(&bounce[i]), CHUNK);
            if (e != cudaSuccess) { bounce[0] = nullptr; return e; }
            cudaEventCreateWithFlags(&done[i], cudaEventDisableTiming);
        }
    }
    const size_t nchunks = (n + CHUNK - 1) / CHUNK;
    for (size_t k = 0; k <= nchunks; k++) {
        if (k < nchunks) {
            const size_t off = k * CHUNK, len = std::min(CHUNK, n - off);
            cudaError_t e = cudaMemcpyAsync(bounce[k & 1], static_cast<const uint8_t *>(d_src) + off, len, cudaMemcpyDeviceToHost, rt.stream);
            if (e != cudaSuccess) return e;
            cudaEventRecord(done[k & 1], rt.stream);
        }
        if (k > 0) {
            const size_t off = (k - 1) * CHUNK, len = std::min(CHUNK, n - off);
            cudaError_t e = cudaEventSynchronize(done[(k - 1) & 1]);
            if (e != cudaSuccess) return e;
            memcpy(static_cast<uint8_t *>(dst) + off, bounce[(k - 1) & 1], len);
        }
    }
    return cudaSuccess;
}

void column_release(Column &c)
{
    if (c.h_comp) cudaFreeHost(c.h_comp);
    cudaFree(c.d_comp); cudaFree(c.d_decoded); cudaFree(c.d_comp_off); cudaFree(c.d_comp_len); cudaFree(c.d_dec_off);
    cudaFree(c.d_origin); cudaFree(c.d_status); cudaFree(c.d_str_off); cudaFree(c.d_skip);
    c.d_skip = nullptr; c.h_skip.clear(); c.h_corrupt.clear(); c.stored_blocks = 0;
    c.h_comp = nullptr; c.d_comp = nullptr; c.d_decoded = nullptr; c.d_comp_off = nullptr; c.d_comp_len = nullptr;
    c.d_dec_off = nullptr; c.d_origin = nullptr; c.d_status = nullptr; c.d_str_off = nullptr;
    c.loaded = false; c.decoded_valid = false; c.dec_lo = c.dec_hi = 0; c.dec_live_gen = 0; c.str_off_valid = false;
}

Geometry make_geometry(const dfdb_table *t)
{
    Geometry g;
    g.nrows_total = t->nrows;
    g.block_size = t->block_size;
    g.blk_lo = t->blk_lo;
    g.dead = nullptr;
    g.nblocks = (int32_t)(t->blk_hi - t->blk_lo);
    g.wpb = (int32_t)((t->block_size + 31) / 32);
    // work units: segments of whole tiles inside a block; a fixed function of the table shape only, so the
    // floating-point combination order does not depend on the GPU or the shard layout
    int64_t tiles_per_block = (t->block_size + TILE_ROWS - 1) / TILE_ROWS;
    int64_t seg_tiles = tiles_per_block;
    while (seg_tiles > 1 && (int64_t)t->nblocks * ((tiles_per_block + seg_tiles - 1) / seg_tiles) < 8192) seg_tiles = (seg_tiles + 1) / 2;
    g.seg_rows = (int32_t)(seg_tiles * TILE_ROWS);
    g.segs_per_block = (int32_t)((t->block_size + g.seg_rows - 1) / g.seg_rows);
    return g;
}

ColView make_view(const Column &c)
{
    ColView v;
    v.base = c.d_decoded;
    v.blk_off = c.d_dec_off;
    v.str_off = c.d_str_off;
    v.kind = c.type.kind;
    v.elsize = c.type.elsize;
    v.nullable = c.type.nullable ? 1 : 0;
    v.cls = value_class(c.type.kind);
    return v;
}

// 16-byte loads of 8-byte values need 16-byte aligned value areas in every block
bool wide_ok(const dfdb_table *t, const Column &c)
{
    if (rt.no_wide || c.type.elsize != 8) return false;
    if (value_class(c.type.kind) == VC_NONE || value_class(c.type.kind) == VC_STR) return false;
    if (!c.type.nullable) return true;
    for (int64_t b = t->blk_lo; b < t->blk_hi; b++) {
        int64_t rows = c.blocks[(size_t)b].rows;
        if ((((rows + 63) / 64) * 8) % 16 != 0) return false;
    }
    return true;
}

// ---- decode ---------------------------------------------------------------------------------------------
// Each K1 decoder, indexed by K1: its dfdb_profile_get name and its launch
const struct {
    const char *name;
    int (*launch)(const DecodeArgs &, unsigned int *counter, int sm_count, cudaStream_t, int cta_limit);
} k1_kernels[K1_COUNT] = {
    {"k1_v3", launch_lz4_decode_v3},
    {"k1_spec", launch_lz4_decode_spec},
    {"k1_long", launch_lz4_decode_long},
    {"k1_bytes", launch_lz4_decode_bytes},
    {"k1_v1", [](const DecodeArgs &a, unsigned int *counter, int sm_count, cudaStream_t stream, int) { return launch_lz4_decode(a, counter, sm_count, stream); }},
    {"k1_lane", launch_lz4_decode_lane},
};

// Option lz4_flavour: 0 = no decoder forced, 1 / 2 = walker (1 was a removed kernel's number), 3 = lane, 4 = spec, 5 = long,
// 6 = bytes.  Any other value is refused.
int set_lz4_flavour(int64_t value)
{
    static const std::optional<K1> forced[] = {std::nullopt, K1::Walker, K1::Walker, K1::Lane, K1::Spec, K1::Long, K1::Bytes};
    if (value < 0 || value > 6) return fail(DFDB_ERR_ARGUMENT, "lz4_flavour %lld is not one of 0 to 6", (long long)value);
    rt.lz4_flavour = forced[value];
    return DFDB_OK;
}

// The decoder the options force on every column, if any: lz4_simple takes precedence over lz4_flavour
std::optional<K1> forced_decoder() { return rt.lz4_simple ? std::optional(K1::Sequential) : rt.lz4_flavour; }

// DecodeArgs::hot of a K1::Lane launch whose columns did (or did not) all sample as K1::Spec: option lane_hot when it is set
int lane_hot(bool sampled_spec) { return rt.lane_hot >= 0 ? (int)rt.lane_hot : sampled_spec ? 1 : 0; }

int launch_decode(const DecodeArgs &a, K1 decoder, cudaStream_t stream = nullptr, int cta_limit = 0, int counter_slot = 0, int64_t bytes = 0)
{
    const int k = (int)decoder;
    rt.k1_launches[k]++;
    rt.k1_bytes[k] += bytes;
    // (launches that may run at the same time need their own job counter)
    return k1_kernels[k].launch(a, rt.d_counter + 4 * counter_slot, rt.sm_count, stream ? stream : rt.stream, cta_limit);
}

// Which decoder suits a column: walk the token stream of one compressed block on the host (done once, at load).  K1::Spec:
// nearly every sequence is plain -- no length extensions -- and makes whole aligned output words; K1::Bytes: nearly every
// sequence is a bare match; K1::Long: long sequences (Union{Float64,Missing} bodies); K1::Walker: everything else.  None when
// the block gives no verdict.
std::optional<K1> sample_flavour(const uint8_t *src, int64_t n, int64_t origin)
{
    int64_t ip = 0, op = 0, nseq = 0, wordform = 0, bare = 0;
    while (ip < n && nseq < 20000) {
        const uint32_t t = src[ip++];
        int64_t L = t >> 4;
        bool plain = true;
        if (L == 15) {
            plain = false;
            for (;;) { if (ip >= n) return std::nullopt; const uint32_t e = src[ip++]; L += e; if (e != 255) break; }
        }
        ip += L;
        op += L;
        if (ip + 2 > n) break;                                   // last sequence
        const uint32_t off = (uint32_t)src[ip] | ((uint32_t)src[ip + 1] << 8);
        ip += 2;
        int64_t M = t & 15;
        if (M == 15) {
            plain = false;
            for (;;) { if (ip >= n) return std::nullopt; const uint32_t e = src[ip++]; M += e; if (e != 255) break; }
        }
        M += 4;
        nseq++;
        // what the spec decoder turns into whole output words without walking: <= 4 literal bytes + match = 8 bytes (or a plain
        // match of 16), offset a multiple of 8, at an aligned output position
        if (plain && L <= 4 && ((off | (op - L)) & 7) == 0 && (L + M == 8 || (L == 0 && M == 16))) wordform++;
        if (plain && L == 0) bare++;                                // a bare match: 3 stream bytes, what the byte-stream decoder verifies in parallel
        op += M;
        if (op > origin) return std::nullopt;
    }
    if (nseq < 64) return op >= 64 * 48 ? std::optional(K1::Long) : std::nullopt;   // (a few very long sequences: a verdict all the same)
    if (wordform * 100 >= nseq * 97) return K1::Spec;
    if (bare * 100 >= nseq * 97) return K1::Bytes;               // match-only byte streams (strings of few distinct values)
    if (op >= nseq * 48) return K1::Long;                        // long sequences (>= 48 output bytes on average): the one-sequence-at-a-time decoder with its stream window
    return K1::Walker;
}

// A column's own decoder, from the token samples of the first, middle and last of its local blocks: the decoder more than half of
// the verdicts name, else the walker (stored blocks are never decoded and give no verdict)
K1 column_decoder(const Column &c, const std::vector<int64_t> &comp_off, const std::vector<int32_t> &comp_len,
                  const std::vector<int32_t> &origin, const std::vector<uint8_t> &stored)
{
    const int64_t nb = (int64_t)stored.size();
    int votes[K1_COUNT] = {0}, verdicts = 0;
    for (const int64_t b : {(int64_t)0, nb / 2, nb - 1})
        if (nb > 0 && !stored[(size_t)b])
            if (const std::optional<K1> v = sample_flavour(c.h_comp + comp_off[(size_t)b], comp_len[(size_t)b], origin[(size_t)b])) { votes[(int)*v]++; verdicts++; }
    // (not the spec decoder for a Union{T,Missing} column: its body starts with its incompressible bitmap -- a long literal run the
    //  spec decoder takes one sequence at a time; measured slower than the walker there: 6.7 against 5.3 ms for 200M
    //  Union{Int64,Missing} rows)
    for (const K1 k : {K1::Spec, K1::Long, K1::Bytes})
        if (2 * votes[(int)k] > verdicts && !(k == K1::Spec && c.type.nullable)) return k;
    return K1::Walker;
}

// Which blocks of its columns a scan's decode covers: the local blocks [lo, hi) that can hold its selected rows, less those
// its zone maps rule out (zone_dead, selection stages) or those without a selected row (live, with the generation of those
// counts, the key of a column's filtered decode: projections).  Made by selection_scope, projection_scope and whole_table.
struct DecodeScope {
    int lo, hi;
    const std::vector<uint8_t> *zone_dead;
    const std::vector<int64_t> *live;
    uint64_t live_gen;
};

// on_part(b0, b1, sms): optional.  Called (once or twice) with consecutive local block ranges that cover the shard, each
// time after work that makes rt.stream wait for the decode of [b0, b1) has been enqueued; `sms` is the number of SMs a
// kernel launched now on rt.stream can expect to find free.  A shard with more blocks to decode than the decoder keeps in
// flight (sm_count x LZ4_SLOTS_PER_SM) decodes in rounds, and its last round is rarely full: the decode of that round is
// given only the SMs it can fill, on a higher-priority stream, and the caller's scan of everything before it runs beside it
// on the others.  Never called when nothing had to be decoded.
using PartFn = std::function<int(int, int, int)>;

// An aggregate's request that the decoder of its predicate's column write the predicate's selection bits (DecodeArgs::bits),
// so that its scan stages only the aggregated column.  ensure_decoded sets `on` before the first on_part call when the
// spec decoder decodes that column in this call, in a launch of its own, in every block the scan visits; else nothing
// writes the bits and the scan evaluates the test itself.
struct BitsReq {
    Column *col;
    ColTest test;
    uint32_t *mask;
    int wpb;
    bool on;
};

int ensure_decoded(dfdb_table *t, const std::vector<int64_t> &col_ids, const DecodeScope &scope, const PartFn *on_part = nullptr,
                   BitsReq *bits = nullptr)
{
    // Only the blocks inside the scope's window are decoded (skip_block / skipblocks in the reference,
    // src/io/blocksiterator.jl:69-78, src/tables/selection.jl:177-184: blocks that a leading range stage rules out are
    // seeked over, not decompressed).  A column remembers which block range of it is currently decoded.
    const int nblocks = (int)(t->blk_hi - t->blk_lo);
    const int wlo = scope.lo, whi = scope.hi;
    std::vector<Column *> cols;
    for (int64_t id : col_ids) {
        Column *c = t->find(id);
        if (!c) return fail(DFDB_ERR_KEY, "unknown column id %lld", (long long)id);
        if (!c->loaded) return fail(DFDB_ERR_STATE, "column %s is not loaded (call dfdb_table_load first)", c->name.c_str());
        const bool have = c->decoded_valid || (c->dec_lo <= wlo && whi <= c->dec_hi) || (scope.live && c->dec_live_gen == scope.live_gen);
        if (!have && std::find(cols.begin(), cols.end(), c) == cols.end()) cols.push_back(c);
    }
    if (cols.empty() || whi == wlo) return DFDB_OK;
    // Projection columns: a block without a selected row is skipped like a block outside the window (skip_cols,
    // blocksiterator.jl:84-95,112-115: `isempty(range) ? skip_cols(proj_cols) : read_cols(proj_cols)`).  The stored-block
    // flags and the scan's per-block survivor counts are merged into one skip list per column for this call.
    const std::vector<int64_t> *live = scope.live && (int)scope.live->size() == nblocks ? scope.live : nullptr;
    const std::vector<uint8_t> *zdead = scope.zone_dead && (int)scope.zone_dead->size() == nblocks ? scope.zone_dead : nullptr;
    // Released on every way out of this call.  The skip lists are freed on rt.stream; decodes queued on the decode streams read
    // them, so unless rt.stream has waited for both streams already, it waits first.
    struct Scratch {
        std::vector<uint8_t *> skips;
        std::vector<cudaEvent_t> events;
        bool decode_streams_busy = false;
        cudaError_t event(cudaEvent_t *e)
        {
            const cudaError_t r = cudaEventCreateWithFlags(e, cudaEventDisableTiming);
            if (r == cudaSuccess) events.push_back(*e);
            return r;
        }
        ~Scratch()
        {
            cudaEvent_t e;
            if (decode_streams_busy)
                for (cudaStream_t ds : {rt.decode_stream, rt.decode_stream2})
                    if (event(&e) != cudaSuccess || cudaEventRecord(e, ds) != cudaSuccess || cudaStreamWaitEvent(rt.stream, e, 0) != cudaSuccess)
                        cudaStreamSynchronize(ds);   // (the host waits instead)
            for (uint8_t *p : skips) scratch_free(p);
            for (cudaEvent_t ev : events) cudaEventDestroy(ev);
        }
    } scratch;
    // One record per column to decode: its skip list on the device, the decoder that decodes it in THIS call, and the count of
    // the blocks it decodes before each block (the host side of its skip list).
    struct Todo {
        Column *c;
        const uint8_t *d_skip;
        K1 decoder;
        std::vector<int> before;   // before[b]: blocks of [0, b) that are decoded
        int64_t work(int b0, int b1) const { return before[(size_t)b1] - before[(size_t)b0]; }
    };
    std::vector<Todo> todo;
    bool filtered = false;
    uint8_t *d_dead = nullptr;           // blocks without a selected row (any column)
    std::vector<uint8_t> dead;
    if (live || zdead) {
        dead.resize((size_t)nblocks);
        for (int b = 0; b < nblocks; b++) dead[(size_t)b] = (live && (*live)[(size_t)b] == 0) || (zdead && (*zdead)[(size_t)b]);
        if (scratch_alloc(reinterpret_cast<void **>(&d_dead), (size_t)nblocks) != cudaSuccess) return fail(DFDB_ERR_NOMEM, "out of device memory for the block skip list");
        scratch.skips.push_back(d_dead);
        CUDA_TRY(cudaMemcpyAsync(d_dead, dead.data(), (size_t)nblocks, cudaMemcpyHostToDevice, rt.stream));
    }
    for (Column *c : cols) {
        Todo r{c, c->d_skip, c->decoder, std::vector<int>((size_t)nblocks + 1, 0)};
        const uint8_t *skip = c->h_skip.data();
        std::vector<uint8_t> sk;
        if (!dead.empty()) {
            sk = c->h_skip;
            for (int b = 0; b < nblocks; b++) if (dead[(size_t)b] && !sk[(size_t)b]) { sk[(size_t)b] = 1; filtered = true; }
            uint8_t *dp = nullptr;
            if (scratch_alloc(reinterpret_cast<void **>(&dp), (size_t)nblocks) != cudaSuccess) return fail(DFDB_ERR_NOMEM, "out of device memory for the block skip list");
            scratch.skips.push_back(dp);
            CUDA_TRY(cudaMemcpyAsync(dp, sk.data(), (size_t)nblocks, cudaMemcpyHostToDevice, rt.stream));
            r.d_skip = dp;
            skip = sk.data();
        }
        for (int b = 0; b < nblocks; b++) r.before[(size_t)b + 1] = r.before[(size_t)b] + (skip[(size_t)b] ? 0 : 1);
        todo.push_back(std::move(r));
    }
    // Transfer-inclusive mode: the compressed blocks live in pinned host memory.  They are copied H2D in
    // block-range chunks on a second stream while the previous chunk is being decoded on the scan stream.
    int64_t host_bytes = 0;
    for (const Todo &r : todo)
        if (r.c->mode == DFDB_LOAD_HOST) host_bytes += (whi < nblocks ? r.c->h_comp_off[(size_t)whi] : (int64_t)r.c->comp_bytes) - r.c->h_comp_off[(size_t)wlo];
    int nchunks = 1;
    if (host_bytes > 0) {
        nchunks = (int)std::min<int64_t>(16, std::max<int64_t>(1, host_bytes / (64ll << 20)));
        if (nchunks > whi - wlo) nchunks = whi - wlo;
    }
    std::vector<cudaEvent_t> copied;
    if (host_bytes > 0) {
        cudaEvent_t start;
        CUDA_TRY(scratch.event(&start));
        CUDA_TRY(cudaEventRecord(start, rt.stream));
        CUDA_TRY(cudaStreamWaitEvent(rt.copy_stream, start, 0));
        PhaseScope ps(PH_H2D, host_bytes, rt.copy_stream);
        for (int k = 0; k < nchunks; k++) {
            const int b0 = wlo + (int)((int64_t)(whi - wlo) * k / nchunks), b1 = wlo + (int)((int64_t)(whi - wlo) * (k + 1) / nchunks);
            for (const Todo &r : todo) {
                Column *c = r.c;
                if (c->mode != DFDB_LOAD_HOST) continue;
                const int64_t lo = c->h_comp_off[(size_t)b0];
                const int64_t hi = b1 < nblocks ? c->h_comp_off[(size_t)b1] : (int64_t)c->comp_bytes;
                CUDA_TRY(cudaMemcpyAsync(c->d_comp + lo, c->h_comp + lo, (size_t)(hi - lo), cudaMemcpyHostToDevice, rt.copy_stream));
            }
            cudaEvent_t e;
            CUDA_TRY(scratch.event(&e));
            CUDA_TRY(cudaEventRecord(e, rt.copy_stream));
            copied.push_back(e);
        }
    }
    // Each column's decoder: the one the options force, else its own.  A column with only a handful of blocks to decode (an
    // incompressible column is stored blocks read in place, plus the odd block LZ4 did shave a few bytes off) is not worth a
    // launch of its own, nor should it keep the others from the decode / scan overlap: it rides in the launch of the column
    // that has the most work, with that column's decoder.
    {
        size_t main_i = 0;
        for (size_t i = 0; i < todo.size(); i++) if (todo[i].work(wlo, whi) > todo[main_i].work(wlo, whi)) main_i = i;
        const std::optional<K1> forced = forced_decoder();
        for (Todo &r : todo)
            r.decoder = forced.value_or(r.work(wlo, whi) * 64 <= todo[main_i].work(wlo, whi) ? todo[main_i].c->decoder : r.c->decoder);
    }
    // Predicate bits: only when the spec decoder decodes every block of the column that the scan visits (no stored block, the
    // whole shard in the window) -- a block it skips, or another decoder, would leave its bits unwritten.  And only for at
    // least two blocks per resident decoder warp: with fewer, each warp decodes a block or two, the decode takes as long as
    // one block does, and the flushes lengthen that by more than the scan saves (B200, rand(1:100) a: 100M rows, 1 526
    // blocks, 2.22 ms with the bits against 2.20 without; 1B rows, 15 259 blocks: 7.91 against 8.24).
    const Todo *bits_todo = nullptr;
    if (bits) {
        bits->on = false;
        for (const Todo &r : todo) if (r.c == bits->col) bits_todo = &r;
        bool ok = bits_todo && wlo == 0 && whi == nblocks && bits_todo->decoder == K1::Spec &&
                  (rt.pred_bits == 1 || bits_todo->work(wlo, whi) >= 2ll * rt.sm_count * LZ4_SPEC_WARPS_PER_SM);
        for (int b = 0; ok && b < nblocks; b++)
            ok = (!dead.empty() && dead[(size_t)b]) || bits_todo->work(b, b + 1) == 1;
        if (!ok) bits_todo = nullptr;
        bits->on = bits_todo != nullptr;
    }
    // One decode launch's arguments: records [q0, q1) of `rs` over local blocks [b0, b1).  Returns the algorithmic bytes of the
    // blocks it decodes (compressed read + decoded written).
    auto fill = [&](DecodeArgs &a, const std::vector<const Todo *> &rs, size_t q0, size_t q1, int b0, int b1) -> int64_t {
        memset(&a, 0, sizeof a);
        a.nblocks = b1 - b0;
        a.blk0 = b0;
        int64_t bytes = 0;
        bool sampled_spec = true;
        for (size_t q = q0; q < q1; q++) {
            const Todo &r = *rs[q];
            Column *c = r.c;
            a.col[a.ncols++] = DecodeCol{c->d_comp, c->d_comp_off, c->d_comp_len, c->d_dec_off, c->d_origin, c->d_decoded, c->d_status, r.d_skip};
            for (int b = b0; b < b1; b++)
                if (r.work(b, b + 1)) bytes += c->blocks[(size_t)(t->blk_lo + b)].compressed + c->blocks[(size_t)(t->blk_lo + b)].origin;
            sampled_spec = sampled_spec && c->decoder == K1::Spec;
        }
        if (rs[q0]->decoder == K1::Lane) a.hot = lane_hot(sampled_spec);
        return bytes;
    };
    // ---- decode / scan overlap (compressed blocks resident, every column on the walker, more than one round of blocks) ----
    bool parted = false;
    if (on_part && host_bytes == 0 && !rt.no_overlap && todo.size() <= (size_t)DECODE_MAX_COLS && !bits_todo) {
        // the walker is the decoder that works in rounds (columns whose blocks are all skipped -- stored bodies read in place --
        // have no say)
        bool walker = true;
        std::vector<const Todo *> all;
        for (const Todo &r : todo) {
            all.push_back(&r);
            walker = walker && (r.work(wlo, whi) == 0 || r.decoder == K1::Walker);
        }
        auto jobs = [&](int b0, int b1) { int64_t n = 0; for (const Todo &r : todo) n += r.work(b0, b1); return n; };
        const int64_t wave = (int64_t)rt.sm_count * LZ4_SLOTS_PER_SM;
        const int64_t real = jobs(wlo, whi);
        // the last round: what is left after the full rounds
        const int64_t last_real = real % wave;
        int split = 0;
        if (walker && real > wave && last_real > 0)
            for (split = wlo; split < whi && jobs(wlo, split) < real - last_real; split++) {}
        const int last_ctas = (int)((last_real + LZ4_SLOTS_PER_SM - 1) / LZ4_SLOTS_PER_SM);
        const int scan_sms = rt.sm_count - last_ctas;
        if (split > wlo && split < whi && scan_sms >= 8) {
            // The full rounds go to one launch (its slots pick up blocks as they finish: no barrier between rounds); the last
            // round is a launch of its own on a second stream, so that its CTAs move in as the first launch's CTAs run out
            // of blocks -- again no barrier -- and it is limited to the SMs it can fill.
            int64_t bytes = 0;
            auto decode_range = [&](int b0, int b1, int cta_limit, cudaStream_t stream, int counter_slot, cudaEvent_t done) -> int {
                DecodeArgs a;
                const int64_t nb = fill(a, all, 0, all.size(), b0, b1);
                bytes += nb;
                LAUNCH(launch_decode(a, K1::Walker, stream, cta_limit, counter_slot, nb));
                CUDA_TRY(cudaEventRecord(done, stream));
                return DFDB_OK;
            };
            cudaEvent_t e0, e1, e2;
            CUDA_TRY(scratch.event(&e0));
            CUDA_TRY(scratch.event(&e1));
            CUDA_TRY(scratch.event(&e2));
            CUDA_TRY(cudaEventRecord(e0, rt.stream));
            CUDA_TRY(cudaStreamWaitEvent(rt.decode_stream, e0, 0));
            CUDA_TRY(cudaStreamWaitEvent(rt.decode_stream2, e0, 0));
            scratch.decode_streams_busy = true;
            // one decode phase record for both launches: from the start of the first to the end of the second
            PhaseRec pr{PH_DECODE, nullptr, nullptr, 2, 0};
            if (rt.profiling) { cudaEventCreate(&pr.a); cudaEventCreate(&pr.b); cudaEventRecord(pr.a, rt.decode_stream); }
            int rc = decode_range(wlo, split, 0, rt.decode_stream, 0, e1);
            if (!rc) rc = decode_range(split, whi, last_ctas, rt.decode_stream2, 1, e2);
            if (pr.a) { cudaEventRecord(pr.b, rt.decode_stream2); pr.bytes = bytes; rt.recs.push_back(pr); }
            if (rc) return rc;
            CUDA_TRY(cudaStreamWaitEvent(rt.stream, e1, 0));
            rc = (*on_part)(wlo, split, scan_sms);
            if (rc) return rc;
            CUDA_TRY(cudaStreamWaitEvent(rt.stream, e2, 0));
            scratch.decode_streams_busy = false;
            rc = (*on_part)(split, whi, rt.sm_count);
            if (rc) return rc;
            parted = true;
        }
    }
    bool chunk_parts = false;
    for (int k = 0; k < nchunks && !parted; k++) {
        const int b0 = wlo + (int)((int64_t)(whi - wlo) * k / nchunks), b1 = wlo + (int)((int64_t)(whi - wlo) * (k + 1) / nchunks);
        if (!copied.empty()) CUDA_TRY(cudaStreamWaitEvent(rt.stream, copied[(size_t)k], 0));
        if (b1 <= b0) continue;
        // columns of one decoder share a launch
        for (int k = 0; k < K1_COUNT; k++) {
          const K1 decoder = (K1)k;
          // (a column whose blocks in this range are all skipped -- stored bodies read in place, blocks without selected rows -- needs no launch)
          std::vector<const Todo *> grp;
          for (const Todo &r : todo) if (r.decoder == decoder && r.work(b0, b1) > 0 && &r != bits_todo) grp.push_back(&r);
          if (bits_todo && bits_todo->decoder == decoder && bits_todo->work(b0, b1) > 0) {
              // the column that writes the predicate's bits: a launch of its own
              DecodeArgs a;
              const int64_t bytes = fill(a, {bits_todo}, 0, 1, b0, b1);
              a.bits = bits->mask;
              a.bits_wpb = bits->wpb;
              a.bits_test = bits->test;
              PhaseScope ps(PH_DECODE, bytes);
              LAUNCH(launch_decode(a, decoder, nullptr, 0, 0, bytes));
          }
          // The walker / consumer decoder works in rounds of sm_count x LZ4_SLOTS_PER_SM blocks, and a block takes about as long
          // whether the round is full or not.  Columns that fit a round each but not together are better off in launches of their
          // own (config 4: Union{Int64,Missing} + Union{Float64,Missing}, 7 630 blocks each: one mixed launch is two rounds in
          // which the slow column's blocks set the pace).  The other decoders have no rounds: their columns share a launch.
          size_t per_launch = DECODE_MAX_COLS;
          if (decoder == K1::Walker && grp.size() > 1) {
              int64_t jobs = 0;
              for (const Todo *r : grp) jobs += r->work(b0, b1);
              if (jobs > (int64_t)rt.sm_count * LZ4_SLOTS_PER_SM) per_launch = 1;
          }
          for (size_t i = 0; i < grp.size(); i += per_launch) {
            DecodeArgs a;
            const int64_t bytes = fill(a, grp, i, std::min(grp.size(), i + per_launch), b0, b1);
            PhaseScope ps(PH_DECODE, bytes);
            LAUNCH(launch_decode(a, decoder, nullptr, 0, 0, bytes));
          }
        }
        // transfer-inclusive mode: the caller's scan of this chunk follows its decode, beside the copy of the next chunks
        if (on_part && nchunks > 1) {
            const int rc = (*on_part)(b0, b1, rt.sm_count);
            if (rc) return rc;
            chunk_parts = true;
        }
    }
    if (on_part && !parted && !chunk_parts) {
        const int rc = (*on_part)(wlo, whi, rt.sm_count);
        if (rc) return rc;
    }
    const Geometry g = make_geometry(t);
    for (const Todo &r : todo)
        if (r.c->type.kind == DFDB_STRING) {
            PhaseScope ps(PH_UNPACK, 0);
            LAUNCH(launch_str_offsets(g, make_view(*r.c), r.c->d_str_off, r.c->d_status, r.c->d_origin, rt.stream, wlo, whi, d_dead));
        }
    // integrity gate (the reference asserts after every block, BlockStreams.jl:112)
    std::vector<int32_t> st((size_t)nblocks);
    for (const Todo &r : todo) {
        Column *c = r.c;
        CUDA_TRY(cudaMemcpyAsync(st.data(), c->d_status, (size_t)nblocks * 4, cudaMemcpyDeviceToHost, rt.stream));
        CUDA_TRY(cudaStreamSynchronize(rt.stream));
        for (int b = wlo; b < whi; b++) {
            // a block the decoder was told to skip (no selected row: skip_cols seeks over it) is not decompressed, hence not judged
            const int32_t verdict = st[(size_t)b] != 0 ? st[(size_t)b] : (!c->h_corrupt.empty() && r.work(b, b + 1) ? c->h_corrupt[(size_t)b] : 0);
            if (verdict != 0)
                return fail(DFDB_ERR_CORRUPT, "decompression error in column %s block %lld (code %d)", c->name.c_str(),
                            (long long)(t->blk_lo + b), verdict);
        }
        // (a decode that skipped blocks without selected rows leaves nothing another scan could rely on)
        c->dec_lo = filtered ? 0 : wlo;
        c->dec_hi = filtered ? 0 : whi;
        c->dec_live_gen = filtered && !zdead ? scope.live_gen : 0;   // (a decode pruned by zone maps is good for that scan only)
        c->decoded_valid = !filtered && wlo == 0 && whi == nblocks;
    }
    return DFDB_OK;
}

void invalidate_decoded(dfdb_table *t)
{
    for (auto &c : t->cols)
        if (c.mode != DFDB_LOAD_DECODED) { c.decoded_valid = false; c.dec_lo = c.dec_hi = 0; c.dec_live_gen = 0; }
}

// a mask (and the counts derived from it) is only good for the shard it was computed on
bool mask_current(const dfdb_scan *s) { return s->mask_valid && s->mask_epoch == s->tbl->epoch; }

// ---- zone maps: which blocks can hold a selected row -----------------------------------------------------------------
// A predicate stage that is a conjunction of `column <cmp> constant` terms (Expr::simple; a missing value compares false)
// selects nothing in a block whose value range [min, max] misses the constant's side for some term, or that holds no
// non-missing value at all.  A dead block is skipped by every stage of the scan, so only stages up to the first range /
// index-vector stage that follows a predicate may prune: that stage ranks the survivors of the stages before it
// (selection.jl:94-111), and a block a later predicate empties may still hold some of those survivors.  A block without
// survivors of the earlier stages contributes nothing to the ranks of the range stages after them, so pruning stays exact
// up to that point.  NaN never satisfies an ordered comparison and is kept out of the range; `!=` only prunes a block whose
// values all equal the constant and that has no NaN.
bool zone_term_dead(const Term &tm, const ZoneEntry &z, int64_t rows)
{
    if (tm.constant_result >= 0) return tm.constant_result == 0;
    if (z.null_count >= rows) return true;
    const bool has = (z.flags & 1) != 0, nan = (z.flags & 2) != 0;
    if (tm.cls == VC_FLT) {
        double mn, mx;
        memcpy(&mn, &z.min_bits, 8);
        memcpy(&mx, &z.max_bits, 8);
        const double c = tm.cf;
        if (c != c) return tm.code != 1;                       // only x != NaN is ever true
        if (tm.code == 1) return has && !nan && mn == c && mx == c;
        if (!has) return true;                                 // only NaN (and missing) values: every ordered comparison is false
        switch (tm.code) {
        case 0: return c < mn || c > mx;
        case 2: return !(mn < c);
        case 3: return !(mn <= c);
        case 4: return !(mx > c);
        default: return !(mx >= c);
        }
    }
    if (!has) return true;
    if (tm.cls == VC_UINT) {
        const uint64_t mn = z.min_bits, mx = z.max_bits, c = (uint64_t)tm.ci;
        switch (tm.code) {
        case 0: return c < mn || c > mx;
        case 1: return mn == c && mx == c;
        case 2: return !(mn < c);
        case 3: return !(mn <= c);
        case 4: return !(mx > c);
        default: return !(mx >= c);
        }
    }
    const int64_t mn = (int64_t)z.min_bits, mx = (int64_t)z.max_bits, c = tm.ci;
    switch (tm.code) {
    case 0: return c < mn || c > mx;
    case 1: return mn == c && mx == c;
    case 2: return !(mn < c);
    case 3: return !(mn <= c);
    case 4: return !(mx > c);
    default: return !(mx >= c);
    }
}

// An `in` stage over a stored numeric column (Expr::inset_slot) selects nothing in a block when no key of the set lies in the
// block's [min, max], unless the set holds missing and the block a missing value (isequal semantics: missing in Set is true),
// or the set holds NaN and the block a NaN (isequal again; under `==` neither can hit).
bool zone_set_dead(const InSet &set, const ZoneEntry &z)
{
    if ((set.flags & SET_MISSING) && (set.flags & SET_ISEQUAL) && z.null_count > 0) return false;
    if (set.has_nan && (z.flags & 2)) return false;
    if (!set.has_range || !(z.flags & 1)) return true;
    if (set.cls == VC_FLT) {
        double kmin, kmax, mn, mx;
        memcpy(&kmin, &set.kmin, 8); memcpy(&kmax, &set.kmax, 8);
        memcpy(&mn, &z.min_bits, 8); memcpy(&mx, &z.max_bits, 8);
        return kmax < mn || kmin > mx;
    }
    if (set.cls == VC_UINT) return set.kmax < z.min_bits || set.kmin > z.max_bits;
    return (int64_t)set.kmax < (int64_t)z.min_bits || (int64_t)set.kmin > (int64_t)z.max_bits;
}

// Fills s->zone_dead (+ the device copy) and s->zone_pruned.  Terms whose class differs from the column's (Int64 column
// against a Float64 constant ...) are left alone: the plan folds those exactly elsewhere.
void zone_prune(dfdb_scan *s)
{
    dfdb_table *t = s->tbl;
    const int nblocks = (int)(t->blk_hi - t->blk_lo);
    s->zone_dead.clear();
    s->zone_pruned = 0;
    if (rt.no_zonemap || nblocks <= 0) return;
    bool any = false;
    std::vector<uint8_t> dead((size_t)nblocks, 0);
    bool after_pred = false;
    for (const Stage &st : s->stages) {
        if (st.kind != ST_PRED) {
            if (after_pred) break;      // this stage ranks earlier survivors: later predicates must not empty their blocks
            continue;
        }
        after_pred = true;
        if (st.e.inset_slot >= 0) {
            const InSet &set = s->sets[(size_t)st.e.sets[0]];
            const Column *c = t->find(s->slots[(size_t)st.e.inset_slot]);
            if (!c || c->zones.size() != c->blocks.size() || value_class(c->type.kind) != set.cls) continue;
            for (int b = 0; b < nblocks; b++) {
                const size_t tb = (size_t)(t->blk_lo + b);
                if (!dead[(size_t)b] && zone_set_dead(set, c->zones[tb])) { dead[(size_t)b] = 1; any = true; s->zone_pruned++; }
            }
            continue;
        }
        if (!st.e.simple) continue;
        for (int i = 0; i < st.e.nterms; i++) {
            const Term &tm = st.e.terms[i];
            const Column *c = t->find(s->slots[(size_t)tm.slot]);
            if (!c || c->zones.size() != c->blocks.size() || value_class(c->type.kind) != tm.cls) continue;
            for (int b = 0; b < nblocks; b++) {
                const size_t tb = (size_t)(t->blk_lo + b);
                if (!dead[(size_t)b] && zone_term_dead(tm, c->zones[tb], c->blocks[tb].rows)) { dead[(size_t)b] = 1; any = true; s->zone_pruned++; }
            }
        }
    }
    if (!any) return;
    s->zone_dead.swap(dead);
    if (!s->d_zone_dead && cudaMalloc(reinterpret_cast<void **>(&s->d_zone_dead), (size_t)nblocks) != cudaSuccess) { s->zone_dead.clear(); s->zone_pruned = 0; return; }
    cudaMemcpyAsync(s->d_zone_dead, s->zone_dead.data(), (size_t)nblocks, cudaMemcpyHostToDevice, rt.stream);
}

const uint8_t *zone_dead_dev(const dfdb_scan *s) { return !s->zone_dead.empty() ? s->d_zone_dead : nullptr; }

// The local blocks that can hold selected rows of a scan: a leading range / index-vector stage works on table row numbers
// (selection.jl:94-111 with offset 0), so the blocks before its first and behind its last row are never decoded.
void scan_window(const dfdb_scan *s, int *wlo, int *whi)
{
    const dfdb_table *t = s->tbl;
    const int64_t nblocks = t->blk_hi - t->blk_lo;
    int64_t lo = 0, hi = nblocks;
    if (!s->stages.empty() && s->stages[0].kind != ST_PRED && t->block_size > 0) {
        const int64_t tb_lo = (s->stages[0].first - 1) / t->block_size, tb_hi = (s->stages[0].last - 1) / t->block_size + 1;
        lo = std::max<int64_t>(lo, tb_lo - t->blk_lo);
        hi = std::min<int64_t>(hi, tb_hi - t->blk_lo);
        if (s->stages[0].first < 1) lo = 0;          // (rows below 1 select nothing; keep the arithmetic simple)
    }
    *wlo = (int)std::min(lo, nblocks);
    *whi = (int)std::max<int64_t>(hi, *wlo);
}

// The decode of a selection stage's columns (and of an aggregate's): the window, less the blocks the scan's zone maps
// ruled out in its last zone_prune.
DecodeScope selection_scope(const dfdb_scan *s)
{
    DecodeScope sc{0, 0, s->zone_dead.empty() ? nullptr : &s->zone_dead, nullptr, 0};
    scan_window(s, &sc.lo, &sc.hi);
    return sc;
}

// The decode of projected columns after select_rows: the window, less the blocks without a selected row while the
// survivor counts are current.
DecodeScope projection_scope(const dfdb_scan *s)
{
    const bool counted = mask_current(s) && s->selected >= 0 && s->live_gen != 0;
    DecodeScope sc{0, 0, nullptr, counted ? &s->blk_live : nullptr, counted ? s->live_gen : 0};
    scan_window(s, &sc.lo, &sc.hi);
    return sc;
}

DecodeScope whole_table(const dfdb_table *t) { return DecodeScope{0, (int)(t->blk_hi - t->blk_lo), nullptr, nullptr, 0}; }

// ---- scan helpers ---------------------------------------------------------------------------------------
int scan_alloc(dfdb_scan *s)
{
    const Geometry g = make_geometry(s->tbl);
    const int64_t words = (int64_t)g.nblocks * g.wpb;
    if (!s->d_mask || s->mask_words != words) {
        cudaFree(s->d_mask);
        s->d_mask = nullptr;
        CUDA_TRY(cudaMalloc(reinterpret_cast<void **>(&s->d_mask), (size_t)std::max<int64_t>(words, 1) * 4));
        CUDA_TRY(cudaMemsetAsync(s->d_mask, 0, (size_t)std::max<int64_t>(words, 1) * 4, rt.stream));
        s->mask_words = words;
        cudaFree(s->d_blk_counts); cudaFree(s->d_blk_base); cudaFree(s->d_blk_bytes);
        CUDA_TRY(cudaMalloc(reinterpret_cast<void **>(&s->d_blk_counts), (size_t)(g.nblocks + 2) * 8));
        CUDA_TRY(cudaMalloc(reinterpret_cast<void **>(&s->d_blk_base), (size_t)(g.nblocks + 2) * 8));
        CUDA_TRY(cudaMalloc(reinterpret_cast<void **>(&s->d_blk_bytes), (size_t)(g.nblocks + 2) * 8 * 2));
        s->mask_valid = false;
    }
    const size_t need = (size_t)std::max(1, g.nblocks * g.segs_per_block) * sizeof(AggPartial);
    if (need > s->partials_cap) {
        cudaFree(s->d_partials);
        CUDA_TRY(cudaMalloc(&s->d_partials, need));
        s->partials_cap = need;
    }
    if (!s->d_result) {
        CUDA_TRY(cudaMalloc(&s->d_result, 256));
        CUDA_TRY(cudaMallocHost(&s->h_result, 256));
    }
    return DFDB_OK;
}

// The device table of an `in` collection, built at the first run that needs it and kept on the handle: one allocation that
// holds the canonical keys as uploaded (String: off | len << 32 words, then the bytes), the slots and the occupancy bits, one
// upload, and the build kernel.  Capacity: the power of two >= 2 keys (load <= 0.5).
int ensure_set(InSet &set)
{
    if (set.d_buf) return DFDB_OK;
    const bool str = set.cls == VC_STR;
    const int64_t n = set.size();
    uint64_t cap = 2;
    while (cap < 2 * (uint64_t)n) cap <<= 1;
    size_t in_bytes = (size_t)n * 8, chars = 0;
    if (str) for (const std::string &k : set.strs) chars += k.size();
    if (chars > 0xFFFFFFFFull) return fail(DFDB_ERR_UNSUPPORTED, "in() collection of more than 4 GiB of String bytes");
    const size_t slots_off = (in_bytes + chars + 15) / 16 * 16;
    const size_t occ_off = slots_off + (size_t)cap * (str ? sizeof(StrSlot) : 8);
    const size_t total = occ_off + (size_t)(cap + 31) / 32 * 4;
    set.h_buf.assign(in_bytes + chars, 0);
    uint8_t *h = set.h_buf.data();
    if (!str) {
        if (n) memcpy(h, set.keys.data(), in_bytes);
    } else {
        uint64_t off = 0;
        for (int64_t i = 0; i < n; i++) {
            const std::string &k = set.strs[(size_t)i];
            const uint64_t w = off | (uint64_t)k.size() << 32;
            memcpy(h + 8 * i, &w, 8);
            memcpy(h + in_bytes + off, k.data(), k.size());
            off += k.size();
        }
    }
    void *d = nullptr;
    if (cudaMalloc(&d, total) != cudaSuccess) {
        cudaGetLastError();
        return fail(DFDB_ERR_NOMEM, "out of device memory for an in() table of %llu slots", (unsigned long long)cap);
    }
    uint8_t *base = static_cast<uint8_t *>(d);
    const SetDesc dev{base + slots_off, reinterpret_cast<const uint32_t *>(base + occ_off), base + in_bytes, cap - 1, set.cls, set.flags};
    const int rc = [&]() -> int {
        if (!set.h_buf.empty()) CUDA_TRY(cudaMemcpyAsync(d, h, set.h_buf.size(), cudaMemcpyHostToDevice, rt.stream));
        CUDA_TRY(cudaMemsetAsync(base + occ_off, 0, total - occ_off, rt.stream));
        const SetBuildArgs a{dev, reinterpret_cast<const unsigned long long *>(d), n};
        if (n) LAUNCH(launch_inset_build(a, rt.stream));
        return DFDB_OK;
    }();
    if (rc) {                    // (the handle keeps no half-built table: the next run starts over)
        cudaStreamSynchronize(rt.stream);
        cudaFree(d);
        return rc;
    }
    set.d_buf = d;
    set.dev = dev;
    return DFDB_OK;
}

// an expression's program on the device, with the tables of its `in` collections
struct DevProg {
    VmProgram *d = nullptr;
    ~DevProg() { cudaFree(d); }
    int upload(dfdb_scan *s, const Expr &e)
    {
        VmProgram p = e.prog;
        for (size_t i = 0; i < e.sets.size(); i++) {
            InSet &set = s->sets[(size_t)e.sets[i]];
            const int rc = ensure_set(set);
            if (rc) return rc;
            p.sets[i] = set.dev;
        }
        CUDA_TRY(cudaMalloc(reinterpret_cast<void **>(&d), sizeof(VmProgram)));
        CUDA_TRY(cudaMemcpyAsync(d, &p, sizeof(VmProgram), cudaMemcpyHostToDevice, rt.stream));
        return DFDB_OK;
    }
};

int fill_slots(dfdb_scan *s, ColView *slots)
{
    for (size_t i = 0; i < s->slots.size(); i++) {
        Column *c = s->tbl->find(s->slots[i]);
        if (!c) return fail(DFDB_ERR_KEY, "unknown column id %lld", (long long)s->slots[i]);
        slots[i] = make_view(*c);
    }
    return DFDB_OK;
}

int check_device_error()
{
    int e = 0;
    CUDA_TRY(cudaMemcpyAsync(&e, rt.d_error, 4, cudaMemcpyDeviceToHost, rt.stream));
    CUDA_TRY(cudaStreamSynchronize(rt.stream));
    if (e) {
        int zero = 0;
        cudaMemcpyAsync(rt.d_error, &zero, 4, cudaMemcpyHostToDevice, rt.stream);
        if (e == DFDB_ERR_DIVIDE) return fail(DFDB_ERR_DIVIDE, "DivideError: integer division error");
        return fail(e, "device-side error %d", e);
    }
    return DFDB_OK;
}

bool fused_terms_wide(dfdb_scan *s, const Expr &e)
{
    for (int i = 0; i < e.nterms; i++) {
        Column *c = s->tbl->find(s->slots[(size_t)e.terms[i].slot]);
        if (!c || !wide_ok(s->tbl, *c)) return false;
    }
    return true;
}

void fill_terms(dfdb_scan *s, const Expr &e, FusedArgs *a)
{
    a->nterms = e.nterms;
    a->const_false = 0;
    for (int i = 0; i < e.nterms; i++) {
        a->term[i] = e.terms[i];
        a->term_col[i] = make_view(*s->tbl->find(s->slots[(size_t)e.terms[i].slot]));
        if (e.terms[i].constant_result == 0) a->const_false = 1;
    }
}

// Runs every selection stage and leaves the selection bitmask in s->d_mask.
// The rank of a surviving row for range stages is global (selection.jl:94-111 running offsets).
int run_selection(dfdb_scan *s)
{
    zone_prune(s);
    const DecodeScope scope = selection_scope(s);
    dfdb_table *t = s->tbl;
    int rc = scan_alloc(s);
    if (rc) return rc;
    Geometry g = make_geometry(t);
    g.dead = zone_dead_dev(s);
    bool dense = true;   // every row of the shard survives so far and the mask is not materialised
    bool used_vm = false;
    int nondense = 0;    // range stages met so far that rank among survivors
    s->exchange_count = -1;
    for (auto &st : s->stages) {
        if (st.kind != ST_PRED) {
            RangeArgs a;
            memset(&a, 0, sizeof a);
            a.g = g; a.mask = s->d_mask; a.kind = st.kind; a.start = st.start; a.step = st.step; a.stop = st.stop;
            if (st.kind == ST_INDEXVEC) {
                if (!st.d_idx) {
                    rc = dev_upload(&st.d_idx, st.idx);
                    if (rc) return rc;
                }
                a.idx = st.d_idx;
                a.nidx = (int64_t)st.idx.size();
            }
            PhaseScope ps(PH_SELECT, 0);
            if (dense) {
                a.dense = 1;
            } else {
                LAUNCH(launch_block_counts(g, s->d_mask, s->d_blk_counts, rt.stream));
                LAUNCH(launch_exclusive_scan(s->d_blk_counts, s->d_blk_base, g.nblocks, rt.stream));
                a.dense = 0;
                a.blk_base = s->d_blk_base;
                if (t->world > 1) {
                    // the rank of a survivor counts the survivors of the lower-ranked shards too (selection.jl:94-111)
                    if ((size_t)nondense >= s->rank_offsets.size()) {
                        CUDA_TRY(cudaMemcpyAsync(s->h_result, s->d_blk_base + g.nblocks, 8, cudaMemcpyDeviceToHost, rt.stream));
                        CUDA_TRY(cudaStreamSynchronize(rt.stream));
                        s->exchange_count = *static_cast<int64_t *>(s->h_result);
                        s->mask_valid = false;
                        return fail(DFDB_NEED_EXCHANGE, "sharded scan: stage %d selects on the global survivor rank; exchange the shard counts first "
                                                        "(dfdb_scan_exchange_count / dfdb_scan_exchange_offset)", nondense);
                    }
                    a.rank_offset = s->rank_offsets[(size_t)nondense];
                }
                nondense++;
            }
            LAUNCH(launch_range_stage(a, rt.stream));
            dense = false;
        } else {
            rc = ensure_decoded(t, st.e.col_ids, scope);
            if (rc) return rc;
            int64_t bytes = 0;
            for (int64_t id : st.e.col_ids) for (int64_t b = t->blk_lo; b < t->blk_hi; b++) bytes += t->find(id)->blocks[(size_t)b].origin;
            PhaseScope ps(PH_SELECT, bytes);
            if (st.e.inset_slot >= 0 && !rt.no_fused) {
                InSet &set = s->sets[(size_t)st.e.sets[0]];
                rc = ensure_set(set);
                if (rc) return rc;
                InSetMaskArgs a;
                memset(&a, 0, sizeof a);
                a.g = g;
                a.col = make_view(*t->find(s->slots[(size_t)st.e.inset_slot]));
                a.set = set.dev;
                a.mask_in = dense ? nullptr : s->d_mask;
                a.mask_out = s->d_mask;
                LAUNCH(launch_inset_mask(a, rt.sm_count, rt.stream));
            } else if (st.e.simple && !rt.no_fused) {
                FusedArgs a;
                memset(&a, 0, sizeof a);
                a.g = g;
                fill_terms(s, st.e, &a);
                a.mask_in = dense ? nullptr : s->d_mask;
                a.mask_out = s->d_mask;
                a.partials = static_cast<AggPartial *>(s->d_partials);
                LAUNCH(launch_fused(a, 0, true, false, rt.sm_count, rt.stream));
            } else {
                VmArgs a;
                memset(&a, 0, sizeof a);
                a.g = g;
                rc = fill_slots(s, a.slot);
                if (rc) return rc;
                DevProg prog;
                rc = prog.upload(s, st.e);
                if (rc) return rc;
                a.prog = prog.d;
                a.mask_in = dense ? nullptr : s->d_mask;
                a.mask_out = s->d_mask;
                a.error_flag = rt.d_error;
                LAUNCH(launch_vm_mask(a, rt.sm_count, rt.stream));
                CUDA_TRY(cudaStreamSynchronize(rt.stream));   // program buffer is freed on scope exit
                used_vm = true;
            }
            dense = false;
        }
    }
    if (dense) {
        PhaseScope ps(PH_SELECT, 0);
        LAUNCH(launch_fill_mask(g, s->d_mask, rt.stream));
    }
    if (used_vm) {
        rc = check_device_error();
        if (rc) return rc;
    }
    s->mask_valid = true;
    s->mask_epoch = t->epoch;
    return DFDB_OK;
}

// Runs the selection, then counts its rows per block (+ exclusive scan: the survivor counts behind projection_scope) and in
// all -> *total.
int select_rows(dfdb_scan *s, int64_t *total)
{
    const int rc = run_selection(s);
    if (rc) return rc;
    const Geometry g = make_geometry(s->tbl);
    {
        PhaseScope ps(PH_CONSUME, (int64_t)g.nblocks * g.wpb * 4);
        LAUNCH(launch_block_counts(g, s->d_mask, s->d_blk_counts, rt.stream));
        LAUNCH(launch_exclusive_scan(s->d_blk_counts, s->d_blk_base, g.nblocks, rt.stream));
    }
    PhaseScope ps(PH_D2H, 8 + (int64_t)g.nblocks * 8);
    s->blk_live.assign((size_t)g.nblocks, 0);
    CUDA_TRY(cudaMemcpyAsync(s->h_result, s->d_blk_base + g.nblocks, 8, cudaMemcpyDeviceToHost, rt.stream));
    if (g.nblocks > 0) CUDA_TRY(cudaMemcpyAsync(s->blk_live.data(), s->d_blk_counts, (size_t)g.nblocks * 8, cudaMemcpyDeviceToHost, rt.stream));
    CUDA_TRY(cudaStreamSynchronize(rt.stream));
    *total = *static_cast<int64_t *>(s->h_result);
    s->selected = *total;
    s->live_gen = rt.next_gen++;       // new counts: a filtered decode keyed on the old ones is not reused
    return DFDB_OK;
}

// Folds the conjunction of terms into one closed interval per column (+ up to two != constants) for the
// TMA-staged kernel.  Returns false when the predicate / columns do not fit that kernel.
bool build_tma_args(dfdb_scan *s, const Expr *e, Column *agg_col, TmaScanArgs *a, bool *const_false)
{
    dfdb_table *t = s->tbl;
    a->ncols = 0;
    a->ntests = 0;
    a->agg_col = -1;
    *const_false = false;
    std::vector<Column *> staged;
    auto stage_col = [&](Column *c) -> int {
        for (size_t i = 0; i < staged.size(); i++) if (staged[i] == c) return (int)i;
        if (staged.size() >= (size_t)TMA_MAX_COLS || !wide_ok(t, *c)) return -1;
        staged.push_back(c);
        a->col[staged.size() - 1] = make_view(*c);
        return (int)staged.size() - 1;
    };
    const int nterms = e ? e->nterms : 0;
    for (int i = 0; i < nterms; i++) {
        const Term &tm = e->terms[i];
        if (tm.constant_result == 0) { *const_false = true; continue; }
        if (tm.constant_result == 1) continue;
        Column *c = t->find(s->slots[(size_t)tm.slot]);
        const int ci = stage_col(c);
        if (ci < 0) return false;
        ColTest *ct = nullptr;
        for (int k = 0; k < a->ntests; k++) if (a->test[k].col == ci) ct = &a->test[k];
        if (!ct) {
            ct = &a->test[a->ntests++];
            memset(ct, 0, sizeof *ct);
            ct->col = ci;
            ct->cls = tm.cls;
            ct->nan_passes = tm.cls == VC_FLT;
            if (tm.cls == VC_INT) { ct->lo_i = INT64_MIN; ct->hi_i = INT64_MAX; }
            else if (tm.cls == VC_UINT) { ct->lo_i = 0; ct->hi_i = -1; }
            else { ct->lo_f = -INFINITY; ct->hi_f = INFINITY; }
        }
        if (tm.cls == VC_FLT) {
            const double c0 = tm.cf;
            if (tm.code == 1) {
                if (c0 != c0) continue;                        // x != NaN is always true
                if (ct->n_ne >= 2) return false;
                ct->ne_f[ct->n_ne++] = c0;
                continue;
            }
            ct->nan_passes = 0;
            if (c0 != c0) { *const_false = true; continue; }   // every ordered comparison with NaN is false
            switch (tm.code) {
            case 0: ct->lo_f = std::max(ct->lo_f, c0); ct->hi_f = std::min(ct->hi_f, c0); break;
            case 2: ct->hi_f = std::min(ct->hi_f, std::nextafter(c0, -INFINITY)); if (c0 == -INFINITY) *const_false = true; break;
            case 3: ct->hi_f = std::min(ct->hi_f, c0); break;
            case 4: ct->lo_f = std::max(ct->lo_f, std::nextafter(c0, INFINITY)); if (c0 == INFINITY) *const_false = true; break;
            default: ct->lo_f = std::max(ct->lo_f, c0); break;
            }
            if (ct->lo_f > ct->hi_f) *const_false = true;
        } else if (tm.cls == VC_INT) {
            const int64_t c0 = tm.ci;
            switch (tm.code) {
            case 0: ct->lo_i = std::max<int64_t>(ct->lo_i, c0); ct->hi_i = std::min<int64_t>(ct->hi_i, c0); break;
            case 1: if (ct->n_ne >= 2) return false; ct->ne_i[ct->n_ne++] = c0; break;
            case 2: if (c0 == INT64_MIN) *const_false = true; else ct->hi_i = std::min<int64_t>(ct->hi_i, c0 - 1); break;
            case 3: ct->hi_i = std::min<int64_t>(ct->hi_i, c0); break;
            case 4: if (c0 == INT64_MAX) *const_false = true; else ct->lo_i = std::max<int64_t>(ct->lo_i, c0 + 1); break;
            default: ct->lo_i = std::max<int64_t>(ct->lo_i, c0); break;
            }
            if (ct->lo_i > ct->hi_i) *const_false = true;
        } else {
            const uint64_t c0 = (uint64_t)tm.ci;
            uint64_t lo = (uint64_t)ct->lo_i, hi = (uint64_t)ct->hi_i;
            switch (tm.code) {
            case 0: lo = std::max(lo, c0); hi = std::min(hi, c0); break;
            case 1: if (ct->n_ne >= 2) return false; ct->ne_i[ct->n_ne++] = (int64_t)c0; break;
            case 2: if (c0 == 0) *const_false = true; else hi = std::min(hi, c0 - 1); break;
            case 3: hi = std::min(hi, c0); break;
            case 4: if (c0 == UINT64_MAX) *const_false = true; else lo = std::max(lo, c0 + 1); break;
            default: lo = std::max(lo, c0); break;
            }
            if (lo > hi) *const_false = true;
            ct->lo_i = (int64_t)lo;
            ct->hi_i = (int64_t)hi;
        }
    }
    if (agg_col) {
        a->agg_col = stage_col(agg_col);
        if (a->agg_col < 0) return false;
    }
    if (staged.empty()) return false;
    a->ncols = (int)staged.size();
    a->nstages = std::min(TMA_MAX_STAGES, (96 * 1024) / (a->ncols * TILE_ROWS * 8));   // two CTAs per SM
    return true;
}

bool single_simple_pred(const dfdb_scan *s)
{
    return !rt.no_fused && s->stages.size() == 1 && s->stages[0].kind == ST_PRED && s->stages[0].e.simple;
}

void agg_to_public(const AggPartial &p, int cls, dfdb_agg *out)
{
    memset(out, 0, sizeof *out);
    out->count = p.count;
    out->nmissing = p.nmissing;
    out->sum_i64 = p.sum_i;
    out->sum_f64 = p.sum_f;
    out->sum_f64_lo = p.sum_lo;
    out->min_i64 = p.min_i; out->max_i64 = p.max_i;
    out->min_f64 = p.min_f; out->max_f64 = p.max_f;
    out->has_nan = p.has_nan;
    const bool any = p.has_value || p.has_nan;
    out->value_class = any ? (cls == VC_FLT ? 3 : cls == VC_UINT ? 2 : cls == VC_BOOL ? 4 : 1) : 0;
}

int run_aggregate(dfdb_scan *s, int32_t proj_idx, bool count_only, AggPartial *host_out, int *cls_out)
{
    zone_prune(s);
    const DecodeScope scope = selection_scope(s);
    dfdb_table *t = s->tbl;
    int rc = scan_alloc(s);
    if (rc) return rc;
    Geometry g = make_geometry(t);
    g.dead = zone_dead_dev(s);
    FusedArgs a;
    memset(&a, 0, sizeof a);
    a.g = g;
    a.partials = static_cast<AggPartial *>(s->d_partials);
    int agg = 0, cls = VC_INT;
    bool wide = true;
    std::vector<int64_t> need;
    Column *ac = nullptr;
    if (!count_only) {
        if (proj_idx < 0 || (size_t)proj_idx >= s->projs.size()) return fail(DFDB_ERR_ARGUMENT, "projection index out of range");
        const Proj &p = s->projs[(size_t)proj_idx];
        if (p.kind != PJ_COL) {
            // a computed column: the VM value of every selected row, folded into the same per-unit partials
            cls = p.e.prog.result_class;
            if (cls == VC_NONE || cls == VC_STR) return fail(DFDB_ERR_UNSUPPORTED, "aggregate over a computed String column");
            rc = run_selection(s);
            if (rc) return rc;
            rc = ensure_decoded(t, p.e.col_ids, scope);
            if (rc) return rc;
            AggVmArgs va;
            memset(&va, 0, sizeof va);
            va.g = g;
            rc = fill_slots(s, va.slot);
            if (rc) return rc;
            DevProg prog;
            rc = prog.upload(s, p.e);
            if (rc) return rc;
            va.prog = prog.d;
            va.mask = s->d_mask;
            va.partials = static_cast<AggPartial *>(s->d_partials);
            va.cls = cls;
            va.error_flag = rt.d_error;
            const int nu = g.nblocks * g.segs_per_block;
            {
                int64_t bytes = 0;
                for (int64_t id : p.e.col_ids) for (int64_t b = t->blk_lo; b < t->blk_hi; b++) bytes += t->find(id)->blocks[(size_t)b].origin;
                PhaseScope ps(PH_CONSUME, bytes);
                CUDA_TRY(cudaMemsetAsync(s->d_partials, 0, (size_t)std::max(nu, 1) * sizeof(AggPartial), rt.stream));
                if (nu > 0) LAUNCH(launch_agg_vm(va, rt.sm_count, rt.stream));
                LAUNCH(launch_agg_finalize(static_cast<AggPartial *>(s->d_partials), nu, cls, static_cast<AggPartial *>(s->d_result), rt.stream));
            }
            CUDA_TRY(cudaMemcpyAsync(s->h_result, s->d_result, sizeof(AggPartial), cudaMemcpyDeviceToHost, rt.stream));
            CUDA_TRY(cudaStreamSynchronize(rt.stream));   // (the program buffer is freed on scope exit)
            rc = check_device_error();                    // DivideError etc. raised by the expression
            if (rc) return rc;
            *host_out = *static_cast<AggPartial *>(s->h_result);
            *cls_out = cls;
            return DFDB_OK;
        }
        ac = t->find(p.col);
        cls = value_class(ac->type.kind);
        if (cls == VC_NONE || cls == VC_STR) return fail(DFDB_ERR_UNSUPPORTED, "aggregate over column %s of type %s", ac->name.c_str(), ac->typestr.c_str());
        agg = cls == VC_FLT ? 2 : 1;
        need.push_back(p.col);
        wide = wide && wide_ok(t, *ac);
    }
    const int nunits = g.nblocks * g.segs_per_block;
    int64_t scan_bytes = 0;
    TmaScanArgs ta, tb;   // tb: the mask-in form, when the decoder writes the predicate's bits
    memset(&ta, 0, sizeof ta);
    memset(&tb, 0, sizeof tb);
    BitsReq bits{nullptr, {}, nullptr, 0, false};
    int64_t bits_bytes = 0;   // the mask-in scan's bytes: the aggregated column + the mask
    bool use_tma = false, scanned = false, finalized = false;
    // the TMA scan of local blocks [b0, b1) on `sms` SMs (partials are per work unit, so parts compose)
    auto scan_part = [&](int b0, int b1, int sms) -> int {
        if (!use_tma || b1 <= b0) return DFDB_OK;
        if (!scanned) {
            // work units that hold no rows (segments past the end of a partial last block) are never visited
            CUDA_TRY(cudaMemsetAsync(s->d_partials, 0, (size_t)std::max(nunits, 1) * sizeof(AggPartial), rt.stream));
            scanned = true;
        }
        TmaScanArgs part = bits.on ? tb : ta;
        if (part.mask_in) part.mask_in += (int64_t)b0 * g.wpb;
        part.g.blk_lo = g.blk_lo + b0;
        part.g.nblocks = b1 - b0;
        for (int c = 0; c < part.ncols; c++) part.col[c].blk_off += b0;
        part.partials = static_cast<AggPartial *>(s->d_partials) + (int64_t)b0 * g.segs_per_block;
        {
            PhaseScope ps(PH_CONSUME, (bits.on ? bits_bytes : scan_bytes) * (b1 - b0) / std::max(g.nblocks, 1));
            LAUNCH(launch_fused_tma(part, agg, sms, rt.stream));
        }
        if (b1 == g.nblocks && !finalized) {
            // the last part: the fold of the partials and the copy of the result follow at once, so that they run (and are
            // covered by the synchronisation of the integrity gate in ensure_decoded) instead of waiting for a host round trip
            {
                PhaseScope ps(PH_CONSUME, 0);
                LAUNCH(launch_agg_finalize(static_cast<AggPartial *>(s->d_partials), nunits, agg == 2 ? VC_FLT : cls, static_cast<AggPartial *>(s->d_result), rt.stream));
            }
            PhaseScope ps(PH_D2H, sizeof(AggPartial));
            CUDA_TRY(cudaMemcpyAsync(s->h_result, s->d_result, sizeof(AggPartial), cudaMemcpyDeviceToHost, rt.stream));
            finalized = true;
        }
        return DFDB_OK;
    };
    const PartFn part_fn = scan_part;
    if (s->stages.empty() || single_simple_pred(s)) {
        if (!s->stages.empty()) for (int64_t id : s->stages[0].e.col_ids) need.push_back(id);
        for (int64_t id : need) {
            Column *c = t->find(id);
            if (!c) return fail(DFDB_ERR_KEY, "unknown column id %lld", (long long)id);
            for (int64_t b = t->blk_lo; b < t->blk_hi; b++) scan_bytes += c->blocks[(size_t)b].origin;
        }
        if (!s->stages.empty()) {
            fill_terms(s, s->stages[0].e, &a);
            wide = wide && fused_terms_wide(s, s->stages[0].e);
        }
        // the fast path is set up before the decode so that it can start on the part of the shard that is decoded
        bool cfalse = false;
        bool loaded = true;
        for (int64_t id : need) loaded = loaded && t->find(id)->loaded;
        use_tma = loaded && wide && !rt.no_tma && nunits > 0 &&
                  build_tma_args(s, s->stages.empty() ? nullptr : &s->stages[0].e, ac, &ta, &cfalse) && !cfalse;
        if (use_tma) {
            ta.g = g;
            ta.agg_cls = cls;
        }
        // The predicate's one column, decoded here, can have its decoder write the selection bits; the scan then stages only
        // the aggregated column (half the bytes of the benchmark's scan).  The bits overwrite the handle's selection mask.
        BitsReq *want = nullptr;
        if (use_tma && ac && ta.ntests == 1 && ta.test[0].col != ta.agg_col && rt.pred_bits != 2 && g.wpb % 4 == 0) {
            const Expr &e = s->stages[0].e;
            Column *pc = nullptr;
            for (int i = 0; i < e.nterms && !pc; i++) if (e.terms[i].constant_result < 0) pc = t->find(s->slots[(size_t)e.terms[i].slot]);
            bool ok = pc && !pc->type.nullable && pc->type.elsize == 8 && pc->mode != DFDB_LOAD_DECODED;
            for (int64_t b = t->blk_lo; ok && b < t->blk_hi; b++) ok = pc->blocks[(size_t)b].origin == block_rows(g, (int)(b - t->blk_lo)) * 8;
            if (ok) {
                tb = ta;
                tb.ncols = 1;
                tb.col[0] = ta.col[ta.agg_col];
                tb.agg_col = 0;
                tb.ntests = 0;
                tb.nstages = TMA_MASK_STAGES;
                tb.mask_in = s->d_mask;
                bits = BitsReq{pc, ta.test[0], s->d_mask, g.wpb, false};
                bits.test.col = 0;
                want = &bits;
                for (int64_t b = t->blk_lo; b < t->blk_hi; b++) bits_bytes += ac->blocks[(size_t)b].origin;
                bits_bytes += (int64_t)g.nblocks * g.wpb * 4;
            }
        }
        rc = ensure_decoded(t, need, scope, use_tma ? &part_fn : nullptr, want);
        if (rc) return rc;
        if (bits.on) s->mask_valid = false;
    } else {
        rc = run_selection(s);
        if (rc) return rc;
        rc = ensure_decoded(t, need, scope);
        if (rc) return rc;
        for (int64_t id : need) for (int64_t b = t->blk_lo; b < t->blk_hi; b++) scan_bytes += t->find(id)->blocks[(size_t)b].origin;
        a.mask_in = s->d_mask;
        wide = false;
    }
    if (ac) { a.agg_col = make_view(*ac); a.agg_cls = cls; }
    {
        if (use_tma) {
            if (!scanned) { rc = scan_part(0, g.nblocks, rt.sm_count); if (rc) return rc; }   // everything was decoded already
        } else if (nunits > 0) {
            PhaseScope ps(PH_CONSUME, scan_bytes);
            LAUNCH(launch_fused(a, agg, false, wide, rt.sm_count, rt.stream));
        }
        if (!finalized) {
            PhaseScope ps(PH_CONSUME, 0);
            LAUNCH(launch_agg_finalize(static_cast<AggPartial *>(s->d_partials), nunits, agg == 2 ? VC_FLT : cls, static_cast<AggPartial *>(s->d_result), rt.stream));
        }
    }
    if (!finalized) {
        PhaseScope ps(PH_D2H, sizeof(AggPartial));
        CUDA_TRY(cudaMemcpyAsync(s->h_result, s->d_result, sizeof(AggPartial), cudaMemcpyDeviceToHost, rt.stream));
    }
    CUDA_TRY(cudaStreamSynchronize(rt.stream));
    *host_out = *static_cast<AggPartial *>(s->h_result);
    *cls_out = cls;
    return DFDB_OK;
}

// ---- result columns: the gather of a row set and the copy to the caller ------------------------------------------------
// a set of rows of the shard: a mask laid out like the selection mask, the exclusive scan of its per-block counts (the total
// at [nblocks]), and 2 * (nblocks + 1) words of String scratch: per-block char bytes | their exclusive scan
struct RowSet {
    const uint32_t *mask;
    const int64_t *blk_base;
    int64_t *blk_bytes;
};

RowSet selection_rows(const dfdb_scan *s) { return RowSet{s->d_mask, s->d_blk_base, s->d_blk_bytes}; }

GatherArgs gather_args(const Geometry &g, const RowSet &rows, const Column &c)
{
    GatherArgs a;
    memset(&a, 0, sizeof a);
    a.g = g;
    a.mask = rows.mask;
    a.blk_base = rows.blk_base;
    a.col = make_view(c);
    return a;
}

// the chars of String column c at `rows`: per-block bytes and their exclusive scan, the bases of gather_rows
int char_bases(const Geometry &g, const RowSet &rows, const Column &c)
{
    LAUNCH(launch_str_block_bytes(gather_args(g, rows, c), rows.blk_bytes, rt.stream));
    LAUNCH(launch_exclusive_scan(rows.blk_bytes, rows.blk_bytes + g.nblocks + 1, g.nblocks, rt.stream));
    return DFDB_OK;
}

// char_bases, and their total to *h (pinned host memory) once the stream gets there
int selected_chars(const Geometry &g, const RowSet &rows, const Column &c, int64_t *h)
{
    const int rc = char_bases(g, rows, c);
    if (rc) return rc;
    CUDA_TRY(cudaMemcpyAsync(h, rows.blk_bytes + g.nblocks + 1 + g.nblocks, 8, cudaMemcpyDeviceToHost, rt.stream));
    return DFDB_OK;
}

// The values of column c at `rows`, in row order, into r (of c's type, allocated for them).  A String column takes the char
// bases that char_bases left in rows.blk_bytes.
int gather_rows(const Geometry &g, const RowSet &rows, const Column &c, ResultCol &r)
{
    GatherArgs a = gather_args(g, rows, c);
    if (r.kind == DFDB_STRING) {
        a.blk_char_base = rows.blk_bytes + g.nblocks + 1;
        a.out_sizes = r.sizes.as<int32_t>();
        a.out_chars = r.chars.as<uint8_t>();
        LAUNCH(launch_gather_strings(a, rt.stream));
    } else {
        a.out_values = r.values.as<uint8_t>();
        a.out_missing = r.missing.as<uint8_t>();
        LAUNCH(launch_gather_fixed(a, rt.stream));
    }
    return DFDB_OK;
}

// Result column r -> the caller's buffers `out`, which must be the ones its type needs (a missing mask is optional).  Each
// array goes by copy_out_queued's rule: into the result arena on the copy stream, anything else before this returns.
// *queued: some array went to the copy stream -- r's buffers are then freed there, and the copy stream is drained before the
// entry point returns.  d2h_bytes >= 0: the copy is profiled as a D2H phase of that many bytes.
int result_copy_out(const ResultCol &r, const dfdb_outcol &out, const char *what, int64_t d2h_bytes, bool *queued)
{
    *queued = false;
    if (r.n == 0) return DFDB_OK;
    const bool str = r.kind == DFDB_STRING;
    if (str ? !out.str_sizes || (r.bytes > 0 && !out.str_chars) : !out.values)
        return fail(DFDB_ERR_ARGUMENT, "%s lacks a buffer its type needs (String: str_sizes and str_chars, else values)", what);
    struct Part { void *dst; const void *src; size_t len; };
    const Part parts[2] = {str ? Part{out.str_sizes, r.sizes.p, (size_t)r.n * 4} : Part{out.values, r.values.p, (size_t)r.n * r.elsize},
                           str ? Part{out.str_chars, r.chars.p, (size_t)r.bytes} : Part{r.nullable ? out.missing : nullptr, r.missing.p, (size_t)r.n}};
    std::optional<PhaseScope> ps;
    if (d2h_bytes >= 0) ps.emplace(PH_D2H, d2h_bytes, arena.pinned(parts[0].dst, parts[0].len) ? rt.copy_stream : rt.stream);
    for (const Part &a : parts) {
        if (!a.dst || a.len == 0) continue;
        cudaError_t e;
        if (copy_out_queued(a.dst, a.src, a.len, &e)) *queued = true;
        if (e != cudaSuccess) return fail(DFDB_ERR_CUDA, "%s copy failed: %s", what, cudaGetErrorString(e));
    }
    return DFDB_OK;
}

// the end of the copies to the caller: the copy stream drained, then the scan stream; rc, the status so far, wins
int copies_done(int rc)
{
    cudaError_t e = cudaStreamSynchronize(rt.copy_stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(rt.stream);
    if (rc) return rc;
    if (e != cudaSuccess) return fail(DFDB_ERR_CUDA, "result copy failed: %s", cudaGetErrorString(e));
    return DFDB_OK;
}

}  // namespace

namespace dfdb {
RuntimeView runtime_view() { return RuntimeView{rt.stream, rt.d_counter + 8, rt.sm_count, rt.inited}; }
void runtime_count_launch() { rt.launches++; }
}  // namespace dfdb

// =================================================================================================
// C ABI
// =================================================================================================
extern "C" {

const char *dfdb_last_error(void) { return dfdb::last_error(); }

int32_t dfdb_init(int32_t device)
{
    if (rt.inited) {
        if (device != rt.device) return fail(DFDB_ERR_STATE, "already initialised on device %d (one process per GPU)", rt.device);
        return DFDB_OK;
    }
    if (const char *fl = getenv("DFDB_LZ4_FLAVOUR"))   // A/B: force one K1 decoder (see dfdb_set_option "lz4_flavour")
        if (const int rc = set_lz4_flavour(atoll(fl))) return rc;
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n == 0) return fail(DFDB_ERR_CUDA, "no CUDA device available: %s", cudaGetErrorString(e));
    if (device < 0 || device >= n) return fail(DFDB_ERR_CUDA, "device %d out of range (%d devices)", device, n);
    CUDA_TRY(cudaSetDevice(device));
    cudaDeviceProp prop;
    CUDA_TRY(cudaGetDeviceProperties(&prop, device));
    if (prop.major < 10) return fail(DFDB_ERR_CUDA, "device %s is sm_%d%d; this library is built for sm_100a only", prop.name, prop.major, prop.minor);
    rt.device = device;
    rt.sm_count = prop.multiProcessorCount;
    // One process per GPU: keep this process's host memory -- above all the pinned staging of the transfer-inclusive mode -- on
    // the NUMA node the GPU hangs off, so that H2D copies do not cross the socket interconnect (measured at 4 and 8 ranks per
    // box: the per-GPU H2D rate halves when every rank's staging sits on one node).  MPOL_PREFERRED: falls back to other nodes
    // when the local one is full.  DFDB_NO_NUMA=1 turns it off.
    rt.numa_node = -1;
    if (!getenv("DFDB_NO_NUMA")) {
        char bus[32] = {0};
        if (cudaDeviceGetPCIBusId(bus, sizeof bus, device) == cudaSuccess) {
            for (char *c = bus; *c; c++) *c = (char)tolower(*c);
            const std::string f = std::string("/sys/bus/pci/devices/") + bus + "/numa_node";
            if (FILE *fp = fopen(f.c_str(), "r")) {
                int node = -1;
                if (fscanf(fp, "%d", &node) == 1 && node >= 0 && node < 64) {
                    unsigned long mask = 1ul << node;
#ifdef SYS_set_mempolicy
                    if (syscall(SYS_set_mempolicy, 1 /* MPOL_PREFERRED */, &mask, 65ul) == 0) rt.numa_node = node;
#endif
                }
                fclose(fp);
            }
        }
    }
    CUDA_TRY(cudaStreamCreateWithFlags(&rt.own_stream, cudaStreamNonBlocking));
    rt.stream = rt.own_stream;
    CUDA_TRY(cudaStreamCreateWithFlags(&rt.copy_stream, cudaStreamNonBlocking));
    {
        int least = 0, greatest = 0;
        CUDA_TRY(cudaDeviceGetStreamPriorityRange(&least, &greatest));
        CUDA_TRY(cudaStreamCreateWithPriority(&rt.decode_stream, cudaStreamNonBlocking, greatest));
        CUDA_TRY(cudaStreamCreateWithPriority(&rt.decode_stream2, cudaStreamNonBlocking, greatest < least - 1 ? greatest + 1 : greatest));
    }
    CUDA_TRY(cudaMalloc(reinterpret_cast<void **>(&rt.d_counter), 64));
    CUDA_TRY(cudaMalloc(reinterpret_cast<void **>(&rt.d_error), 64));
    CUDA_TRY(cudaMemset(rt.d_error, 0, 64));
    if (const char *ov = getenv("DFDB_NO_OVERLAP")) rt.no_overlap = atoll(ov);       // A/B: decode / scan overlap off
    rt.inited = true;
    return DFDB_OK;
}

int32_t dfdb_shutdown(void)
{
    if (!rt.inited) return DFDB_OK;
    cudaStreamSynchronize(rt.stream);
    dfdb_comm_destroy();
    profile_collect();
    cudaFree(rt.d_counter);
    cudaFree(rt.d_error);
    { std::lock_guard<std::mutex> lk(arena.mu); arena.trim(0); }
    cudaStreamDestroy(rt.own_stream);
    cudaStreamDestroy(rt.copy_stream);
    cudaStreamDestroy(rt.decode_stream);
    cudaStreamDestroy(rt.decode_stream2);
    rt.inited = false;
    return DFDB_OK;
}

int32_t dfdb_set_stream(void *cuda_stream)
{
    int rc = need_init();
    if (rc) return rc;
    cudaStreamSynchronize(rt.stream);
    rt.stream = cuda_stream ? static_cast<cudaStream_t>(cuda_stream) : rt.own_stream;
    return DFDB_OK;
}

int32_t dfdb_synchronize(void)
{
    int rc = need_init();
    if (rc) return rc;
    CUDA_TRY(cudaStreamSynchronize(rt.stream));
    return DFDB_OK;
}

int64_t dfdb_kernel_launches(void) { return rt.launches.load(); }
int32_t dfdb_numa_node(void) { return rt.numa_node; }

int32_t dfdb_set_option(const char *name, int64_t value)
{
    std::string n(name ? name : "");
    if (n == "lz4_simple") rt.lz4_simple = value;
    else if (n == "no_wide") rt.no_wide = value;
    else if (n == "no_fused") rt.no_fused = value;
    else if (n == "no_tma") rt.no_tma = value;
    else if (n == "pred_bits") rt.pred_bits = value;
    else if (n == "lz4_flavour") return set_lz4_flavour(value);
    else if (n == "no_overlap") rt.no_overlap = value;
    else if (n == "no_alias") rt.no_alias = value;
    else if (n == "lane_hot") rt.lane_hot = value;
    else if (n == "no_zonemap") rt.no_zonemap = value;
    else if (n == "host_arena_cap_mb") { std::lock_guard<std::mutex> lk(arena.mu); arena.cap_bytes = (size_t)std::max<int64_t>(value, 0) << 20; arena.trim(arena.cap_bytes); }
    else return fail(DFDB_ERR_ARGUMENT, "unknown option %s", n.c_str());
    return DFDB_OK;
}

int32_t dfdb_profile_enable(int32_t on) { rt.profiling = on != 0; return DFDB_OK; }
int32_t dfdb_profile_reset(void)
{
    if (rt.inited) { cudaStreamSynchronize(rt.stream); profile_collect(); }
    for (int i = 0; i < PH_COUNT; i++) { rt.acc_ms[i] = 0; rt.acc_launches[i] = 0; rt.acc_bytes[i] = 0; }
    for (int64_t &n : rt.k1_launches) n = 0;
    for (int64_t &n : rt.k1_bytes) n = 0;
    return DFDB_OK;
}
int32_t dfdb_profile_get(const char *phase, double *total_ms, int64_t *launches, int64_t *bytes)
{
    if (rt.inited) profile_collect();
    for (int i = 0; i < PH_COUNT; i++)
        if (strcmp(phase, k_phases[i]) == 0) {
            if (total_ms) *total_ms = rt.acc_ms[i];
            if (launches) *launches = rt.acc_launches[i];
            if (bytes) *bytes = rt.acc_bytes[i];
            return DFDB_OK;
        }
    // decode launches and bytes per K1 decoder since the last reset, by the names in k1_kernels
    for (int i = 0; i < K1_COUNT; i++)
        if (strcmp(phase, k1_kernels[i].name) == 0) {
            if (total_ms) *total_ms = 0;
            if (launches) *launches = rt.k1_launches[i];
            if (bytes) *bytes = rt.k1_bytes[i];
            return DFDB_OK;
        }
    return fail(DFDB_ERR_ARGUMENT, "unknown phase %s", phase);
}

// ---- table ------------------------------------------------------------------------------------------
int32_t dfdb_table_open(const char *path, dfdb_table **out)
{
    if (!path || !out) return fail(DFDB_ERR_ARGUMENT, "null argument");
    return table_open_host(path, out);
}

int32_t dfdb_table_close(dfdb_table *t)
{
    if (!t) return DFDB_OK;
    if (rt.inited) cudaStreamSynchronize(rt.stream);
    for (auto &c : t->cols) column_release(c);
    delete t;
    return DFDB_OK;
}

int64_t dfdb_table_nrows(const dfdb_table *t) { return t->nrows; }
int64_t dfdb_table_ncols(const dfdb_table *t) { return (int64_t)t->cols.size(); }
int64_t dfdb_table_block_size(const dfdb_table *t) { return t->block_size; }
int64_t dfdb_table_nblocks(const dfdb_table *t) { return t->nblocks; }

int32_t dfdb_table_column(const dfdb_table *t, int32_t index, int64_t *id, char *name, int32_t name_cap, char *typestring,
                          int32_t ts_cap, int32_t *kind, int32_t *nullable, int32_t *elsize)
{
    if (index < 0 || (size_t)index >= t->cols.size()) return fail(DFDB_ERR_KEY, "column index %d out of range", index);
    const Column &c = t->cols[(size_t)index];
    if (id) *id = c.id;
    if (name && name_cap > 0) snprintf(name, (size_t)name_cap, "%s", c.name.c_str());
    if (typestring && ts_cap > 0) snprintf(typestring, (size_t)ts_cap, "%s", c.typestr.c_str());
    if (kind) *kind = c.type.kind;
    if (nullable) *nullable = c.type.nullable;
    if (elsize) *elsize = c.type.elsize;
    return DFDB_OK;
}

int32_t dfdb_table_column_stats(const dfdb_table *t, int64_t col_id, int64_t *compressed, int64_t *uncompressed)
{
    const Column *c = const_cast<dfdb_table *>(t)->find(col_id);
    if (!c) return fail(DFDB_ERR_KEY, "unknown column id %lld", (long long)col_id);
    int64_t cs = 0, us = 0;
    for (int64_t b = t->blk_lo; b < t->blk_hi; b++) { cs += c->blocks[(size_t)b].compressed; us += c->blocks[(size_t)b].origin; }
    if (compressed) *compressed = cs;
    if (uncompressed) *uncompressed = us;
    return DFDB_OK;
}

int32_t dfdb_table_column_stored(const dfdb_table *t, int64_t col_id, int64_t *blocks, int64_t *bytes)
{
    const Column *c = const_cast<dfdb_table *>(t)->find(col_id);
    if (!c) return fail(DFDB_ERR_KEY, "unknown column id %lld", (long long)col_id);
    int64_t nb = 0, by = 0;
    for (size_t b = 0; b < c->h_skip.size(); b++)
        if (c->h_skip[b]) { nb++; by += c->blocks[(size_t)t->blk_lo + b].origin; }
    if (blocks) *blocks = nb;
    if (bytes) *bytes = by;
    return DFDB_OK;
}

int32_t dfdb_table_set_shard(dfdb_table *t, int32_t rank, int32_t world)
{
    if (world < 1 || rank < 0 || rank >= world) return fail(DFDB_ERR_ARGUMENT, "bad shard %d of %d", rank, world);
    for (auto &c : t->cols) if (c.loaded) column_release(c);
    t->rank = rank;
    t->world = world;
    t->epoch++;                        // masks, survivor counts and filtered decodes of the old shard are stale
    t->blk_lo = t->nblocks * rank / world;
    t->blk_hi = t->nblocks * (rank + 1) / world;
    return DFDB_OK;
}

int32_t dfdb_table_shard_range(const dfdb_table *t, int64_t *block_lo, int64_t *block_hi, int64_t *row_lo, int64_t *row_hi)
{
    if (block_lo) *block_lo = t->blk_lo;
    if (block_hi) *block_hi = t->blk_hi;
    if (row_lo) *row_lo = std::min(t->nrows, t->blk_lo * t->block_size);
    if (row_hi) *row_hi = std::min(t->nrows, t->blk_hi * t->block_size);
    return DFDB_OK;
}

int32_t dfdb_table_load(dfdb_table *t, const int64_t *col_ids, int32_t n, int32_t mode)
{
    int rc = need_init();
    if (rc) return rc;
    if (mode < DFDB_LOAD_HOST || mode > DFDB_LOAD_DECODED) return fail(DFDB_ERR_ARGUMENT, "bad residency mode %d", mode);
    std::vector<Column *> cols;
    if (n <= 0) for (auto &c : t->cols) cols.push_back(&c);
    else
        for (int i = 0; i < n; i++) {
            Column *c = t->find(col_ids[i]);
            if (!c) return fail(DFDB_ERR_KEY, "unknown column id %lld", (long long)col_ids[i]);
            cols.push_back(c);
        }
    const int64_t nb = t->blk_hi - t->blk_lo;
    for (Column *c : cols) {
        if (c->loaded && c->mode == mode) continue;
        column_release(*c);
        std::vector<int64_t> comp_off((size_t)nb), dec_off((size_t)nb), lit_start((size_t)nb, 0);
        std::vector<int32_t> comp_len((size_t)nb), origin((size_t)nb);
        std::vector<uint8_t> stored((size_t)nb, 0);
        int64_t cpos = 0, dpos = 0;
        const std::string colfile = t->path + "/" + std::to_string(c->id) + ".bin";
        int fd = open(colfile.c_str(), O_RDONLY);
        if (fd < 0) return fail(DFDB_ERR_IO, "cannot open %s", colfile.c_str());
        std::vector<uint8_t> head;
        c->stored_blocks = 0;
        for (int64_t b = 0; b < nb; b++) {
            const BlockInfo &bi = c->blocks[(size_t)(t->blk_lo + b)];
            if (c->type.kind == DFDB_STRING && bi.origin < 4 + 4 * (int64_t)bi.rows) {
                close(fd);
                return fail(DFDB_ERR_CORRUPT, "column %s block %lld: string body smaller than its size table", c->name.c_str(), (long long)(t->blk_lo + b));
            }
            if (c->type.kind != DFDB_STRING) {
                int64_t expect = (int64_t)bi.rows * c->type.elsize + (c->type.nullable ? ((bi.rows + 63) / 64) * 8 : 0);
                if (bi.origin != expect) {
                    close(fd);
                    return fail(DFDB_ERR_CORRUPT, "column %s block %lld: body is %lld bytes, expected %lld", c->name.c_str(),
                                (long long)(t->blk_lo + b), (long long)bi.origin, (long long)expect);
                }
            }
            // A stored block -- what LZ4 emits for incompressible data -- is one literal run: token 0xF?, the length
            // extension bytes, then the body itself.  Its body is referenced in place (no copy); the payload is
            // placed so that the body starts on a 256-byte boundary like every decoded slot.
            if (!rt.no_alias && bi.origin >= 15) {
                const int64_t q = (bi.origin - 15) / 255, r = (bi.origin - 15) % 255, ls = 1 + q + 1;
                if (bi.compressed == ls + bi.origin) {
                    head.resize((size_t)ls);
                    bool ok = pread(fd, head.data(), (size_t)ls, bi.file_off) == (ssize_t)ls && (head[0] >> 4) == 15 && head[(size_t)ls - 1] == (uint8_t)r;
                    for (int64_t i = 1; ok && i <= q; i++) ok = head[(size_t)i] == 255;
                    if (ok) { stored[(size_t)b] = 1; lit_start[(size_t)b] = ls; c->stored_blocks++; }
                }
            }
            if (stored[(size_t)b]) {
                // the payload of a stored block is never parsed on the device, so only its body needs alignment
                const int64_t ls = lit_start[(size_t)b];
                cpos = ((cpos + ls + 255) & ~(int64_t)255) - ls;
            }
            comp_off[(size_t)b] = cpos;
            comp_len[(size_t)b] = (int32_t)bi.compressed;
            cpos = (cpos + bi.compressed + 15) & ~(int64_t)15;
            origin[(size_t)b] = (int32_t)bi.origin;
            if (!stored[(size_t)b]) {
                dec_off[(size_t)b] = dpos;
                dpos += (bi.origin + 255) & ~(int64_t)255;
            }
        }
        c->comp_bytes = (size_t)cpos + 4096;       // slack for the decoder's aligned window over-read
        c->decoded_bytes = (size_t)dpos + 256;
        c->h_comp_off = comp_off;
        CUDA_TRY(cudaMallocHost(reinterpret_cast<void **>(&c->h_comp), c->comp_bytes));
        memset(c->h_comp + cpos, 0, 4096);
        int64_t prev_end = 0;
        for (int64_t b = 0; b < nb; b++) {
            const BlockInfo &bi = c->blocks[(size_t)(t->blk_lo + b)];
            if (comp_off[(size_t)b] > prev_end) memset(c->h_comp + prev_end, 0, (size_t)(comp_off[(size_t)b] - prev_end));   // alignment gap
            prev_end = comp_off[(size_t)b] + bi.compressed;
            int64_t got = 0;
            while (got < bi.compressed) {
                ssize_t r = pread(fd, c->h_comp + comp_off[(size_t)b] + got, (size_t)(bi.compressed - got), bi.file_off + got);
                if (r <= 0) { close(fd); return fail(DFDB_ERR_IO, "short read in %s", colfile.c_str()); }
                got += r;
            }
        }
        close(fd);
        if (cpos > prev_end) memset(c->h_comp + prev_end, 0, (size_t)(cpos - prev_end));
        c->decoder = column_decoder(*c, comp_off, comp_len, origin, stored);
        CUDA_TRY(cudaMalloc(reinterpret_cast<void **>(&c->d_comp), c->comp_bytes));
        if ((rc = dev_upload(&c->d_comp_off, comp_off))) return rc;
        if ((rc = dev_upload(&c->d_comp_len, comp_len))) return rc;
        if ((rc = dev_upload(&c->d_origin, origin))) return rc;
        if ((rc = dev_upload(&c->d_skip, stored))) return rc;
        c->h_skip = stored;
        CUDA_TRY(cudaMalloc(reinterpret_cast<void **>(&c->d_status), (size_t)std::max<int64_t>(nb, 1) * 4));
        CUDA_TRY(cudaMemset(c->d_status, 0, (size_t)std::max<int64_t>(nb, 1) * 4));
        CUDA_TRY(cudaMalloc(reinterpret_cast<void **>(&c->d_decoded), c->decoded_bytes));
        // body offsets are relative to d_decoded; a stored block's body lives inside the compressed buffer
        for (int64_t b = 0; b < nb; b++)
            if (stored[(size_t)b]) dec_off[(size_t)b] = (int64_t)((c->d_comp + comp_off[(size_t)b] + lit_start[(size_t)b]) - c->d_decoded);
        c->h_dec_off = dec_off;
        if ((rc = dev_upload(&c->d_dec_off, dec_off))) return rc;
        if (c->type.kind == DFDB_STRING)
            CUDA_TRY(cudaMalloc(reinterpret_cast<void **>(&c->d_str_off), (size_t)std::max<int64_t>(nb, 1) * (size_t)t->block_size * 4));
        CUDA_TRY(cudaMemcpy(c->d_comp, c->h_comp, c->comp_bytes, cudaMemcpyHostToDevice));
        // Acceptance.  The reference asserts the result of LZ4_decompress_safe for every block it reads (BlockStreams.jl:110-112);
        // the walker / consumer decoders are memory-safe but do not enforce liblz4's end-of-block rules, so the verdict for every
        // block is taken once, here, from the lane-per-block decoder (lz4_decode_lane.cu), which implements those rules exactly
        // (tests: identical accept / reject with the CPU codec on fuzzed streams).  Scans consult it in their integrity gate.
        c->h_corrupt.clear();
        if (nb > 0) {
            DecodeArgs va;
            memset(&va, 0, sizeof va);
            va.ncols = 1;
            va.nblocks = (int)nb;
            va.hot = c->decoder == K1::Spec ? 1 : 0;
            va.col[0] = DecodeCol{c->d_comp, c->d_comp_off, c->d_comp_len, c->d_dec_off, c->d_origin, c->d_decoded, c->d_status, c->d_skip};
            LAUNCH(launch_lz4_decode_lane(va, rt.d_counter, rt.sm_count, rt.stream));
            c->h_corrupt.assign((size_t)nb, 0);
            CUDA_TRY(cudaMemcpyAsync(c->h_corrupt.data(), c->d_status, (size_t)nb * 4, cudaMemcpyDeviceToHost, rt.stream));
            CUDA_TRY(cudaMemsetAsync(c->d_status, 0, (size_t)nb * 4, rt.stream));
            CUDA_TRY(cudaStreamSynchronize(rt.stream));
            // (blocks beyond the lane decoder's 32 MB position range are not judged here; the walker decoders' own checks apply)
            for (int64_t b = 0; b < nb; b++)
                if (origin[(size_t)b] >= (1 << 25) || comp_len[(size_t)b] >= (1 << 25)) c->h_corrupt[(size_t)b] = 0;
        }
        if (mode != DFDB_LOAD_HOST) {
            cudaFreeHost(c->h_comp);
            c->h_comp = nullptr;
        }
        c->mode = mode;
        c->loaded = true;
        c->decoded_valid = false;
        c->dec_lo = c->dec_hi = 0;
        c->dec_live_gen = 0;
    }
    return DFDB_OK;
}

int32_t dfdb_table_drop_decoded(dfdb_table *t)
{
    for (auto &c : t->cols) { c.decoded_valid = false; c.dec_lo = c.dec_hi = 0; c.dec_live_gen = 0; }
    return DFDB_OK;
}

// ---- zone maps ------------------------------------------------------------------------------------------
int32_t dfdb_table_build_zonemaps(dfdb_table *t, const int64_t *col_ids, int32_t n)
{
    int rc = need_init();
    if (rc) return rc;
    if (!t) return fail(DFDB_ERR_ARGUMENT, "null argument");
    if (t->world != 1) return fail(DFDB_ERR_STATE, "zone maps are built on the unsharded table (the sidecar covers every block)");
    std::vector<Column *> cols;
    if (n <= 0) {
        for (auto &c : t->cols) {
            const int cls = value_class(c.type.kind);
            if (c.type.elsize > 0 && c.type.elsize <= 8 && (cls == VC_INT || cls == VC_UINT || cls == VC_FLT || cls == VC_BOOL)) cols.push_back(&c);
        }
    } else {
        for (int i = 0; i < n; i++) {
            Column *c = t->find(col_ids[i]);
            if (!c) return fail(DFDB_ERR_KEY, "unknown column id %lld", (long long)col_ids[i]);
            const int cls = value_class(c->type.kind);
            if (!(c->type.elsize > 0 && c->type.elsize <= 8 && (cls == VC_INT || cls == VC_UINT || cls == VC_FLT || cls == VC_BOOL)))
                return fail(DFDB_ERR_UNSUPPORTED, "zone maps need a fixed-width numeric column; %s is %s", c->name.c_str(), c->typestr.c_str());
            cols.push_back(c);
        }
    }
    const Geometry g = make_geometry(t);
    const int nb = g.nblocks;
    ZoneOut *d_out = nullptr;
    if (nb > 0) CUDA_TRY(cudaMalloc(reinterpret_cast<void **>(&d_out), (size_t)nb * sizeof(ZoneOut)));
    std::vector<ZoneOut> h((size_t)nb);
    for (Column *c : cols) {
        if (!c->loaded) { int64_t id = c->id; rc = dfdb_table_load(t, &id, 1, DFDB_LOAD_HBM); if (rc) { cudaFree(d_out); return rc; } }
        invalidate_decoded(t);
        rc = ensure_decoded(t, {c->id}, whole_table(t));
        if (rc) { cudaFree(d_out); return rc; }
        if (nb > 0) {
            if (launch_zone_map(g, make_view(*c), d_out, rt.stream) != 0) { cudaFree(d_out); return fail(DFDB_ERR_CUDA, "zone map launch failed"); }
            rt.launches++;
            cudaMemcpyAsync(h.data(), d_out, (size_t)nb * sizeof(ZoneOut), cudaMemcpyDeviceToHost, rt.stream);
            if (cudaStreamSynchronize(rt.stream) != cudaSuccess) { cudaFree(d_out); return fail(DFDB_ERR_CUDA, "zone map kernel failed"); }
        }
        c->zones.assign((size_t)nb, ZoneEntry());
        for (int b = 0; b < nb; b++) {
            c->zones[(size_t)b].min_bits = h[(size_t)b].min_bits; c->zones[(size_t)b].max_bits = h[(size_t)b].max_bits;
            c->zones[(size_t)b].null_count = h[(size_t)b].null_count; c->zones[(size_t)b].flags = h[(size_t)b].flags;
        }
        rc = zonemap_write(t, *c);
        if (rc) { cudaFree(d_out); return rc; }
    }
    cudaFree(d_out);
    return DFDB_OK;
}

int32_t dfdb_table_zonemap(const dfdb_table *t, int64_t col_id, int64_t block, dfdb_zone *out)
{
    const Column *c = const_cast<dfdb_table *>(t)->find(col_id);
    if (!c || !out) return fail(DFDB_ERR_KEY, "unknown column id %lld", (long long)col_id);
    if (c->zones.size() != c->blocks.size()) return fail(DFDB_ERR_STATE, "column %s has no zone map (dfdb_table_build_zonemaps)", c->name.c_str());
    if (block < 0 || (size_t)block >= c->zones.size()) return fail(DFDB_ERR_ARGUMENT, "block %lld out of range", (long long)block);
    const ZoneEntry &z = c->zones[(size_t)block];
    memset(out, 0, sizeof *out);
    out->rows = c->blocks[(size_t)block].rows;
    out->null_count = z.null_count;
    out->has_value = z.flags & 1;
    out->has_nan = (z.flags >> 1) & 1;
    if (value_class(c->type.kind) == VC_FLT) { memcpy(&out->min_f64, &z.min_bits, 8); memcpy(&out->max_f64, &z.max_bits, 8); }
    else { out->min_i64 = (int64_t)z.min_bits; out->max_i64 = (int64_t)z.max_bits; }
    return DFDB_OK;
}

int32_t dfdb_scan_pruned(const dfdb_scan *s, int64_t *pruned, int64_t *blocks)
{
    if (!s) return fail(DFDB_ERR_ARGUMENT, "null argument");
    if (pruned) *pruned = s->zone_pruned;
    if (blocks) *blocks = s->tbl->blk_hi - s->tbl->blk_lo;
    return DFDB_OK;
}

// ---- scan ---------------------------------------------------------------------------------------------
int32_t dfdb_scan_prepare(dfdb_table *t, const uint8_t *plan, int64_t plan_len, dfdb_scan **out)
{
    if (!t || !plan || !out) return fail(DFDB_ERR_ARGUMENT, "null argument");
    auto *s = new dfdb_scan();
    s->tbl = t;
    int rc = plan_parse(t, plan, plan_len, s);
    if (rc) { delete s; return rc; }
    *out = s;
    return DFDB_OK;
}

int32_t dfdb_scan_free(dfdb_scan *s)
{
    if (!s) return DFDB_OK;
    if (rt.inited) cudaStreamSynchronize(rt.stream);
    cudaFree(s->d_mask); cudaFree(s->d_blk_counts); cudaFree(s->d_blk_base); cudaFree(s->d_blk_bytes);
    cudaFree(s->d_partials); cudaFree(s->d_result); cudaFree(s->d_zone_dead);
    if (s->h_result) cudaFreeHost(s->h_result);
    for (auto &st : s->stages) cudaFree(st.d_idx);
    for (auto &set : s->sets) cudaFree(set.d_buf);
    delete s;
    return DFDB_OK;
}

int32_t dfdb_scan_nproj(const dfdb_scan *s) { return (int32_t)s->projs.size(); }

int32_t dfdb_scan_proj_type(const dfdb_scan *s, int32_t proj_idx, int32_t *kind, int32_t *nullable, int32_t *elsize)
{
    if (proj_idx < 0 || (size_t)proj_idx >= s->projs.size()) return fail(DFDB_ERR_ARGUMENT, "projection index out of range");
    const ColType &t = s->projs[(size_t)proj_idx].type;
    if (kind) *kind = t.kind;
    if (nullable) *nullable = t.nullable;
    if (elsize) *elsize = t.elsize;
    return DFDB_OK;
}

int32_t dfdb_scan_count(dfdb_scan *s, int64_t *n)
{
    int rc = need_init();
    if (rc) return rc;
    dfdb_table *t = s->tbl;
    invalidate_decoded(t);
    if (s->stages.empty()) {
        // isonly_range with an empty queue: header-only count (blocksiterator.jl:135)
        *n = std::min(t->nrows, t->blk_hi * t->block_size) - std::min(t->nrows, t->blk_lo * t->block_size);
        return DFDB_OK;
    }
    if (single_simple_pred(s)) {
        AggPartial p;
        int cls;
        rc = run_aggregate(s, -1, true, &p, &cls);
        if (rc) return rc;
        *n = p.count;
        return DFDB_OK;
    }
    return select_rows(s, n);
}

int32_t dfdb_scan_aggregate(dfdb_scan *s, int32_t proj_idx, dfdb_agg *out)
{
    int rc = need_init();
    if (rc) return rc;
    invalidate_decoded(s->tbl);
    AggPartial p;
    int cls;
    rc = run_aggregate(s, proj_idx, false, &p, &cls);
    if (rc) return rc;
    agg_to_public(p, cls, out);
    return DFDB_OK;
}

int32_t dfdb_scan_aggregate_device(dfdb_scan *s, int32_t proj_idx, void *device_out)
{
    dfdb_agg a;
    int rc = dfdb_scan_aggregate(s, proj_idx, &a);
    if (rc) return rc;
    CUDA_TRY(cudaMemcpyAsync(device_out, &a, sizeof a, cudaMemcpyHostToDevice, rt.stream));
    CUDA_TRY(cudaStreamSynchronize(rt.stream));
    return DFDB_OK;
}

int32_t dfdb_agg_fold(const dfdb_agg *partials, int32_t n, dfdb_agg *out)
{
    // fixed rank-order fold (the device fold of merged groups runs the same two functions)
    dfdb_agg r;
    memset(&r, 0, sizeof r);
    for (int i = 0; i < n; i++) dfdb_agg_fold_step(r, partials[i]);
    dfdb_agg_fold_finish(r);
    *out = r;
    return DFDB_OK;
}

int32_t dfdb_scan_exchange_count(dfdb_scan *s, int64_t *local_survivors, int32_t *pending)
{
    int rc = need_init();
    if (rc) return rc;
    if (!s || !local_survivors || !pending) return fail(DFDB_ERR_ARGUMENT, "null argument");
    invalidate_decoded(s->tbl);
    rc = run_selection(s);
    if (rc == DFDB_NEED_EXCHANGE) {
        *local_survivors = s->exchange_count;
        *pending = 1;
        return DFDB_OK;
    }
    *local_survivors = 0;
    *pending = 0;
    return rc;
}

int32_t dfdb_scan_exchange_offset(dfdb_scan *s, int64_t survivors_in_lower_ranks)
{
    if (!s) return fail(DFDB_ERR_ARGUMENT, "null argument");
    if (s->exchange_count < 0) return fail(DFDB_ERR_STATE, "no exchange is pending on this scan (call dfdb_scan_exchange_count first)");
    if (survivors_in_lower_ranks < 0) return fail(DFDB_ERR_ARGUMENT, "negative survivor count");
    s->rank_offsets.push_back(survivors_in_lower_ranks);
    s->exchange_count = -1;
    s->mask_valid = false;
    s->selected = -1;
    s->live_gen = 0;
    return DFDB_OK;
}

int32_t dfdb_scan_mask(dfdb_scan *s, uint64_t *words, int64_t nwords)
{
    int rc = need_init();
    if (rc) return rc;
    dfdb_table *t = s->tbl;
    invalidate_decoded(t);
    rc = run_selection(s);
    if (rc) return rc;
    const Geometry g = make_geometry(t);
    std::vector<uint32_t> h((size_t)std::max<int64_t>(s->mask_words, 1));
    {
        PhaseScope ps(PH_D2H, s->mask_words * 4);
        CUDA_TRY(cudaMemcpyAsync(h.data(), s->d_mask, (size_t)s->mask_words * 4, cudaMemcpyDeviceToHost, rt.stream));
        CUDA_TRY(cudaStreamSynchronize(rt.stream));
    }
    if (nwords < (t->nrows + 63) / 64) return fail(DFDB_ERR_ARGUMENT, "mask buffer too small: need %lld words", (long long)((t->nrows + 63) / 64));
    memset(words, 0, (size_t)nwords * 8);
    for (int lb = 0; lb < g.nblocks; lb++) {
        const int64_t row0 = (g.blk_lo + lb) * g.block_size;
        const int64_t rows = block_rows(g, lb);
        if ((row0 & 31) == 0) {
            // word-aligned block: copy 32-bit words straight into the little-endian 64-bit layout
            uint32_t *w32 = reinterpret_cast<uint32_t *>(words);
            for (int64_t w = 0; w * 32 < rows; w++) w32[(row0 >> 5) + w] = h[(size_t)((int64_t)lb * g.wpb + w)];
        } else {
            for (int64_t r = 0; r < rows; r++)
                if ((h[(size_t)((int64_t)lb * g.wpb + (r >> 5))] >> (r & 31)) & 1u) words[(row0 + r) >> 6] |= 1ull << ((row0 + r) & 63);
        }
    }
    return DFDB_OK;
}

int32_t dfdb_scan_indices(dfdb_scan *s, int64_t *idx, int64_t cap, int64_t *n)
{
    int rc = need_init();
    if (rc) return rc;
    invalidate_decoded(s->tbl);
    int64_t total = 0;
    rc = select_rows(s, &total);
    if (rc) return rc;
    if (n) *n = total;
    if (total > cap) return fail(DFDB_ERR_ARGUMENT, "index buffer too small: need %lld", (long long)total);
    if (total == 0) return DFDB_OK;
    int64_t *d_out = nullptr;
    CUDA_TRY(cudaMalloc(reinterpret_cast<void **>(&d_out), (size_t)total * 8));
    GatherArgs a;
    memset(&a, 0, sizeof a);
    a.g = make_geometry(s->tbl);
    a.mask = s->d_mask;
    a.blk_base = s->d_blk_base;
    a.out_indices = d_out;
    if (launch_gather_indices(a, rt.stream) != 0) { cudaFree(d_out); return fail(DFDB_ERR_CUDA, "gather_indices launch failed"); }
    rt.launches++;
    cudaError_t e = cudaMemcpyAsync(idx, d_out, (size_t)total * 8, cudaMemcpyDeviceToHost, rt.stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(rt.stream);
    cudaFree(d_out);
    if (e != cudaSuccess) return fail(DFDB_ERR_CUDA, "indices copy failed: %s", cudaGetErrorString(e));
    return DFDB_OK;
}

int32_t dfdb_scan_materialize_sizes(dfdb_scan *s, int64_t *nrows, int64_t *str_bytes_per_col)
{
    int rc = need_init();
    if (rc) return rc;
    dfdb_table *t = s->tbl;
    invalidate_decoded(t);
    int64_t total = 0;
    rc = select_rows(s, &total);
    if (rc) return rc;
    if (nrows) *nrows = total;
    s->str_bytes.assign(s->projs.size(), 0);
    const Geometry g = make_geometry(t);
    const DecodeScope scope = projection_scope(s);
    for (size_t i = 0; i < s->projs.size(); i++) {
        const Proj &p = s->projs[i];
        if (p.kind == PJ_COL && p.type.kind == DFDB_STRING && total > 0) {
            rc = ensure_decoded(t, {p.col}, scope);
            if (rc) return rc;
            PhaseScope ps(PH_CONSUME, 0);
            if ((rc = selected_chars(g, selection_rows(s), *t->find(p.col), static_cast<int64_t *>(s->h_result)))) return rc;
            CUDA_TRY(cudaStreamSynchronize(rt.stream));
            s->str_bytes[i] = *static_cast<int64_t *>(s->h_result);
        }
        if (str_bytes_per_col) str_bytes_per_col[i] = s->str_bytes[i];
    }
    return DFDB_OK;
}

int32_t dfdb_scan_materialize(dfdb_scan *s, dfdb_outcol *cols, int32_t ncols)
{
    int rc = need_init();
    if (rc) return rc;
    dfdb_table *t = s->tbl;
    if ((size_t)ncols != s->projs.size()) return fail(DFDB_ERR_ARGUMENT, "expected %zu output columns, got %d", s->projs.size(), ncols);
    if (!mask_current(s) || s->selected < 0) {
        rc = dfdb_scan_materialize_sizes(s, nullptr, nullptr);
        if (rc) return rc;
    }
    const int64_t total = s->selected;
    const Geometry g = make_geometry(t);
    if (total == 0) return DFDB_OK;
    const DecodeScope scope = projection_scope(s);
    struct CopyDrain { ~CopyDrain() { cudaStreamSynchronize(rt.copy_stream); } } drain;   // no queued copy outlives this call, on any path
    const RowSet rows = selection_rows(s);
    for (size_t i = 0; i < s->projs.size(); i++) {
        const Proj &p = s->projs[i];
        ResultCol r;
        r.set_type(p.type);
        if (p.kind == PJ_COL) {
            rc = ensure_decoded(t, {p.col}, scope);
            if (rc) return rc;
            const Column &c = *t->find(p.col);
            if ((rc = r.alloc(total, s->str_bytes[i]))) return rc;
            {
                PhaseScope ps(PH_CONSUME, c.total_origin + total * r.elsize);
                if (r.kind == DFDB_STRING) rc = char_bases(g, rows, c);   // (the scratch holds the last String column's)
                if (!rc) rc = gather_rows(g, rows, c, r);
            }
            if (rc) return rc;
        } else {
            rc = ensure_decoded(t, p.e.col_ids, scope);
            if (rc) return rc;
            ProjVmArgs a;
            memset(&a, 0, sizeof a);
            a.g = g;
            rc = fill_slots(s, a.slot);
            if (rc) return rc;
            DevProg prog;
            rc = prog.upload(s, p.e);
            if (rc) return rc;
            if ((rc = r.alloc(total, 0))) return rc;
            a.prog = prog.d;
            a.mask = rows.mask;
            a.blk_base = rows.blk_base;
            a.out_values = r.values.as<uint8_t>();
            a.out_missing = r.missing.as<uint8_t>();
            a.elsize = r.elsize;
            a.error_flag = rt.d_error;
            LAUNCH(launch_proj_vm(a, rt.stream));
            if ((rc = check_device_error())) return rc;
        }
        // stored columns are profiled as D2H phases of their values / sizes + chars
        const int64_t d2h = p.kind != PJ_COL ? -1 : r.kind == DFDB_STRING ? total * 4 + r.bytes : total * r.elsize;
        bool queued = false;
        rc = result_copy_out(r, cols[i], "output column", d2h, &queued);
        const cudaError_t e = queued ? cudaSuccess : cudaStreamSynchronize(rt.stream);
        if (queued) r.release(rt.copy_stream);
        if (rc) return rc;
        if (e != cudaSuccess) return fail(DFDB_ERR_CUDA, "materialize failed: %s", cudaGetErrorString(e));
    }
    return copies_done(DFDB_OK);
}

// ---- communicator: NCCL, bound at run time -------------------------------------------------------------
// (declarations restated from nccl.h so that the library builds without it; the ABI of these five entry points is stable
// across NCCL 2.x: ncclUniqueId is 128 bytes passed by value, ncclInt8 = 0)
namespace {
struct NcclId { char internal[DFDB_COMM_ID_BYTES]; };
struct Nccl {
    void *lib = nullptr;
    int (*GetUniqueId)(NcclId *) = nullptr;
    int (*CommInitRank)(void **, int, NcclId, int) = nullptr;
    int (*AllGather)(const void *, void *, size_t, int, void *, cudaStream_t) = nullptr;
    int (*CommDestroy)(void *) = nullptr;
    const char *(*GetErrorString)(int) = nullptr;
    void *comm = nullptr;
    int rank = 0, world = 0;
    uint8_t *d_buf = nullptr;      // world + 1 records of an exchange: [0] = this rank's contribution, [1..] = gathered
    uint8_t *h_buf = nullptr;      // pinned mirror
} nccl;

int nccl_bind()
{
    if (nccl.lib) return DFDB_OK;
    const char *names[] = {getenv("DFDB_NCCL_LIB"), "libnccl.so.2", "libnccl.so"};
    for (const char *n : names) {
        if (!n || !*n) continue;
        nccl.lib = dlopen(n, RTLD_NOW | RTLD_GLOBAL);
        if (nccl.lib) break;
    }
    if (!nccl.lib) return fail(DFDB_ERR_STATE, "cannot open libnccl.so.2 (%s); set DFDB_NCCL_LIB", dlerror());
    nccl.GetUniqueId = reinterpret_cast<decltype(nccl.GetUniqueId)>(dlsym(nccl.lib, "ncclGetUniqueId"));
    nccl.CommInitRank = reinterpret_cast<decltype(nccl.CommInitRank)>(dlsym(nccl.lib, "ncclCommInitRank"));
    nccl.AllGather = reinterpret_cast<decltype(nccl.AllGather)>(dlsym(nccl.lib, "ncclAllGather"));
    nccl.CommDestroy = reinterpret_cast<decltype(nccl.CommDestroy)>(dlsym(nccl.lib, "ncclCommDestroy"));
    nccl.GetErrorString = reinterpret_cast<decltype(nccl.GetErrorString)>(dlsym(nccl.lib, "ncclGetErrorString"));
    if (!nccl.GetUniqueId || !nccl.CommInitRank || !nccl.AllGather || !nccl.CommDestroy) {
        dlclose(nccl.lib);
        nccl.lib = nullptr;
        return fail(DFDB_ERR_STATE, "libnccl does not export the expected entry points");
    }
    return DFDB_OK;
}

#define NCCL_TRY(expr)                                                                                              \
    do {                                                                                                            \
        int _r = (expr);                                                                                            \
        if (_r != 0) return fail(DFDB_ERR_CUDA, "%s failed: %s", #expr, nccl.GetErrorString ? nccl.GetErrorString(_r) : "?"); \
    } while (0)

// An exchange record on the wire: the rank's status (8 bytes), then the payload, padded to whole 128-byte slots.  The largest
// is an order statistics round's {count, counts}; the communicator's buffers hold world + 1 of those.
constexpr size_t COMM_SLOT = 128;
constexpr size_t comm_record_bytes(size_t len) { return (8 + len + COMM_SLOT - 1) / COMM_SLOT * COMM_SLOT; }
constexpr size_t COMM_RECORD_MAX = comm_record_bytes(8 * (1 + DFDB_ORDER_MAX_COUNTS));
static_assert(comm_record_bytes(sizeof(dfdb_agg)) == COMM_SLOT, "a partial and its status fit one slot");

// every rank's payload after comm_exchange, in rank order (valid until the next exchange)
struct Records {
    const uint8_t *first = nullptr;
    size_t stride = 0;
    const void *of(int r) const { return first + stride * (size_t)r; }
};

// The record exchange of the _all entry points: one ncclAllGather on the scan stream of every rank's status and `len` bytes of
// `mine` (the same len on every rank: each caller sends a fixed record).  The status travels with the record, so that a rank
// whose local pass failed makes every rank fail instead of leaving the others waiting in the next collective: a local error
// is returned as it is (its message stays the thread's last error), another rank's is DFDB_ERR_STATE.
int comm_exchange(int status, const void *mine, size_t len, const char *what, Records *all)
{
    const size_t rec = comm_record_bytes(len);
    const int64_t st = status;
    memcpy(nccl.h_buf, &st, 8);
    memcpy(nccl.h_buf + 8, mine, len);
    memset(nccl.h_buf + 8 + len, 0, rec - 8 - len);
    CUDA_TRY(cudaMemcpyAsync(nccl.d_buf, nccl.h_buf, rec, cudaMemcpyHostToDevice, rt.stream));
    NCCL_TRY(nccl.AllGather(nccl.d_buf, nccl.d_buf + rec, rec, /*ncclInt8*/ 0, nccl.comm, rt.stream));
    CUDA_TRY(cudaMemcpyAsync(nccl.h_buf + rec, nccl.d_buf + rec, rec * (size_t)nccl.world, cudaMemcpyDeviceToHost, rt.stream));
    CUDA_TRY(cudaStreamSynchronize(rt.stream));
    if (status) return status;
    for (int r = 0; r < nccl.world; r++) {
        int64_t theirs;
        memcpy(&theirs, nccl.h_buf + rec * (size_t)(1 + r), 8);
        if (theirs) return fail(DFDB_ERR_STATE, "%s failed on rank %d (status %lld)", what, r, (long long)theirs);
    }
    all->first = nccl.h_buf + rec + 8;
    all->stride = rec;
    return DFDB_OK;
}

// The rule of every _all entry point: an exchange is needed when the table is sharded or a communicator exists, and then the
// communicator must serve this table's shard (its rank and world)
int comm_rule(const dfdb_scan *s, bool *exchange)
{
    *exchange = s->tbl->world > 1 || nccl.comm;
    if (*exchange && (!nccl.comm || nccl.world != s->tbl->world || nccl.rank != s->tbl->rank))
        return fail(DFDB_ERR_STATE, "the table is shard %d of %d but the communicator is rank %d of %d", s->tbl->rank, s->tbl->world, nccl.rank, nccl.world);
    return DFDB_OK;
}

// the start of every _all entry point: the rule, then the survivor-count exchanges the plan needs
int exchange_prologue(dfdb_scan *s, bool *exchange)
{
    int rc = comm_rule(s, exchange);
    if (rc || !*exchange) return rc;
    return dfdb_scan_resolve_exchange(s);
}

// every rank's agg (with the status of the local pass that made it), folded in rank order
int fold_all(int status, const dfdb_agg &mine, const char *what, dfdb_agg *whole)
{
    Records all;
    int rc = comm_exchange(status, &mine, sizeof mine, what, &all);
    if (rc) return rc;
    std::vector<dfdb_agg> parts((size_t)nccl.world);
    for (int r = 0; r < nccl.world; r++) parts[(size_t)r] = *static_cast<const dfdb_agg *>(all.of(r));
    return dfdb_agg_fold(parts.data(), nccl.world, whole);
}
}  // namespace

int32_t dfdb_comm_unique_id(uint8_t *id)
{
    if (!id) return fail(DFDB_ERR_ARGUMENT, "null argument");
    int rc = nccl_bind();
    if (rc) return rc;
    NcclId u;
    NCCL_TRY(nccl.GetUniqueId(&u));
    memcpy(id, u.internal, DFDB_COMM_ID_BYTES);
    return DFDB_OK;
}

int32_t dfdb_comm_init(int32_t rank, int32_t world, const uint8_t *id)
{
    int rc = need_init();
    if (rc) return rc;
    if (!id || world < 1 || rank < 0 || rank >= world) return fail(DFDB_ERR_ARGUMENT, "bad communicator arguments (rank %d of %d)", rank, world);
    if (nccl.comm) return fail(DFDB_ERR_STATE, "a communicator already exists (dfdb_comm_destroy first)");
    rc = nccl_bind();
    if (rc) return rc;
    NcclId u;
    memcpy(u.internal, id, DFDB_COMM_ID_BYTES);
    CUDA_TRY(cudaSetDevice(rt.device));
    NCCL_TRY(nccl.CommInitRank(&nccl.comm, world, u, rank));
    nccl.rank = rank;
    nccl.world = world;
    CUDA_TRY(cudaMalloc(reinterpret_cast<void **>(&nccl.d_buf), COMM_RECORD_MAX * (size_t)(world + 1)));
    CUDA_TRY(cudaMallocHost(reinterpret_cast<void **>(&nccl.h_buf), COMM_RECORD_MAX * (size_t)(world + 1)));
    return DFDB_OK;
}

int32_t dfdb_comm_destroy(void)
{
    if (!nccl.comm) return DFDB_OK;
    if (rt.inited) cudaStreamSynchronize(rt.stream);
    nccl.CommDestroy(nccl.comm);
    nccl.comm = nullptr;
    nccl.world = 0;
    cudaFree(nccl.d_buf);
    cudaFreeHost(nccl.h_buf);
    nccl.d_buf = nccl.h_buf = nullptr;
    return DFDB_OK;
}

int32_t dfdb_comm_info(int32_t *rank, int32_t *world)
{
    if (rank) *rank = nccl.comm ? nccl.rank : 0;
    if (world) *world = nccl.comm ? nccl.world : 0;
    return DFDB_OK;
}

int32_t dfdb_scan_resolve_exchange(dfdb_scan *s)
{
    int rc = need_init();
    if (rc) return rc;
    if (!s) return fail(DFDB_ERR_ARGUMENT, "null argument");
    {
        // only a range / index-vector stage that follows another stage ranks rows among ALL survivors; every other plan is
        // shard-local and must not pay a selection pass here
        size_t ranked = 0;
        for (size_t i = 1; i < s->stages.size(); i++) ranked += s->stages[i].kind != ST_PRED;
        if (ranked <= s->rank_offsets.size()) return DFDB_OK;
    }
    bool exchange = false;
    if ((rc = comm_rule(s, &exchange)) || !exchange) return rc;
    for (int stage = 0; stage < 64; stage++) {
        // every rank runs the same plan, so every rank has the same number of pending stages; the flag travels with the
        // count all the same so that a disagreement is an error, not a hang
        struct Pending { int64_t count, pending; } mine = {0, 0};
        int32_t pending = 0;
        rc = dfdb_scan_exchange_count(s, &mine.count, &pending);
        mine.pending = pending;
        Records all;
        if ((rc = comm_exchange(rc, &mine, sizeof mine, "the survivor count", &all))) return rc;
        int64_t lower = 0;
        for (int r = 0; r < nccl.world; r++) {
            const Pending &theirs = *static_cast<const Pending *>(all.of(r));
            if (theirs.pending != pending) return fail(DFDB_ERR_STATE, "ranks disagree on the plan: rank %d has %s exchange pending", r, theirs.pending ? "an" : "no");
            if (r < nccl.rank) lower += theirs.count;
        }
        if (!pending) return DFDB_OK;
        rc = dfdb_scan_exchange_offset(s, lower);
        if (rc) return rc;
    }
    return fail(DFDB_ERR_STATE, "too many exchange stages");
}

int32_t dfdb_scan_aggregate_all(dfdb_scan *s, int32_t proj_idx, dfdb_agg *out)
{
    int rc = need_init();
    if (rc) return rc;
    if (!s || !out) return fail(DFDB_ERR_ARGUMENT, "null argument");
    bool exchange = false;
    if ((rc = exchange_prologue(s, &exchange))) return rc;
    if (!exchange) return dfdb_scan_aggregate(s, proj_idx, out);     // unsharded, no communicator: the local result is the result
    dfdb_agg mine{};
    rc = dfdb_scan_aggregate(s, proj_idx, &mine);
    return fold_all(rc, mine, "aggregate", out);
}

int32_t dfdb_scan_row_offset_all(dfdb_scan *s, int64_t *local, int64_t *row_offset, int64_t *total)
{
    int rc = need_init();
    if (rc) return rc;
    if (!s) return fail(DFDB_ERR_ARGUMENT, "null argument");
    bool exchange = false;
    if ((rc = exchange_prologue(s, &exchange))) return rc;
    int64_t n = 0;
    rc = dfdb_scan_count(s, &n);
    int64_t lower = 0, all = n;
    if (exchange) {
        Records counts;
        rc = comm_exchange(rc, &n, sizeof n, "count", &counts);
        all = 0;
        for (int r = 0; !rc && r < nccl.world; r++) {
            const int64_t c = *static_cast<const int64_t *>(counts.of(r));
            if (r < nccl.rank) lower += c;
            all += c;
        }
    }
    if (rc) return rc;
    if (local) *local = n;
    if (row_offset) *row_offset = lower;
    if (total) *total = all;
    return DFDB_OK;
}

int32_t dfdb_scan_count_all(dfdb_scan *s, int64_t *n)
{
    if (!n) return fail(DFDB_ERR_ARGUMENT, "null argument");
    return dfdb_scan_row_offset_all(s, nullptr, nullptr, n);
}

// ---- group table: hash table of the selected rows by key (group-by reduce, unique) ------------------------
namespace {
constexpr long long GROUP_UNUSED = 0x7f7f7f7f7f7f7f7fll;     // `first` of a slot no group took

struct GroupTable {
    long long *rep = nullptr, *first = nullptr;
    GroupAcc *acc = nullptr;             // cap x nvals; none without value columns
    int *flag = nullptr;                 // [0] overflow, [2..3] group counter
    uint64_t cap = 0;
    unsigned long long ngroups = 0;
    void release()
    {
        cudaFree(rep); cudaFree(first); cudaFree(acc); cudaFree(flag);
        rep = first = nullptr; acc = nullptr; flag = nullptr;
    }
    ~GroupTable() { release(); }
};

// Builds the table over key columns kc[0..nkeys) with the accumulators of value columns vc[0..nvals) for the selected rows
// (s->d_mask).  It starts near the size the data suggests and grows fourfold while it overflows or is more than half full, up to
// max_cap slots; max_cap = 0: as many slots as free device memory holds at 16 bytes each (a table without value columns).
int build_group_table(const dfdb_scan *s, const Geometry &g, Column *const *kc, int nkeys, Column *const *vc, int nvals, int64_t total, uint64_t max_cap,
                      GroupTable *gt)
{
    if (max_cap == 0) {
        // device memory the scratch pool holds but does not use is not free to cudaMalloc; hand it back first, so that the
        // ceiling (and the table) can use it
        CUDA_TRY(cudaStreamSynchronize(rt.stream));
        cudaMemPool_t pool;
        if (cudaDeviceGetDefaultMemPool(&pool, rt.device) == cudaSuccess) cudaMemPoolTrimTo(pool, 0);
        size_t free_b = 0, total_b = 0;
        CUDA_TRY(cudaMemGetInfo(&free_b, &total_b));
        max_cap = 1;
        while (max_cap * 2 * 16 <= free_b) max_cap *= 2;
    }
    for (uint64_t cap = 1u << 16; cap <= max_cap; cap <<= 2) {
        if (cap < (uint64_t)std::min<int64_t>(total, 1 << 26) / 64) continue;       // (start near the size the data suggests)
        gt->release();
        gt->cap = cap;
        if (cudaMalloc(reinterpret_cast<void **>(&gt->rep), cap * 8) != cudaSuccess || cudaMalloc(reinterpret_cast<void **>(&gt->first), cap * 8) != cudaSuccess ||
            (nvals > 0 && cudaMalloc(reinterpret_cast<void **>(&gt->acc), cap * nvals * sizeof(GroupAcc)) != cudaSuccess) ||
            cudaMalloc(reinterpret_cast<void **>(&gt->flag), 16) != cudaSuccess) {
            gt->release();
            cudaGetLastError();
            return fail(DFDB_ERR_NOMEM, "out of device memory for a group table of %llu slots", (unsigned long long)cap);
        }
        cudaMemsetAsync(gt->rep, 0xff, cap * 8, rt.stream);
        cudaMemsetAsync(gt->first, 0x7f, cap * 8, rt.stream);
        cudaMemsetAsync(gt->flag, 0, 16, rt.stream);
        GroupArgs a;
        memset(&a, 0, sizeof a);
        a.g = g; a.mask = s->d_mask; a.nkeys = nkeys; a.nvals = nvals;
        for (int i = 0; i < nkeys; i++) a.key[i] = make_view(*kc[i]);
        for (int i = 0; i < nvals; i++) a.val[i] = make_view(*vc[i]);
        a.rep = gt->rep; a.first = gt->first; a.acc = gt->acc; a.cap_mask = cap - 1; a.overflow = gt->flag;
        a.ngroups = reinterpret_cast<unsigned long long *>(gt->flag + 2);
        if (nvals > 0) {
            // min / max start at the identities of their order
            int cls4[4] = {VC_INT, VC_INT, VC_INT, VC_INT};
            for (int i = 0; i < nvals; i++) cls4[i] = value_class(vc[i]->type.kind);
            if (launch_group_init(gt->acc, (long long)(cap * nvals), nvals, cls4, rt.stream) != 0) return fail(DFDB_ERR_CUDA, "group-by launch failed");
            rt.launches++;
        }
        {
            PhaseScope ps(PH_CONSUME, 0);
            if (launch_group_reduce(a, rt.sm_count, rt.stream) != 0) return fail(DFDB_ERR_CUDA, "group-by launch failed");
            rt.launches++;
        }
        int flag[4] = {0, 0, 0, 0};
        cudaMemcpyAsync(flag, gt->flag, 16, cudaMemcpyDeviceToHost, rt.stream);
        if (cudaStreamSynchronize(rt.stream) != cudaSuccess) return fail(DFDB_ERR_CUDA, "group-by kernel failed: %s", cudaGetErrorString(cudaGetLastError()));
        unsigned long long ng;
        memcpy(&ng, flag + 2, 8);
        if (flag[0] || ng * 2 > cap) continue;                                         // too full: a table four times the size
        gt->ngroups = ng;
        return DFDB_OK;
    }
    gt->release();
    return fail(DFDB_ERR_NOMEM, "more groups than the largest group table holds");
}
}  // namespace

// ---- results in materialize's layout on the device (unique; group-by keys) and their cross-shard merge ---------------
namespace {
// The lowest selected row of every group of a group table, set in a mask laid out like the selection mask, with the mask's
// per-block counts and their exclusive scan.  Its own buffers: s->d_mask / d_blk_base stay the selection's, so that a
// materialize on the same handle is unaffected.
struct FirstRows {
    PoolBuf mask, blk;               // blk: per-block counts | their exclusive scan | string bytes per block | their scan
    RowSet rows{};
};
int first_rows_mask(const dfdb_scan *s, const Geometry &g, const GroupTable &gt, FirstRows *fr)
{
    const size_t nb2 = (size_t)g.nblocks + 2, words = (size_t)std::max<int64_t>(s->mask_words, 1);
    if (fr->mask.alloc(words * 4) != cudaSuccess || fr->blk.alloc(nb2 * 4 * 8) != cudaSuccess)
        return fail(DFDB_ERR_NOMEM, "out of device memory for the first-row mask");
    uint32_t *mask = fr->mask.as<uint32_t>();
    int64_t *blk = fr->blk.as<int64_t>();
    fr->rows = RowSet{mask, blk + nb2, blk + 2 * nb2};
    CUDA_TRY(cudaMemsetAsync(mask, 0, words * 4, rt.stream));
    PhaseScope ps(PH_CONSUME, 0);
    LAUNCH(launch_unique_first_mask(gt.first, (long long)gt.cap, GROUP_UNUSED, g, mask, rt.stream));
    LAUNCH(launch_block_counts(g, mask, blk, rt.stream));
    LAUNCH(launch_exclusive_scan(blk, blk + nb2, g.nblocks, rt.stream));
    CUDA_TRY(cudaStreamSynchronize(rt.stream));          // (the caller frees the table next)
    return DFDB_OK;
}

// The values of column c at the rows of `fr`, in row order -- the order of first appearance -- into r (of c's type)
int gather_first_rows(dfdb_scan *s, const Geometry &g, const FirstRows &fr, const Column &c, ResultCol &r)
{
    const bool str = r.kind == DFDB_STRING;
    int64_t *h = static_cast<int64_t *>(s->h_result);
    CUDA_TRY(cudaMemcpyAsync(h, fr.rows.blk_base + g.nblocks, 8, cudaMemcpyDeviceToHost, rt.stream));
    int rc = str ? selected_chars(g, fr.rows, c, h + 1) : DFDB_OK;
    if (rc) return rc;
    CUDA_TRY(cudaStreamSynchronize(rt.stream));
    if ((rc = r.alloc(h[0], str ? h[1] : 0))) return rc;
    {
        PhaseScope ps(PH_CONSUME, 0);
        rc = gather_rows(g, fr.rows, c, r);
    }
    if (rc) return rc;
    CUDA_TRY(cudaStreamSynchronize(rt.stream));
    return DFDB_OK;
}

// an empty result column of r's type
ResultCol typed_like(const ResultCol &r)
{
    ResultCol t;
    t.kind = r.kind;
    t.elsize = r.elsize;
    t.nullable = r.nullable;
    return t;
}

// group-by's share of a merge: each position's first row and nvals aggregates (device arrays) and the part sizes in rank
// order; the kept positions' first rows and the folded aggregates of every merged group come back on the host
struct GroupParts {
    const long long *first;
    const dfdb_agg *aggs;
    int nvals;
    std::vector<int64_t> part_n;
    std::vector<int64_t> *first_out;
    std::vector<dfdb_agg> *aggs_out;
};

// Cross-shard merge: in[0..nkeys) hold the rank-order concatenation of the local results (device arrays of the types of
// res[]); every key tuple is kept where it first occurs, and the merged columns replace res[]
int merge_device(ResultCol *res, const ResultCol *in, int nkeys, const GroupParts *gp)
{
    for (int k = 0; k < nkeys; k++) res[k].release();
    if (gp) { gp->first_out->clear(); gp->aggs_out->clear(); }
    const long long n = in[0].n;
    if (n == 0) return DFDB_OK;
    unsigned long long cap = 1024;
    while (cap < 2ull * (unsigned long long)n) cap <<= 1;
    MergeArgs a;
    memset(&a, 0, sizeof a);
    a.n = n; a.nkeys = nkeys; a.cap_mask = cap - 1;
    const size_t n1 = (size_t)n + 1;
    PoolBuf rep, slot, keep_buf, scan_buf, kept_bytes[GROUP_MAX_KEYS], char_off[GROUP_MAX_KEYS];
    if (rep.alloc(cap * 8) != cudaSuccess || slot.alloc((size_t)n * 8) != cudaSuccess || keep_buf.alloc(n1 * 8) != cudaSuccess ||
        scan_buf.alloc((size_t)scan_i64_tmp_len(n) * 8) != cudaSuccess)
        return fail(DFDB_ERR_NOMEM, "out of device memory for merging %lld values", n);
    a.rep = rep.as<long long>();
    a.slot = slot.as<long long>();
    int64_t *keep = keep_buf.as<int64_t>(), *scan_tmp = scan_buf.as<int64_t>();
    for (int k = 0; k < nkeys; k++) {
        MergeKey &K = a.key[k];
        K.kind = res[k].kind; K.elsize = res[k].elsize;
        K.values = in[k].values.as<uint8_t>(); K.missing = res[k].nullable ? in[k].missing.as<uint8_t>() : nullptr;
        if (res[k].kind != DFDB_STRING) continue;
        K.sizes = in[k].sizes.as<int32_t>(); K.chars = in[k].chars.as<uint8_t>();
        if (kept_bytes[k].alloc(n1 * 8) != cudaSuccess || char_off[k].alloc(n1 * 8) != cudaSuccess)
            return fail(DFDB_ERR_NOMEM, "out of device memory for merging %lld values", n);
        K.kept_bytes = kept_bytes[k].as<int64_t>();
        K.char_off = char_off[k].as<int64_t>();
    }
    CUDA_TRY(cudaMemsetAsync(a.rep, 0xff, cap * 8, rt.stream));
    {
        PhaseScope ps(PH_CONSUME, 0);
        for (int k = 0; k < nkeys; k++) {
            if (!char_off[k].p) continue;
            LAUNCH(launch_str_lengths(a.key[k].sizes, n, char_off[k].as<int64_t>(), rt.stream));
            LAUNCH(launch_scan_i64(char_off[k].as<int64_t>(), n, scan_tmp, rt.stream));
        }
        LAUNCH(launch_merge_insert(a, rt.stream));
        LAUNCH(launch_merge_keep(a, keep, rt.stream));
        LAUNCH(launch_scan_i64(keep, n, scan_tmp, rt.stream));
        for (int k = 0; k < nkeys; k++)
            if (a.key[k].kept_bytes) LAUNCH(launch_scan_i64(a.key[k].kept_bytes, n, scan_tmp, rt.stream));
    }
    int64_t h[1 + GROUP_MAX_KEYS] = {0, 0, 0};     // kept positions, their char bytes per key (its own buffer: a handle that
    CUDA_TRY(cudaMemcpyAsync(h, keep + n, 8, cudaMemcpyDeviceToHost, rt.stream));      // never ran a scan has no pinned mirror)
    for (int k = 0; k < nkeys; k++)
        if (a.key[k].kept_bytes) CUDA_TRY(cudaMemcpyAsync(h + 1 + k, a.key[k].kept_bytes + n, 8, cudaMemcpyDeviceToHost, rt.stream));
    CUDA_TRY(cudaStreamSynchronize(rt.stream));
    const int64_t m = h[0];
    ResultCol out[GROUP_MAX_KEYS];                 // the merged columns: res[]'s once complete
    for (int k = 0; k < nkeys; k++) {
        out[k] = typed_like(res[k]);
        const int rc = out[k].alloc(m, h[1 + k]);
        if (rc) return rc;
        MergeKey &K = a.key[k];
        K.out_values = out[k].values.as<uint8_t>(); K.out_missing = out[k].missing.as<uint8_t>();
        K.out_sizes = out[k].sizes.as<int32_t>(); K.out_chars = out[k].chars.as<uint8_t>();
    }
    PoolBuf first_buf, aggs_buf, dup_buf;
    const int nv = gp ? gp->nvals : 0;
    if (gp && (first_buf.alloc((size_t)m * 8) != cudaSuccess || dup_buf.alloc(4) != cudaSuccess ||
               (nv > 0 && aggs_buf.alloc((size_t)m * nv * sizeof(dfdb_agg)) != cudaSuccess)))
        return fail(DFDB_ERR_NOMEM, "out of device memory for %lld merged groups", (long long)m);
    long long *d_first = first_buf.as<long long>();
    dfdb_agg *d_aggs = aggs_buf.as<dfdb_agg>();
    int *d_dup = dup_buf.as<int>();
    {
        PhaseScope ps(PH_CONSUME, 0);
        LAUNCH(launch_merge_emit(a, keep, gp ? gp->first : nullptr, d_first, rt.stream));
        if (nv > 0) {
            // rank order: one launch per part, each folding into slots no other thread of it touches
            CUDA_TRY(cudaMemsetAsync(d_aggs, 0, (size_t)m * nv * sizeof(dfdb_agg), rt.stream));
            CUDA_TRY(cudaMemsetAsync(d_dup, 0, 4, rt.stream));
            long long lo = 0;
            for (int64_t pn : gp->part_n) {
                LAUNCH(launch_merge_fold(a, keep, gp->aggs, nv, lo, lo + pn, d_aggs, d_dup, rt.stream));
                lo += pn;
            }
            LAUNCH(launch_merge_fold_finish(d_aggs, (long long)m * nv, rt.stream));
        }
    }
    int dup = 0;
    if (gp) {
        gp->first_out->resize((size_t)m);
        gp->aggs_out->resize((size_t)m * nv);
        CUDA_TRY(cudaMemcpyAsync(gp->first_out->data(), d_first, (size_t)m * 8, cudaMemcpyDeviceToHost, rt.stream));
        if (nv > 0) {
            CUDA_TRY(cudaMemcpyAsync(gp->aggs_out->data(), d_aggs, (size_t)m * nv * sizeof(dfdb_agg), cudaMemcpyDeviceToHost, rt.stream));
            CUDA_TRY(cudaMemcpyAsync(&dup, d_dup, 4, cudaMemcpyDeviceToHost, rt.stream));
        }
    }
    CUDA_TRY(cudaStreamSynchronize(rt.stream));
    if (dup) {
        gp->first_out->clear();
        gp->aggs_out->clear();
        return fail(DFDB_ERR_ARGUMENT, "a part holds one key twice (a part is one rank's groups, whose keys are distinct)");
    }
    for (int k = 0; k < nkeys; k++) res[k] = std::move(out[k]);
    return DFDB_OK;
}

// All-gather of one device array over the communicator: rank r contributes len[r] bytes (on the wire every part is padded to
// the largest); *packed receives the parts back to back in rank order
int allgather_packed(const void *local, const std::vector<size_t> &len, PoolBuf *packed)
{
    const int world = nccl.world;
    size_t most = 0, all = 0;
    for (size_t l : len) { most = std::max(most, l); all += l; }
    if (packed->alloc(all) != cudaSuccess) return fail(DFDB_ERR_NOMEM, "out of device memory for the gathered results");
    if (most == 0) return DFDB_OK;
    PoolBuf send, recv;
    if (send.alloc(most) != cudaSuccess || recv.alloc(most * (size_t)world) != cudaSuccess)
        return fail(DFDB_ERR_NOMEM, "out of device memory for the all-gather");
    if (len[(size_t)nccl.rank] > 0) CUDA_TRY(cudaMemcpyAsync(send.p, local, len[(size_t)nccl.rank], cudaMemcpyDeviceToDevice, rt.stream));
    NCCL_TRY(nccl.AllGather(send.p, recv.p, most, /*ncclInt8*/ 0, nccl.comm, rt.stream));
    size_t at = 0;
    for (int r = 0; r < world; r++) {
        if (len[(size_t)r] > 0)
            CUDA_TRY(cudaMemcpyAsync(packed->as<uint8_t>() + at, recv.as<uint8_t>() + most * (size_t)r, len[(size_t)r], cudaMemcpyDeviceToDevice, rt.stream));
        at += len[(size_t)r];
    }
    CUDA_TRY(cudaStreamSynchronize(rt.stream));
    return DFDB_OK;
}

// all-gather of one column of the local results (rank r: cnt[r] values, cb[r] chars) into `in` (u's type)
int allgather_result(const ResultCol &u, const std::vector<int64_t> &cnt, const std::vector<int64_t> &cb, ResultCol &in)
{
    const int world = nccl.world;
    in = typed_like(u);
    std::vector<size_t> per_value((size_t)world), chars((size_t)world);
    for (int r = 0; r < world; r++) {
        in.n += cnt[(size_t)r];
        chars[(size_t)r] = (size_t)cb[(size_t)r];
        if (u.kind == DFDB_STRING) in.bytes += cb[(size_t)r];
    }
    auto scaled = [&](size_t elem) { for (int r = 0; r < world; r++) per_value[(size_t)r] = (size_t)cnt[(size_t)r] * elem; return per_value; };
    if (u.kind == DFDB_STRING) {
        const int rc = allgather_packed(u.sizes.p, scaled(4), &in.sizes);
        return rc ? rc : allgather_packed(u.chars.p, chars, &in.chars);
    }
    const int rc = allgather_packed(u.values.p, scaled((size_t)u.elsize), &in.values);
    return rc || !u.nullable ? rc : allgather_packed(u.missing.p, scaled(1), &in.missing);
}

// A merge's parts carried by the host, checked and copied to the device: part r holds part_n[r] values of every key column k,
// in parts[r * nkeys + k] (and part_str_bytes[r * nkeys + k] chars for a String column); in[k], typed already, receives
// their rank-order concatenation
int upload_parts(ResultCol *in, int nkeys, const dfdb_outcol *parts, const int64_t *part_n, const int64_t *part_str_bytes, int32_t nparts)
{
    int64_t total = 0;
    for (int32_t r = 0; r < nparts; r++) {
        if (part_n[r] < 0) return fail(DFDB_ERR_ARGUMENT, "negative part size");
        total += part_n[r];
    }
    for (int k = 0; k < nkeys; k++) {
        const bool str = in[k].kind == DFDB_STRING;
        if (str && !part_str_bytes) return fail(DFDB_ERR_ARGUMENT, "String columns need their parts' char byte counts");
        int64_t bytes = 0;
        for (int32_t r = 0; r < nparts; r++) {
            const dfdb_outcol &p = parts[(size_t)r * nkeys + k];
            const int64_t pb = str ? part_str_bytes[(size_t)r * nkeys + k] : 0;
            if (pb < 0) return fail(DFDB_ERR_ARGUMENT, "negative part size");
            if (part_n[r] > 0 && (str ? !p.str_sizes || (pb > 0 && !p.str_chars) : !p.values || (in[k].nullable && !p.missing)))
                return fail(DFDB_ERR_ARGUMENT, "key %d of part %d lacks a buffer its column type needs", k, r);
            bytes += pb;
        }
        const int rc = in[k].alloc(total, bytes);
        if (rc) return rc;
        int64_t at = 0, at_b = 0;
        for (int32_t r = 0; r < nparts; r++) {
            const dfdb_outcol &p = parts[(size_t)r * nkeys + k];
            const int64_t cnt = part_n[r], pb = str ? part_str_bytes[(size_t)r * nkeys + k] : 0;
            if (cnt > 0 && str) {
                CUDA_TRY(cudaMemcpyAsync(in[k].sizes.as<int32_t>() + at, p.str_sizes, (size_t)cnt * 4, cudaMemcpyHostToDevice, rt.stream));
                if (pb > 0) CUDA_TRY(cudaMemcpyAsync(in[k].chars.as<uint8_t>() + at_b, p.str_chars, (size_t)pb, cudaMemcpyHostToDevice, rt.stream));
            } else if (cnt > 0) {
                CUDA_TRY(cudaMemcpyAsync(in[k].values.as<uint8_t>() + at * in[k].elsize, p.values, (size_t)cnt * in[k].elsize, cudaMemcpyHostToDevice, rt.stream));
                if (in[k].nullable) CUDA_TRY(cudaMemcpyAsync(in[k].missing.as<uint8_t>() + at, p.missing, (size_t)cnt, cudaMemcpyHostToDevice, rt.stream));
            }
            at += cnt;
            at_b += pb;
        }
    }
    return DFDB_OK;
}

// unique_all / groupreduce_all after the local pass (`status`): every rank's result sizes travel with its status, then every
// rank's key columns -- with group-by's first rows and nvals aggregates -- are all-gathered and merged on the device; the merged
// result replaces the handle's
int merge_all(int status, dfdb_scan *s, bool group, int nkeys, int nvals)
{
    ResultCol *keys = group ? s->group_keys : &s->uniq;
    struct Sizes { int64_t n, bytes[GROUP_MAX_KEYS]; } mine = {};
    for (int k = 0; !status && k < nkeys; k++) {
        mine.n = keys[k].n;
        mine.bytes[k] = keys[k].bytes;
    }
    Records all;
    int rc = comm_exchange(status, &mine, sizeof mine, group ? "group-by" : "unique", &all);
    if (rc) return rc;
    const int world = nccl.world;
    std::vector<int64_t> cnt((size_t)world);
    std::vector<std::vector<int64_t>> cb((size_t)nkeys, std::vector<int64_t>((size_t)world));
    for (int r = 0; r < world; r++) {
        const Sizes &theirs = *static_cast<const Sizes *>(all.of(r));
        cnt[(size_t)r] = theirs.n;
        for (int k = 0; k < nkeys; k++) cb[(size_t)k][(size_t)r] = theirs.bytes[k];
    }
    if (group) s->group_nkeys = 0;                                   // (the local result is the merge's input now)
    ResultCol in[GROUP_MAX_KEYS];
    for (int k = 0; k < nkeys; k++)
        if ((rc = allgather_result(keys[k], cnt, cb[(size_t)k], in[k]))) return rc;
    if (!group) return merge_device(keys, in, nkeys, nullptr);
    // first rows and aggregates: the local ones to the device, then gathered like the keys
    const size_t mine_n = s->group_first.size();
    PoolBuf lfirst, laggs, first, aggs;
    if (lfirst.alloc(mine_n * 8) != cudaSuccess || laggs.alloc(mine_n * nvals * sizeof(dfdb_agg)) != cudaSuccess)
        return fail(DFDB_ERR_NOMEM, "out of device memory for the local group results");
    if (mine_n > 0) CUDA_TRY(cudaMemcpyAsync(lfirst.p, s->group_first.data(), mine_n * 8, cudaMemcpyHostToDevice, rt.stream));
    if (mine_n > 0 && nvals > 0) CUDA_TRY(cudaMemcpyAsync(laggs.p, s->group_aggs.data(), mine_n * nvals * sizeof(dfdb_agg), cudaMemcpyHostToDevice, rt.stream));
    std::vector<size_t> len8((size_t)world), len_agg((size_t)world);
    for (int r = 0; r < world; r++) {
        len8[(size_t)r] = (size_t)cnt[(size_t)r] * 8;
        len_agg[(size_t)r] = (size_t)cnt[(size_t)r] * nvals * sizeof(dfdb_agg);
    }
    if ((rc = allgather_packed(lfirst.p, len8, &first)) || (rc = allgather_packed(laggs.p, len_agg, &aggs))) return rc;
    const GroupParts gp{first.as<const long long>(), aggs.as<const dfdb_agg>(), nvals, cnt, &s->group_first, &s->group_aggs};
    if ((rc = merge_device(keys, in, nkeys, &gp))) return rc;
    s->group_nkeys = nkeys;
    return DFDB_OK;
}

// the stored column of projection pi, when group-by can take it as a key (value = false) or a value column
int group_column(const dfdb_scan *s, int32_t pi, bool value, Column **out)
{
    if (pi < 0 || (size_t)pi >= s->projs.size()) return fail(DFDB_ERR_ARGUMENT, "projection index out of range");
    const Proj &p = s->projs[(size_t)pi];
    if (p.kind != PJ_COL) return fail(DFDB_ERR_UNSUPPORTED, "group-by keys and values are stored columns (materialize a computed column with add_column first)");
    Column *c = s->tbl->find(p.col);
    const int cls = value_class(c->type.kind);
    if (cls == VC_NONE || c->type.elsize > 8) return fail(DFDB_ERR_UNSUPPORTED, "column %s of type %s cannot be grouped", c->name.c_str(), c->typestr.c_str());
    if (value && cls == VC_STR) return fail(DFDB_ERR_UNSUPPORTED, "aggregate over column %s of type %s", c->name.c_str(), c->typestr.c_str());
    *out = c;
    return DFDB_OK;
}

int group_limits(int32_t nkeys, int32_t nvals)
{
    if (nkeys < 1 || nkeys > GROUP_MAX_KEYS || nvals < 0 || nvals > GROUP_MAX_VALS)
        return fail(DFDB_ERR_UNSUPPORTED, "group-by takes 1..%d key and 0..%d value columns", GROUP_MAX_KEYS, GROUP_MAX_VALS);
    return DFDB_OK;
}
}  // namespace

// ---- group-by reduce ------------------------------------------------------------------------------------
int32_t dfdb_scan_groupreduce(dfdb_scan *s, const int32_t *key_proj, int32_t nkeys, const int32_t *val_proj, int32_t nvals, int64_t *ngroups)
{
    int rc = need_init();
    if (rc) return rc;
    if (!s || !key_proj || !ngroups) return fail(DFDB_ERR_ARGUMENT, "null argument");
    if ((rc = group_limits(nkeys, nvals))) return rc;
    dfdb_table *t = s->tbl;
    Column *kc[GROUP_MAX_KEYS] = {nullptr, nullptr}, *vc[GROUP_MAX_VALS] = {nullptr, nullptr, nullptr, nullptr};
    std::vector<int64_t> need;
    for (int i = 0; i < nkeys; i++) {
        if ((rc = group_column(s, key_proj[i], false, &kc[i]))) return rc;
        need.push_back(kc[i]->id);
    }
    for (int i = 0; i < nvals; i++) {
        if ((rc = group_column(s, val_proj[i], true, &vc[i]))) return rc;
        need.push_back(vc[i]->id);
    }
    s->group_nkeys = 0;                                                          // (no result until this call succeeds)
    for (int i = 0; i < nkeys; i++) {
        s->group_keys[i].release();
        s->group_keys[i].set_type(kc[i]->type);
    }
    invalidate_decoded(t);
    int64_t total = 0;
    rc = select_rows(s, &total);
    if (rc) return rc;
    s->group_first.clear();
    s->group_aggs.clear();
    *ngroups = 0;
    if (total == 0) {
        s->group_nkeys = nkeys;
        return DFDB_OK;
    }
    rc = ensure_decoded(t, need, projection_scope(s));
    if (rc) return rc;
    const Geometry g = make_geometry(t);
    GroupTable gt;
    rc = build_group_table(s, g, kc, nkeys, vc, nvals, total, 1ull << 28, &gt);
    if (rc) return rc;
    const int nv = nvals;
    const unsigned long long ng = gt.ngroups;
    // ---- results to the host, groups in order of first appearance: the used slots are packed on the device first ----
    long long *d_pfirst = nullptr;
    GroupAcc *d_pacc = nullptr;
    const size_t ngz = (size_t)std::max<unsigned long long>(ng, 1);
    if (cudaMalloc(reinterpret_cast<void **>(&d_pfirst), ngz * 8) != cudaSuccess ||
        (nv > 0 && cudaMalloc(reinterpret_cast<void **>(&d_pacc), ngz * nv * sizeof(GroupAcc)) != cudaSuccess)) {
        cudaFree(d_pfirst);
        cudaGetLastError();
        return fail(DFDB_ERR_NOMEM, "out of device memory for %llu group results", ng);
    }
    cudaMemsetAsync(gt.flag + 2, 0, 8, rt.stream);                              // (the group counter is the pack cursor now)
    if (launch_group_compact(gt.first, gt.acc, (long long)gt.cap, nv, GROUP_UNUSED, reinterpret_cast<unsigned long long *>(gt.flag + 2), d_pfirst, d_pacc, rt.stream) != 0) {
        cudaFree(d_pfirst); cudaFree(d_pacc);
        return fail(DFDB_ERR_CUDA, "group-by launch failed");
    }
    rt.launches++;
    std::vector<long long> first(ngz);
    std::vector<GroupAcc> acc(ngz * (size_t)std::max(nv, 1));
    cudaMemcpyAsync(first.data(), d_pfirst, (size_t)ng * 8, cudaMemcpyDeviceToHost, rt.stream);
    if (nv > 0) cudaMemcpyAsync(acc.data(), d_pacc, (size_t)ng * nv * sizeof(GroupAcc), cudaMemcpyDeviceToHost, rt.stream);
    cudaError_t e = cudaStreamSynchronize(rt.stream);
    cudaFree(d_pfirst); cudaFree(d_pacc);
    if (e != cudaSuccess) return fail(DFDB_ERR_CUDA, "group-by results: %s", cudaGetErrorString(e));
    // the key values of the groups, in group order: a merge with other shards' groups has no rows to materialize them from
    FirstRows fr;
    {
        PhaseScope ps(PH_GROUP_KEYS, 0);
        rc = first_rows_mask(s, g, gt, &fr);
    }
    gt.release();
    if (rc) return rc;
    {
        PhaseScope ps(PH_GROUP_KEYS, 0);
        for (int i = 0; i < nkeys && !rc; i++) rc = gather_first_rows(s, g, fr, *kc[i], s->group_keys[i]);
    }
    if (rc) return rc;
    std::vector<std::pair<long long, size_t>> order;
    for (size_t sl = 0; sl < (size_t)ng; sl++) order.emplace_back(first[sl], sl);
    std::sort(order.begin(), order.end());
    s->group_first.resize(order.size());
    s->group_aggs.assign(order.size() * (size_t)nvals, dfdb_agg());
    for (size_t gi = 0; gi < order.size(); gi++) {
        s->group_first[gi] = t->blk_lo * t->block_size + order[gi].first + 1;
        for (int v = 0; v < nvals; v++) {
            const GroupAcc &ga = acc[order[gi].second * (size_t)nv + (size_t)v];
            dfdb_agg &o = s->group_aggs[gi * (size_t)nvals + (size_t)v];
            memset(&o, 0, sizeof o);
            const int cls = value_class(vc[v]->type.kind);
            o.count = (int64_t)ga.count; o.nmissing = (int64_t)ga.nmissing; o.sum_i64 = ga.sum_i; o.sum_f64 = ga.sum_f; o.has_nan = (ga.flags >> 1) & 1;
            if (cls == VC_FLT) {
                auto undo = [](long long k) { const long long b = k < 0 ? (long long)(0x8000000000000000ull - (unsigned long long)k) : k; double d; memcpy(&d, &b, 8); return d; };
                if (ga.flags & 1) { o.min_f64 = undo(ga.min_k); o.max_f64 = undo(ga.max_k); }
                if (ga.flags & 2) { o.min_f64 = o.max_f64 = NAN; }              // NaN propagates through Julia's min / max
            } else if (ga.flags & 1) { o.min_i64 = ga.min_k; o.max_i64 = ga.max_k; }
            o.value_class = (ga.flags & 3) ? (cls == VC_FLT ? 3 : cls == VC_UINT ? 2 : cls == VC_BOOL ? 4 : 1) : 0;
        }
    }
    *ngroups = (int64_t)order.size();
    s->group_nkeys = nkeys;
    return DFDB_OK;
}

int32_t dfdb_scan_group_results(dfdb_scan *s, int64_t *first_rows, dfdb_agg *aggs)
{
    if (!s) return fail(DFDB_ERR_ARGUMENT, "null argument");
    if (first_rows && !s->group_first.empty()) memcpy(first_rows, s->group_first.data(), s->group_first.size() * 8);
    if (aggs && !s->group_aggs.empty()) memcpy(aggs, s->group_aggs.data(), s->group_aggs.size() * sizeof(dfdb_agg));
    return DFDB_OK;
}

int32_t dfdb_scan_group_key_bytes(dfdb_scan *s, int64_t *str_bytes_per_key)
{
    if (!s || !str_bytes_per_key) return fail(DFDB_ERR_ARGUMENT, "null argument");
    if (s->group_nkeys == 0) return fail(DFDB_ERR_STATE, "no group-by result on this scan (call dfdb_scan_groupreduce first)");
    for (int i = 0; i < s->group_nkeys; i++) str_bytes_per_key[i] = s->group_keys[i].bytes;
    return DFDB_OK;
}

int32_t dfdb_scan_group_keys(dfdb_scan *s, dfdb_outcol *keys, int32_t nkeys)
{
    int rc = need_init();
    if (rc) return rc;
    if (!s || !keys) return fail(DFDB_ERR_ARGUMENT, "null argument");
    if (s->group_nkeys == 0) return fail(DFDB_ERR_STATE, "no group-by result on this scan (call dfdb_scan_groupreduce first)");
    if (nkeys != s->group_nkeys) return fail(DFDB_ERR_ARGUMENT, "the group-by result has %d key columns, not %d", s->group_nkeys, nkeys);
    bool queued;
    for (int i = 0; i < nkeys && !rc; i++) rc = result_copy_out(s->group_keys[i], keys[i], "group key column", -1, &queued);
    return copies_done(rc);
}

int32_t dfdb_scan_groupreduce_merge(dfdb_scan *s, const int32_t *key_proj, int32_t nkeys, int32_t nvals, const dfdb_outcol *keys, const int64_t *first_rows,
                                    const dfdb_agg *aggs, const int64_t *part_n, const int64_t *part_str_bytes, int32_t nparts, int64_t *ngroups)
{
    int rc = need_init();
    if (rc) return rc;
    if (!s || !key_proj || !ngroups || nparts < 0 || (nparts > 0 && (!keys || !part_n))) return fail(DFDB_ERR_ARGUMENT, "null argument");
    if ((rc = group_limits(nkeys, nvals))) return rc;
    Column *kc[GROUP_MAX_KEYS] = {nullptr, nullptr};
    ResultCol in[GROUP_MAX_KEYS];
    for (int k = 0; k < nkeys; k++) {
        if ((rc = group_column(s, key_proj[k], false, &kc[k]))) return rc;
        in[k].set_type(kc[k]->type);
    }
    if ((rc = upload_parts(in, nkeys, keys, part_n, part_str_bytes, nparts))) return rc;
    const int64_t total = in[0].n;
    if (total > 0 && (!first_rows || (nvals > 0 && !aggs))) return fail(DFDB_ERR_ARGUMENT, "the parts need their first rows and aggregates");
    PoolBuf d_first, d_aggs;
    if (d_first.alloc((size_t)total * 8) != cudaSuccess || d_aggs.alloc((size_t)total * nvals * sizeof(dfdb_agg)) != cudaSuccess)
        return fail(DFDB_ERR_NOMEM, "out of device memory for %lld groups to merge", (long long)total);
    if (total > 0) CUDA_TRY(cudaMemcpyAsync(d_first.p, first_rows, (size_t)total * 8, cudaMemcpyHostToDevice, rt.stream));
    if (total > 0 && nvals > 0) CUDA_TRY(cudaMemcpyAsync(d_aggs.p, aggs, (size_t)total * nvals * sizeof(dfdb_agg), cudaMemcpyHostToDevice, rt.stream));
    s->group_nkeys = 0;
    for (int k = 0; k < nkeys; k++) s->group_keys[k].set_type(kc[k]->type);
    const GroupParts gp{d_first.as<const long long>(), d_aggs.as<const dfdb_agg>(), nvals, std::vector<int64_t>(part_n, part_n + nparts), &s->group_first,
                        &s->group_aggs};
    if ((rc = merge_device(s->group_keys, in, nkeys, &gp))) return rc;
    s->group_nkeys = nkeys;
    *ngroups = (int64_t)s->group_first.size();
    return DFDB_OK;
}

int32_t dfdb_scan_groupreduce_all(dfdb_scan *s, const int32_t *key_proj, int32_t nkeys, const int32_t *val_proj, int32_t nvals, int64_t *ngroups)
{
    int rc = need_init();
    if (rc) return rc;
    if (!s || !ngroups) return fail(DFDB_ERR_ARGUMENT, "null argument");
    bool exchange = false;
    if ((rc = exchange_prologue(s, &exchange))) return rc;
    if (!exchange) return dfdb_scan_groupreduce(s, key_proj, nkeys, val_proj, nvals, ngroups);   // unsharded, no communicator: the local result is the result
    rc = dfdb_scan_groupreduce(s, key_proj, nkeys, val_proj, nvals, ngroups);
    if ((rc = merge_all(rc, s, true, nkeys, nvals))) return rc;
    *ngroups = (int64_t)s->group_first.size();
    return DFDB_OK;
}

// ---- unique -------------------------------------------------------------------------------------------------
namespace {
// the stored column of projection proj_idx, when unique can take it
int unique_column(dfdb_scan *s, int32_t proj_idx, Column **out)
{
    if (proj_idx < 0 || (size_t)proj_idx >= s->projs.size()) return fail(DFDB_ERR_ARGUMENT, "projection index out of range");
    const Proj &p = s->projs[(size_t)proj_idx];
    if (p.kind != PJ_COL) return fail(DFDB_ERR_UNSUPPORTED, "unique takes a stored column (materialize a computed column with add_column first)");
    Column *c = s->tbl->find(p.col);
    const int k = c->type.kind;
    if ((value_class(k) == VC_NONE && k != DFDB_F16 && k != DFDB_CHAR) || (k != DFDB_STRING && c->type.elsize > 8))
        return fail(DFDB_ERR_UNSUPPORTED, "unique over column %s of type %s", c->name.c_str(), c->typestr.c_str());
    *out = c;
    return DFDB_OK;
}
}  // namespace

int32_t dfdb_scan_unique(dfdb_scan *s, int32_t proj_idx, int64_t *n, int64_t *str_bytes)
{
    int rc = need_init();
    if (rc) return rc;
    if (!s || !n) return fail(DFDB_ERR_ARGUMENT, "null argument");
    Column *c = nullptr;
    if ((rc = unique_column(s, proj_idx, &c))) return rc;
    dfdb_table *t = s->tbl;
    ResultCol &u = s->uniq;
    u.release();
    u.set_type(c->type);
    *n = 0;
    if (str_bytes) *str_bytes = 0;
    invalidate_decoded(t);
    int64_t total = 0;
    rc = select_rows(s, &total);
    if (rc) return rc;
    if (total == 0) return DFDB_OK;
    rc = ensure_decoded(t, {c->id}, projection_scope(s));
    if (rc) return rc;
    const Geometry g = make_geometry(t);
    // the first selected row of every distinct value
    FirstRows fr;
    {
        GroupTable gt;
        Column *kc[1] = {c};
        rc = build_group_table(s, g, kc, 1, nullptr, 0, total, 0, &gt);
        if (rc) return rc;
        rc = first_rows_mask(s, g, gt, &fr);
        if (rc) return rc;
    }                                                          // (the table is freed before the values are gathered)
    rc = gather_first_rows(s, g, fr, *c, u);
    if (rc) return rc;
    *n = u.n;
    if (str_bytes) *str_bytes = u.bytes;
    return DFDB_OK;
}

int32_t dfdb_scan_unique_values(dfdb_scan *s, dfdb_outcol *out)
{
    int rc = need_init();
    if (rc) return rc;
    if (!s || !out) return fail(DFDB_ERR_ARGUMENT, "null argument");
    if (s->uniq.kind == 0) return fail(DFDB_ERR_STATE, "no unique result on this scan (call dfdb_scan_unique first)");
    bool queued;
    return copies_done(result_copy_out(s->uniq, *out, "unique values", -1, &queued));
}

int32_t dfdb_scan_unique_merge(dfdb_scan *s, const dfdb_outcol *parts, const int64_t *part_n, const int64_t *part_str_bytes, int32_t nparts, int64_t *n,
                               int64_t *str_bytes)
{
    int rc = need_init();
    if (rc) return rc;
    if (!s || !n || nparts < 0 || (nparts > 0 && (!parts || !part_n))) return fail(DFDB_ERR_ARGUMENT, "null argument");
    ResultCol &u = s->uniq;
    if (u.kind == 0) {                         // no local result yet: the parts are of projection 0
        Column *c = nullptr;
        if ((rc = unique_column(s, 0, &c))) return rc;
        u.set_type(c->type);
    }
    ResultCol in = typed_like(u);
    if ((rc = upload_parts(&in, 1, parts, part_n, part_str_bytes, nparts))) return rc;
    if ((rc = merge_device(&u, &in, 1, nullptr))) return rc;
    *n = u.n;
    if (str_bytes) *str_bytes = u.bytes;
    return DFDB_OK;
}

int32_t dfdb_scan_unique_all(dfdb_scan *s, int32_t proj_idx, int64_t *n, int64_t *str_bytes)
{
    int rc = need_init();
    if (rc) return rc;
    if (!s || !n) return fail(DFDB_ERR_ARGUMENT, "null argument");
    bool exchange = false;
    if ((rc = exchange_prologue(s, &exchange))) return rc;
    if (!exchange) return dfdb_scan_unique(s, proj_idx, n, str_bytes);     // unsharded, no communicator: the local result is the result
    rc = dfdb_scan_unique(s, proj_idx, n, str_bytes);
    if ((rc = merge_all(rc, s, false, 1, 0))) return rc;
    *n = s->uniq.n;
    if (str_bytes) *str_bytes = s->uniq.bytes;
    return DFDB_OK;
}

// ---- order statistics: exact k-th smallest values by MSD radix select ---------------------------------------------------
namespace {
// the stored column of projection pi when order statistics take it
int order_column(const dfdb_scan *s, int32_t pi, Column **out)
{
    if (pi < 0 || (size_t)pi >= s->projs.size()) return fail(DFDB_ERR_ARGUMENT, "projection index out of range");
    const Proj &p = s->projs[(size_t)pi];
    if (p.kind != PJ_COL) return fail(DFDB_ERR_UNSUPPORTED, "median / quantile take a stored column (materialize a computed column with add_column first)");
    Column *c = s->tbl->find(p.col);
    switch (c->type.kind) {
    case DFDB_I8: case DFDB_I16: case DFDB_I32: case DFDB_I64: case DFDB_U8: case DFDB_U16: case DFDB_U32: case DFDB_U64:
    case DFDB_F32: case DFDB_F64: case DFDB_BOOL:
        *out = c;
        return DFDB_OK;
    default:
        return fail(DFDB_ERR_UNSUPPORTED, "median / quantile over column %s of type %s", c->name.c_str(), c->typestr.c_str());
    }
}

// the isless key of a value's bits at width W = 8 * elsize (see OrderHistArgs) and its inverse
uint64_t order_key(uint64_t b, int kind, int elsize)
{
    const int w = elsize * 8;
    const uint64_t ones = w == 64 ? ~0ull : (1ull << w) - 1, sign = 1ull << (w - 1);
    b &= ones;
    if (kind == DFDB_F32 || kind == DFDB_F64) return b ^ ((b & sign) ? ones : sign);
    if (kind >= DFDB_I8 && kind <= DFDB_I64) return b ^ sign;
    return b;
}
uint64_t order_unkey(uint64_t k, int kind, int elsize)
{
    const int w = elsize * 8;
    const uint64_t ones = w == 64 ? ~0ull : (1ull << w) - 1, sign = 1ull << (w - 1);
    if (kind == DFDB_F32 || kind == DFDB_F64) return (k & sign) ? k ^ sign : k ^ ones;
    if (kind >= DFDB_I8 && kind <= DFDB_I64) return k ^ sign;
    return k;
}

// the key of an agg's minimum / maximum; a zero bound is taken as -0.0 (min) / 0.0 (max) so that both zeros lie inside
uint64_t order_bound_key(const dfdb_agg &w, int kind, int elsize, bool max)
{
    uint64_t b;
    if (kind == DFDB_F64 || kind == DFDB_F32) {
        double d = max ? w.max_f64 : w.min_f64;
        if (d == 0.0) d = max ? 0.0 : -0.0;
        if (kind == DFDB_F64) {
            memcpy(&b, &d, 8);
        } else {
            const float f = (float)d;
            uint32_t u;
            memcpy(&u, &f, 4);
            b = u;
        }
    } else {
        b = (uint64_t)(max ? w.max_i64 : w.min_i64);
    }
    return order_key(b, kind, elsize);
}

// one round over this shard's candidates: the histogram of the next digit of every open prefix (compacting the candidates
// first-hand when they are few), its counts into o.local
int order_launch_round(OrderState &o)
{
    o.open.clear();
    for (uint64_t p : o.pre) o.open.push_back(p);
    std::sort(o.open.begin(), o.open.end());
    o.open.erase(std::unique(o.open.begin(), o.open.end()), o.open.end());
    const int64_t np = (int64_t)o.open.size();
    int bits = 1;
    while (bits < 12 && (np << (bits + 1)) <= ORDER_MAX_BINS) bits++;
    bits = std::min(bits, o.lo);
    o.bits = bits;
    const int64_t nbins = np << bits;
    o.local.assign((size_t)nbins, 0);
    const bool keyed = o.nkeys >= 0;
    const int64_t source = keyed ? o.nkeys : o.col.n;
    // once the open prefixes hold an eighth of the candidates or fewer, this round also writes their keys to a smaller buffer
    // that the later rounds read instead
    const bool compact = o.cand >= 0 && o.cand * 8 <= source && source > 0;
    PoolBuf pre, counts, out;
    if (pre.alloc((size_t)np * 8) != cudaSuccess || counts.alloc((size_t)nbins * 8 + 8) != cudaSuccess)
        return fail(DFDB_ERR_NOMEM, "out of device memory for the radix-select counts");
    if (compact && o.cand > 0 && out.alloc((size_t)o.cand * 8) != cudaSuccess)
        return fail(DFDB_ERR_NOMEM, "out of device memory for %lld candidate keys", (long long)o.cand);
    uint64_t *d_pre = pre.as<uint64_t>(), *d_counts = counts.as<uint64_t>();
    CUDA_TRY(cudaMemcpyAsync(d_pre, o.open.data(), (size_t)np * 8, cudaMemcpyHostToDevice, rt.stream));
    CUDA_TRY(cudaMemsetAsync(d_counts, 0, (size_t)nbins * 8 + 8, rt.stream));
    OrderHistArgs a;
    memset(&a, 0, sizeof a);
    a.values = keyed ? nullptr : o.col.values.as<uint8_t>();
    a.missing = keyed ? nullptr : o.col.missing.as<uint8_t>();
    a.keys = o.keys.as<unsigned long long>();
    a.n = source;
    a.kind = o.col.kind;
    a.elsize = o.col.elsize;
    a.prefixes = reinterpret_cast<const unsigned long long *>(d_pre);
    a.nprefix = (int)np;
    a.hi_shift = o.lo;
    a.bits = bits;
    a.counts = reinterpret_cast<unsigned long long *>(d_counts);
    if (compact) {
        a.out_keys = out.as<unsigned long long>();
        a.out_n = reinterpret_cast<unsigned long long *>(d_counts + nbins);
    }
    {
        PhaseScope ps(PH_ORDER, source * (keyed ? 8 : o.col.elsize + o.col.nullable));
        LAUNCH(launch_order_hist(a, rt.stream));
    }
    int64_t written = 0;
    CUDA_TRY(cudaMemcpyAsync(o.local.data(), d_counts, (size_t)nbins * 8, cudaMemcpyDeviceToHost, rt.stream));
    CUDA_TRY(cudaMemcpyAsync(&written, d_counts + nbins, 8, cudaMemcpyDeviceToHost, rt.stream));
    CUDA_TRY(cudaStreamSynchronize(rt.stream));
    o.round++;
    if (compact) {
        if (written != o.cand) return fail(DFDB_ERR_STATE, "radix select: %lld candidate keys written, %lld expected", (long long)written, (long long)o.cand);
        o.keys = std::move(out);
        o.nkeys = o.cand;
    }
    return DFDB_OK;
}

// takes the global counts of the round in flight: every wanted rank moves to the digit that holds it
int order_advance(OrderState &o, const int64_t *g, int64_t ng)
{
    const int64_t nbins = (int64_t)o.local.size();
    if (ng != nbins) return fail(DFDB_ERR_ARGUMENT, "expected %lld global counts, got %lld", (long long)nbins, (long long)ng);
    if (o.round == 1) {
        int64_t sum = 0;
        for (int64_t i = 0; i < ng; i++) sum += g[i];
        if (sum != o.expect)
            return fail(DFDB_ERR_ARGUMENT, "the global counts hold %lld values but `whole` has %lld non-missing ones (whole is not the fold of every rank's prepare)",
                        (long long)sum, (long long)o.expect);
    }
    const int64_t span = 1ll << o.bits;
    std::vector<int64_t> chosen;                   // bins that hold a wanted rank
    for (size_t i = 0; i < o.pre.size(); i++) {
        const int64_t idx = std::lower_bound(o.open.begin(), o.open.end(), o.pre[i]) - o.open.begin();
        const int64_t *c = g + idx * span;
        int64_t d = 0, cum = 0;
        while (d < span && cum + c[d] < o.rem[i]) cum += c[d++];
        if (d == span) return fail(DFDB_ERR_ARGUMENT, "the global counts do not hold rank %lld (they are not the sum of every rank's local counts)", (long long)o.rem[i]);
        o.rem[i] -= cum;
        o.pre[i] = (o.pre[i] << o.bits) | (uint64_t)d;
        chosen.push_back(idx * span + d);
    }
    std::sort(chosen.begin(), chosen.end());
    chosen.erase(std::unique(chosen.begin(), chosen.end()), chosen.end());
    o.cand = 0;
    for (int64_t b : chosen) o.cand += o.local[(size_t)b];
    o.lo -= o.bits;
    return DFDB_OK;
}

int order_finish(OrderState &o, int64_t *nlocal)
{
    o.result.resize(o.pre.size());
    for (size_t i = 0; i < o.pre.size(); i++) o.result[i] = order_unkey(o.pre[i], o.col.kind, o.col.elsize);
    o.phase = 2;
    o.local.clear();
    *nlocal = 0;
    return DFDB_OK;
}
}  // namespace

int32_t dfdb_scan_order_prepare(dfdb_scan *s, int32_t proj_idx, dfdb_agg *local)
{
    int rc = need_init();
    if (rc) return rc;
    if (!s || !local) return fail(DFDB_ERR_ARGUMENT, "null argument");
    Column *c = nullptr;
    if ((rc = order_column(s, proj_idx, &c))) return rc;
    OrderState &o = s->order;
    o = OrderState();
    // the agg first: it is dfdb_scan_aggregate's, bit for bit (its scan leaves the selection mask alone)
    dfdb_agg agg;
    if ((rc = dfdb_scan_aggregate(s, proj_idx, &agg))) return rc;
    dfdb_table *t = s->tbl;
    int64_t total = 0;
    rc = select_rows(s, &total);                           // (no invalidate_decoded: the aggregate's decode of the column may serve)
    if (rc) return rc;
    ResultCol col;                                         // (the handle's once complete)
    col.set_type(c->type);
    if (total > 0) {
        rc = ensure_decoded(t, {c->id}, projection_scope(s));
        if (rc) return rc;
        if ((rc = col.alloc(total, 0))) return rc;
        {
            PhaseScope ps(PH_CONSUME, total * col.elsize);
            rc = gather_rows(make_geometry(t), selection_rows(s), *c, col);
        }
        if (rc) return rc;
        const cudaError_t e = cudaStreamSynchronize(rt.stream);
        if (e != cudaSuccess) return fail(DFDB_ERR_CUDA, "gather failed: %s", cudaGetErrorString(e));
    }
    o.col = std::move(col);
    o.whole = agg;
    *local = agg;
    return DFDB_OK;
}

int32_t dfdb_scan_order_prepare_all(dfdb_scan *s, int32_t proj_idx, dfdb_agg *whole)
{
    int rc = need_init();
    if (rc) return rc;
    if (!s || !whole) return fail(DFDB_ERR_ARGUMENT, "null argument");
    bool exchange = false;
    if ((rc = exchange_prologue(s, &exchange))) return rc;
    if (!exchange) return dfdb_scan_order_prepare(s, proj_idx, whole);     // unsharded, no communicator: the local agg is the whole
    dfdb_agg mine{};
    rc = dfdb_scan_order_prepare(s, proj_idx, &mine);
    if ((rc = fold_all(rc, mine, "order statistics prepare", whole))) return rc;
    s->order.whole = *whole;
    return DFDB_OK;
}

int32_t dfdb_scan_order_round(dfdb_scan *s, const dfdb_agg *whole, const int64_t *ranks, int32_t nranks, const int64_t *global_counts, int64_t nglobal,
                              int64_t *local_counts, int64_t cap, int64_t *nlocal)
{
    int rc = need_init();
    if (rc) return rc;
    if (!s || !local_counts || !nlocal) return fail(DFDB_ERR_ARGUMENT, "null argument");
    if (cap < DFDB_ORDER_MAX_COUNTS) return fail(DFDB_ERR_ARGUMENT, "local_counts holds %lld counts; a round needs DFDB_ORDER_MAX_COUNTS (%d)", (long long)cap, DFDB_ORDER_MAX_COUNTS);
    OrderState &o = s->order;
    if (o.col.kind == 0) return fail(DFDB_ERR_STATE, "no values prepared on this scan (call dfdb_scan_order_prepare first)");
    *nlocal = 0;
    if (!global_counts) {
        // a new query over the prepared values
        if (!whole || !ranks) return fail(DFDB_ERR_ARGUMENT, "the first round needs `whole` and the ranks");
        if (nranks < 1 || nranks > DFDB_ORDER_MAX_RANKS) return fail(DFDB_ERR_ARGUMENT, "%d ranks (1 to %d per call)", nranks, DFDB_ORDER_MAX_RANKS);
        o.phase = 0;
        if (whole->has_nan) return fail(DFDB_ERR_ARGUMENT, "the column holds NaN: its order statistics are undefined");
        const int64_t n = whole->count - whole->nmissing;
        for (int32_t i = 0; i < nranks; i++)
            if (ranks[i] < 1 || ranks[i] > n) return fail(DFDB_ERR_ARGUMENT, "rank %lld outside [1, %lld]", (long long)ranks[i], (long long)n);
        o.expect = n;
        o.rem.assign(ranks, ranks + nranks);
        const uint64_t kmin = order_bound_key(*whole, o.col.kind, o.col.elsize, false), kmax = order_bound_key(*whole, o.col.kind, o.col.elsize, true);
        if (kmin > kmax) return fail(DFDB_ERR_ARGUMENT, "`whole` has its minimum above its maximum");
        // digits start at the highest bit where min and max differ: every value shares the bits above it
        int b = 0;
        while (b < 64 && ((kmin ^ kmax) >> b) != 0) b++;
        o.lo = b;
        o.pre.assign((size_t)nranks, b >= 64 ? 0 : kmin >> b);
        o.round = 0;
        o.cand = -1;
        o.keys.reset();
        o.nkeys = -1;
        if (o.lo == 0) return order_finish(o, nlocal);         // every value is the same
    } else {
        if (o.phase != 1) return fail(DFDB_ERR_STATE, "no radix-select round is in flight on this scan (start one with global_counts = NULL)");
        o.phase = 0;
        if ((rc = order_advance(o, global_counts, nglobal))) return rc;
        if (o.lo == 0) return order_finish(o, nlocal);
    }
    if ((rc = order_launch_round(o))) return rc;
    memcpy(local_counts, o.local.data(), o.local.size() * 8);
    *nlocal = (int64_t)o.local.size();
    o.phase = 1;
    return DFDB_OK;
}

int32_t dfdb_scan_order_values(dfdb_scan *s, void *values)
{
    if (!s || !values) return fail(DFDB_ERR_ARGUMENT, "null argument");
    const OrderState &o = s->order;
    if (o.phase != 2) return fail(DFDB_ERR_STATE, "the radix select on this scan is not done (run dfdb_scan_order_round until *nlocal == 0)");
    uint8_t *out = static_cast<uint8_t *>(values);
    for (size_t i = 0; i < o.result.size(); i++) memcpy(out + i * (size_t)o.col.elsize, &o.result[i], (size_t)o.col.elsize);   // (little-endian: the low bytes)
    return DFDB_OK;
}

int32_t dfdb_scan_order_stats_all(dfdb_scan *s, const int64_t *ranks, int32_t nranks, void *values)
{
    int rc = need_init();
    if (rc) return rc;
    if (!s || !ranks || !values) return fail(DFDB_ERR_ARGUMENT, "null argument");
    OrderState &o = s->order;
    if (o.col.kind == 0) return fail(DFDB_ERR_STATE, "no values prepared on this scan (call dfdb_scan_order_prepare_all first)");
    bool exchange = false;
    if ((rc = exchange_prologue(s, &exchange))) return rc;
    const dfdb_agg whole = o.whole;
    // record per rank: count of counts | counts (fixed size, so that every rank's all-gather has the same shape)
    std::vector<int64_t> mine(1 + DFDB_ORDER_MAX_COUNTS), sum(DFDB_ORDER_MAX_COUNTS);
    int64_t nlocal = 0;
    const int64_t *global = nullptr;
    for (int round = 0;; round++) {
        rc = dfdb_scan_order_round(s, &whole, ranks, nranks, global, global ? nlocal : 0, mine.data() + 1, DFDB_ORDER_MAX_COUNTS, &nlocal);
        if (exchange) {
            mine[0] = nlocal;
            Records all;
            if ((rc = comm_exchange(rc, mine.data(), mine.size() * 8, "an order statistics round", &all))) return rc;
            std::fill(sum.begin(), sum.end(), 0);
            for (int r = 0; r < nccl.world; r++) {
                const int64_t *theirs = static_cast<const int64_t *>(all.of(r));
                if (theirs[0] != nlocal) return fail(DFDB_ERR_STATE, "ranks disagree on round %d: rank %d has %lld counts, this rank %lld", round, r, (long long)theirs[0], (long long)nlocal);
                for (int64_t i = 0; i < nlocal; i++) sum[(size_t)i] += theirs[1 + i];
            }
            global = sum.data();
        } else {
            if (rc) return rc;
            global = mine.data() + 1;
        }
        if (nlocal == 0) break;
    }
    return dfdb_scan_order_values(s, values);
}

// ---- result arena ------------------------------------------------------------------------------------
int32_t dfdb_host_alloc(int64_t bytes, void **ptr)
{
    int rc = need_init();
    if (rc) return rc;
    if (!ptr || bytes < 0) return fail(DFDB_ERR_ARGUMENT, "bad host allocation request");
    const size_t want = ((size_t)std::max<int64_t>(bytes, 1) + ((1u << 21) - 1)) & ~(size_t)((1u << 21) - 1);   // whole 2 MB pages
    void *p = nullptr;
    size_t cap = 0;
    {
        std::lock_guard<std::mutex> lk(arena.mu);
        auto it = arena.spare.lower_bound(want);
        if (it != arena.spare.end() && it->first <= want + want / 2) {                     // a close enough fit
            p = it->second;
            cap = it->first;
            arena.spare_bytes -= cap;
            arena.spare.erase(it);
        }
    }
    if (!p) {
        cudaError_t e = cudaHostAlloc(&p, want, cudaHostAllocDefault);
        if (e != cudaSuccess) {
            { std::lock_guard<std::mutex> lk(arena.mu); arena.trim(0); }
            e = cudaHostAlloc(&p, want, cudaHostAllocDefault);
        }
        if (e != cudaSuccess) { cudaGetLastError(); return fail(DFDB_ERR_NOMEM, "cannot pin %zu bytes of host memory: %s", want, cudaGetErrorString(e)); }
        cap = want;
    }
    std::lock_guard<std::mutex> lk(arena.mu);
    arena.live[reinterpret_cast<uintptr_t>(p)] = cap;
    *ptr = p;
    return DFDB_OK;
}

int32_t dfdb_host_free(void *ptr)
{
    if (!ptr) return DFDB_OK;
    std::lock_guard<std::mutex> lk(arena.mu);
    auto it = arena.live.find(reinterpret_cast<uintptr_t>(ptr));
    if (it == arena.live.end()) return fail(DFDB_ERR_ARGUMENT, "not a dfdb_host_alloc buffer");
    const size_t cap = it->second;
    arena.live.erase(it);
    if (rt.inited && arena.spare_bytes + cap <= arena.cap_bytes) {
        arena.spare.emplace(cap, ptr);
        arena.spare_bytes += cap;
    } else {
        cudaFreeHost(ptr);
    }
    return DFDB_OK;
}

int32_t dfdb_lz4_classify_block(const uint8_t *comp, int64_t comp_len, int64_t origin)
{
    if (!comp || comp_len < 0 || origin < 0) { fail(DFDB_ERR_ARGUMENT, "bad block"); return -2; }   // (not a DFDB_ERR_* value: those are positive, like the decoders)
    // the header's numbers: 1 = walker, 2 = spec, 3 = long, 4 = bytes (K1's first four), -1 = no verdict
    const std::optional<K1> k = sample_flavour(comp, comp_len, origin);
    return k ? (int)*k + 1 : -1;
}

// ---- codec hook ---------------------------------------------------------------------------------------
int32_t dfdb_lz4_decode_blocks(const uint8_t *comp, const int64_t *comp_off, const int64_t *comp_len, uint8_t *out,
                               const int64_t *out_off, const int64_t *origin, int32_t n, int32_t *status)
{
    int rc = need_init();
    if (rc) return rc;
    if (n <= 0) return DFDB_OK;
    std::vector<int64_t> coff((size_t)n), doff((size_t)n);
    std::vector<int32_t> clen((size_t)n), orig((size_t)n);
    int64_t cpos = 0, dpos = 0;
    for (int i = 0; i < n; i++) {
        if (comp_len[i] < 0 || origin[i] < 0 || comp_len[i] > 0x7F000000LL || origin[i] > 0x7E000000LL) return fail(DFDB_ERR_ARGUMENT, "bad block sizes");
        coff[(size_t)i] = cpos; clen[(size_t)i] = (int32_t)comp_len[i]; cpos += (comp_len[i] + 15) & ~(int64_t)15;
        doff[(size_t)i] = dpos; orig[(size_t)i] = (int32_t)origin[i]; dpos += (origin[i] + 255) & ~(int64_t)255;
    }
    std::vector<uint8_t> packed((size_t)cpos + 4096, 0);
    for (int i = 0; i < n; i++) memcpy(packed.data() + coff[(size_t)i], comp + comp_off[i], (size_t)comp_len[i]);
    uint8_t *d_comp = nullptr, *d_out = nullptr;
    int64_t *d_coff = nullptr, *d_doff = nullptr;
    int32_t *d_clen = nullptr, *d_orig = nullptr, *d_status = nullptr;
    auto cleanup = [&]() { cudaFree(d_comp); cudaFree(d_out); cudaFree(d_coff); cudaFree(d_doff); cudaFree(d_clen); cudaFree(d_orig); cudaFree(d_status); };
    rc = DFDB_OK;
    if (cudaMalloc(reinterpret_cast<void **>(&d_comp), packed.size()) != cudaSuccess ||
        cudaMalloc(reinterpret_cast<void **>(&d_out), (size_t)dpos + 256) != cudaSuccess ||
        cudaMalloc(reinterpret_cast<void **>(&d_status), (size_t)n * 4) != cudaSuccess) {
        cleanup();
        return fail(DFDB_ERR_NOMEM, "out of device memory");
    }
    if ((rc = dev_upload(&d_coff, coff)) || (rc = dev_upload(&d_doff, doff)) || (rc = dev_upload(&d_clen, clen)) || (rc = dev_upload(&d_orig, orig))) {
        cleanup();
        return rc;
    }
    cudaMemcpyAsync(d_comp, packed.data(), packed.size(), cudaMemcpyHostToDevice, rt.stream);
    cudaMemsetAsync(d_status, 0xff, (size_t)n * 4, rt.stream);
    DecodeArgs a;
    memset(&a, 0, sizeof a);
    a.ncols = 1;
    a.nblocks = n;
    a.col[0] = DecodeCol{d_comp, d_coff, d_clen, d_doff, d_orig, d_out, d_status, nullptr};
    // acceptance first (the lane-per-block decoder: LZ4_decompress_safe's rules exactly), then the forced decoder or the walker
    const K1 decoder = forced_decoder().value_or(K1::Walker);
    if (decoder == K1::Lane) a.hot = lane_hot(false);
    std::vector<int32_t> verdict((size_t)n, 0);
    if (decoder != K1::Lane) {
        DecodeArgs va = a;
        if (launch_lz4_decode_lane(va, rt.d_counter, rt.sm_count, rt.stream) != 0) { cleanup(); return fail(DFDB_ERR_CUDA, "decode launch failed"); }
        rt.launches++;
        cudaMemcpyAsync(verdict.data(), d_status, (size_t)n * 4, cudaMemcpyDeviceToHost, rt.stream);
        cudaMemsetAsync(d_status, 0xff, (size_t)n * 4, rt.stream);
        cudaStreamSynchronize(rt.stream);
    }
    if (launch_decode(a, decoder) != 0) { cleanup(); return fail(DFDB_ERR_CUDA, "decode launch failed"); }
    rt.launches++;
    std::vector<uint8_t> hout((size_t)dpos + 256);
    cudaMemcpyAsync(hout.data(), d_out, hout.size(), cudaMemcpyDeviceToHost, rt.stream);
    cudaMemcpyAsync(status, d_status, (size_t)n * 4, cudaMemcpyDeviceToHost, rt.stream);
    cudaError_t e = cudaStreamSynchronize(rt.stream);
    cleanup();
    if (e != cudaSuccess) return fail(DFDB_ERR_CUDA, "decode failed: %s", cudaGetErrorString(e));
    for (int i = 0; i < n; i++) {
        if (status[i] == 0 && verdict[(size_t)i] == 0) memcpy(out + out_off[i], hout.data() + doff[(size_t)i], (size_t)origin[i]);
        else status[i] = DFDB_ERR_CORRUPT;
    }
    return DFDB_OK;
}

}  // extern "C"
