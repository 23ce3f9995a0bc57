// lz4_decode_spec.cu -- K1 for word-regular columns: one warp per column block, token positions VERIFIED instead of walked.
//
// Replaces read_block's LZ4_decompress_safe call (/root/reference/src/io/BlockStreams.jl:101-119) for the column kind that
// dominates the benchmark: 8-byte values whose LZ4 stream is almost entirely "plain" sequences -- token 0x04 / 0x0C (no
// literals, match of 8 or 16 bytes), a two-byte offset that is a multiple of 8.  Such a sequence is exactly 3 stream bytes, so
// inside a run of them token k sits at p0 + 3k: nobody has to walk the chain.  Every lane reads the three bytes at its assumed
// position and checks that they ARE a plain sequence; by induction from lane 0 (whose position is known) the first lane that
// fails the check ends the run, and every lane before it is a real sequence.  Lane = sequence = output word.  A source word
// before the batch is final in global memory (L2); a source word inside the batch is another lane's word, and chains of those
// collapse by pointer jumping over warp shuffles.  The run may be closed by one sequence of the "word form" -- up to 5 literal
// bytes followed by a match, 8 or 16 bytes in all ((1, 7), (2, 6), (0, 16) ...) -- which its own lane expands.  One coalesced
// store per batch; the next batch's stream bytes are requested before this batch's sources are waited for.  Anything else --
// length extensions, unaligned offsets, the last sequences of the block -- is decoded one sequence at a time by the whole
// warp (decode_one_sequence, lz4_common.cuh).
//
// Three batch shapes, in order of frequency on rand(1:100): 32 one-word sequences (the full batch, compiled on its own: ~71
// instructions + 6 per jump round for 256 output bytes); a full batch that holds ONE two-word sequence (match of 16 - L0 bytes:
// same stream stride, the lanes behind it shift by one word); a run that ends inside the batch, with its closing sequence.
// Against the walker / consumer kernel (lz4_decode_v3.cu, ~350 warp instructions per 32 tokens: ring entries, polls, dependency
// waves) this is ~125 instructions per batch on average, 5 CTAs x 8 warps per SM at 48 registers; the kernel is issue-bound
// (IPC 2.95) and its time follows its instruction count: 5.66 ms per 1e9 rows against 13.1 ms (DESIGN.md has the history).  The
// kernel is memory-safe on any input (every access is bounds-checked, errors set a per-block status); the accept / reject
// verdict of damaged streams is the lane decoder's, taken at load (api.cu).  The same file holds the long-sequence decoder
// (lz4_decode_long_kernel).
//
// Algorithmic bytes per block (roofline): compressed bytes read + origin bytes written.
#include <cuda_runtime.h>

#include <type_traits>

#include "kernels.cuh"
#include "lz4_common.cuh"

namespace dfdb {
namespace {

using namespace lz4;

constexpr int SPEC_WARPS = 8;
static_assert(SPEC_WARPS * 5 == LZ4_SPEC_WARPS_PER_SM, "the launch bounds below keep 5 CTAs per SM");
constexpr uint32_t SPEC_RING = 512;      // per warp: the last output words of its block, in shared memory (match sources are nearly always recent)
constexpr uint32_t SPEC_SMEM = (SPEC_WARPS + 1) * SPEC_RING * 8;   // dynamic shared memory per CTA: the rings + alignment slack
constexpr uint32_t SPEC_NEAR = SPEC_RING - 64;   // a source at most this many words back is read from the ring (the margin keeps this batch's stores off it)

__device__ __forceinline__ uint32_t ldg_u32(const uint8_t *p) { return __ldg(reinterpret_cast<const unsigned int *>(p)); }

// the 8 stream bytes at tp = ip + stride * lane (three aligned words; payload buffers carry slack behind the last block, so reading a
// few words past this block's payload is safe -- such bytes are never USED: the fast path checks the positions first)
__device__ __forceinline__ uint64_t load_stream_at(const uint8_t *__restrict__ src, uint32_t tp)
{
    const uint8_t *a = src + (tp & ~3u);
    const uint32_t sh = tp * 8u;             // (the funnel shift takes it modulo 32)
    const uint32_t w0 = ldg_u32(a), w1 = ldg_u32(a + 4), w2 = ldg_u32(a + 8);
    return (uint64_t)__funnelshift_r(w0, w1, sh) | ((uint64_t)__funnelshift_r(w1, w2, sh) << 32);
}

// Requests the 512-byte group g + 2 of the stream (four 128-byte lines) from HBM into L2, ahead of the position.  A real call on
// purpose: inlined, the few instructions are predicated and cost their issue slots in every batch; as a call they cost a branch
// that is taken once in about five batches.
static __device__ __noinline__ void prefetch_group(const uint8_t *src, uint32_t g, uint32_t lane)
{
    if (lane < 4u) asm volatile("prefetch.global.L2 [%0];" ::"l"(src + ((g + 2u) << 9) + 128u * lane));
}

// Predicate bits (DecodeArgs::bits): the verdict of bits_test on output words [w0, w1) of the block (w0 a multiple of 32), one
// mask word per 32 words, bits at and past w1 zero.  A word at or past ring_from is read from the ring -- the caller
// guarantees it is still there --, any other from global memory (final there: the warp wrote it before its last __syncwarp).
// Real calls, like prefetch_group: the batch loop pays one compare and a branch taken once in eight batches.
static __device__ __noinline__ void flush_bits(const DecodeArgs &args, const unsigned long long *out64, uint32_t *mw, uint32_t w0, uint32_t w1,
                                               uint32_t ring_from)
{
    extern __shared__ unsigned char spec_dyn[];
    const uint32_t ring_s = ((smem_addr(spec_dyn) + SPEC_RING * 8u - 1u) & ~(SPEC_RING * 8u - 1u)) + (threadIdx.x >> 5) * (SPEC_RING * 8u);
    const uint32_t lane = lane_id();
    for (uint32_t g = w0; g < w1; g += 32u) {
        const uint32_t w = g + lane;
        bool p = false;
        if (w < w1) {
            unsigned long long v;
            if (w >= ring_from) asm volatile("ld.shared.u64 %0, [%1];" : "=l"(v) : "r"(((w << 3) & ((SPEC_RING - 1u) << 3)) | ring_s) : "memory");
            else v = __ldcg(out64 + w);
            p = coltest_pass(args.bits_test, v);
        }
        const uint32_t m = __ballot_sync(FULL, p);
        if (lane == 0) mw[g >> 5] = m;
    }
}
// The flush a batch makes with an integer interval test (BITS == 1): the whole 256-word chunk at w0, all in the ring (2 KB
// of its 4 KB, in one piece): eight shared loads at fixed offsets, a subtract + compare and a ballot each, two 16-byte stores
// (the block's mask words are a multiple of four).  The interval comes in registers: the test's fields are kernel
// parameters, which a called function could only read through generic loads.
static __device__ __noinline__ void flush_chunk(uint32_t *mw, uint32_t w0, unsigned long long lo, unsigned long long span)
{
    extern __shared__ unsigned char spec_dyn[];
    const uint32_t ring_s = ((smem_addr(spec_dyn) + SPEC_RING * 8u - 1u) & ~(SPEC_RING * 8u - 1u)) + (threadIdx.x >> 5) * (SPEC_RING * 8u);
    const uint32_t lane = lane_id();
    const uint32_t a0 = ring_s + ((w0 & (SPEC_RING - 1u)) + lane) * 8u;
    uint32_t m[8];
#pragma unroll
    for (int k = 0; k < 8; k++) {
        unsigned long long v;
        asm volatile("ld.shared.u64 %0, [%1];" : "=l"(v) : "r"(a0 + 256u * k) : "memory");
        m[k] = __ballot_sync(FULL, v - lo <= span);
    }
    if (lane == 0) {
        uint4 *d = reinterpret_cast<uint4 *>(mw + (w0 >> 5));
        d[0] = make_uint4(m[0], m[1], m[2], m[3]);
        d[1] = make_uint4(m[4], m[5], m[6], m[7]);
    }
}

// one block, whole warp; returns E_*.  (Positions are 32-bit in the batch loop: column blocks are far below 4 GB; the kernel
// is instruction-bound -- IPC 2.9 per SM in the first profile -- so the loop is kept lean.)
//
// Fusing the predicate + aggregate scan into this kernel was built in three forms; each lost to a decode followed by a separate
// scan and was removed (DESIGN.md section 8 has the measurements).  What stayed is BITS: the decoder evaluates the predicate
// on the words it has just written, still in its ring, and writes the selection bits, so that the scan reads only the
// aggregated column.  Each 256-word chunk of the output is flushed once, by the step that moves the position past its end:
// a batch (at most 33 words, so the chunk is still in the ring) or a one-sequence step (from global memory).  The caller
// flushes the last partial chunk.  BITS: 0 = the plain decoder, 1 = an integer interval test, 2 = any test.
template <int BITS>
__device__ int decode_block_spec(const DecodeArgs &args, uint32_t *mw, const uint8_t *__restrict__ src, uint32_t comp_len, uint8_t *dst, uint32_t origin,
                                 uint32_t ring_s)
{
    uint32_t lane = lane_id();
    asm volatile("" : "+r"(lane));           // (kept in a register instead of an S2R in every batch)
    uint32_t ip = 0, op = 0;
    bool done = false;
    unsigned long long *out64 = reinterpret_cast<unsigned long long *>(dst);
    // A run is a stretch of sequences of ONE shape: L0 literal bytes (0..4) + a match of 8 - L0 bytes, offset a multiple of 8,
    // at an aligned output position -- 3 + L0 stream bytes and one output word each.  rand(1:100) Int64 columns are runs of
    // L0 = 0 (token 0x04), sorted Int64 columns runs of L0 = 2 (token 0x22).  The stride of the last run is assumed for the next
    // batch (its bytes are requested early); two sequences of another shape in a row switch the run's shape.
    uint32_t L0 = 0, pendL = 0xffu;
    uint32_t tok0 = 0x04u, sh0 = 8u;       // the run's token, where its offset sits in the lane's stream bytes, the bytes a word takes from its source
    unsigned long long kp0 = ~0ull;
    uint32_t ring_from = 0;            // output words >= this one (and within SPEC_RING of the position) are in the ring
    // a match never writes the block's last 12 bytes in the fast path (the end-of-block rules stay with the one-sequence path):
    // an output word w may be written when w < lim_w; and the fast path needs 7 * 32 + 16 stream bytes ahead
    uint32_t lim_w = origin >= 12u ? (origin - 12u) >> 3 : 0u;
    asm volatile("" : "+r"(lim_w));          // (kept in a register: ptxas otherwise recomputes it -- and ring_s, 11 instructions -- in every batch)
    int32_t ip_lim = comp_len >= 7u * 32u + 16u ? (int32_t)(comp_len - (7u * 32u + 16u)) : -1;     // (-1: the block is too short for the fast path)
    asm volatile("" : "+r"(ip_lim));         // (kept in a register: ptxas otherwise recomputes it in every batch)
    // a source word: from the ring when it is recent, else from global memory (final there: L2).  ring_s, the ring's address in
    // the shared window, is a multiple of the ring's 4 KB (the kernel aligns it at run time), so a word's slot is one LOP3 away
    // from its index.
    asm volatile("" : "+r"(ring_s));
    auto ring_slot = [&](uint32_t w) -> uint32_t { return ((w << 3) & ((SPEC_RING - 1u) << 3)) | ring_s; };
    auto source = [&](uint32_t sw, uint32_t opw) -> unsigned long long {
        unsigned long long v;
        if (sw >= ring_from && opw - sw <= SPEC_NEAR) asm volatile("ld.shared.u64 %0, [%1];" : "=l"(v) : "r"(ring_slot(sw)) : "memory");
        else v = __ldcg(out64 + sw);
        return v;
    };
    auto put = [&](uint32_t w, unsigned long long v) {
        out64[w] = v;
        asm volatile("st.shared.u64 [%0], %1;" ::"r"(ring_slot(w)), "l"(v) : "memory");
    };
    // the compressed bytes are read exactly once, so each batch would wait a DRAM round trip for its own bytes: the stream is
    // pulled from HBM into L2 two to three 512-byte groups ahead of the position, one request per 128-byte line
    if (lane < 12u) asm volatile("prefetch.global.L2 [%0];" ::"l"(src + 128u * lane));
    uint32_t tp = 3u * lane;                 // where this lane's sequence starts in the stream: ip + stride * lane
    uint64_t x = load_stream_at(src, tp);
    // What every batch does once it knows its shape: ask for the next batch's stream bytes (they travel while this batch's
    // sources do) and, on entering a new 512-byte group of the stream, for the group after the next.
    auto advance_stream = [&](uint32_t adv, bool restride) -> uint64_t {
        const uint32_t nip = ip + adv;
        tp = restride ? nip + (3u + L0) * lane : tp + adv;
        const uint64_t nx = load_stream_at(src, tp);
        if ((nip ^ ip) >> 9) prefetch_group(src, nip >> 9, lane);
        ip = nip;
        return nx;
    };
    // what every batch does last: move the position, and flush the chunk it finishes
    auto advance_op = [&](uint32_t adv) {
        const uint32_t nop = op + adv;
        if (BITS && ((nop ^ op) >> 11)) {
            const uint32_t w0 = ((nop >> 11) << 8) - 256u;
            if (BITS == 1 && w0 >= ring_from)
                flush_chunk(mw, w0, (unsigned long long)args.bits_test.lo_i, (unsigned long long)args.bits_test.hi_i - (unsigned long long)args.bits_test.lo_i);
            else
                flush_bits(args, out64, mw, w0, w0 + 256u, ring_from);
        }
        op = nop;
    };
    while (!done) {
        bool batch = false;
        if ((op & 7u) == 0 && (int32_t)ip <= ip_lim) {
            const uint32_t opw = op >> 3;
            const uint32_t tok = (uint32_t)x & 0xffu;
            const uint32_t off = (uint32_t)(x >> sh0) & 0xffffu;
            // offset a multiple of 8, not zero, inside the output: rotate the low three bits to the top -- any of them set, or a
            // zero offset (minus one wraps), fails the one comparison; for the lanes that pass, offr is the offset in words
            const uint32_t offr = __funnelshift_r(off, off, 3);
            const bool okp = tok == tok0 && offr - 1u < opw + lane && opw + lane < lim_w;
            const uint32_t badp = ~__ballot_sync(FULL, okp);
            if (!badp) {
                // ---- a full batch of 32 one-word sequences: lane = sequence = output word ----
                pendL = 0xffu;
                const uint64_t nx = advance_stream(32u * (3u + L0), false);
                // Sources.  A source inside the batch is another lane's word, and only the bytes behind the literal bytes come
                // from it, so a chain of in-batch sources ends in the word of its far root: the chains collapse by pointer jumping
                // over the word INDEX (<= 5 rounds, one shuffle each), and every lane then fetches its root itself.
                const uint32_t myw = opw + lane;
                uint32_t s = myw - offr;
                bool inb = s >= opw;
                while (__any_sync(FULL, inb)) {
                    const uint32_t t = __shfl_sync(FULL, s, s - opw);
                    if (inb) { s = t; inb = s >= opw; }
                }
                const unsigned long long v = source(s, opw);
                put(myw, (v & kp0) | ((unsigned long long)(x >> 8) & ~kp0));
                __syncwarp();                                                   // the batch's words are visible to the whole warp
                advance_op(256u);
                x = nx;
                batch = true;
            } else {
                // One lane fails, and only because its match is 16 - L0 bytes instead of 8 - L0 -- same stream stride, two output
                // words, 1 % of the tokens of rand(1:100) and the end of a quarter of its batches --, with both sources before the
                // batch: the batch stays whole.  Lanes behind it sit one word further on; the owner of an in-batch source word q is
                // lane q up to it, lane q - 1 behind it, and word z + 1 is that sequence's second word (source: the word after its first).
                uint32_t z = 32u;
                if ((badp & (badp - 1u)) == 0) {
                    const uint32_t zz = (uint32_t)__ffs(badp) - 1u;
                    const bool two = lane == zz && tok == tok0 + 8u && offr - 1u < opw + lane && offr >= zz + 2u;
                    if (__ballot_sync(FULL, two) && opw + 33u <= lim_w) z = zz;
                }
                // Or the one lane that fails is a (1, 7) sequence in a run of plain matches (L0 = 0: LZ4 missed a value and emitted
                // its first byte as a literal): one stream byte more, so the lanes behind it find their sequence one byte further on
                // -- in the eight stream bytes they already hold -- and one output word like everybody else.  The batch stays whole
                // if they all check out from there and none of them copies that word (its literal byte is not in its source).
                uint32_t zb = 32u;
                const uint32_t offr1 = __funnelshift_r((uint32_t)(x >> 16) & 0xffffu, (uint32_t)(x >> 16) & 0xffffu, 3);
                if (z == 32u && tok0 == 0x04u) {
                    const uint32_t zz = (uint32_t)__ffs(badp) - 1u;
                    const bool pos_ok = offr1 - 1u < opw + lane && opw + lane < lim_w;
                    const bool c = lane < zz || (pos_ok && (lane == zz ? tok == 0x13u : (((uint32_t)(x >> 8) & 0xffu) == 0x04u && offr1 != lane - zz)));
                    if (__all_sync(FULL, c)) zb = zz;
                }
                if (zb < 32u) {
                    // ---- a full batch with one (1, 7) sequence in it ----
                    pendL = 0xffu;
                    const uint64_t nx = advance_stream(32u * 3u + 1u, false);
                    const uint32_t myw = opw + lane;
                    uint32_t s = myw - (lane >= zb ? offr1 : offr);
                    bool inb = s >= opw;
                    while (__any_sync(FULL, inb)) {
                        const uint32_t t = __shfl_sync(FULL, s, s - opw);
                        if (inb) { s = t; inb = s >= opw; }
                    }
                    unsigned long long v = source(s, opw);
                    if (lane == zb) v = (v & ~0xffull) | ((unsigned long long)(x >> 8) & 0xffull);
                    put(myw, v);
                    __syncwarp();                                               // the batch's words are visible to the whole warp
                    advance_op(256u);
                    x = nx;
                    batch = true;
                } else if (z < 32u) {
                    // ---- a full batch with one two-word sequence in it ----
                    pendL = 0xffu;
                    const uint64_t nx = advance_stream(32u * (3u + L0), false);
                    const uint32_t myw = opw + lane + (lane > z ? 1u : 0u);
                    uint32_t s = myw - offr;
                    bool inb = s >= opw;                                            // (never lane z)
                    while (__any_sync(FULL, inb)) {
                        const uint32_t q = s - opw;
                        const uint32_t t = __shfl_sync(FULL, s, q - (q > z ? 1u : 0u));
                        if (inb) { s = t + (q == z + 1u ? 1u : 0u); inb = s >= opw; }
                    }
                    const unsigned long long v = source(s, opw);
                    put(myw, (v & kp0) | ((unsigned long long)(x >> 8) & ~kp0));
                    if (lane == z) put(myw + 1u, source(s + 1u, opw));
                    __syncwarp();                                                   // the batch's words are visible to the whole warp
                    advance_op(264u);
                    x = nx;
                    batch = true;
                } else {
                    // ---- the run ends inside the batch: n one-word sequences, then maybe one closing sequence of another word form ----
                    // (Keeping sequences of 16 - L0 match bytes -- two words, same stream stride -- inside the run was built and
                    // measured: 13 % fewer batches, but the bookkeeping (first-word masks, owner lookup, truncation at 32 words) made
                    // every such batch dearer; 5.6 G instead of 4.9 G warp instructions per 1e9 rows.  They close the run like any
                    // other shape.)
                    const uint32_t n = (uint32_t)__ffs(badp) - 1u;
                    const uint32_t myw = opw + lane;
                    // the sequence that ends the run, analysed by its own lane: any "word form" -- L <= 5 literal bytes + match, 8 or 16 bytes in all
                    const uint32_t L = tok >> 4, LM = L + (tok & 15u) + 4u;
                    // (its offset: stream bytes L + 1 and L + 2 of the lane's eight, picked by one PRMT -- a 64-bit variable shift is a dozen instructions)
                    const uint32_t off_s = __byte_perm((uint32_t)x, (uint32_t)(x >> 32), 0x4421u + 0x11u * L) & 0xffffu, offw_s = off_s >> 3;
                    const uint32_t Wc = LM >> 3;
                    const bool sp = lane == n && L <= 5u && (LM == 8u || LM == 16u) && (off_s & 7u) == 0 && off_s != 0 &&
                                    offw_s <= myw && offw_s >= lane + Wc &&                    // sources inside the output and final (before the batch)
                                    myw + Wc <= lim_w;
                    uint32_t hdr_s = 0, W_s = 0;
                    if (__ballot_sync(FULL, sp)) {
                        const uint32_t pk = __shfl_sync(FULL, (L << 8) | Wc, n);
                        hdr_s = 3u + (pk >> 8);
                        W_s = pk & 0xffu;
                    }
                    if (n + W_s > 0) {
                        const uint32_t stride = 3u + L0;
                        const unsigned long long kp = sp ? ~0ull << (8u * L) : kp0;   // the bytes a word takes from its source (the others are literals)
                        // a sequence of another one-word shape alone at the head of a batch is just the closing sequence of an empty run;
                        // two of the same shape in a row are a new run: switch (the bytes requested next use the new stride)
                        if (n == 0 && W_s == 1u) {
                            const uint32_t Lh = hdr_s - 3u;
                            if (Lh == pendL && Lh <= 4u) {
                                L0 = Lh;
                                tok0 = (L0 << 4) | (4u - L0); sh0 = 8u + 8u * L0; kp0 = ~0ull << (8u * L0);
                            }
                            pendL = Lh;
                        } else {
                            pendL = 0xffu;
                        }
                        const uint64_t nx = advance_stream(stride * n + hdr_s, stride != 3u + L0);
                        const bool mine = lane < n;
                        uint32_t s = myw - (sp ? offw_s : offr);
                        bool inb = mine && s >= opw;
                        while (__any_sync(FULL, inb)) {
                            const uint32_t t = __shfl_sync(FULL, s, s - opw);
                            if (inb) { s = t; inb = s >= opw; }
                        }
                        if (mine || sp) {
                            const unsigned long long v = source(s, opw);
                            put(myw, (v & kp) | ((unsigned long long)(x >> 8) & ~kp));
                        }
                        if (W_s == 2u && sp) put(myw + 1u, source(s + 1u, opw));    // a closing sequence of two words
                        __syncwarp();                                               // the batch's words are visible to the whole warp
                        advance_op(8u * (n + W_s));
                        x = nx;
                        batch = true;
                    }
                }
            }
        }
        if (!batch) {
            // ---- anything else: one sequence, whole warp ----
            int64_t ip64 = ip, op64 = op;
            const int e = decode_one_sequence(src, comp_len, dst, origin, ip64, op64, done);
            if (e) return e;
            ip = (uint32_t)ip64;
            if (BITS && ((op ^ (uint32_t)op64) >> 11)) flush_bits(args, out64, mw, (op >> 11) << 8, ((uint32_t)op64 >> 11) << 8, ~0u);
            op = (uint32_t)op64;
            ring_from = (op + 7u) >> 3;                                         // (what this path wrote is in global memory only)
            tp = ip + (3u + L0) * lane;
            x = load_stream_at(src, tp);
        }
    }
    return (op == origin && ip == comp_len) ? E_OK : E_SIZE;
}

// ---- long-sequence columns: one sequence at a time, the stream parsed out of shared memory -------------------------------------
// Union{Float64,Missing} bodies, decimal strings, anything whose sequences are long (tens of bytes: a literal run with a length
// extension, a match): there are few tokens per output byte, so the token chain is not the problem -- the LATENCY of reading it is.
// decode_one_sequence fetches token, extension bytes and offset from global memory, three dependent round trips to L2 per
// sequence (~2 000 cycles); the walker / consumer kernel parks its walker lane at every length extension.  Here the warp keeps a
// 4 KB circular window of the stream in shared memory (the spec decoder's ring, unused in this mode), filled 512 bytes at a time
// with cp.async two kilobytes ahead of the position, and parses the headers out of it: a sequence costs a few shared-memory
// reads plus its copies, which are fire-and-forget (literals: stream -> output, the lines are in L2 because the window fetched
// them; match: output -> output through L2, ordered by __syncwarp).  Same safety contract as every decoder here.
constexpr uint32_t LW = SPEC_RING * 8u;      // window bytes (4 KB), a power of two
constexpr uint32_t LW_CHUNK = 512u;          // one warp-wide cp.async: 32 lanes x 16 bytes
constexpr uint32_t LW_AHEAD = 2048u;         // how far ahead of the position the window is requested

__device__ int decode_block_long(const uint8_t *__restrict__ src, uint32_t comp_len, uint8_t *dst, uint32_t origin, uint32_t win_s)
{
    const uint32_t lane = lane_id();
    uint32_t ip = 0, op = 0;
    uint32_t issued = 0;                     // stream bytes [.., issued) are in the window or on their way (multiple of LW_CHUNK)
    uint32_t ready = 0;                      // stream bytes [.., ready) are in the window for sure
    auto request = [&](uint32_t upto) {      // ask for chunks until `upto` is covered (the payload slot is padded, the buffer has slack behind it)
        while (issued < upto) {
            const uint32_t pos = issued + 16u * lane;
            asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(win_s + (pos & (LW - 1u))), "l"(src + pos) : "memory");
            asm volatile("cp.async.commit_group;" ::: "memory");        // one group per chunk: chunks complete in order
            issued += LW_CHUNK;
        }
    };
    auto need = [&](uint32_t upto) {         // make sure bytes [ip, upto) can be read from the window
        if (upto > ready) {
            if (upto > issued) request((upto + LW_CHUNK - 1u) & ~(LW_CHUNK - 1u));
            // wait for no more than the chunks that are needed: the youngest ones (requested LW_AHEAD ahead) stay in flight
            const uint32_t young = (issued - upto) / LW_CHUNK;          // whole chunks behind `upto` that may remain pending
            if (young >= 3u) { asm volatile("cp.async.wait_group 3;" ::: "memory"); ready = issued - 3u * LW_CHUNK; }
            else if (young == 2u) { asm volatile("cp.async.wait_group 2;" ::: "memory"); ready = issued - 2u * LW_CHUNK; }
            else if (young == 1u) { asm volatile("cp.async.wait_group 1;" ::: "memory"); ready = issued - LW_CHUNK; }
            else { asm volatile("cp.async.wait_group 0;" ::: "memory"); ready = issued; }
            __syncwarp();
        }
    };
    auto wbyte = [&](uint32_t pos) -> uint32_t {
        uint32_t v;
        asm volatile("ld.shared.u8 %0, [%1];" : "=r"(v) : "r"(win_s + (pos & (LW - 1u))) : "memory");
        return v;
    };
    // length extension bytes (add bytes while they are 255), 32 at a time out of the window
    auto length_ext = [&](uint32_t &len) -> bool {
        for (;;) {
            need(ip + 32u);
            const uint32_t p = ip + lane;
            const uint32_t b = p < comp_len ? wbyte(p) : 0u;          // past the end reads as a terminator and is caught below
            const uint32_t stop = __ballot_sync(FULL, b != 255u);
            if (stop == 0) { len += 255u * 32u; ip += 32u; if (ip >= comp_len || len > 0x7f000000u) return false; continue; }
            const uint32_t f = (uint32_t)__ffs(stop) - 1u;
            const uint32_t last = __shfl_sync(FULL, b, f);
            if (ip + f >= comp_len) return false;
            len += 255u * f + last;
            ip += f + 1u;
            return true;
        }
    };
    // four stream bytes at any position of the window (two aligned words, funnel shift)
    auto wword = [&](uint32_t pos) -> uint32_t {
        uint32_t w0, w1;
        asm volatile("ld.shared.u32 %0, [%1];" : "=r"(w0) : "r"(win_s + (pos & (LW - 4u))) : "memory");
        asm volatile("ld.shared.u32 %0, [%1];" : "=r"(w1) : "r"(win_s + ((pos + 4u) & (LW - 4u))) : "memory");
        return __funnelshift_r(w0, w1, pos * 8u);
    };
    // A short match (<= 32 bytes: one byte per lane) is loaded when it is parsed and STORED two sequences later, after the headers
    // of the next two have been parsed: the L2 round trip of its source runs under those parses instead of stalling the warp.
    // Nothing can observe the delay: a pending match is stored before anything reads what it writes (the check below), and
    // stores of different sequences never overlap.  Two slots that swap roles from one sequence to the next (the loop body is
    // instantiated twice) -- moving a pending value from a "younger" to an "older" register would wait for its load.
    struct Pend { uint32_t pos = 0, len = 0, val = 0; };
    Pend pa, pb;
    auto store = [&](Pend &p) {
        if (p.len) {
            if (lane < p.len) dst[p.pos + lane] = (uint8_t)p.val;
            p.len = 0;
            __syncwarp();
        }
    };
    // one sequence; `mine` holds the match of two sequences ago (stored here, then reused), `other` the previous one's.
    // returns 0: go on, 1: the block's last sequence is done, < 0: -E_*
    auto step = [&](Pend &mine, Pend &other) -> int {
        // keep the window LW_AHEAD ahead; never request past what the window can hold beyond the position
        if (issued < ip + LW_AHEAD && issued + LW_CHUNK <= (ip & ~(LW_CHUNK - 1u)) + LW) request(issued + LW_CHUNK);
        if (ip >= comp_len) return -E_TRUNCATED;
        need(ip + 4u);
        const uint32_t token = wbyte(ip);
        ip += 1u;
        uint32_t L = token >> 4;
        if (L == 15u && !length_ext(L)) return -E_TRUNCATED;
        if (L > comp_len - ip) return -E_TRUNCATED;
        if (L > origin - op) return -E_OVERFLOW;
        store(mine);
        if (L > 0) {
            if (L <= 1024u) {
                // literals out of the window (they are stream bytes, no round trip to L2): bytes up to the output's next 4-byte
                // boundary, whole words, the bytes behind the last whole word
                need(ip + L);
                uint8_t *d = dst + op;
                const uint32_t head = min((uint32_t)(-(intptr_t)d) & 3u, L), words = (L - head) >> 2, tail0 = head + 4u * words;
                if (lane < head) d[lane] = (uint8_t)wbyte(ip + lane);
#pragma unroll 1
                for (uint32_t i = lane; i < words; i += 32u) reinterpret_cast<uint32_t *>(d + head)[i] = wword(ip + head + 4u * i);
                if (lane < L - tail0) d[tail0 + lane] = (uint8_t)wbyte(ip + tail0 + lane);
            } else {
                warp_copy(dst + op, src + ip, (int64_t)L);
            }
        }
        ip += L;
        op += L;
        if (ip == comp_len) return 1;                                  // last sequence: literals only
        if (ip + 2u > comp_len) return -E_TRUNCATED;
        if (ip >= issued) {                                            // a long literal run left the window behind: restart it at the position
            asm volatile("cp.async.wait_all;" ::: "memory");
            __syncwarp();
            issued = ready = ip & ~(LW_CHUNK - 1u);
        }
        need(ip + 3u);
        const uint32_t off = wbyte(ip) | (wbyte(ip + 1u) << 8);
        ip += 2u;
        uint32_t M = token & 15u;
        if (M == 15u && !length_ext(M)) return -E_TRUNCATED;
        M += 4u;
        if (off == 0 || off > op) return -E_OFFSET;
        if (M > origin - op) return -E_OVERFLOW;
        // a source that the previous sequence's pending match has yet to write: store that one first
        // (source = [op - off, op - off + min(M, off)), pending = [other.pos, other.pos + other.len))
        if (other.len && off > op - (other.pos + other.len) && off - min(M, off) < op - other.pos) store(other);
        __syncwarp();                                                  // literal bytes (and stored matches) visible to the whole warp
        // every source byte is < op, i.e. already final or just stored: the copy is fully parallel even when it overlaps
        const uint8_t *m_src = dst + op - off;
        if (M <= 32u) {
            if (off >= M) { if (lane < M) mine.val = __ldcg(m_src + lane); }
            else if (lane < M) mine.val = __ldcg(m_src + lane % off);
            mine.pos = op;
            mine.len = M;
        } else {
            store(other);
            uint8_t *m_dst = dst + op;
            if (off >= M) {
#pragma unroll 2
                for (uint32_t i = lane; i < M; i += 32u) m_dst[i] = __ldcg(m_src + i);
            } else {
#pragma unroll 1
                for (uint32_t i = lane; i < M; i += 32u) m_dst[i] = __ldcg(m_src + (i % off));
            }
            __syncwarp();
        }
        op += M;
        return 0;
    };
    request(LW_AHEAD);
    for (;;) {
        int r = step(pa, pb);
        if (r == 0) r = step(pb, pa);
        if (r < 0) return -r;
        if (r > 0) break;
    }
    store(pa);
    store(pb);
    asm volatile("cp.async.wait_all;" ::: "memory");
    return (op == origin && ip == comp_len) ? E_OK : E_SIZE;
}

// 5 CTAs x 8 warps per SM at 48 registers (DESIGN.md has the measurements of 4 and 6).  BITS != 0: args.bits is set (one
// column), see decode_block_spec.
template <int BITS>
__global__ void __launch_bounds__(SPEC_WARPS * 32, 5) lz4_decode_spec_kernel(const __grid_constant__ DecodeArgs args, unsigned int *counter)
{
    // the rings: dynamic shared memory, aligned HERE to the ring size (the shared window starts behind the 1 KB the system
    // reserves, so a declared alignment does not give an aligned address; the launcher adds one ring of slack)
    extern __shared__ unsigned char spec_dyn[];
    const uint32_t ring_s = ((smem_addr(spec_dyn) + SPEC_RING * 8u - 1u) & ~(SPEC_RING * 8u - 1u)) + (threadIdx.x >> 5) * (SPEC_RING * 8u);
    const uint32_t lane = lane_id();
    const long long njobs = (long long)args.ncols * args.nblocks;
    for (;;) {
        unsigned int job = 0;
        if (lane == 0) job = atomicAdd(counter, 1u);
        job = __shfl_sync(FULL, job, 0);
        if ((long long)job >= njobs) return;
        const int c = (int)(job % args.ncols);
        const int b = args.blk0 + (int)(job / args.ncols);
        const DecodeCol &col = args.col[c];
        if (col.skip && col.skip[b]) continue;
        const uint8_t *src = col.comp + col.comp_off[b];
        uint8_t *dst = col.out + col.dec_off[b];
        const uint32_t comp_len = (uint32_t)col.comp_len[b], origin = (uint32_t)col.origin[b];
        uint32_t *mw = BITS ? args.bits + (size_t)b * args.bits_wpb : nullptr;
        int e;
        if (origin == 0) e = (comp_len == 1 && src[0] == 0) ? E_OK : E_SIZE;
        else if (comp_len == 0) e = E_TRUNCATED;
        else if (((uintptr_t)src & 3u) || ((uintptr_t)dst & 7u)) e = decode_simple(src, comp_len, dst, origin);
        else e = decode_block_spec<BITS>(args, mw, src, comp_len, dst, origin, ring_s);
        // the chunks that no step finished: the last partial one, or all of them after the one-sequence decoder (its output
        // slots are 8-byte aligned in every layout that asks for bits)
        if (BITS && e == E_OK) {
            const uint32_t from = ((uintptr_t)src & 3u) ? 0u : (origin >> 11) << 8;
            flush_bits(args, reinterpret_cast<const unsigned long long *>(dst), mw, from, origin >> 3, ~0u);
        }
        if (lane == 0) col.status[b] = e;
        __syncwarp();
    }
}

}  // namespace

namespace {
// the long-sequence decoder as a kernel of its own (inside the spec kernel its registers spilled the batch loop): same job queue,
// one warp per block, 8 warps per CTA, the 4 KB window per warp in dynamic shared memory
__global__ void __launch_bounds__(SPEC_WARPS * 32, 3) lz4_decode_long_kernel(const __grid_constant__ DecodeArgs args, unsigned int *counter)
{
    extern __shared__ unsigned char spec_dyn[];
    const uint32_t win_s = ((smem_addr(spec_dyn) + LW - 1u) & ~(LW - 1u)) + (threadIdx.x >> 5) * LW;
    const uint32_t lane = lane_id();
    const long long njobs = (long long)args.ncols * args.nblocks;
    for (;;) {
        unsigned int job = 0;
        if (lane == 0) job = atomicAdd(counter, 1u);
        job = __shfl_sync(FULL, job, 0);
        if ((long long)job >= njobs) return;
        const int c = (int)(job % args.ncols);
        const int b = args.blk0 + (int)(job / args.ncols);
        const DecodeCol &col = args.col[c];
        if (col.skip && col.skip[b]) continue;
        const uint8_t *src = col.comp + col.comp_off[b];
        uint8_t *dst = col.out + col.dec_off[b];
        const uint32_t comp_len = (uint32_t)col.comp_len[b], origin = (uint32_t)col.origin[b];
        int e;
        if (origin == 0) e = (comp_len == 1 && src[0] == 0) ? E_OK : E_SIZE;
        else if (comp_len == 0) e = E_TRUNCATED;
        else if ((uintptr_t)src & 15u) e = decode_simple(src, comp_len, dst, origin);
        else e = decode_block_long(src, comp_len, dst, origin, win_s);
        if (lane == 0) col.status[b] = e;
        __syncwarp();
    }
}

}  // namespace

int launch_lz4_decode_long(const DecodeArgs &args, unsigned int *d_counter, int sm_count, cudaStream_t stream, int cta_limit)
{
    const long long njobs = (long long)args.ncols * args.nblocks;
    if (njobs <= 0) return 0;
    cudaMemsetAsync(d_counter, 0, sizeof(unsigned int), stream);
    long long ctas = (njobs + SPEC_WARPS - 1) / SPEC_WARPS;
    const long long max_ctas = cta_limit > 0 ? cta_limit : (long long)sm_count * 3;
    if (ctas > max_ctas) ctas = max_ctas;
    lz4_decode_long_kernel<<<(unsigned int)ctas, SPEC_WARPS * 32, SPEC_SMEM, stream>>>(args, d_counter);
    return cudaGetLastError() == cudaSuccess ? 0 : 1;
}

int launch_lz4_decode_spec(const DecodeArgs &args, unsigned int *d_counter, int sm_count, cudaStream_t stream, int cta_limit)
{
    const long long njobs = (long long)args.ncols * args.nblocks;
    if (njobs <= 0) return 0;
    cudaMemsetAsync(d_counter, 0, sizeof(unsigned int), stream);
    long long ctas = (njobs + SPEC_WARPS - 1) / SPEC_WARPS;
    const long long max_ctas = cta_limit > 0 ? cta_limit : (long long)sm_count * 5;   // persistent over the job queue
    if (ctas > max_ctas) ctas = max_ctas;
    if (ctas < 1) ctas = 1;
    if (!args.bits) lz4_decode_spec_kernel<0><<<(unsigned int)ctas, SPEC_WARPS * 32, SPEC_SMEM, stream>>>(args, d_counter);
    else if (args.bits_test.cls != VC_FLT && args.bits_test.n_ne == 0) lz4_decode_spec_kernel<1><<<(unsigned int)ctas, SPEC_WARPS * 32, SPEC_SMEM, stream>>>(args, d_counter);
    else lz4_decode_spec_kernel<2><<<(unsigned int)ctas, SPEC_WARPS * 32, SPEC_SMEM, stream>>>(args, d_counter);
    return cudaGetLastError() == cudaSuccess ? 0 : 1;
}

}  // namespace dfdb
