// lz4_decode_lane.cu -- K1 (third generation): raw LZ4 block decode on sm_100a, ONE LANE PER COLUMN BLOCK.
//
// Replaces read_block's LZ4_decompress_safe call (/root/reference/src/io/BlockStreams.jl:101-119, liblz4 via
// CodecLz4) for whole batches of independent column blocks, same safety contract and the same acceptance rules
// (lz4_lane_core.cuh): never reads outside the compressed payload slot, never writes outside the decoded slot,
// per-block status instead of the reference's `@assert size == sizes.origin "decompression error"`.
//
// Why this shape.  The serial part of an LZ4 block is its token chain; the walker / consumer kernels
// (lz4_decode_v3.cu) spend ~350 warp instructions per 256 output bytes on handing the chain's
// result from one warp to another (ring entries, polls, per-batch prefix work).  Here nothing is handed over:
// every lane runs the whole decoder of its own block as a two-stage software pipeline in registers
// (parse -> DEPTH-deep piece queue -> emit, lz4_lane_core.cuh), one piece of at most 8 output bytes per lane
// per step, all 32 lanes of a warp converged on the same step whatever their blocks contain.  The step loop is
// rolled (one copy of the code, piece data in a shared-memory queue): with one warp per SM sub-partition an
// unrolled loop misses the instruction cache on every line (measured: 1 350 cycles per step, 10x the walker
// kernels, for the 58 KB body of an 8x unrolled loop).
// A 1B-row column is 15 259 blocks = 3.2 warps per SM, so the kernel is latency-bound by design and gives each
// lane a large private working set in shared memory instead of occupancy:
//   * a 176-word history ring (the last 1.4 KB of output): match sources are LDS, not global loads;
//   * a 256-byte window of the compressed stream, refilled 128 bytes at a time.
// Global traffic is warp-cooperative and fully coalesced: every ROUND steps the warp flushes each lane's complete
// 128-byte output unit (8 lanes x 16 bytes per unit, read back from that lane's ring) and refills each lane's
// window with cp.async (8 lanes x 16 bytes per lane).  Match sources older than the ring are final in global
// memory (written by this warp, made visible by __syncwarp) and are fetched with an 8-byte cp.async into the
// piece queue when the piece is parsed, DEPTH steps before they are needed.
//
// Algorithmic bytes per block (roofline): compressed bytes read + origin bytes written.
#include <cuda_runtime.h>
#include <math_constants.h>

#include <cstdio>
#include <cstdlib>

#include "kernels.cuh"
#include "lz4_lane_core.cuh"

namespace dfdb {

namespace {

using namespace lane;

constexpr unsigned FULL = 0xffffffffu;
constexpr int LANE_WARPS = 4;
constexpr int LANE_THREADS = LANE_WARPS * 32;
struct LaneSmem {
    __align__(16) uint8_t win[LANE_THREADS][WIN_BYTES];
    uint64_t ring[LANE_THREADS][RING_STRIDE];
    uint64_t qd[LANE_WARPS][SUBS * DEPTH][32];   // piece queue: the data bytes of K_DATA / K_WORDQ pieces and the literal bytes of K_WORD pieces
    uint32_t qm[LANE_WARPS][SUBS * DEPTH][32];   // piece queue: the descriptors
    // per-warp mailboxes of the cooperative rounds (owner lane writes, the 8 serving lanes read)
    uint64_t fl_addr[LANE_WARPS][32];     // global address of the unit to flush (0 = none)
    uint64_t rf_addr[LANE_WARPS][32];     // global address of the next stream chunk
    uint32_t fl_slot[LANE_WARPS][32];     // ring slot where the unit starts
    uint32_t rf_meta[LANE_WARPS][32];     // window byte offset | chunks << 16
};

__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ uint64_t lds64(uint32_t sa)
{
    uint64_t v;
    asm volatile("ld.shared.u64 %0, [%1];" : "=l"(v) : "r"(sa) : "memory");
    return v;
}
__device__ __forceinline__ void sts64(uint32_t sa, uint64_t v) { asm volatile("st.shared.u64 [%0], %1;" ::"r"(sa), "l"(v) : "memory"); }
__device__ __forceinline__ uint32_t lds32(uint32_t sa)
{
    uint32_t v;
    asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(sa) : "memory");
    return v;
}
__device__ __forceinline__ void sts32(uint32_t sa, uint32_t v) { asm volatile("st.shared.u32 [%0], %1;" ::"r"(sa), "r"(v) : "memory"); }
__device__ __forceinline__ void cp_async16(uint32_t dst_sa, const void *src)
{
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst_sa), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async8(uint32_t dst_sa, const void *src)
{
    asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(dst_sa), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

struct DevMem {
    uint32_t win_sa, ring_sa, q_sa;
    const uint8_t *out;
    __device__ __forceinline__ void put_data(uint32_t slot, uint64_t d) const { sts64(q_sa + slot * 256u, d); }
    __device__ __forceinline__ void put_far(uint32_t slot, uint32_t src) const { cp_async8(q_sa + slot * 256u, out + src); }
    __device__ __forceinline__ uint64_t get_data(uint32_t slot) const { return lds64(q_sa + slot * 256u); }
    __device__ __forceinline__ uint64_t win_read(uint32_t pos) const { return lds64(win_sa + (pos & (uint32_t)(WIN_BYTES - 1))); }
    __device__ __forceinline__ uint64_t ring_load(uint32_t s) const { return lds64(ring_sa + s * 8u); }
    __device__ __forceinline__ void ring_store(uint32_t s, uint64_t v) const { sts64(ring_sa + s * 8u, v); }
    __device__ __forceinline__ uint64_t out_load(uint32_t pos) const { return __ldcg(reinterpret_cast<const unsigned long long *>(out + pos)); }
};

__global__ void __launch_bounds__(LANE_THREADS, 1) lz4_decode_lane_kernel(const DecodeArgs A, unsigned int *counter, unsigned int first_dynamic)
{
    extern __shared__ __align__(128) uint8_t smem_raw[];
    LaneSmem &S = *reinterpret_cast<LaneSmem *>(smem_raw);

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const long long njobs = (long long)A.ncols * A.nblocks;
    const long long nlanes = (long long)gridDim.x * LANE_THREADS;
    const long long g = (long long)blockIdx.x * LANE_THREADS + tid;

    DevMem mem;
    mem.win_sa = smem_u32(&S.win[tid][0]);
    mem.ring_sa = smem_u32(&S.ring[tid][0]);
    mem.q_sa = smem_u32(&S.qd[warp][0][lane]);
    mem.out = nullptr;

    Parser P;
    Emitter E;
    P.reset(0, 0);
    P.st = PS_IDLE;
    E.reset();
    const uint32_t qm_sa = smem_u32(&S.qm[warp][0][lane]);
#pragma unroll
    for (int u = 0; u < SUBS * DEPTH; u++) sts32(qm_sa + u * 128u, K_NONE);

    const uint8_t *comp = nullptr;
    int32_t *status = nullptr;
    uint32_t win_req = 0, comp_padded = 0;
    bool active = false, exhausted = false;

    // the first pass of jobs is assigned statically (spread over all lanes when there are fewer jobs than lanes)
    long long next_job = -1;
    if (njobs <= nlanes) {
        const long long j0 = g * njobs / nlanes, j1 = (g + 1) * njobs / nlanes;
        if (j1 > j0) next_job = j0;
    } else {
        next_job = g;
    }

    auto pickup = [&]() {
        for (;;) {
            long long job = next_job;
            next_job = -1;
            if (job < 0) job = (long long)first_dynamic + atomicAdd(counter, 1u);
            if (job >= njobs) { exhausted = true; return; }
            const int c = (int)(job % A.ncols);
            const int lb = A.blk0 + (int)(job / A.ncols);
            const DecodeCol &col = A.col[c];
            if (col.skip && col.skip[lb]) continue;
            const uint32_t clen = (uint32_t)col.comp_len[lb], origin = (uint32_t)col.origin[lb];
            const uint8_t *src = col.comp + col.comp_off[lb];
            int32_t *st = col.status + lb;
            if (origin == 0) { *st = (clen == 1 && src[0] == 0) ? E_OK : E_SIZE; continue; }
            if (clen == 0) { *st = E_TRUNCATED; continue; }
            if (clen >= MAX_POS || origin >= MAX_POS || ((uintptr_t)src & 15u)) { *st = E_INTERNAL; continue; }
            comp = src;
            status = st;
            mem.out = col.out + col.dec_off[lb];
            comp_padded = (clen + 15u) & ~15u;
            win_req = 0;
            P.reset(clen, origin);
            E.reset();
            active = true;
            return;
        }
    };
    pickup();

    const int grp = lane >> 3, pc = lane & 7;
    const bool hot = A.hot != 0;
    const uint32_t ring_warp_sa = smem_u32(&S.ring[warp * 32][0]);
    const uint32_t win_warp_sa = smem_u32(&S.win[warp * 32][0]);

    for (;;) {
        if (!__any_sync(FULL, active)) break;
        // ---- the window refill requested a round ago has landed: every step waits for all but the DEPTH - 1 newest copy groups ----
        __syncwarp();
        P.win_fill = win_req;
        // ---- cooperative window refill for the next round: whole 16-byte chunks, at most 8 per lane, never over bytes the parser
        //      still needs; the copies land while this round's steps run ----
        {
            uint32_t m = 0;
            if (active) {
                m = ((uint32_t)WIN_BYTES - (win_req - (P.ip & ~15u))) >> 4;
                m = umin(m, 8u);
                m = umin(m, (comp_padded - win_req) >> 4);
            }
            if (__any_sync(FULL, m != 0)) {
                S.rf_addr[warp][lane] = (uint64_t)(uintptr_t)(comp + win_req);
                S.rf_meta[warp][lane] = (win_req & (uint32_t)(WIN_BYTES - 1)) | (m << 16);
                __syncwarp();
#pragma unroll
                for (int j = 0; j < 8; j++) {
                    const int t = 4 * j + grp;
                    const uint32_t meta = S.rf_meta[warp][t];
                    if ((uint32_t)pc < (meta >> 16))
                        cp_async16(win_warp_sa + (uint32_t)t * WIN_BYTES + (((meta & 0xffffu) + 16u * pc) & (uint32_t)(WIN_BYTES - 1)),
                                   reinterpret_cast<const uint8_t *>((uintptr_t)S.rf_addr[warp][t]) + 16u * pc);
                }
                cp_async_commit();
                win_req += m << 4;
            }
        }
        // ---- ROUND steps of the two-stage pipeline ----
        //      Each step emits the two pieces parsed DEPTH steps ago and parses two new ones into the same queue slots.  Word pieces
        //      take the straight-line fast path, lane by lane; the general step runs only when some lane of the warp needs it.
#pragma unroll 1
        for (uint32_t v = 0; v < (uint32_t)ROUND; v++) {
            const uint32_t slotA = (uint32_t)SUBS * (v & (uint32_t)(DEPTH - 1)), slotB = slotA + 1;
            cp_async_wait<DEPTH - 1>();            // the far sources fetched when these two pieces were parsed have landed
            const uint32_t mA = lds32(qm_sa + slotA * 128u), mB = lds32(qm_sa + slotB * 128u);
            if (hot && (v & (uint32_t)(HOT_PERIOD - 1)) != (uint32_t)(HOT_PERIOD - 1)) {
                // hot step (word-regular columns): two plain tokens per lane or nothing; a lane that meets anything else waits for the next full step
                uint32_t nA, nB;
                E.fast2(mem, mA, mB, slotA, slotB);
                P.fast2(mem, E.flushed, slotA, slotB, nA, nB);
                sts32(qm_sa + slotA * 128u, nA);
                sts32(qm_sa + slotB * 128u, nB);
                cp_async_commit();
                continue;
            }
            const bool eA = E.fast(mem, mA, slotA);
            if (__any_sync(FULL, !eA)) { if (!eA) E.step(mem, mA, slotA); }
            const bool eB = E.fast(mem, mB, slotB);
            if (__any_sync(FULL, !eB)) { if (!eB) E.step(mem, mB, slotB); }
            uint32_t nA = K_NONE, nB = K_NONE;
            const bool pA = P.fast(mem, E.flushed, slotA, nA);
            if (__any_sync(FULL, !pA)) { if (!pA) nA = P.step(mem, E.flushed, slotA); }
            const bool pB = P.fast(mem, E.flushed, slotB, nB);
            if (__any_sync(FULL, !pB)) { if (!pB) nB = P.step(mem, E.flushed, slotB); }
            sts32(qm_sa + slotA * 128u, nA);
            sts32(qm_sa + slotB * 128u, nB);
            cp_async_commit();
        }
        const bool fin = active && (P.st == PS_ERR || (P.st == PS_END && E.op == P.opp));
        // ---- cooperative flush of complete units (the last, partial unit of a finished block too: slots are padded) ----
        for (;;) {
            const bool want = active && P.st != PS_ERR && (E.unit_ready() || (fin && E.flushed < E.op));
            if (!__any_sync(FULL, want)) break;
            S.fl_addr[warp][lane] = want ? (uint64_t)(uintptr_t)(mem.out + E.flushed) : 0ull;
            S.fl_slot[warp][lane] = E.flush_slot();
            __syncwarp();
#pragma unroll
            for (int j = 0; j < 8; j++) {
                const int t = 4 * j + grp;
                const uint64_t a = S.fl_addr[warp][t];
                if (a) {
                    const uint32_t sa = ring_warp_sa + (uint32_t)t * (RING_STRIDE * 8u) + (S.fl_slot[warp][t] + 2u * pc) * 8u;
                    ulonglong2 v;
                    v.x = lds64(sa);
                    v.y = lds64(sa + 8);
                    *reinterpret_cast<ulonglong2 *>((uintptr_t)a + 16u * pc) = v;
                }
            }
            __syncwarp();
            if (want) E.flushed += UNIT_BYTES;
        }
        if (fin) {
            *status = P.st == PS_ERR ? (int32_t)P.err : ((E.op == P.op_end && P.ip == P.ip_end) ? E_OK : E_SIZE);
            active = false;
            P.st = PS_IDLE;
#pragma unroll
            for (int u = 0; u < SUBS * DEPTH; u++) sts32(qm_sa + u * 128u, K_NONE);   // (pieces of a block that failed are dropped)
        }
        if (!active && !exhausted) pickup();
    }
}

}  // namespace

size_t lane_smem_bytes() { return sizeof(LaneSmem) + 128; }

int launch_lz4_decode_lane(const DecodeArgs &args, unsigned int *d_counter, int sm_count, cudaStream_t stream, int cta_limit)
{
    static bool configured = false;
    const int smem = (int)lane_smem_bytes();
    if (!configured) {
        if (cudaFuncSetAttribute(lz4_decode_lane_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem) != cudaSuccess) return 1;
        configured = true;
    }
    const long long njobs = (long long)args.ncols * args.nblocks;
    if (njobs <= 0) return 0;
    // one CTA per SM, every SM: with fewer jobs than lanes the jobs are spread so that every block gets as much of an SM as possible
    int ctas = sm_count;
    if (cta_limit > 0 && ctas > cta_limit) ctas = cta_limit;
    if ((long long)ctas > njobs) ctas = (int)njobs;
    if (ctas < 1) ctas = 1;
    const long long nlanes = (long long)ctas * LANE_THREADS;
    const unsigned int first_dynamic = (unsigned int)(njobs <= nlanes ? njobs : nlanes);
    cudaMemsetAsync(d_counter, 0, sizeof(unsigned int), stream);
    lz4_decode_lane_kernel<<<ctas, LANE_THREADS, smem, stream>>>(args, d_counter, first_dynamic);
    return cudaGetLastError() == cudaSuccess ? 0 : 1;
}

}  // namespace dfdb
