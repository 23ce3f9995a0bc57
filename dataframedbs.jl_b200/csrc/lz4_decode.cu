// lz4_decode.cu -- K1, sequential baseline: one warp per compressed column block, one sequence at a time (decode_simple,
// lz4_common.cuh).
//
// Replaces read_block's LZ4_decompress_safe call (/root/reference/src/io/BlockStreams.jl:101-119,
// liblz4 through CodecLz4) for whole batches of independent column blocks.  Like the _safe decoder it
// never reads outside the compressed payload nor writes outside `origin` bytes, and it reports a
// per-block status instead of the reference's `@assert size == sizes.origin "decompression error"`.
// It runs when the option lz4_simple is set: the one way to run decode_simple, which the spec / long / bytes / v3
// decoders fall back to for unaligned blocks, over every body kind.
//
// Algorithmic bytes per block (roofline): compressed bytes read + origin bytes written.
#include <cuda_runtime.h>

#include "kernels.cuh"
#include "lz4_common.cuh"

namespace dfdb {

namespace {

using namespace lz4;

constexpr int WARPS_PER_CTA = 8;

}  // namespace

__global__ void __launch_bounds__(WARPS_PER_CTA * 32, 4) lz4_decode_kernel(DecodeArgs args, unsigned int *counter)
{
    const uint32_t lane = lane_id();
    const unsigned int njobs = (unsigned int)args.ncols * (unsigned int)args.nblocks;
    for (;;) {
        unsigned int job = 0;
        if (lane == 0) job = atomicAdd(counter, 1u);
        job = __shfl_sync(0xffffffffu, job, 0);
        if (job >= njobs) break;
        const int c = (int)(job % (unsigned int)args.ncols);
        const int b = args.blk0 + (int)(job / (unsigned int)args.ncols);
        const DecodeCol &col = args.col[c];
        if (col.skip && col.skip[b]) continue;     // stored block whose body is referenced in place
        const uint8_t *src = col.comp + col.comp_off[b];
        uint8_t *dst = col.out + col.dec_off[b];
        const int64_t comp_len = col.comp_len[b], origin = col.origin[b];
        const int e = decode_simple(src, comp_len, dst, origin);
        if (lane == 0) col.status[b] = e;
        __syncwarp();
    }
}

int launch_lz4_decode(const DecodeArgs &args, unsigned int *d_counter, int sm_count, cudaStream_t stream)
{
    cudaMemsetAsync(d_counter, 0, sizeof(unsigned int), stream);
    const long long njobs = (long long)args.ncols * args.nblocks;
    long long ctas = (njobs + WARPS_PER_CTA - 1) / WARPS_PER_CTA;
    const long long max_ctas = (long long)sm_count * 4;     // 32 resident warps per SM, persistent over the job queue
    if (ctas > max_ctas) ctas = max_ctas;
    if (ctas < 1) ctas = 1;
    lz4_decode_kernel<<<(unsigned int)ctas, WARPS_PER_CTA * 32, 0, stream>>>(args, d_counter);
    return cudaGetLastError() == cudaSuccess ? 0 : 1;
}

}  // namespace dfdb
