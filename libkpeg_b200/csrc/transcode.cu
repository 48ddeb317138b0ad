// transcode.cu -- TG, the one kernel of its own the lossless transcoder (kpeg_cuda_transcode, kpeg_cuda.cu) runs between
// the decoder's K0..K2 (coefficient tiles) and the encoder's coded stages (EH / EB, E3..E5, encode.cu).
//
//   TG tc_gather_kernel  tiles -> coef [nblk][64] zig-zag and dc [nblk] in OUTPUT block order, each block moved by the
//                        transform (transcode_core.h), and the range rules checked in the output's order (flag word)
//
// Memory-bound: 128 bytes read (one source block's tile line; its chunks are only swizzled inside the line) and 130
// written per block, plus a 2-byte read of the previous output block's DC.  One CTA stages TG_BLOCKS source blocks in
// shared memory through coalesced 16-byte loads (eight threads per 128-byte line), then every thread gathers its output
// chunk of eight coefficients from there and stores it with one 16-byte store.
#include <cuda_runtime.h>

#include "encode.cuh"
#include "entropy_core.h"
#include "kernels.cuh"
#include "transcode_core.h"

namespace kpeg {
namespace tc {
namespace {

constexpr int TG_THREADS = 256;
constexpr int TG_BLOCKS = TG_THREADS / 8; // output blocks per CTA: one thread per 16-byte chunk
constexpr uint32_t BIAS2 = COEF_BIAS | (COEF_BIAS << 16);

__constant__ XformTable c_xform = make_xform_table();

__device__ __forceinline__ int tile_dc(const uint4 *tiles, uint64_t b)
{
    const uint16_t v = __ldg(reinterpret_cast<const uint16_t *>(tiles + coef_tile_chunk((uint32_t)b, 0u)));
    return (int)(int16_t)(uint16_t)(v ^ COEF_BIAS);
}

__global__ void __launch_bounds__(TG_THREADS) tc_gather_kernel(TcGeom g, const uint4 *__restrict__ tiles, int16_t *__restrict__ coef,
                                                               int16_t *__restrict__ dc, uint32_t *__restrict__ fail)
{
    __shared__ uint4 sm[TG_BLOCKS * 8];
    const uint32_t j = threadIdx.x >> 3, k = threadIdx.x & 7u;
    const uint64_t ob = (uint64_t)blockIdx.x * TG_BLOCKS + j;
    const bool live = ob < g.out.nblk;
    if (live) {
        const uint4 v = __ldg(tiles + coef_tile_chunk((uint32_t)source_index(g, ob), k));
        sm[j * 8u + k] = make_uint4(v.x ^ BIAS2, v.y ^ BIAS2, v.z ^ BIAS2, v.w ^ BIAS2);
    }
    __syncthreads();
    if (!live)
        return;
    alignas(16) int16_t o[8];
    bool ok = gather_chunk(c_xform, g.xform, reinterpret_cast<const int16_t *>(&sm[j * 8u]), (int)k, o);
    reinterpret_cast<uint4 *>(coef)[ob * 8u + k] = *reinterpret_cast<const uint4 *>(o);
    if (k == 0u) {
        dc[ob] = o[0];
        ok = ok && dc_in_range(g, ob, o[0], [&](uint64_t pb) { return tile_dc(tiles, source_index(g, pb)); });
    }
    if (!ok)
        atomicOr(fail, 1u);
}

} // namespace

void launch_gather(const TcGeom &g, const void *tiles, int16_t *coef, int16_t *dc, uint32_t *fail, cudaStream_t s, uint32_t *launches)
{
    const uint64_t grid = (g.out.nblk + TG_BLOCKS - 1) / TG_BLOCKS;
    tc_gather_kernel<<<(unsigned)grid, TG_THREADS, 0, s>>>(g, reinterpret_cast<const uint4 *>(tiles), coef, dc, fail);
    ++*launches;
}

} // namespace tc
} // namespace kpeg
