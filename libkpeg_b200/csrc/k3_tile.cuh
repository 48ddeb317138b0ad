// k3_tile.cuh -- stage 0 of the reconstruction kernels (idct_kernel in k3_fused.cu, idct_scaled_kernel in k3_scaled.cu):
// a strip's coefficient tile and a quantiser table arrive in shared memory by bulk copies of the copy engine
// (cp.async.bulk + mbarrier, SASS UBLKCP), and the tile of the strip that will run in this CTA's slot next is pulled into L2.
#ifndef KPEG_K3_TILE_CUH
#define KPEG_K3_TILE_CUH

#include <stdint.h>

#include "kernels.cuh"

namespace kpeg {

#ifndef KPEG_IDCT_PREFETCH_AHEAD
#define KPEG_IDCT_PREFETCH_AHEAD 1184
#endif
constexpr uint32_t IDCT_PREFETCH_AHEAD = KPEG_IDCT_PREFETCH_AHEAD; // strips: 148 SMs x 8 CTAs, the strip that runs in this CTA's slot next

__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity)
{
    asm volatile("{\n"
                 ".reg .pred p;\n"
                 "KPEG_MBAR_WAIT:\n"
                 "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
                 "@p bra KPEG_MBAR_DONE;\n"
                 "bra KPEG_MBAR_WAIT;\n"
                 "KPEG_MBAR_DONE:\n"
                 "}" ::"r"(bar), "r"(parity) : "memory");
}
__device__ __forceinline__ void bulk_load(uint32_t dst, const void *src, uint32_t bytes, uint32_t bar)
{
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(dst), "l"(src), "r"(bytes), "r"(bar) : "memory");
}

// Issued by one thread: the tile of `strip` (NC * IDCT_MCUS_PER_CTA blocks of 128 bytes) -> tile_smem and table_bytes of
// `table` -> table_smem, both completing on the barrier `bar` (wait with mbar_wait(bar, 0)).  Addresses and sizes are
// multiples of 16 bytes.
template <int NC>
__device__ __forceinline__ void k3_load_strip(const void *tiles, uint32_t strip, uint32_t nstrips, void *tile_smem, const void *table,
                                              uint32_t table_bytes, void *table_smem, uint32_t bar)
{
    constexpr uint32_t tile_bytes = NC * IDCT_MCUS_PER_CTA * 128u;
    const char *tile = reinterpret_cast<const char *>(tiles) + (size_t)strip * tile_bytes;
    mbar_init(bar, 1);
    mbar_expect_tx(bar, table_bytes + tile_bytes);
    bulk_load(smem_u32(tile_smem), tile, tile_bytes, bar);
    bulk_load(smem_u32(table_smem), table, table_bytes, bar);
    // the tile of the strip that will run in this CTA's slot next: DRAM -> L2 now
    if (strip + IDCT_PREFETCH_AHEAD < nstrips)
        asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(tile + (size_t)IDCT_PREFETCH_AHEAD * tile_bytes), "r"(tile_bytes) : "memory");
}

} // namespace kpeg
#endif
