// k3_tile.cuh -- stage 0 of the reconstruction kernels (idct_kernel in k3_fused.cu, idct_scaled_kernel in k3_scaled.cu):
// a strip's coefficient tile and a quantiser table arrive in shared memory by bulk copies of the copy engine
// (cp.async.bulk + mbarrier, SASS UBLKCP), and the tile of the strip that will run in this CTA's slot next is pulled into L2.
#ifndef KPEG_K3_TILE_CUH
#define KPEG_K3_TILE_CUH

#include <stdint.h>

#include <type_traits>

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
// multiples of 16 bytes.  LISTED (crop decode): the CTAs run the strips of `list` (n entries; this is entry blockIdx.x), and
// the prefetch looks ahead in the list; otherwise CTA i runs strip i of n.
template <int NC, bool LISTED = false>
__device__ __forceinline__ void k3_load_strip(const void *tiles, uint32_t strip, uint32_t nstrips, void *tile_smem, const void *table,
                                              uint32_t table_bytes, void *table_smem, uint32_t bar, const uint32_t *list = nullptr)
{
    constexpr uint32_t tile_bytes = NC * IDCT_MCUS_PER_CTA * 128u;
    const char *tile = reinterpret_cast<const char *>(tiles) + (size_t)strip * tile_bytes;
    mbar_init(bar, 1);
    mbar_expect_tx(bar, table_bytes + tile_bytes);
    bulk_load(smem_u32(tile_smem), tile, tile_bytes, bar);
    bulk_load(smem_u32(table_smem), table, table_bytes, bar);
    // the tile of the strip that will run in this CTA's slot next: DRAM -> L2 now
    if constexpr (LISTED) {
        if (blockIdx.x + IDCT_PREFETCH_AHEAD < nstrips)
            asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(reinterpret_cast<const char *>(tiles) +
                                                                               (size_t)__ldg(list + blockIdx.x + IDCT_PREFETCH_AHEAD) * tile_bytes),
                         "r"(tile_bytes) : "memory");
    } else if (strip + IDCT_PREFETCH_AHEAD < nstrips) {
        asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(tile + (size_t)IDCT_PREFETCH_AHEAD * tile_bytes), "r"(tile_bytes) : "memory");
    }
}

// The strip CTA blockIdx.x reconstructs, the strips of the launch and their list (nullptr: CTA i runs strip i): crop
// decodes run the listed strips only (IdctCropArgs), whole-image decodes every strip (IdctArgs).
template <class A>
__device__ __forceinline__ uint32_t k3_strip(const A &a)
{
    if constexpr (std::is_same_v<A, IdctCropArgs>)
        return __ldg(a.strip_list + blockIdx.x);
    else
        return blockIdx.x;
}
template <class A>
__device__ __forceinline__ uint32_t k3_nstrips(const A &a)
{
    if constexpr (std::is_same_v<A, IdctCropArgs>)
        return a.nlisted;
    else
        return a.nstrips;
}
template <class A>
__device__ __forceinline__ const uint32_t *k3_list(const A &a)
{
    if constexpr (std::is_same_v<A, IdctCropArgs>)
        return a.strip_list;
    else
        return nullptr;
}
template <bool CROP>
using K3Args = std::conditional_t<CROP, IdctCropArgs, IdctArgs>;

} // namespace kpeg
#endif
