// k3_scaled.cu -- the reconstruction stage of a reduced-size decode (KPEG_FLAG_SCALE_1_2 / _1_4 / _1_8) as one sm_100a
// kernel, in place of K3 (idct_kernel + idct_patch_kernel): dequantisation, libjpeg-turbo's reduced IDCT with its
// range-limit table, libjpeg's integer YCbCr -> RGB and the interleaved store at the reduced size.  K0..K2 run unchanged
// and leave the same coefficient tiles (kernels.cuh) whatever the scale.
//
// One CTA per strip of IDCT_MCUS_PER_CTA MCUs, as K3:
//   stage 0  the strip's tile and the plain quantisers (DeviceTables::qint) by bulk copies (k3_tile.cuh, shared with K3)
//   stage 1  one thread = one 8x8 block: the coefficients the transform reads, straight from the swizzled tile,
//            dequantised, through the reduced transform (idct_reduced.h) -> K x K samples in shared memory (K = 8 / S)
//   stage 2  one thread per output pixel of the strip: colour (three components) and the store, clipped at the right and
//            bottom edges of each image (a batch's images lie back to back at the reduced size)
// Everything is integer arithmetic with a unique result, so there is no tie band and no patch pass: one launch.
#include <cuda_runtime.h>
#include <stddef.h>
#include <stdint.h>

#include <type_traits>

#include "entropy_core.h"
#include "idct_reduced.h"
#include "k3_tile.cuh"
#include "kernels.cuh"
#include "kpeg_common.h"

namespace kpeg {

static_assert(offsetof(DeviceTables, qint) % 16 == 0, "qint is staged by a bulk copy");

// CROP: CTA i reconstructs strip a.strip_list[i], and stores only the pixels inside a.crop[image] (crop_geom.h)
template <int NC, int S, bool CROP>
__global__ void __launch_bounds__(NC * IDCT_MCUS_PER_CTA) idct_scaled_kernel(K3Args<CROP> a)
{
    constexpr int NM = IDCT_MCUS_PER_CTA;
    constexpr int NB = NM * NC;
    constexpr int K = 8 / S;
    __shared__ __align__(128) uint4 coef[NB * 8]; // the tile image: [block][chunk ^ (block & 7)], biased 16-bit, zig-zag
    __shared__ __align__(16) int32_t q[NC][64];   // plain quantisers, zig-zag order
    __shared__ uint8_t samp[NC][NM][K * K];       // range-limited samples of every block
    __shared__ __align__(8) unsigned long long mbar;

    const int t = threadIdx.x;
    const int comp = t / NM;
    const int ml = t % NM;
    const int bl = ml * NC + comp;
    const uint32_t total_mcus = a.g.nimages * a.g.mcus_per_image;
    const uint32_t strip = k3_strip(a);
    const uint32_t mcu0 = strip * NM;

    // ---- stage 0 ----------------------------------------------------------------------------------------------
    const uint32_t bar = smem_u32(&mbar);
    if (t == 0) {
        k3_load_strip<NC, CROP>(a.tiles, strip, k3_nstrips(a), coef, a.tables->qint, NC * 64u * 4u, q, bar, k3_list(a));
        mbar_wait(bar, 0);
    }
    __syncthreads();

    // ---- stage 1: one thread = one block ------------------------------------------------------------------------
    if (mcu0 + (uint32_t)ml < total_mcus) {
        const unsigned char *tile = reinterpret_cast<const unsigned char *>(coef);
        const int32_t *qc = q[comp];
        auto dq = [&](int zz) -> int32_t {
            const uint32_t v = *reinterpret_cast<const uint16_t *>(tile + coef_tile_byte((uint32_t)bl * 64u + (uint32_t)zz));
            return ((int32_t)v - (int32_t)COEF_BIAS) * qc[zz];
        };
        red::idct_reduced<S>(dq, samp[comp][ml]);
    }
    __syncthreads();

    // ---- stage 2: colour and store ------------------------------------------------------------------------------
    const OutGeom o = out_geom(a.g);
    for (uint32_t p = (uint32_t)t; p < (uint32_t)(NM * K * K); p += (uint32_t)NB) {
        const red::StripPixel px = red::strip_pixel(p, K, NM);
        const uint32_t m = mcu0 + px.ml;
        if (m >= total_mcus)
            continue;
        uint64_t off;
        if constexpr (CROP)
            off = red::scaled_crop_offset(a.g, o, a.crop, m, px.r, px.c);
        else
            off = red::scaled_pixel_offset(a.g, o, m, px.r, px.c);
        if (off == ~(uint64_t)0)
            continue;
        const int s = (int)(px.r * K + px.c);
        uint8_t *dst = a.pixels + off;
        if constexpr (NC == 3) {
            const uint32_t v = red::ycc_rgb(samp[0][px.ml][s], samp[1][px.ml][s], samp[2][px.ml][s]);
            dst[0] = (uint8_t)v;
            dst[1] = (uint8_t)(v >> 8);
            dst[2] = (uint8_t)(v >> 16);
        } else {
            dst[0] = samp[0][px.ml][s];
        }
    }
}

cudaError_t launch_idct_scaled(const IdctCropArgs &a, cudaStream_t s, uint32_t *launches)
{
    const uint32_t total_mcus = a.g.nimages * a.g.mcus_per_image;
    const uint32_t S = scale_denom(a.g.flags);
    const bool rgb = a.g.ncomp == 3, crop = a.crop != nullptr;
    const uint32_t grid = crop ? a.nlisted : (total_mcus + IDCT_MCUS_PER_CTA - 1) / IDCT_MCUS_PER_CTA;
    const uint32_t threads = a.g.ncomp * IDCT_MCUS_PER_CTA;
    auto go = [&](auto NCC, auto SC, auto CC) {
        constexpr bool CROP = decltype(CC)::value;
        idct_scaled_kernel<decltype(NCC)::value, decltype(SC)::value, CROP><<<grid, threads, 0, s>>>(static_cast<const K3Args<CROP> &>(a));
    };
    using C1 = std::integral_constant<int, 1>;
    using C3 = std::integral_constant<int, 3>;
    auto by_scale = [&](auto NCC, auto CC) {
        if (S == 2)
            go(NCC, std::integral_constant<int, 2>{}, CC);
        else if (S == 4)
            go(NCC, std::integral_constant<int, 4>{}, CC);
        else
            go(NCC, std::integral_constant<int, 8>{}, CC);
    };
    if (S != 2 && S != 4 && S != 8)
        return cudaErrorInvalidValue;
    if (crop)
        rgb ? by_scale(C3{}, std::true_type{}) : by_scale(C1{}, std::true_type{});
    else
        rgb ? by_scale(C3{}, std::false_type{}) : by_scale(C1{}, std::false_type{});
    ++*launches;
    return cudaSuccess;
}

} // namespace kpeg
