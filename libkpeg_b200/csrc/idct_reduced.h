// idct_reduced.h -- per-block and per-pixel arithmetic of the reduced-size decode (KPEG_FLAG_SCALE_1_2 / _1_4 / _1_8):
// libjpeg-turbo's reduced IDCTs (jidctred.c: jpeg_idct_4x4, jpeg_idct_2x2, jpeg_idct_1x1) with its post-IDCT range-limit
// table, and libjpeg's integer YCbCr -> RGB (jdcolor.c ycc_rgb_convert).  KPEG_HD: the same source runs in
// idct_scaled_kernel (k3_scaled.cu) and in the CPU replay of tests/emu/emu_scaled.cpp.
//
// Integer widths are libjpeg's on LP64: the dequantised coefficient is an int (16-bit coefficient x 8-bit quantiser),
// every product and sum of a pass is 64-bit (JLONG), the workspace between the passes is int.  With a crafted stream a
// dequantised coefficient reaches 32767 x 255, and pass 2's sums then need more than 32 bits.
#ifndef KPEG_IDCT_REDUCED_H
#define KPEG_IDCT_REDUCED_H

#include <stdint.h>

#include "crop_geom.h"
#include "kpeg_common.h"

#ifdef __CUDA_ARCH__
#define KPEG_RED_UNROLL _Pragma("unroll") // device pass only: the workspace must stay in registers
#else
#define KPEG_RED_UNROLL
#endif

namespace kpeg {
namespace red {

constexpr int CONST_BITS = 13, PASS1_BITS = 2;
// FIX(x) = (int64) (x * 2^13 + 0.5), jidctred.c
constexpr int64_t FIX_0_211164243 = 1730, FIX_0_509795579 = 4176, FIX_0_601344887 = 4926, FIX_0_720959822 = 5906,
                  FIX_0_765366865 = 6270, FIX_0_850430095 = 6967, FIX_0_899976223 = 7373, FIX_1_061594337 = 8697,
                  FIX_1_272758580 = 10426, FIX_1_451774981 = 11893, FIX_1_847759065 = 15137, FIX_2_172734803 = 17799,
                  FIX_2_562915447 = 20995, FIX_3_624509785 = 29692;

KPEG_HD int64_t descale(int64_t x, int n) { return (x + ((int64_t)1 << (n - 1))) >> n; }

// libjpeg's IDCT_range_limit table (prepare_range_limit_table) indexed with (x & RANGE_MASK): it WRAPS, it does not clamp.
KPEG_HD uint32_t range_limit(int64_t x)
{
    const uint32_t t = (uint32_t)x & 1023u;
    return t < 128u ? t + 128u : t < 512u ? 255u : t < 896u ? 0u : t - 896u;
}

// zig-zag index of natural position (row r, column c): diagonal s = r + c, odd diagonals run down, even ones up
KPEG_HD constexpr int zz_of_nat(int r, int c)
{
    const int s = r + c;
    const int base = s < 8 ? s * (s + 1) / 2 : 64 - (15 - s) * (16 - s) / 2;
    const int rmin = s > 7 ? s - 7 : 0, rmax = s < 7 ? s : 7;
    return base + ((s & 1) ? r - rmin : rmax - r);
}

// The reduced transforms.  dq(zz) is the dequantised coefficient of zig-zag index zz (an int); out receives the K x K
// output samples row by row (K = 8 / S), already through the range-limit table.
template <class DQ>
KPEG_HD void idct_4x4(DQ dq, uint8_t *out)
{
    int ws[8 * 4];
KPEG_RED_UNROLL
    for (int col = 0; col < 8; ++col) {
        if (col == 4) // the second pass does not read column 4
            continue;
        int64_t tmp0 = (int64_t)dq(zz_of_nat(0, col)) * ((int64_t)1 << (CONST_BITS + 1));
        int64_t tmp2 = (int64_t)dq(zz_of_nat(2, col)) * FIX_1_847759065 + (int64_t)dq(zz_of_nat(6, col)) * -FIX_0_765366865;
        const int64_t tmp10 = tmp0 + tmp2, tmp12 = tmp0 - tmp2;
        const int64_t z1 = dq(zz_of_nat(7, col)), z2 = dq(zz_of_nat(5, col)), z3 = dq(zz_of_nat(3, col)), z4 = dq(zz_of_nat(1, col));
        tmp0 = z1 * -FIX_0_211164243 + z2 * FIX_1_451774981 + z3 * -FIX_2_172734803 + z4 * FIX_1_061594337;
        tmp2 = z1 * -FIX_0_509795579 + z2 * -FIX_0_601344887 + z3 * FIX_0_899976223 + z4 * FIX_2_562915447;
        constexpr int sh = CONST_BITS - PASS1_BITS + 1;
        ws[0 * 8 + col] = (int)descale(tmp10 + tmp2, sh);
        ws[3 * 8 + col] = (int)descale(tmp10 - tmp2, sh);
        ws[1 * 8 + col] = (int)descale(tmp12 + tmp0, sh);
        ws[2 * 8 + col] = (int)descale(tmp12 - tmp0, sh);
    }
KPEG_RED_UNROLL
    for (int row = 0; row < 4; ++row) {
        const int *w = ws + row * 8;
        int64_t tmp0 = (int64_t)w[0] * ((int64_t)1 << (CONST_BITS + 1));
        int64_t tmp2 = (int64_t)w[2] * FIX_1_847759065 + (int64_t)w[6] * -FIX_0_765366865;
        const int64_t tmp10 = tmp0 + tmp2, tmp12 = tmp0 - tmp2;
        const int64_t z1 = w[7], z2 = w[5], z3 = w[3], z4 = w[1];
        tmp0 = z1 * -FIX_0_211164243 + z2 * FIX_1_451774981 + z3 * -FIX_2_172734803 + z4 * FIX_1_061594337;
        tmp2 = z1 * -FIX_0_509795579 + z2 * -FIX_0_601344887 + z3 * FIX_0_899976223 + z4 * FIX_2_562915447;
        constexpr int sh = CONST_BITS + PASS1_BITS + 3 + 1;
        out[row * 4 + 0] = (uint8_t)range_limit(descale(tmp10 + tmp2, sh));
        out[row * 4 + 3] = (uint8_t)range_limit(descale(tmp10 - tmp2, sh));
        out[row * 4 + 1] = (uint8_t)range_limit(descale(tmp12 + tmp0, sh));
        out[row * 4 + 2] = (uint8_t)range_limit(descale(tmp12 - tmp0, sh));
    }
}

template <class DQ>
KPEG_HD void idct_2x2(DQ dq, uint8_t *out)
{
    int ws[8 * 2];
KPEG_RED_UNROLL
    for (int col = 0; col < 8; ++col) {
        if (col == 2 || col == 4 || col == 6) // the second pass reads columns 0, 1, 3, 5, 7 only
            continue;
        const int64_t tmp10 = (int64_t)dq(zz_of_nat(0, col)) * ((int64_t)1 << (CONST_BITS + 2));
        const int64_t tmp0 = (int64_t)dq(zz_of_nat(7, col)) * -FIX_0_720959822 + (int64_t)dq(zz_of_nat(5, col)) * FIX_0_850430095 +
                             (int64_t)dq(zz_of_nat(3, col)) * -FIX_1_272758580 + (int64_t)dq(zz_of_nat(1, col)) * FIX_3_624509785;
        constexpr int sh = CONST_BITS - PASS1_BITS + 2;
        ws[0 * 8 + col] = (int)descale(tmp10 + tmp0, sh);
        ws[1 * 8 + col] = (int)descale(tmp10 - tmp0, sh);
    }
KPEG_RED_UNROLL
    for (int row = 0; row < 2; ++row) {
        const int *w = ws + row * 8;
        const int64_t tmp10 = (int64_t)w[0] * ((int64_t)1 << (CONST_BITS + 2));
        const int64_t tmp0 = (int64_t)w[7] * -FIX_0_720959822 + (int64_t)w[5] * FIX_0_850430095 + (int64_t)w[3] * -FIX_1_272758580 +
                             (int64_t)w[1] * FIX_3_624509785;
        constexpr int sh = CONST_BITS + PASS1_BITS + 3 + 2;
        out[row * 2 + 0] = (uint8_t)range_limit(descale(tmp10 + tmp0, sh));
        out[row * 2 + 1] = (uint8_t)range_limit(descale(tmp10 - tmp0, sh));
    }
}

template <class DQ>
KPEG_HD void idct_1x1(DQ dq, uint8_t *out)
{
    out[0] = (uint8_t)range_limit((int)descale((int64_t)dq(0), 3));
}

// scale S = 2, 4, 8 -> the transform of 8 / S output samples per side
template <int S, class DQ>
KPEG_HD void idct_reduced(DQ dq, uint8_t *out)
{
    static_assert(S == 2 || S == 4 || S == 8, "reduced scales are 1/2, 1/4, 1/8");
    if constexpr (S == 2)
        idct_4x4(dq, out);
    else if constexpr (S == 4)
        idct_2x2(dq, out);
    else
        idct_1x1(dq, out);
}

// jdcolor.c ycc_rgb_convert with SCALEBITS 16 (FIX(1.40200) = 91881, FIX(0.71414) = 46802, FIX(0.34414) = 22554,
// FIX(1.77200) = 116130), each channel clamped by the sample range-limit table -> R | G << 8 | B << 16
KPEG_HD uint32_t clamp255(int v) { return v < 0 ? 0u : v > 255 ? 255u : (uint32_t)v; }
KPEG_HD uint32_t ycc_rgb(int y, int cb, int cr)
{
    cb -= 128;
    cr -= 128;
    const uint32_t r = clamp255(y + ((91881 * cr + 32768) >> 16));
    const uint32_t g = clamp255(y + ((-46802 * cr - 22554 * cb + 32768) >> 16));
    const uint32_t b = clamp255(y + ((116130 * cb + 32768) >> 16));
    return r | g << 8 | b << 16;
}

// ---- where a strip's output goes -----------------------------------------------------------------------------------
// A strip of NM consecutive MCUs (MCU-interleaved blocks) gives NM x K x K output pixels; work item p of the strip is
// pixel (row r, column c) of the K x K square of strip MCU ml, ordered row, then MCU, then column, so that consecutive
// items of one MCU row land next to each other in the output.
struct StripPixel {
    uint32_t ml, r, c;
};
KPEG_HD StripPixel strip_pixel(uint32_t p, uint32_t K, uint32_t NM)
{
    const uint32_t r = p / (NM * K), rem = p - r * NM * K;
    return StripPixel{rem / K, r, rem - (rem / K) * K};
}

// Byte offset in the job's output of pixel (r, c) of MCU m (index in the job), or UINT64_MAX when it falls beyond the
// right or bottom edge (the output is ceil(W / S) x ceil(H / S): a ragged edge block contributes part of its square).
KPEG_HD uint64_t scaled_pixel_offset(const JobGeom &g, const OutGeom &o, uint32_t m, uint32_t r, uint32_t c)
{
    const uint32_t K = 8u / o.scale;
    const uint32_t img = m / g.mcus_per_image, mi = m - img * g.mcus_per_image;
    const uint32_t by = mi / g.mcus_x, bx = mi - by * g.mcus_x;
    const uint32_t oy = by * K + r, ox = bx * K + c;
    if (ox >= o.width || oy >= o.height)
        return ~(uint64_t)0;
    return (uint64_t)img * o.bytes() + (uint64_t)oy * o.row_bytes() + (uint64_t)ox * o.ncomp;
}

// The same pixel in a crop decode's output (crop_geom.h): its byte offset in the crop of its image, or CROP_SKIP outside
// the rectangle (which lies inside the output image: the ragged edge needs no test of its own).
KPEG_HD uint64_t scaled_crop_offset(const JobGeom &g, const OutGeom &o, const CropWin *crop, uint32_t m, uint32_t r, uint32_t c)
{
    const uint32_t K = 8u / o.scale;
    const uint32_t img = m / g.mcus_per_image, mi = m - img * g.mcus_per_image;
    const uint32_t by = mi / g.mcus_x, bx = mi - by * g.mcus_x;
    return crop_pixel_offset(crop[img], o.ncomp, bx * K + c, by * K + r);
}

} // namespace red
} // namespace kpeg
#endif
