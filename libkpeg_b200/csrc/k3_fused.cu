// k3_fused.cu -- K3 of the B200 decode path as ONE sm_100a kernel: dequantisation, de-zigzag, 8x8 IDCT, level shift,
// YCbCr->RGB and the interleaved store, with the exact re-evaluation of the samples near a rounding tie in the same kernel.
//
// What it replaces in the reference: the dequantisation and de-zigzag of MCU::constructMCU (src/MCU.cpp:110-120),
// MCU::computeIDCT (:172-216), performLevelShift (:218-245), convertYCbCrToRGB (:247-279) and
// Image::createImageFromMCUs (src/Image.cpp:51-70).
//
// One CTA reconstructs a strip of IDCT_MCUS_PER_CTA consecutive MCUs from the strip's coefficient tile, which K2
// (k2_expand.cu) left in global memory as the image of this kernel's shared-memory tile (kernels.cuh).
//
//   stage 0  by the copy engine: the tile (12 KB for RGB) and the quantiser table arrive with bulk copies
//            (cp.async.bulk + mbarrier, SASS UBLKCP); the tile that will run in this CTA's slot next is pulled into L2
//            (k3_tile.cuh, shared with the reduced-size kernel of k3_scaled.cu)
//   stage 1  one thread = one 8x8 block, all 64 values in registers, two fp32 lanes per instruction (FADD2 / FMUL2 /
//            FFMA2): biased 16-bit -> fp32 by byte permute + one packed subtract (no I2F), dequantise (AAN prescale
//            folded into the quantiser), de-zigzag by register renaming, separable fp32 IDCT, rounding, tie-band test;
//            blocks without AC coefficients take the reference's one-term evaluation directly
//   stage 2  per pixel row: YCbCr -> RGB on pixel pairs (fp32 with proven margin, double otherwise), pack, store
//   stage 3  the samples inside the tie band (0.1 % .. 0.7 %) need the reference's own operation order: the strip lists
//            their pixels (one record per pixel: where it is, which components are tied, the three fast samples) and
//            idct_patch_kernel re-evaluates them afterwards from the coefficient tiles with full warps.  (Resolved inside
//            this kernel -- one warp, six lanes busy on average, the CTA's slot held for a 64-term serial chain, and the
//            unrolled chain in this kernel's instruction stream -- it cost 21 % of the stall samples and a third of the
//            instruction-cache misses.)  Only a strip with more ties than its list holds resolves them itself.
//
// All file:line citations are relative to /root/reference.
#include <cuda_runtime.h>
#include <stddef.h>
#include <stdint.h>

#include <algorithm>
#include <utility>

#include "entropy_core.h"
#include "idct_core.h"
#include "k3_tile.cuh"
#include "kernels.cuh"
#include "kpeg_common.h"

namespace kpeg {

template <int NAT>
struct NatZz {
    static constexpr int value = make_zigzag_tables().nat2zz[NAT];
};

#ifndef KPEG_EXACT_SKIP_ZERO
#define KPEG_EXACT_SKIP_ZERO 1 // the exact evaluation skips the accumulation of zero terms (same bits, shorter dependent chain)
#endif

#ifndef KPEG_EXACT_WIDEN_INT
#define KPEG_EXACT_WIDEN_INT 0 // 1: the exact evaluation widens float -> double by integer arithmetic (idct_core.h widen_f32) instead of F2F
#endif

#ifndef KPEG_IDCT_MIN_CTAS
#define KPEG_IDCT_MIN_CTAS 8
#endif

// Per-block facts the colour stage needs, derived from A = sum |dequantised coefficient| (every sample of the
// block is bounded by A / 4: the 64 basis functions are bounded by 1/4):
//   BLK_NONZERO  some coefficient is non-zero (otherwise all 64 samples are 0)
//   BLK_WIDE     A > COLOUR_SAFE_A: samples may leave the range the fp32 colour path is proven for
//   BLK_HUGE     samples may not fit the 16-bit fields of a tie record: the MCU is reconstructed wholesale on the exact path
constexpr uint32_t BLK_NONZERO = 1u, BLK_WIDE = 2u, BLK_HUGE = 4u;
constexpr float COLOUR_SAFE_A = 4.0f * (COLOUR_FAST_RANGE - 8.0f);
constexpr float SAMPLE_SAFE_A = 4.0f * 32000.0f;

// A biased 16-bit coefficient c + COEF_BIAS placed in the low mantissa bits of RINT_MAGIC's pattern is the float
// RINT_MAGIC + COEF_BIAS + c: subtracting SAMPLE_MAGIC gives c (exactly).
constexpr float SAMPLE_MAGIC = RINT_MAGIC + 32768.0f;

// Bit layout of a block's 64-bit tie mask (x = rows 0..3, y = rows 4..7): the bit of sample (row, col) in its word.
// The upper 16 bits hold columns 0..3, the lower 16 columns 4..7; inside, earlier samples sit higher.
__host__ __device__ constexpr int tie_bit(int row, int col) { return ((col & 4) ? 0 : 16) + 15 - (4 * (row & 3) + (col & 3)); }
// inverse: bit index b of word w (0 = rows 0..3, 1 = rows 4..7) -> sample index row * 8 + col
__device__ __forceinline__ int tie_sample(int w, int b)
{
    const int k = 15 - (b & 15);
    return (4 * w + (k >> 2)) * 8 + ((b & 16) ? 0 : 4) + (k & 3);
}

constexpr int TIE_LIST_CAP = IDCT_TIE_LIST_CAP; // (block, sample) entries per strip; a strip with more walks its blocks' masks instead
constexpr uint32_t TIE_EMPTY = 0xFFFFFFFFu;     // tie record without a pixel

template <int NC>
struct IdctSmem {
    static constexpr int NM = IDCT_MCUS_PER_CTA;
    static constexpr int NB = NM * NC;
    // The coefficient tile and the sample tile share their memory: every thread pulls its block into registers, a CTA
    // barrier, and the samples go where the coefficients were.  (The rare paths that need coefficients again -- the exact
    // evaluation of a strip with more ties than its list holds -- fetch them from the tile in global memory.)
    union {
        uint4 coef[NB * 8];           // [block][chunk ^ (block & 7)]: eight biased 16-bit coefficients per chunk, zig-zag order
        float4 samp[NC * 8 * 2 * NM]; // [comp][row][half][mcu] -> four rounded, unshifted samples (integer-valued floats)
    };
    float2 qpair[NC][32];         // prescaled quantisers in the pair order of the transform (pair_nat)
    uint2 tiemask[NB];            // per block: its tie mask (bit layout: tie_bit), for the flags of a tied pixel's other components
    uint16_t ties[TIE_LIST_CAP];  // block in strip | sample << 7
    uint8_t flag[NB];             // per block: BLK_*
    uint32_t ntie, any_huge;
    uint32_t img0, by0, bx0, mi0; // image / block row / block column / MCU-in-image of the strip's first MCU
    unsigned long long mbar;      // completion barrier of the stage-0 bulk copies
};
// eight strips per SM: 228 KB of shared memory, 1 KB of each CTA's share taken by the driver
static_assert(sizeof(IdctSmem<3>) <= (233472 / 8 - 1024), "idct_kernel<3> no longer fits eight CTAs per SM");

// ---- two fp32 lanes per instruction (sm_100a FADD2 / FMUL2 / FFMA2) -------------------------------
// K3 is bound by instruction issue, and most of what it issues are fp32 adds of the IDCT butterflies.  Blackwell's
// packed fp32 instructions do two independent IEEE lanes per issue slot, so the transform, the dequantisation, the
// rounding and the colour arithmetic run on register pairs.  A pair is a 64-bit register; packing / unpacking is
// register naming (mov.b64), not arithmetic.
struct F2 {
    unsigned long long v;
};
__device__ __forceinline__ F2 pack2(float lo, float hi)
{
    F2 r;
    asm("mov.b64 %0, {%1, %2};" : "=l"(r.v) : "f"(lo), "f"(hi));
    return r;
}
__device__ __forceinline__ void unpack2(F2 a, float &lo, float &hi) { asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(a.v)); }
__device__ __forceinline__ float lo2(F2 a)
{
    float lo, hi;
    unpack2(a, lo, hi);
    return lo;
}
__device__ __forceinline__ float hi2(F2 a)
{
    float lo, hi;
    unpack2(a, lo, hi);
    return hi;
}
__device__ __forceinline__ F2 splat2(float k) { return pack2(k, k); }
__device__ __forceinline__ F2 lane_add(F2 a, F2 b)
{
    F2 r;
    asm("add.rn.f32x2 %0, %1, %2;" : "=l"(r.v) : "l"(a.v), "l"(b.v));
    return r;
}
__device__ __forceinline__ F2 lane_sub(F2 a, F2 b)
{
    F2 r;
    asm("sub.rn.f32x2 %0, %1, %2;" : "=l"(r.v) : "l"(a.v), "l"(b.v));
    return r;
}
__device__ __forceinline__ F2 lane_mul(F2 a, F2 b)
{
    F2 r;
    asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(r.v) : "l"(a.v), "l"(b.v));
    return r;
}
__device__ __forceinline__ F2 lane_fma(F2 a, F2 b, F2 c)
{
    F2 r;
    asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r.v) : "l"(a.v), "l"(b.v), "l"(c.v));
    return r;
}
__device__ __forceinline__ F2 lane_mul_k(F2 a, float k) { return lane_mul(a, splat2(k)); }
__device__ __forceinline__ F2 lane_fma_k(F2 a, float k, F2 c) { return lane_fma(a, splat2(k), c); }

// Biased 16-bit value `h` (0 = low half, 1 = high half) of word w -> the float RINT_MAGIC + value + COEF_BIAS, by ONE byte
// permute: the 16 bits become the low mantissa bits of 0x4B40xxxx.  Subtracting SAMPLE_MAGIC (packed, two at a time)
// gives the value itself -- no I2F, which runs on the quarter-rate XU pipe.
__device__ __forceinline__ float biased16_as_magic(uint32_t w, int h)
{
    return __uint_as_float(__byte_perm(w, (uint32_t)RINT_MAGIC_BITS, h ? 0x7632u : 0x7610u));
}

// word holding coefficient I (zig-zag index) of a block held as eight 16-byte chunks
template <int I>
__device__ __forceinline__ uint32_t chunk_word(const uint4 (&ch)[8])
{
    constexpr int k = I >> 3, j = (I & 7) >> 1;
    return j == 0 ? ch[k].x : (j == 1 ? ch[k].y : (j == 2 ? ch[k].z : ch[k].w));
}

// Dequantise (AAN prescale folded into q; q arrives in pair order, see IdctSmem::qpair) and de-zigzag by register
// renaming; on the way, A = sum |c_i| * q_i, the magnitude the tie band is proportional to: |f| * (1 / prescale)
// with the reciprocal an immediate and the absolute value a free operand modifier -- one FFMA per coefficient.
// (fp32 accumulation is off by < 1e-5 relative; the band carries a 10 % margin.)  The DC term is kept apart:
// a_ac is a sum of non-negative terms, so it is zero exactly when every AC coefficient is.
template <int... Ps>
__device__ __forceinline__ void dequant_dezigzag(const uint4 (&ch)[8], const float2 *qpair, F2 (&P)[32], float &a_ac, float &a_dc,
                                                 std::integer_sequence<int, Ps...>)
{
    float A[4] = {0.0f, 0.0f, 0.0f, 0.0f}; // four short dependent chains instead of one of 64
    const F2 unbias = splat2(SAMPLE_MAGIC);
    float dcterm = 0.0f;
    auto one = [&](auto PI) {
        constexpr int p = decltype(PI)::value;
        constexpr int n0 = pair_nat(p, 0), n1 = pair_nat(p, 1);
        constexpr int z0 = NatZz<n0>::value, z1 = NatZz<n1>::value;
        const float2 q = qpair[p];
        const F2 c = lane_sub(pack2(biased16_as_magic(chunk_word<z0>(ch), z0 & 1), biased16_as_magic(chunk_word<z1>(ch), z1 & 1)), unbias);
        P[p] = lane_mul(c, pack2(q.x, q.y));
        if (n0 == 0)
            dcterm = fabsf(lo2(P[p])) * aan_unscale(n0);
        else
            A[p & 1] = fmaf(fabsf(lo2(P[p])), aan_unscale(n0), A[p & 1]);
        if (n1 == 0)
            dcterm = fabsf(hi2(P[p])) * aan_unscale(n1);
        else
            A[2 + (p & 1)] = fmaf(fabsf(hi2(P[p])), aan_unscale(n1), A[2 + (p & 1)]);
    };
    (one(std::integral_constant<int, Ps>{}), ...);
    a_ac = (A[0] + A[1]) + (A[2] + A[3]);
    a_dc = dcterm;
}

// Packed 2-D transform, first half: the row pass, two rows per instruction.
// P[rp * 8 + c] = rows pair_row(rp, 0), pair_row(rp, 1) at column c, in place.
__device__ __forceinline__ void idct_rows_packed(F2 (&P)[32])
{
#pragma unroll
    for (int rp = 0; rp < 4; ++rp)
        idct8_aan(P[rp * 8 + 0], P[rp * 8 + 1], P[rp * 8 + 2], P[rp * 8 + 3], P[rp * 8 + 4], P[rp * 8 + 5],
                  P[rp * 8 + 6], P[rp * 8 + 7]);
}

// Second half, one column: idct8_aan (idct_core.h) over the eight rows, same operations in the same order.
// With X = (v0, v1), Y = (v4, v7), X2 = (v2, v5), Y2 = (v6, v3) the first two butterfly stages of the even part
// (low lanes) and of the odd part (high lanes) are the same instruction, so they run packed; the rest is scalar on
// the halves.  Nothing is moved between registers.  v[r] = row r of this column.
__device__ __forceinline__ void idct8_column(F2 X, F2 Y, F2 X2, F2 Y2, float (&v)[8])
{
    const F2 S1 = lane_add(X, Y), D1 = lane_sub(X, Y);     // (t10, z11)  (t11, z12)
    const F2 S2 = lane_add(X2, Y2), D2 = lane_sub(X2, Y2); // (t13, z13)  (v2 - v6, z10)
    const F2 E = lane_add(S1, S2), F = lane_sub(S1, S2);   // (e0, o7)    (e3, z11 - z13)
    // even part
    const float t11 = lo2(D1), t13 = lo2(S2), e0 = lo2(E), e3 = lo2(F);
    const float n12 = lane_fma_k(lo2(D2), -1.414213562373095f, t13); // -(t12)
    const float e1 = lane_sub(t11, n12), e2 = lane_add(t11, n12);
    // odd part
    const float z12 = hi2(D1), z10 = hi2(D2), o7 = hi2(E);
    const float z5 = lane_mul_k(lane_add(z10, z12), 1.847759065022573f);
    const float t20 = lane_fma_k(z12, -1.082392200292394f, z5);
    const float t22 = lane_fma_k(z10, -2.613125929752753f, z5);
    const float o6 = lane_sub(t22, o7);
    const float n5 = lane_fma_k(hi2(F), -1.414213562373095f, o6); // -(o5)
    const float o4 = lane_add(t20, n5);
    v[0] = lane_add(e0, o7);
    v[7] = lane_sub(e0, o7);
    v[1] = lane_add(e1, o6);
    v[6] = lane_sub(e1, o6);
    v[2] = lane_sub(e2, n5);
    v[5] = lane_add(e2, n5);
    v[3] = lane_add(e3, o4);
    v[4] = lane_sub(e3, o4);
}

// Four ints -> four bytes with unsigned saturation (cvt.pack.sat: two values per instruction).
__device__ __forceinline__ uint32_t pack4_sat(int a, int b, int c, int d)
{
    // cvt.pack.sat.u8.s32.b32 d, x, y, z:  d = (z << 16) | (sat(x) << 8) | sat(y)
    uint32_t hi, r;
    asm("cvt.pack.sat.u8.s32.b32 %0, %1, %2, 0;" : "=r"(hi) : "r"(d), "r"(c));
    asm("cvt.pack.sat.u8.s32.b32 %0, %1, %2, %3;" : "=r"(r) : "r"(b), "r"(a), "r"(hi));
    return r;
}

// Rare path (G within 1e-3 of an integer, or samples out of the fp32-safe range): the reference's
// own double expression.  Out of line: several call sites.
__device__ __noinline__ uint32_t colour_exact_int(int y, int cb, int cr)
{
    int R, G, B;
    ycc_to_rgb_exact(y, cb, cr, R, G, B); // clamped to [0,255]
    return (uint32_t)R | ((uint32_t)G << 8) | ((uint32_t)B << 16);
}
__device__ __forceinline__ uint32_t colour_exact_px(float y, float cb, float cr) { return colour_exact_int((int)y, (int)cb, (int)cr); }

// pixel (unshifted integer samples) -> packed bytes, fast path with exact fallback
template <int NC>
__device__ __forceinline__ uint32_t colour_px(int y, int cb, int cr)
{
    if (NC == 1)
        return (uint32_t)clamp_u8(y + 128);
    int R, G, B;
    if (!ycc_to_rgb_fast((float)y, (float)cb, (float)cr, R, G, B))
        return colour_exact_int(y, cb, cr);
    return (uint32_t)clamp_u8(R) | ((uint32_t)clamp_u8(G) << 8) | ((uint32_t)clamp_u8(B) << 16);
}

// ---- colour of one pixel row of an MCU ---------------------------------------------------------------
// Colour of the eight pixels of one row of an MCU -> 24 channel values, three variants chosen per MCU:
//   COLOUR_PLAIN    ycc_to_rgb_fast's arithmetic on pixel pairs (FFMA2 / FADD2); its range precondition holds for
//                   the whole MCU (no block is BLK_WIDE) and its flat-chroma special case cannot occur unnoticed
//                   (a pixel with Cb = Cr = 0 fails the G test and takes the exact expression, which is right too)
//   COLOUR_FLAT     both chroma blocks are all-zero (gray-as-YCbCr content): R = G = B = Y + 128
//   COLOUR_GENERAL  ycc_to_rgb_fast itself, pixel by pixel, with its range and flat tests
enum { COLOUR_PLAIN = 0, COLOUR_FLAT = 1, COLOUR_GENERAL = 2 };

// bits 0..23 = R, G, B; bit 24 set when the double expression was needed
__device__ __noinline__ uint32_t colour_px_general(float y, float cb, float cr)
{
    int R, G, B;
    if (!ycc_to_rgb_fast(y, cb, cr, R, G, B))
        return colour_exact_px(y, cb, cr) | (1u << 24);
    return (uint32_t)clamp_u8(R) | ((uint32_t)clamp_u8(G) << 8) | ((uint32_t)clamp_u8(B) << 16);
}

// eight samples of a row (two float4 halves) -> four pairs: register naming only
__device__ __forceinline__ void row_pairs(const float4 &h0, const float4 &h1, F2 (&v)[4])
{
    v[0] = pack2(h0.x, h0.y);
    v[1] = pack2(h0.z, h0.w);
    v[2] = pack2(h1.x, h1.y);
    v[3] = pack2(h1.z, h1.w);
}

// -> the row's 24 bytes as six words; returns the number of pixels that took the double expression.
// redo (COLOUR_PLAIN only): bit j set = pixel j of the row must be replaced by colour_exact_px.
template <int MODE>
__device__ __forceinline__ uint32_t colour_row8(const F2 (&yy)[4], const F2 (&bb)[4], const F2 (&cc)[4], uint32_t (&out)[6],
                                                uint32_t &redo)
{
    uint32_t exact = 0;
    if constexpr (MODE == COLOUR_GENERAL) {
        uint32_t p[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            const float y = (j & 1) ? hi2(yy[j >> 1]) : lo2(yy[j >> 1]);
            const float cb = (j & 1) ? hi2(bb[j >> 1]) : lo2(bb[j >> 1]);
            const float cr = (j & 1) ? hi2(cc[j >> 1]) : lo2(cc[j >> 1]);
            p[j] = colour_px_general(y, cb, cr);
            exact += p[j] >> 24;
            p[j] &= 0xFFFFFFu;
        }
#pragma unroll
        for (int q = 0; q < 2; ++q) {
            out[3 * q + 0] = p[4 * q] | (p[4 * q + 1] << 24);
            out[3 * q + 1] = (p[4 * q + 1] >> 8) | (p[4 * q + 2] << 16);
            out[3 * q + 2] = (p[4 * q + 2] >> 16) | (p[4 * q + 3] << 8);
        }
        return exact;
    }
    int px[24];
    if constexpr (MODE == COLOUR_FLAT) {
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            const float y = (j & 1) ? hi2(yy[j >> 1]) : lo2(yy[j >> 1]);
            px[3 * j] = px[3 * j + 1] = px[3 * j + 2] = float_bits(y + (RINT_MAGIC + 128.0f)) - RINT_MAGIC_BITS;
        }
    } else {
        const F2 magic = splat2(RINT_MAGIC);
        const F2 tiny = splat2(__int_as_float(1)); // 2^-149
        F2 dg[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const F2 y = yy[k], cb = bb[k], cr = cc[k];
            // ycc_to_rgb_fast (idct_core.h), two pixels per instruction
            const F2 yr = lane_add(y, splat2(127.501f));
            const F2 yg = lane_add(y, splat2(127.5f));
            const F2 r = lane_fma_k(cr, 1.402f, yr);
            const F2 b = lane_fma_k(cb, 1.772f, yr);
            const F2 g = lane_fma_k(cr, -0.714136f, lane_fma_k(cb, -0.344136f, yg));
            dg[k] = lane_sub(g, lane_sub(lane_add(g, magic), magic));
            // rint() to an integer WITHOUT the magic-number bias: v * 2^-149 is a denormal whose bit pattern is
            // rint(v) itself (round to nearest even, like the magic add) when v >= 0, and has the sign bit set -- a
            // large negative int -- when v < 0, which the saturating pack turns into 0 just as it would -|v|.
            const F2 ri = lane_mul(r, tiny), gi = lane_mul(g, tiny), bi = lane_mul(b, tiny);
#pragma unroll
            for (int h = 0; h < 2; ++h) {
                const int j = 2 * k + h;
                px[3 * j] = float_bits(h ? hi2(ri) : lo2(ri));
                px[3 * j + 1] = float_bits(h ? hi2(gi) : lo2(gi));
                px[3 * j + 2] = float_bits(h ? hi2(bi) : lo2(bi));
            }
        }
        // G within COLOUR_G_BAND of an integer somewhere in the row (0.2 % of the pixels): ONE test per row on the
        // largest |dg|; the caller replaces the listed pixels by the double expression after the row is stored
        float worst = fmaxf(fabsf(lo2(dg[0])), fabsf(hi2(dg[0])));
#pragma unroll
        for (int k = 1; k < 4; ++k)
            worst = fmaxf(worst, fmaxf(fabsf(lo2(dg[k])), fabsf(hi2(dg[k]))));
        if (!(worst < 0.5f - COLOUR_G_BAND)) {
#pragma unroll
            for (int j = 0; j < 8; ++j)
                if (!(fabsf((j & 1) ? hi2(dg[j >> 1]) : lo2(dg[j >> 1])) < 0.5f - COLOUR_G_BAND))
                    redo |= 1u << j;
        }
    }
#pragma unroll
    for (int k = 0; k < 6; ++k)
        out[k] = pack4_sat(px[4 * k], px[4 * k + 1], px[4 * k + 2], px[4 * k + 3]);
    return exact;
}

// ---- exact evaluation (stage 3) ------------------------------------------------------------------------
// coefficient I (zig-zag index) of a block held as eight 16-byte chunks of biased 16-bit values, as an integer
template <int I>
__device__ __forceinline__ int chunk_coef_int(const uint4 (&ch)[8])
{
    const uint32_t w = chunk_word<I>(ch);
    return (int)((I & 1) ? (w >> 16) : (w & 0xFFFFu)) - (int)COEF_BIAS;
}

// The 64 terms of the reference's sum (idct_core.h exact_sample, MCU.cpp:184-198) in ascending natural order
// (== u outer, v inner), fully unrolled: every index is a compile-time constant, the block stays in registers, and
// there is no branch and no load of the block in the chain.  A zero coefficient contributes +-0, which leaves the float
// accumulator unchanged, so evaluating all 64 terms gives the same bits as skipping the zero ones.
template <int... Ns>
__device__ __forceinline__ float exact_terms(const uint4 (&ch)[8], const int32_t *q, const double (&cx)[8],
                                             const double (&cy)[8], float c00, float c01, std::integer_sequence<int, Ns...>)
{
    float sum = 0.0f;
    auto term = [&](auto N) {
        constexpr int nat = decltype(N)::value, zi = NatZz<nat>::value, u = nat >> 3, v = nat & 7;
        const int F = chunk_coef_int<zi>(ch) * __ldg(q + zi);                           // MCU.cpp:110-112, :115-120
        const float cc = (u == 0 && v == 0) ? c00 : ((u == 0 || v == 0) ? c01 : 1.0f); // Cu * Cv
        const float t = mul_f32(cc, (float)F);
#if KPEG_EXACT_WIDEN_INT
        const double d = mul_f64(mul_f64(widen_f32(t), cx[u]), cy[v]);
        sum = (float)add_f64(widen_f32(sum), d); // float accumulator, rounded every term
#else
        const double d = mul_f64(mul_f64((double)t, cx[u]), cy[v]);
#if KPEG_EXACT_SKIP_ZERO
        // a zero coefficient contributes +-0, which leaves the float accumulator unchanged: the add is predicated off,
        // so the lane's dependent chain is as long as its block has non-zero coefficients, not 64 terms (the kernel is
        // bound by the latency of that chain; at low quality settings the tied samples sit in blocks with a handful)
        if (F != 0)
            sum = (float)add_f64((double)sum, d);
#else
        sum = (float)add_f64((double)sum, d); // float accumulator, rounded every term
#endif
#endif
    };
    (term(std::integral_constant<int, Ns>{}), ...);
    return sum;
}

// The reference's evaluation of sample s of block gb (index in the job, component comp) from the coefficient tiles in global
// memory (DC value already in slot 0, AC coefficients already dropped where the F1 rule says so); defined below.
template <int NC>
__device__ __noinline__ int exact_sample_global(const uint4 *tiles, const DeviceTables *T, uint32_t gb, uint32_t comp, int s);

__device__ __forceinline__ void st_shared_u16(uint32_t addr, uint32_t v)
{
    asm volatile("st.shared.u16 [%0], %1;" ::"r"(addr), "h"((uint16_t)v) : "memory");
}

// CROP (crop decode, crop_geom.h): CTA i reconstructs strip a.strip_list[i], and every store -- the rows of stage 2, the
// colour-exact rewrites, the tie records and the pixels stage 3 repaints -- keeps to a.crop[image]
template <int NC, bool CROP>
__global__ void __launch_bounds__(NC * IDCT_MCUS_PER_CTA, NC == 3 ? KPEG_IDCT_MIN_CTAS : 16) idct_kernel(K3Args<CROP> a)
{
    constexpr int NM = IDCT_MCUS_PER_CTA;
    constexpr int NB = NM * NC;
    extern __shared__ __align__(128) unsigned char smem_raw[];
    IdctSmem<NC> &sm = *reinterpret_cast<IdctSmem<NC> *>(smem_raw);

    const int t = threadIdx.x;
    const int comp = t / NM; // warp-uniform
    const int ml = t % NM;   // == lane
    const int bl = ml * NC + comp; // block index inside the CTA's strip (MCU-interleaved)
    const uint32_t total_mcus = a.g.nimages * a.g.mcus_per_image;
    const uint32_t strip = k3_strip(a);
    const uint32_t mcu0 = strip * NM;
    const uint32_t m = mcu0 + ml;
    const bool active = m < total_mcus;

    // ---- stage 0: tile and quantisers by the copy engine, strip origin ------------------------------------------
    const uint32_t bar = smem_u32(&sm.mbar);
    if (t == 0) {
        k3_load_strip<NC, CROP>(a.tiles, strip, k3_nstrips(a), sm.coef, a.tables->qpair, NC * 64u * 4u, sm.qpair, bar, k3_list(a));
        sm.ntie = 0;
        sm.any_huge = 0;
        const uint32_t img = mcu0 / a.g.mcus_per_image, mi = mcu0 - img * a.g.mcus_per_image;
        sm.img0 = img;
        sm.mi0 = mi;
        sm.by0 = mi / a.g.mcus_x;
        sm.bx0 = mi - sm.by0 * a.g.mcus_x;
        mbar_wait(bar, 0); // the barrier below hands the data on
    }
    __syncthreads();

    // ---- stage 1: one thread = one 8x8 block ------------------------------------------------------
    uint4 ch[8];
#pragma unroll
    for (int k = 0; k < 8; ++k)
        ch[k] = sm.coef[bl * 8 + (k ^ (bl & 7))];
    __syncthreads(); // every block is in registers: the samples may overwrite the tile
    uint32_t tie_lo = 0, tie_hi = 0; // this block's tie mask (bit layout: tie_bit)
    if (active) {
        F2 P[32];
        float a_ac, a_dc;
        dequant_dezigzag(ch, sm.qpair[comp], P, a_ac, a_dc, std::make_integer_sequence<int, 32>{});
        const float A = a_ac + a_dc;
        uint32_t flag = (A != 0.0f ? BLK_NONZERO : 0u) | (A > COLOUR_SAFE_A ? BLK_WIDE : 0u);
        if (A > SAMPLE_SAFE_A) {
            // samples that may not fit 16 bits (no 8-bit image has them): the MCU is redone wholesale in stage 3
            flag |= BLK_HUGE;
            sm.any_huge = 1u;
        } else if (a_ac == 0.0f) {
            // DC only (flat blocks are common, and for suitable DC values EVERY sample is an exact tie): the reference's
            // sum has one non-zero term, float(C0 * C0 * F), whatever the sample (cos 0 = 1): MCU.cpp:190-198, :228
            const int dcv = (int)(ch[0].x & 0xFFFFu) - (int)COEF_BIAS;
            const int F = dcv * __ldg(&a.tables->qint[comp][0]);
            const float tt = mul_f32(__ldg(&a.tables->cc[0][0]), (float)F);
            const float b = (float)round_half_away(0.25f * tt);
            const float4 row = make_float4(b, b, b, b);
#pragma unroll
            for (int i = 0; i < 16; ++i)
                sm.samp[(comp * 16 + i) * NM + ml] = row;
        } else {
            const float thresh = 0.5f - tie_band(A);
            idct_rows_packed(P);
            // (x + M) - M == rint(x) for |x| < 2^22.  A sample is inside the tie band when its distance d from the
            // rounded value exceeds thresh, i.e. when d*d - thresh^2 >= 0: one FFMA2 per sample pair, and the
            // complement of the sign bit is shifted into the block's mask with one funnel shift per sample (no
            // compares, no predicates).  thresh^2 is taken a hair low, so the packed test can only flag more than
            // |d| > thresh does.  (x + M) - M, an integer-valued float, is the sample the tile keeps.
            const float t2 = thresh > 0.0f ? thresh * thresh * (1.0f - 1.0f / 2097152.0f) : 0.0f;
            const F2 neg_t2 = splat2(-t2);
            const F2 magic = splat2(RINT_MAGIC);
            uint32_t keep[2][2]; // [half][word]: sign bits = "outside the band", 16 per half and word
            auto half_block = [&](auto HALF) { // columns 4 half .. 4 half + 3 of all eight rows
                constexpr int half = decltype(HALF)::value;
                float v[4][8]; // [column - 4 half][row]
#pragma unroll
                for (int c = 0; c < 4; ++c)
                    idct8_column(P[0 * 8 + 4 * half + c], P[1 * 8 + 4 * half + c], P[2 * 8 + 4 * half + c], P[3 * 8 + 4 * half + c], v[c]);
                uint32_t kl = 0, kh = 0;
#pragma unroll
                for (int row = 0; row < 8; ++row) {
                    F2 w[2];
#pragma unroll
                    for (int k = 0; k < 2; ++k) {
                        const F2 x = pack2(v[2 * k][row], v[2 * k + 1][row]);
                        w[k] = lane_sub(lane_add(x, magic), magic);
                        const F2 d = lane_sub(x, w[k]);
                        const F2 e = lane_fma(d, d, neg_t2);
                        if (row < 4) {
                            kl = __funnelshift_l((uint32_t)float_bits(lo2(e)), kl, 1);
                            kl = __funnelshift_l((uint32_t)float_bits(hi2(e)), kl, 1);
                        } else {
                            kh = __funnelshift_l((uint32_t)float_bits(lo2(e)), kh, 1);
                            kh = __funnelshift_l((uint32_t)float_bits(hi2(e)), kh, 1);
                        }
                    }
                    sm.samp[((comp * 8 + row) * 2 + half) * NM + ml] = make_float4(lo2(w[0]), hi2(w[0]), lo2(w[1]), hi2(w[1]));
                }
                keep[half][0] = kl;
                keep[half][1] = kh;
            };
            half_block(std::integral_constant<int, 0>{});
            half_block(std::integral_constant<int, 1>{});
            // 16 bits per (half, word), first sample shifted in ends up highest: bit 15 - (4 (row & 3) + (col & 3))
            tie_lo = ~((keep[0][0] << 16) | (keep[1][0] & 0xFFFFu));
            tie_hi = ~((keep[0][1] << 16) | (keep[1][1] & 0xFFFFu));
            // queue the samples inside the band for stage 3 (most blocks have none)
            uint32_t lo = tie_lo, hi = tie_hi;
            while (lo | hi) {
                int w, b;
                if (lo) {
                    w = 0;
                    b = __ffs((int)lo) - 1;
                    lo &= lo - 1u;
                } else {
                    w = 1;
                    b = __ffs((int)hi) - 1;
                    hi &= hi - 1u;
                }
                const uint32_t at = atomicAdd(&sm.ntie, 1u);
                if (at < (uint32_t)TIE_LIST_CAP)
                    sm.ties[at] = (uint16_t)((uint32_t)bl | ((uint32_t)tie_sample(w, b) << 7));
            }
        }
        sm.flag[bl] = (uint8_t)flag;
    }
    sm.tiemask[bl] = make_uint2(tie_lo, tie_hi);
    __syncthreads();

    // ---- stage 2: colour conversion + interleaved store -------------------------------------------
    // position of MCU `mm_l` of the strip (no division when the strip wraps at most once)
    auto mcu_origin = [&](uint32_t mm_l, uint32_t &img, uint32_t &by, uint32_t &bx) {
        img = sm.img0, by = sm.by0, bx = sm.bx0 + mm_l;
        if (a.g.mcus_x >= (uint32_t)NM) {
            if (bx >= a.g.mcus_x) {
                bx -= a.g.mcus_x;
                if (++by == a.g.mcus_y) {
                    by = 0;
                    ++img;
                }
            }
        } else { // images narrower than a strip
            const uint32_t mg = mcu0 + mm_l;
            img = mg / a.g.mcus_per_image;
            const uint32_t mi = mg - img * a.g.mcus_per_image;
            by = mi / a.g.mcus_x;
            bx = mi - by * a.g.mcus_x;
        }
    };
    const uint32_t W = a.g.width, H = a.g.height;
    uint32_t colour_exact = 0;
    if (active) {
        uint32_t img, by, bx;
        mcu_origin((uint32_t)ml, img, by, bx);
        uint8_t *img_base = a.pixels + (size_t)img * W * H * NC;
        const bool full_w = bx * 8u + 8u <= W;
        // crop: the block's columns [c_lo, c_hi) lie inside the rectangle; 8-byte stores when all eight do and the
        // rectangle keeps them aligned
        CropWin win = {};
        uint32_t c_lo = 0, c_hi = 0;
        if constexpr (CROP) {
            win = a.crop[img];
            const uint32_t x = bx * 8u;
            c_lo = win.x0 > x ? min(win.x0 - x, 8u) : 0u;
            c_hi = win.x0 + win.w > x ? min(win.x0 + win.w - x, 8u) : 0u;
        }
        const bool vec_ok = CROP ? c_lo == 0u && c_hi == 8u && ((win.x0 | win.w) & 7u) == 0u &&
                                       (((reinterpret_cast<uintptr_t>(a.pixels) | win.out_off) & 7u) == 0u)
                                 : full_w && (W % 8u == 0u) && ((reinterpret_cast<uintptr_t>(a.pixels) & 7u) == 0);
        int mode = COLOUR_PLAIN;
        if constexpr (NC == 3) {
            const uint32_t f0 = sm.flag[ml * NC], f1 = sm.flag[ml * NC + 1], f2 = sm.flag[ml * NC + 2];
            mode = ((f0 | f1 | f2) & BLK_WIDE) ? COLOUR_GENERAL : (((f1 | f2) & BLK_NONZERO) ? COLOUR_PLAIN : COLOUR_FLAT);
        }
        for (int row = comp; row < 8; row += NC) { // the NC warps of the CTA share the 8 pixel rows
            const uint32_t y = by * 8u + row;
            if (y >= H)
                continue;
            if constexpr (CROP)
                if (y - win.y0 >= win.h || c_lo >= c_hi)
                    continue;
            const float4 y0 = sm.samp[((0 * 8 + row) * 2 + 0) * NM + ml], y1 = sm.samp[((0 * 8 + row) * 2 + 1) * NM + ml];
            uint32_t out[2 * NC];
            uint32_t redo = 0;
            if constexpr (NC == 3) {
                F2 yy[4], bb[4], cc[4];
                row_pairs(y0, y1, yy);
                row_pairs(sm.samp[((1 * 8 + row) * 2 + 0) * NM + ml], sm.samp[((1 * 8 + row) * 2 + 1) * NM + ml], bb);
                row_pairs(sm.samp[((2 * 8 + row) * 2 + 0) * NM + ml], sm.samp[((2 * 8 + row) * 2 + 1) * NM + ml], cc);
                uint32_t o6[6];
                if (mode == COLOUR_PLAIN)
                    colour_exact += colour_row8<COLOUR_PLAIN>(yy, bb, cc, o6, redo);
                else if (mode == COLOUR_FLAT)
                    colour_exact += colour_row8<COLOUR_FLAT>(yy, bb, cc, o6, redo);
                else
                    colour_exact += colour_row8<COLOUR_GENERAL>(yy, bb, cc, o6, redo);
#pragma unroll
                for (int k = 0; k < 6; ++k)
                    out[k] = o6[k];
            } else {
                // gray: the reference's colour path with Cb = Cr = 128 gives R = G = B = clamp(Y) (SURVEY A.8)
                const float f8[8] = {y0.x, y0.y, y0.z, y0.w, y1.x, y1.y, y1.z, y1.w};
                int v[8];
#pragma unroll
                for (int j = 0; j < 8; ++j) // integer-valued floats: the magic add is exact
                    v[j] = float_bits(f8[j] + (RINT_MAGIC + 128.0f)) - RINT_MAGIC_BITS;
                out[0] = pack4_sat(v[0], v[1], v[2], v[3]);
                out[1] = pack4_sat(v[4], v[5], v[6], v[7]);
            }
            uint8_t *dst = img_base + ((size_t)y * W + bx * 8u) * NC;
            if constexpr (CROP) // where column bx * 8 of row y would be in the crop (the bytes before c_lo are not stored)
                dst = a.pixels + (long long)(win.out_off + ((uint64_t)(y - win.y0) * win.w + bx * 8u) * NC) - (long long)win.x0 * NC;
            if (vec_ok) {
#pragma unroll
                for (int k = 0; k < NC; ++k)
                    reinterpret_cast<uint2 *>(dst)[k] = make_uint2(out[2 * k], out[2 * k + 1]);
            } else if constexpr (CROP) {
#pragma unroll
                for (int j = 0; j < 8 * NC; ++j)
                    if ((uint32_t)j >= c_lo * NC && (uint32_t)j < c_hi * NC)
                        dst[j] = (uint8_t)(out[j >> 2] >> (8 * (j & 3)));
            } else {
                const uint32_t nbytes = (full_w ? 8u : W - bx * 8u) * NC;
#pragma unroll
                for (int j = 0; j < 8 * NC; ++j) // compile-time indices: `out` stays in registers
                    if ((uint32_t)j < nbytes)
                        dst[j] = (uint8_t)(out[j >> 2] >> (8 * (j & 3)));
            }
            while (redo) { // rare: this thread's own later byte stores replace what it has just written
                const int j = __ffs((int)redo) - 1;
                redo &= redo - 1u;
                if (bx * 8u + (uint32_t)j >= W)
                    continue;
                if constexpr (CROP)
                    if ((uint32_t)j < c_lo || (uint32_t)j >= c_hi)
                        continue;
                const float *sp = reinterpret_cast<const float *>(sm.samp);
                const int sy = (int)sp[(((0 * 8 + row) * 2 + (j >> 2)) * NM + ml) * 4 + (j & 3)];
                const int sb = (int)sp[(((1 * 8 + row) * 2 + (j >> 2)) * NM + ml) * 4 + (j & 3)];
                const int sr = (int)sp[((((NC - 1) * 8 + row) * 2 + (j >> 2)) * NM + ml) * 4 + (j & 3)];
                const uint32_t e = colour_exact_int(sy, sb, sr);
                dst[3 * j] = (uint8_t)e;
                dst[3 * j + 1] = (uint8_t)(e >> 8);
                dst[3 * j + 2] = (uint8_t)(e >> 16);
                ++colour_exact;
            }
        }
    }
    __syncthreads();

    // ---- stage 3: the samples inside the tie band ------------------------------------------------------------
    const uint32_t ntie = sm.ntie;
    if (ntie == 0u && sm.any_huge == 0u) {
        if (t == 0)
            a.tie_cnt[strip] = 0u;
        if (colour_exact)
            atomicAdd(&a.meta->colour_exact, colour_exact);
        return;
    }
    float *spf = reinterpret_cast<float *>(sm.samp);
    const uint4 *gtiles = reinterpret_cast<const uint4 *>(a.tiles);
    const uint32_t blk0 = mcu0 * (uint32_t)NC; // first block of the strip in the job
    auto samp_index = [&](uint32_t c, uint32_t mm_l, int s) { // index of sample s of component c of MCU mm_l in the sample tile
        return ((((c * 8u + (uint32_t)(s >> 3)) * 2u + (uint32_t)((s & 7) >> 2)) * NM + mm_l) * 4u) + (uint32_t)(s & 3);
    };
    auto resolve = [&](uint32_t b, int s) { // exact sample -> sample tile
        const uint32_t c = b % NC, mm_l = b / NC;
        const int e = exact_sample_global<NC>(gtiles, a.tables, blk0 + b, c, s);
        spf[samp_index(c, mm_l, s)] = (float)e;
    };
    auto repaint = [&](uint32_t b, int s) { // pixel of sample s of block b's MCU from the (now exact) sample tile
        const uint32_t mm_l = b / NC;
        if (mcu0 + mm_l >= total_mcus)
            return;
        uint32_t img, by, bx;
        mcu_origin(mm_l, img, by, bx);
        const uint32_t px = bx * 8u + (uint32_t)(s & 7), py = by * 8u + (uint32_t)(s >> 3);
        if (px >= W || py >= H)
            return;
        uint64_t coff = 0;
        if constexpr (CROP) {
            coff = crop_pixel_offset(a.crop[img], NC, px, py);
            if (coff == CROP_SKIP)
                return;
        }
        const int y = (int)spf[samp_index(0, mm_l, s)];
        int cb = 0, cr = 0;
        if (NC == 3) {
            cb = (int)spf[samp_index(1, mm_l, s)];
            cr = (int)spf[samp_index(NC - 1, mm_l, s)];
        }
        const uint32_t v = colour_px<NC>(y, cb, cr);
        uint8_t *dst = CROP ? a.pixels + coff : a.pixels + ((size_t)img * W * H + (size_t)py * W + px) * NC;
        dst[0] = (uint8_t)v;
        if (NC == 3) {
            dst[1] = (uint8_t)(v >> 8);
            dst[2] = (uint8_t)(v >> 16);
        }
    };
    if (ntie <= (uint32_t)TIE_LIST_CAP) {
        // the common case: one record per tied PIXEL for idct_patch_kernel.  A pixel may be tied in more than one
        // component: the entry of the lowest tied component carries the flags of all of them, the others stay empty.
        // Pixels of an MCU that is redone wholesale below (BLK_HUGE) and pixels outside the image are not listed.
        for (uint32_t i = (uint32_t)t; i < ntie; i += (uint32_t)NB) {
            const uint32_t e = sm.ties[i], b = e & 127u, mm_l = b / NC, c = b % NC;
            const int sidx = (int)(e >> 7);
            // which components of this pixel are tied: one bit of each block's mask
            const int tbit = tie_bit(sidx >> 3, sidx & 7);
            uint32_t flags = 0, huge = 0;
#pragma unroll
            for (int cc = 0; cc < NC; ++cc) {
                const uint2 tm = sm.tiemask[mm_l * NC + cc];
                flags |= ((((sidx >> 3) & 4) ? tm.y : tm.x) >> tbit & 1u) << cc;
                huge |= sm.flag[mm_l * NC + cc];
            }
            uint4 r = make_uint4(TIE_EMPTY, 0, 0, 0);
            uint32_t img, by, bx;
            mcu_origin(mm_l, img, by, bx);
            const uint32_t px = bx * 8u + (uint32_t)(sidx & 7), py = by * 8u + (uint32_t)(sidx >> 3);
            bool listed = (flags & (0u - flags)) == (1u << c) && !(huge & BLK_HUGE) && mcu0 + mm_l < total_mcus && px < W && py < H;
            uint64_t coff = 0;
            if constexpr (CROP) { // a pixel outside the rectangle is not listed
                coff = listed ? crop_pixel_offset(a.crop[img], NC, px, py) : CROP_SKIP;
                listed = coff != CROP_SKIP;
            }
            if (listed) {
                r.x = img * W * H + py * W + px; // pixels of a job are < 2^32 (host_tables.h)
                if constexpr (CROP)
                    r.x = (uint32_t)(coff / NC); // the pixel's index in the crop output
                r.y = mcu0 + mm_l;
                auto biased = [&](uint32_t c) { return ((uint32_t)(int)spf[samp_index(c, mm_l, sidx)] + COEF_BIAS) & 0xFFFFu; };
                r.z = (uint32_t)sidx | (flags << 8) | (biased(0) << 16);
                r.w = NC == 3 ? biased(1) | (biased(2) << 16) : 0u;
            }
            a.tie_rec[(size_t)strip * TIE_LIST_CAP + i] = r;
        }
        if (t == 0)
            a.tie_cnt[strip] = ntie;
    } else {
        // more ties than the list holds (flat or synthetic content): every thread walks the mask of its own block and
        // resolves its ties here, from the tile, which is still in shared memory
        if (t == 0)
            a.tie_cnt[strip] = 0u;
        for (int pass = 0; pass < 2; ++pass) {
            uint32_t lo = tie_lo, hi = tie_hi;
            while (lo | hi) {
                int w, b;
                if (lo) {
                    w = 0;
                    b = __ffs((int)lo) - 1;
                    lo &= lo - 1u;
                } else {
                    w = 1;
                    b = __ffs((int)hi) - 1;
                    hi &= hi - 1u;
                }
                if (pass == 0)
                    resolve((uint32_t)bl, tie_sample(w, b));
                else
                    repaint((uint32_t)bl, tie_sample(w, b));
            }
            __syncthreads();
        }
    }
    if (sm.any_huge) {
        // MCUs with a block whose samples may not fit the sample tile (garbage-sized coefficients): every pixel from the
        // exact sample evaluation and the double colour expression, nothing through the 16-bit tile
        __syncthreads();
        for (uint32_t i = (uint32_t)t; i < (uint32_t)NM * 64u; i += (uint32_t)NB) {
            const uint32_t mm_l = i >> 6;
            const int s = (int)(i & 63u);
            uint32_t fl = 0;
            for (int c = 0; c < NC; ++c)
                fl |= sm.flag[mm_l * NC + c];
            if (!(fl & BLK_HUGE) || mcu0 + mm_l >= total_mcus)
                continue;
            uint32_t img, by, bx;
            mcu_origin(mm_l, img, by, bx);
            const uint32_t px = bx * 8u + (uint32_t)(s & 7), py = by * 8u + (uint32_t)(s >> 3);
            if (px >= W || py >= H)
                continue;
            uint64_t coff = 0;
            if constexpr (CROP) {
                coff = crop_pixel_offset(a.crop[img], NC, px, py);
                if (coff == CROP_SKIP)
                    continue;
            }
            int e[3] = {0, 0, 0};
            for (int c = 0; c < NC; ++c)
                e[c] = exact_sample_global<NC>(gtiles, a.tables, blk0 + mm_l * NC + (uint32_t)c, (uint32_t)c, s);
            const uint32_t v = NC == 3 ? colour_exact_int(e[0], e[1], e[2]) : (uint32_t)clamp_u8(e[0] + 128);
            uint8_t *dst = CROP ? a.pixels + coff : a.pixels + ((size_t)img * W * H + (size_t)py * W + px) * NC;
            dst[0] = (uint8_t)v;
            if (NC == 3) {
                dst[1] = (uint8_t)(v >> 8);
                dst[2] = (uint8_t)(v >> 16);
            }
        }
    }
    if (t == 0)
        atomicAdd(&a.meta->exact_samples, ntie);
    if (colour_exact)
        atomicAdd(&a.meta->colour_exact, colour_exact);
}

// ---- the tied pixels, re-evaluated in the reference's own operation order (MCU.cpp:184-198, :228) ---------------
// Tie record (uint4): x = pixel index in the job (image-major, row-major) or TIE_EMPTY, y = MCU index in the job,
// z = sample index | tied components << 8 | fast Y sample << 16, w = fast Cb sample | fast Cr sample << 16 (samples
// biased by COEF_BIAS).  A warp takes the records of 32 strips at a time and hands them out 32 per pass, so the long
// serial evaluation always runs with (nearly) full warps.
template <int NC>
__device__ __noinline__ int exact_sample_global(const uint4 *tiles, const DeviceTables *T, uint32_t gb, uint32_t comp, int s)
{
    uint4 ch[8];
#pragma unroll
    for (int k = 0; k < 8; ++k)
        ch[k] = __ldg(tiles + coef_tile_chunk(gb, (uint32_t)k));
    const int x = s >> 3, y = s & 7;
    double cx[8], cy[8];
#pragma unroll
    for (int k = 0; k < 8; ++k) {
        cx[k] = __ldg(&T->cosd[x][k]);
        cy[k] = __ldg(&T->cosd[y][k]);
    }
    const float sum = exact_terms(ch, T->qint[comp], cx, cy, __ldg(&T->cc[0][0]), __ldg(&T->cc[0][1]),
                                  std::make_integer_sequence<int, 64>{});
    const float out = (float)mul_f64(0.25, (double)sum);
    return round_half_away(out);
}

constexpr int PATCH_WARPS = 8;

// CROP: the strips are those of a.strip_list (the tie counts of the others are stale from earlier jobs); the records hold
// pixel indices in the crop output already
template <int NC, bool CROP>
__global__ void __launch_bounds__(PATCH_WARPS * 32) idct_patch_kernel(K3Args<CROP> a)
{
    // one CTA per 32 strips; its warps share the passes over the group's records (a pass = 32 records, one per lane):
    // every pass is a long serial chain, so it is the number of warps in flight that hides it
    const uint32_t lane = threadIdx.x & 31u, wl = threadIdx.x >> 5;
    const uint4 *tiles = reinterpret_cast<const uint4 *>(a.tiles);
    const uint32_t nstrips = k3_nstrips(a);
    for (uint32_t s0 = blockIdx.x * 32u; s0 < nstrips; s0 += gridDim.x * 32u) {
        uint32_t strip = s0 + lane;
        if constexpr (CROP)
            strip = s0 + lane < nstrips ? __ldg(a.strip_list + s0 + lane) : 0u;
        const uint32_t cnt = (CROP ? s0 + lane : strip) < nstrips ? min(__ldg(a.tie_cnt + strip), (uint32_t)TIE_LIST_CAP) : 0u;
        uint32_t incl = cnt; // inclusive scan of the 32 strips' counts
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const uint32_t o = __shfl_up_sync(0xffffffffu, incl, d);
            if ((int)lane >= d)
                incl += o;
        }
        const uint32_t total = __shfl_sync(0xffffffffu, incl, 31);
        for (uint32_t e0 = wl * 32u; e0 < total; e0 += PATCH_WARPS * 32u) {
            const uint32_t e = e0 + lane;
            // the strip record e belongs to: the first lane whose inclusive count exceeds e (five shuffle steps)
            uint32_t lo = 0;
#pragma unroll
            for (int step = 16; step >= 1; step >>= 1) {
                const uint32_t v = __shfl_sync(0xffffffffu, incl, (int)(lo + (uint32_t)step - 1u));
                if (v <= e)
                    lo += (uint32_t)step;
            }
            const uint32_t before = __shfl_sync(0xffffffffu, incl - cnt, (int)min(lo, 31u));
            uint32_t rstrip = s0 + lo;
            if constexpr (CROP)
                rstrip = __shfl_sync(0xffffffffu, strip, (int)min(lo, 31u));
            if (e >= total)
                continue;
            const uint4 r = __ldg(a.tie_rec + (size_t)rstrip * TIE_LIST_CAP + (e - before));
            if (r.x == TIE_EMPTY)
                continue;
            const int s = (int)(r.z & 63u);
            const uint32_t flags = (r.z >> 8) & 7u;
            int v[3] = {(int)(r.z >> 16) - (int)COEF_BIAS, (int)(r.w & 0xFFFFu) - (int)COEF_BIAS, (int)(r.w >> 16) - (int)COEF_BIAS};
            // nearly every tied pixel is tied in ONE component, a different one from lane to lane: every lane evaluates its
            // own lowest tied component in the same call (a loop over the components with a test per lane ran the 64-term
            // chain three times with a third of the lanes each: 11 of 32 lanes active on average)
            for (uint32_t left = flags; left != 0u; left &= left - 1u) {
                const uint32_t c = (uint32_t)__ffs((int)left) - 1u;
                const int ex = exact_sample_global<NC>(tiles, a.tables, r.y * NC + c, c, s);
                v[0] = c == 0u ? ex : v[0];
                v[1] = c == 1u ? ex : v[1];
                v[2] = c == 2u ? ex : v[2];
            }
            const uint32_t px = colour_px<NC>(v[0], v[1], v[2]);
            uint8_t *dst = a.pixels + (size_t)r.x * NC;
            dst[0] = (uint8_t)px;
            if (NC == 3) {
                dst[1] = (uint8_t)(px >> 8);
                dst[2] = (uint8_t)(px >> 16);
            }
        }
    }
}

void k3_configure()
{
    cudaFuncSetAttribute(idct_kernel<3, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(IdctSmem<3>));
    cudaFuncSetAttribute(idct_kernel<1, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(IdctSmem<1>));
    cudaFuncSetAttribute(idct_kernel<3, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(IdctSmem<3>));
    cudaFuncSetAttribute(idct_kernel<1, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(IdctSmem<1>));
}

uint32_t k3_strip_slots(uint32_t ncomp) { return (uint32_t)IDCT_MCUS_PER_CTA * ncomp * 64u; }

cudaError_t launch_idct(const IdctCropArgs &a_in, cudaStream_t s, uint32_t *launches)
{
    if (scale_denom(a_in.g.flags) != 1u)
        return launch_idct_scaled(a_in, s, launches);
    const IdctCropArgs &a = a_in;
    const IdctArgs &whole = a;
    const uint32_t total_mcus = a.g.nimages * a.g.mcus_per_image;
    const bool crop = a.crop != nullptr;
    const uint32_t grid = crop ? a.nlisted : (total_mcus + IDCT_MCUS_PER_CTA - 1) / IDCT_MCUS_PER_CTA;
    if (a.g.ncomp == 3)
        crop ? idct_kernel<3, true><<<grid, 3 * IDCT_MCUS_PER_CTA, sizeof(IdctSmem<3>), s>>>(a)
             : idct_kernel<3, false><<<grid, 3 * IDCT_MCUS_PER_CTA, sizeof(IdctSmem<3>), s>>>(whole);
    else
        crop ? idct_kernel<1, true><<<grid, IDCT_MCUS_PER_CTA, sizeof(IdctSmem<1>), s>>>(a)
             : idct_kernel<1, false><<<grid, IDCT_MCUS_PER_CTA, sizeof(IdctSmem<1>), s>>>(whole);
    ++*launches;
    // the pixels inside the tie band: a small grid (a few records per strip), full warps
    const uint32_t pgrid = std::min<uint32_t>((grid + 31u) / 32u, 148u * 16u);
    if (a.g.ncomp == 3)
        crop ? idct_patch_kernel<3, true><<<pgrid, PATCH_WARPS * 32, 0, s>>>(a) : idct_patch_kernel<3, false><<<pgrid, PATCH_WARPS * 32, 0, s>>>(whole);
    else
        crop ? idct_patch_kernel<1, true><<<pgrid, PATCH_WARPS * 32, 0, s>>>(a) : idct_patch_kernel<1, false><<<pgrid, PATCH_WARPS * 32, 0, s>>>(whole);
    ++*launches;
    return cudaSuccess;
}

} // namespace kpeg
