/* ref_scaled.c -- host reference of the reduced-size decode (KPEG_FLAG_SCALE_*), restated from libjpeg-turbo's C code:
 * jidctred.c (jpeg_idct_4x4, jpeg_idct_2x2, jpeg_idct_1x1, including their zero-AC shortcuts), jdmaster.c
 * (prepare_range_limit_table) and jdcolor.c (build_ycc_rgb_table, ycc_rgb_convert, grayscale_convert), with LP64 types
 * (JLONG = 64 bits).  Written independently of libkpeg_b200/csrc/idct_reduced.h, which the kernel and the replay share:
 * the tests hold the two against each other.
 *
 * kpo_reconstruct_scaled: quantised coefficients (the oracle's: [block][64] zig-zag, blocks MCU-interleaved, any parity
 * mode) and quantisers ([component][64] zig-zag) of `nimages` images of one geometry -> the images at 1/scale the size,
 * back to back, interleaved R,G,B or gray.  Returns 0, or -1 for bad arguments. */
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

typedef long long JLONG;
typedef unsigned char JSAMPLE;
#define MAXJSAMPLE 255
#define CENTERJSAMPLE 128
#define DCTSIZE 8
#define CONST_BITS 13
#define PASS1_BITS 2
#define RANGE_MASK (MAXJSAMPLE * 4 + 3)
#define ONE ((JLONG)1)
#define DESCALE(x, n) (((x) + (ONE << ((n) - 1))) >> (n))
#define LEFT_SHIFT(a, b) ((JLONG)((unsigned long long)(a) << (b)))
#define MULTIPLY(var, c) ((var) * (c))
#define DEQUANTIZE(coef, quantval) (((int)(coef)) * (quantval))

#define FIX_0_211164243 ((JLONG)1730)
#define FIX_0_509795579 ((JLONG)4176)
#define FIX_0_601344887 ((JLONG)4926)
#define FIX_0_720959822 ((JLONG)5906)
#define FIX_0_765366865 ((JLONG)6270)
#define FIX_0_850430095 ((JLONG)6967)
#define FIX_0_899976223 ((JLONG)7373)
#define FIX_1_061594337 ((JLONG)8697)
#define FIX_1_272758580 ((JLONG)10426)
#define FIX_1_451774981 ((JLONG)11893)
#define FIX_1_847759065 ((JLONG)15137)
#define FIX_2_172734803 ((JLONG)17799)
#define FIX_2_562915447 ((JLONG)20995)
#define FIX_3_624509785 ((JLONG)29692)

static const int natural_order[64] = {0,  1,  8,  16, 9,  2,  3,  10, 17, 24, 32, 25, 18, 11, 4,  5,  12, 19, 26, 33, 40, 48,
                                      41, 34, 27, 20, 13, 6,  7,  14, 21, 28, 35, 42, 49, 56, 57, 50, 43, 36, 29, 22, 15, 23,
                                      30, 37, 44, 51, 58, 59, 52, 45, 38, 31, 39, 46, 53, 60, 61, 54, 47, 55, 62, 63};

/* jdmaster.c prepare_range_limit_table: sample_range_limit, IDCT range limit = sample_range_limit + CENTERJSAMPLE */
static JSAMPLE range_table[5 * (MAXJSAMPLE + 1) + CENTERJSAMPLE];
static const JSAMPLE *sample_range_limit;

static void prepare_range_limit_table(void)
{
    JSAMPLE *table = range_table + (MAXJSAMPLE + 1);
    int i;
    sample_range_limit = table;
    memset(table - (MAXJSAMPLE + 1), 0, (MAXJSAMPLE + 1));
    for (i = 0; i <= MAXJSAMPLE; i++)
        table[i] = (JSAMPLE)i;
    table += CENTERJSAMPLE;
    for (i = CENTERJSAMPLE; i < 2 * (MAXJSAMPLE + 1); i++)
        table[i] = MAXJSAMPLE;
    memset(table + 2 * (MAXJSAMPLE + 1), 0, 2 * (MAXJSAMPLE + 1) - CENTERJSAMPLE);
    memcpy(table + (4 * (MAXJSAMPLE + 1) - CENTERJSAMPLE), sample_range_limit, CENTERJSAMPLE);
}

/* coef_block: natural order, as jdcoefct.c hands it to the IDCT; quantptr: natural order */
static void jpeg_idct_4x4(const int16_t *coef_block, const int *quantptr, JSAMPLE *out /* 4 x 4 */)
{
    const JSAMPLE *range_limit = sample_range_limit + CENTERJSAMPLE;
    int workspace[DCTSIZE * 4];
    const int16_t *inptr = coef_block;
    const int *qp = quantptr;
    int *wsptr = workspace;
    JLONG tmp0, tmp2, tmp10, tmp12, z1, z2, z3, z4;
    int ctr;
    for (ctr = DCTSIZE; ctr > 0; inptr++, qp++, wsptr++, ctr--) {
        if (ctr == DCTSIZE - 4)
            continue;
        if (inptr[DCTSIZE * 1] == 0 && inptr[DCTSIZE * 2] == 0 && inptr[DCTSIZE * 3] == 0 && inptr[DCTSIZE * 5] == 0 &&
            inptr[DCTSIZE * 6] == 0 && inptr[DCTSIZE * 7] == 0) {
            int dcval = (int)LEFT_SHIFT(DEQUANTIZE(inptr[DCTSIZE * 0], qp[DCTSIZE * 0]), PASS1_BITS);
            wsptr[DCTSIZE * 0] = dcval;
            wsptr[DCTSIZE * 1] = dcval;
            wsptr[DCTSIZE * 2] = dcval;
            wsptr[DCTSIZE * 3] = dcval;
            continue;
        }
        tmp0 = DEQUANTIZE(inptr[DCTSIZE * 0], qp[DCTSIZE * 0]);
        tmp0 = LEFT_SHIFT(tmp0, CONST_BITS + 1);
        z2 = DEQUANTIZE(inptr[DCTSIZE * 2], qp[DCTSIZE * 2]);
        z3 = DEQUANTIZE(inptr[DCTSIZE * 6], qp[DCTSIZE * 6]);
        tmp2 = MULTIPLY(z2, FIX_1_847759065) + MULTIPLY(z3, -FIX_0_765366865);
        tmp10 = tmp0 + tmp2;
        tmp12 = tmp0 - tmp2;
        z1 = DEQUANTIZE(inptr[DCTSIZE * 7], qp[DCTSIZE * 7]);
        z2 = DEQUANTIZE(inptr[DCTSIZE * 5], qp[DCTSIZE * 5]);
        z3 = DEQUANTIZE(inptr[DCTSIZE * 3], qp[DCTSIZE * 3]);
        z4 = DEQUANTIZE(inptr[DCTSIZE * 1], qp[DCTSIZE * 1]);
        tmp0 = MULTIPLY(z1, -FIX_0_211164243) + MULTIPLY(z2, FIX_1_451774981) + MULTIPLY(z3, -FIX_2_172734803) +
               MULTIPLY(z4, FIX_1_061594337);
        tmp2 = MULTIPLY(z1, -FIX_0_509795579) + MULTIPLY(z2, -FIX_0_601344887) + MULTIPLY(z3, FIX_0_899976223) +
               MULTIPLY(z4, FIX_2_562915447);
        wsptr[DCTSIZE * 0] = (int)DESCALE(tmp10 + tmp2, CONST_BITS - PASS1_BITS + 1);
        wsptr[DCTSIZE * 3] = (int)DESCALE(tmp10 - tmp2, CONST_BITS - PASS1_BITS + 1);
        wsptr[DCTSIZE * 1] = (int)DESCALE(tmp12 + tmp0, CONST_BITS - PASS1_BITS + 1);
        wsptr[DCTSIZE * 2] = (int)DESCALE(tmp12 - tmp0, CONST_BITS - PASS1_BITS + 1);
    }
    wsptr = workspace;
    for (ctr = 0; ctr < 4; ctr++) {
        JSAMPLE *outptr = out + ctr * 4;
        if (wsptr[1] == 0 && wsptr[2] == 0 && wsptr[3] == 0 && wsptr[5] == 0 && wsptr[6] == 0 && wsptr[7] == 0) {
            JSAMPLE outval = range_limit[(int)DESCALE((JLONG)wsptr[0], PASS1_BITS + 3) & RANGE_MASK];
            outptr[0] = outptr[1] = outptr[2] = outptr[3] = outval;
            wsptr += DCTSIZE;
            continue;
        }
        tmp0 = LEFT_SHIFT((JLONG)wsptr[0], CONST_BITS + 1);
        tmp2 = MULTIPLY((JLONG)wsptr[2], FIX_1_847759065) + MULTIPLY((JLONG)wsptr[6], -FIX_0_765366865);
        tmp10 = tmp0 + tmp2;
        tmp12 = tmp0 - tmp2;
        z1 = (JLONG)wsptr[7];
        z2 = (JLONG)wsptr[5];
        z3 = (JLONG)wsptr[3];
        z4 = (JLONG)wsptr[1];
        tmp0 = MULTIPLY(z1, -FIX_0_211164243) + MULTIPLY(z2, FIX_1_451774981) + MULTIPLY(z3, -FIX_2_172734803) +
               MULTIPLY(z4, FIX_1_061594337);
        tmp2 = MULTIPLY(z1, -FIX_0_509795579) + MULTIPLY(z2, -FIX_0_601344887) + MULTIPLY(z3, FIX_0_899976223) +
               MULTIPLY(z4, FIX_2_562915447);
        outptr[0] = range_limit[(int)DESCALE(tmp10 + tmp2, CONST_BITS + PASS1_BITS + 3 + 1) & RANGE_MASK];
        outptr[3] = range_limit[(int)DESCALE(tmp10 - tmp2, CONST_BITS + PASS1_BITS + 3 + 1) & RANGE_MASK];
        outptr[1] = range_limit[(int)DESCALE(tmp12 + tmp0, CONST_BITS + PASS1_BITS + 3 + 1) & RANGE_MASK];
        outptr[2] = range_limit[(int)DESCALE(tmp12 - tmp0, CONST_BITS + PASS1_BITS + 3 + 1) & RANGE_MASK];
        wsptr += DCTSIZE;
    }
}

static void jpeg_idct_2x2(const int16_t *coef_block, const int *quantptr, JSAMPLE *out /* 2 x 2 */)
{
    const JSAMPLE *range_limit = sample_range_limit + CENTERJSAMPLE;
    int workspace[DCTSIZE * 2];
    const int16_t *inptr = coef_block;
    const int *qp = quantptr;
    int *wsptr = workspace;
    JLONG tmp0, tmp10, z1;
    int ctr;
    for (ctr = DCTSIZE; ctr > 0; inptr++, qp++, wsptr++, ctr--) {
        if (ctr == DCTSIZE - 2 || ctr == DCTSIZE - 4 || ctr == DCTSIZE - 6)
            continue;
        if (inptr[DCTSIZE * 1] == 0 && inptr[DCTSIZE * 3] == 0 && inptr[DCTSIZE * 5] == 0 && inptr[DCTSIZE * 7] == 0) {
            int dcval = (int)LEFT_SHIFT(DEQUANTIZE(inptr[DCTSIZE * 0], qp[DCTSIZE * 0]), PASS1_BITS);
            wsptr[DCTSIZE * 0] = dcval;
            wsptr[DCTSIZE * 1] = dcval;
            continue;
        }
        z1 = DEQUANTIZE(inptr[DCTSIZE * 0], qp[DCTSIZE * 0]);
        tmp10 = LEFT_SHIFT(z1, CONST_BITS + 2);
        z1 = DEQUANTIZE(inptr[DCTSIZE * 7], qp[DCTSIZE * 7]);
        tmp0 = MULTIPLY(z1, -FIX_0_720959822);
        z1 = DEQUANTIZE(inptr[DCTSIZE * 5], qp[DCTSIZE * 5]);
        tmp0 += MULTIPLY(z1, FIX_0_850430095);
        z1 = DEQUANTIZE(inptr[DCTSIZE * 3], qp[DCTSIZE * 3]);
        tmp0 += MULTIPLY(z1, -FIX_1_272758580);
        z1 = DEQUANTIZE(inptr[DCTSIZE * 1], qp[DCTSIZE * 1]);
        tmp0 += MULTIPLY(z1, FIX_3_624509785);
        wsptr[DCTSIZE * 0] = (int)DESCALE(tmp10 + tmp0, CONST_BITS - PASS1_BITS + 2);
        wsptr[DCTSIZE * 1] = (int)DESCALE(tmp10 - tmp0, CONST_BITS - PASS1_BITS + 2);
    }
    wsptr = workspace;
    for (ctr = 0; ctr < 2; ctr++) {
        JSAMPLE *outptr = out + ctr * 2;
        if (wsptr[1] == 0 && wsptr[3] == 0 && wsptr[5] == 0 && wsptr[7] == 0) {
            JSAMPLE outval = range_limit[(int)DESCALE((JLONG)wsptr[0], PASS1_BITS + 3) & RANGE_MASK];
            outptr[0] = outptr[1] = outval;
            wsptr += DCTSIZE;
            continue;
        }
        tmp10 = LEFT_SHIFT((JLONG)wsptr[0], CONST_BITS + 2);
        tmp0 = MULTIPLY((JLONG)wsptr[7], -FIX_0_720959822) + MULTIPLY((JLONG)wsptr[5], FIX_0_850430095) +
               MULTIPLY((JLONG)wsptr[3], -FIX_1_272758580) + MULTIPLY((JLONG)wsptr[1], FIX_3_624509785);
        outptr[0] = range_limit[(int)DESCALE(tmp10 + tmp0, CONST_BITS + PASS1_BITS + 3 + 2) & RANGE_MASK];
        outptr[1] = range_limit[(int)DESCALE(tmp10 - tmp0, CONST_BITS + PASS1_BITS + 3 + 2) & RANGE_MASK];
        wsptr += DCTSIZE;
    }
}

static void jpeg_idct_1x1(const int16_t *coef_block, const int *quantptr, JSAMPLE *out)
{
    const JSAMPLE *range_limit = sample_range_limit + CENTERJSAMPLE;
    int dcval = DEQUANTIZE(coef_block[0], quantptr[0]);
    dcval = (int)DESCALE((JLONG)dcval, 3);
    out[0] = range_limit[dcval & RANGE_MASK];
}

/* jdcolor.c build_ycc_rgb_table */
#define SCALEBITS 16
#define ONE_HALF ((JLONG)1 << (SCALEBITS - 1))
#define FIX(x) ((JLONG)((x) * (1L << SCALEBITS) + 0.5))
static int Cr_r_tab[256], Cb_b_tab[256];
static JLONG Cr_g_tab[256], Cb_g_tab[256];

static void build_ycc_rgb_table(void)
{
    int i;
    JLONG x;
    for (i = 0, x = -CENTERJSAMPLE; i <= MAXJSAMPLE; i++, x++) {
        Cr_r_tab[i] = (int)((FIX(1.40200) * x + ONE_HALF) >> SCALEBITS);
        Cb_b_tab[i] = (int)((FIX(1.77200) * x + ONE_HALF) >> SCALEBITS);
        Cr_g_tab[i] = (-FIX(0.71414)) * x;
        Cb_g_tab[i] = (-FIX(0.34414)) * x + ONE_HALF;
    }
}

int kpo_reconstruct_scaled(const int16_t *coef, const uint16_t *qt, int width, int height, int ncomp, int nimages, int scale,
                           uint8_t *out)
{
    if (!coef || !qt || !out || width < 1 || height < 1 || (ncomp != 1 && ncomp != 3) || nimages < 1 ||
        (scale != 2 && scale != 4 && scale != 8))
        return -1;
    prepare_range_limit_table();
    build_ycc_rgb_table();
    const int k = 8 / scale, mx = (width + 7) / 8, my = (height + 7) / 8;
    const int ow = (width + scale - 1) / scale, oh = (height + scale - 1) / scale;
    const int pw = mx * k, ph = my * k; /* whole-block planes, cropped on output */
    JSAMPLE *planes = (JSAMPLE *)malloc((size_t)ncomp * pw * ph);
    if (!planes)
        return -1;
    int q[3][64];
    for (int c = 0; c < ncomp; ++c)
        for (int i = 0; i < 64; ++i)
            q[c][natural_order[i]] = qt[c * 64 + i];
    for (int img = 0; img < nimages; ++img) {
        for (int by = 0; by < my; ++by)
            for (int bx = 0; bx < mx; ++bx)
                for (int c = 0; c < ncomp; ++c) {
                    const int16_t *zz = coef + ((((size_t)img * my + by) * mx + bx) * ncomp + c) * 64;
                    int16_t nat[64];
                    JSAMPLE blk[16];
                    for (int i = 0; i < 64; ++i)
                        nat[natural_order[i]] = zz[i];
                    if (scale == 2)
                        jpeg_idct_4x4(nat, q[c], blk);
                    else if (scale == 4)
                        jpeg_idct_2x2(nat, q[c], blk);
                    else
                        jpeg_idct_1x1(nat, q[c], blk);
                    for (int r = 0; r < k; ++r)
                        for (int x = 0; x < k; ++x)
                            planes[((size_t)c * ph + by * k + r) * pw + bx * k + x] = blk[r * k + x];
                }
        uint8_t *o = out + (size_t)img * ow * oh * ncomp;
        for (int y = 0; y < oh; ++y)
            for (int x = 0; x < ow; ++x) {
                const int Y = planes[(size_t)y * pw + x];
                if (ncomp == 1) {
                    o[(size_t)y * ow + x] = (uint8_t)Y; /* grayscale_convert: a copy */
                    continue;
                }
                const int cb = planes[((size_t)ph + y) * pw + x], cr = planes[((size_t)2 * ph + y) * pw + x];
                uint8_t *p = o + ((size_t)y * ow + x) * 3;
                p[0] = sample_range_limit[Y + Cr_r_tab[cr]];
                p[1] = sample_range_limit[Y + (int)((Cb_g_tab[cb] + Cr_g_tab[cr]) >> SCALEBITS)];
                p[2] = sample_range_limit[Y + Cb_b_tab[cb]];
            }
    }
    free(planes);
    return 0;
}
