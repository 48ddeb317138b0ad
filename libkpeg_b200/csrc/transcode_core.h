// transcode_core.h -- per-block logic of the lossless transcoder (csrc/transcode.cu, kpeg_cuda_transcode), written as
// KPEG_HD code so tests/emu/emu_transcode.cpp replays exactly what TG runs.
//
// TG (tc_gather_kernel) turns the decoder's coefficient tiles (K2's output: biased by COEF_BIAS, zig-zag, 16-byte chunks
// swizzled, kernels.cuh) into the encoder's input (coef [nblk][64] zig-zag, dc [nblk]) in OUTPUT block order, moving
// every block by one of the eight lossless transforms (KPEG_XFORM_*, include/kpeg_cuda.h):
//   - the block grid: output block (bx, by) comes from source block source_block(t, bx, by);
//   - inside a block: output zig-zag position i takes source position kXform.e[t][i] & 63, negated when bit 7 is set
//     (u is the vertical frequency, v the horizontal one: a horizontal flip negates odd v, a vertical flip odd u, a
//     transpose swaps F[u][v] and F[v][u]).
// It also checks the baseline range rules in the output's block order and segmentation (every DC difference of category
// <= 11, every AC coefficient within +-1023): the coded stages index their tables by category and the encoder's scratch
// is sized by the bound those rules give, so a violation is reported before anything is coded.
#ifndef KPEG_TRANSCODE_CORE_H
#define KPEG_TRANSCODE_CORE_H

#include <stdint.h>

#include "encode_core.h"
#include "kpeg_common.h"
#include "kpeg_cuda.h"

namespace kpeg {
namespace tc {

constexpr int NXFORM = 8;

KPEG_HD bool transposes(uint32_t t)
{
    return t == KPEG_XFORM_TRANSPOSE || t == KPEG_XFORM_TRANSVERSE || t == KPEG_XFORM_ROT90 || t == KPEG_XFORM_ROT270;
}

// jpegtran -perfect: a flip may not move a partial edge block.  w, h: the input's size.
KPEG_HD bool xform_allowed(uint32_t t, uint32_t w, uint32_t h)
{
    const bool w8 = w % 8u == 0u, h8 = h % 8u == 0u;
    switch (t) {
    case KPEG_XFORM_NONE:
    case KPEG_XFORM_TRANSPOSE: return true;
    case KPEG_XFORM_FLIP_H: return w8;
    case KPEG_XFORM_FLIP_V: return h8;
    case KPEG_XFORM_TRANSVERSE:
    case KPEG_XFORM_ROT180: return w8 && h8;
    case KPEG_XFORM_ROT90: return h8;
    case KPEG_XFORM_ROT270: return w8;
    default: return false;
    }
}

// Source block of output block (bx, by); smx, smy: the source's block grid.
KPEG_HD void source_block(uint32_t t, uint32_t bx, uint32_t by, uint32_t smx, uint32_t smy, uint32_t &sx, uint32_t &sy)
{
    switch (t) {
    case KPEG_XFORM_FLIP_H: sx = smx - 1u - bx; sy = by; break;
    case KPEG_XFORM_FLIP_V: sx = bx; sy = smy - 1u - by; break;
    case KPEG_XFORM_TRANSPOSE: sx = by; sy = bx; break;
    case KPEG_XFORM_TRANSVERSE: sx = smx - 1u - by; sy = smy - 1u - bx; break;
    case KPEG_XFORM_ROT90: sx = by; sy = smy - 1u - bx; break;
    case KPEG_XFORM_ROT180: sx = smx - 1u - bx; sy = smy - 1u - by; break;
    case KPEG_XFORM_ROT270: sx = smx - 1u - by; sy = bx; break;
    default: sx = bx; sy = by; break;
    }
}

// ---- the in-block permutation and signs, one 64-entry table per transform -------------------------------------
struct XformTable {
    uint8_t e[NXFORM][64]; // output zig-zag i -> source zig-zag index | 0x80 when the value is negated
};

constexpr XformTable make_xform_table()
{
    int nat[64] = {}, zz[64] = {}; // zig-zag <-> natural (row * 8 + column)
    int i = 0;
    for (int d = 0; d < 15; ++d) {
        const int lo = d < 8 ? 0 : d - 7, hi = d < 8 ? d : 7;
        for (int k = lo; k <= hi; ++k) {
            const int r = (d & 1) ? k : (hi + lo - k);
            nat[i] = r * 8 + (d - r);
            zz[nat[i]] = i;
            ++i;
        }
    }
    XformTable T = {};
    for (int t = 0; t < NXFORM; ++t) {
        const bool tr = t == 3 || t == 4 || t == 5 || t == 7;
        const bool neg_v = t == 1 || t == 4 || t == 5 || t == 6; // of the output's horizontal frequency
        const bool neg_u = t == 2 || t == 4 || t == 6 || t == 7; // of the output's vertical frequency
        for (int o = 0; o < 64; ++o) {
            const int u = nat[o] >> 3, v = nat[o] & 7;
            const int src = tr ? zz[v * 8 + u] : o;
            const bool neg = ((neg_v && (v & 1)) != (neg_u && (u & 1)));
            T.e[t][o] = (uint8_t)(src | (neg ? 0x80 : 0));
        }
    }
    return T;
}

// Largest magnitudes the baseline tables code: DC difference category <= 11, AC category <= 10 (T.81 F.1.2).
constexpr int MAX_DC_DIFF = 2047;
constexpr int MAX_AC = 1023;

// What TG needs: the output geometry (EncGeom with the output's size and restart interval) and the source grid.
struct TcGeom {
    enc::EncGeom out;
    uint32_t smx, smy; // source block grid
    uint32_t xform;
};

// Source block (MCU-interleaved index) of output block ob.
KPEG_HD uint64_t source_index(const TcGeom &g, uint64_t ob)
{
    const uint64_t m = ob / g.out.ncomp, c = ob - m * g.out.ncomp;
    uint32_t sx, sy;
    source_block(g.xform, (uint32_t)(m % g.out.mx), (uint32_t)(m / g.out.mx), g.smx, g.smy, sx, sy);
    return ((uint64_t)sy * g.smx + sx) * g.out.ncomp + c;
}

// Output zig-zag positions 8k .. 8k+7 of a block from its source block's 64 plain coefficients (zig-zag).  Returns
// false when one of them is an AC coefficient beyond MAX_AC.
KPEG_HD bool gather_chunk(const XformTable &T, uint32_t t, const int16_t *src, int k, int16_t o[8])
{
    bool ok = true;
    for (int j = 0; j < 8; ++j) {
        const int i = 8 * k + j;
        const uint32_t e = T.e[t][i];
        const int v = (e & 0x80u) ? -(int)src[e & 63u] : (int)src[e & 63u];
        o[j] = (int16_t)v;
        if (i && (v > MAX_AC || v < -MAX_AC))
            ok = false;
    }
    return ok;
}

// The DC difference of output block ob under the output's segmentation is within range.  dc_of(block) gives the
// absolute DC of an output block.
template <class DcOf>
KPEG_HD bool dc_in_range(const TcGeom &g, uint64_t ob, int dc, const DcOf &dc_of)
{
    const uint64_t m = ob / g.out.ncomp;
    const int diff = dc - (enc::starts_segment(g.out, m) ? 0 : dc_of(ob - g.out.ncomp));
    return diff <= MAX_DC_DIFF && diff >= -MAX_DC_DIFF;
}

} // namespace tc
} // namespace kpeg
#endif
