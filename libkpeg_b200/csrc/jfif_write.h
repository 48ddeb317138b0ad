// jfif_write.h -- host-only pieces every baseline-JPEG writer of this project shares: the ITU-T T.81
// Annex K quantisation and Huffman tables, the zig-zag order, the IJG quality scaling, the double
// FDCT cosine table and the container header (lena's segment order, SURVEY F7).
//
// Used by the synthetic reference encoder (host/synth_encoder.cpp) and by the GPU encoder's host side
// (csrc/encode_tables.cpp).  Both are compiled with -ffp-contract=off: the cosine table is evaluated
// here with the host libm, once, and the GPU encoder uploads it, so the two encoders multiply by the
// very same doubles.
#ifndef KPEG_JFIF_WRITE_H
#define KPEG_JFIF_WRITE_H

#include <stdint.h>

#include <cmath>
#include <cstring>
#include <vector>

#include "huff_opt.h"

namespace kpeg {
namespace jfif {

// ---- ITU-T T.81 Annex K tables (public standard constants) -------------------------------------

inline constexpr uint8_t kLumaQ[64] = {16, 11, 10, 16, 24,  40,  51,  61,  12, 12, 14, 19, 26,  58,  60,  55,
                                       14, 13, 16, 24, 40,  57,  69,  56,  14, 17, 22, 29, 51,  87,  80,  62,
                                       18, 22, 37, 56, 68,  109, 103, 77,  24, 35, 55, 64, 81,  104, 113, 92,
                                       49, 64, 78, 87, 103, 121, 120, 101, 72, 92, 95, 98, 112, 100, 103, 99};
inline constexpr uint8_t kChromaQ[64] = {17, 18, 24, 47, 99, 99, 99, 99, 18, 21, 26, 66, 99, 99, 99, 99,
                                         24, 26, 56, 99, 99, 99, 99, 99, 47, 66, 99, 99, 99, 99, 99, 99,
                                         99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99,
                                         99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99};

inline constexpr uint8_t kDcLumaBits[16] = {0, 1, 5, 1, 1, 1, 1, 1, 1, 0, 0, 0, 0, 0, 0, 0};
inline constexpr uint8_t kDcChromaBits[16] = {0, 3, 1, 1, 1, 1, 1, 1, 1, 1, 1, 0, 0, 0, 0, 0};
inline constexpr uint8_t kDcVals[12] = {0, 1, 2, 3, 4, 5, 6, 7, 8, 9, 10, 11};
inline constexpr uint8_t kAcLumaBits[16] = {0, 2, 1, 3, 3, 2, 4, 3, 5, 5, 4, 4, 0, 0, 1, 0x7d};
inline constexpr uint8_t kAcLumaVals[162] = {
    0x01, 0x02, 0x03, 0x00, 0x04, 0x11, 0x05, 0x12, 0x21, 0x31, 0x41, 0x06, 0x13, 0x51, 0x61, 0x07, 0x22, 0x71,
    0x14, 0x32, 0x81, 0x91, 0xa1, 0x08, 0x23, 0x42, 0xb1, 0xc1, 0x15, 0x52, 0xd1, 0xf0, 0x24, 0x33, 0x62, 0x72,
    0x82, 0x09, 0x0a, 0x16, 0x17, 0x18, 0x19, 0x1a, 0x25, 0x26, 0x27, 0x28, 0x29, 0x2a, 0x34, 0x35, 0x36, 0x37,
    0x38, 0x39, 0x3a, 0x43, 0x44, 0x45, 0x46, 0x47, 0x48, 0x49, 0x4a, 0x53, 0x54, 0x55, 0x56, 0x57, 0x58, 0x59,
    0x5a, 0x63, 0x64, 0x65, 0x66, 0x67, 0x68, 0x69, 0x6a, 0x73, 0x74, 0x75, 0x76, 0x77, 0x78, 0x79, 0x7a, 0x83,
    0x84, 0x85, 0x86, 0x87, 0x88, 0x89, 0x8a, 0x92, 0x93, 0x94, 0x95, 0x96, 0x97, 0x98, 0x99, 0x9a, 0xa2, 0xa3,
    0xa4, 0xa5, 0xa6, 0xa7, 0xa8, 0xa9, 0xaa, 0xb2, 0xb3, 0xb4, 0xb5, 0xb6, 0xb7, 0xb8, 0xb9, 0xba, 0xc2, 0xc3,
    0xc4, 0xc5, 0xc6, 0xc7, 0xc8, 0xc9, 0xca, 0xd2, 0xd3, 0xd4, 0xd5, 0xd6, 0xd7, 0xd8, 0xd9, 0xda, 0xe1, 0xe2,
    0xe3, 0xe4, 0xe5, 0xe6, 0xe7, 0xe8, 0xe9, 0xea, 0xf1, 0xf2, 0xf3, 0xf4, 0xf5, 0xf6, 0xf7, 0xf8, 0xf9, 0xfa};
inline constexpr uint8_t kAcChromaBits[16] = {0, 2, 1, 2, 4, 4, 3, 4, 7, 5, 4, 4, 0, 1, 2, 0x77};
inline constexpr uint8_t kAcChromaVals[162] = {
    0x00, 0x01, 0x02, 0x03, 0x11, 0x04, 0x05, 0x21, 0x31, 0x06, 0x12, 0x41, 0x51, 0x07, 0x61, 0x71, 0x13, 0x22,
    0x32, 0x81, 0x08, 0x14, 0x42, 0x91, 0xa1, 0xb1, 0xc1, 0x09, 0x23, 0x33, 0x52, 0xf0, 0x15, 0x62, 0x72, 0xd1,
    0x0a, 0x16, 0x24, 0x34, 0xe1, 0x25, 0xf1, 0x17, 0x18, 0x19, 0x1a, 0x26, 0x27, 0x28, 0x29, 0x2a, 0x35, 0x36,
    0x37, 0x38, 0x39, 0x3a, 0x43, 0x44, 0x45, 0x46, 0x47, 0x48, 0x49, 0x4a, 0x53, 0x54, 0x55, 0x56, 0x57, 0x58,
    0x59, 0x5a, 0x63, 0x64, 0x65, 0x66, 0x67, 0x68, 0x69, 0x6a, 0x73, 0x74, 0x75, 0x76, 0x77, 0x78, 0x79, 0x7a,
    0x82, 0x83, 0x84, 0x85, 0x86, 0x87, 0x88, 0x89, 0x8a, 0x92, 0x93, 0x94, 0x95, 0x96, 0x97, 0x98, 0x99, 0x9a,
    0xa2, 0xa3, 0xa4, 0xa5, 0xa6, 0xa7, 0xa8, 0xa9, 0xaa, 0xb2, 0xb3, 0xb4, 0xb5, 0xb6, 0xb7, 0xb8, 0xb9, 0xba,
    0xc2, 0xc3, 0xc4, 0xc5, 0xc6, 0xc7, 0xc8, 0xc9, 0xca, 0xd2, 0xd3, 0xd4, 0xd5, 0xd6, 0xd7, 0xd8, 0xd9, 0xda,
    0xe2, 0xe3, 0xe4, 0xe5, 0xe6, 0xe7, 0xe8, 0xe9, 0xea, 0xf2, 0xf3, 0xf4, 0xf5, 0xf6, 0xf7, 0xf8, 0xf9, 0xfa};

// zig-zag index -> natural (row*8+col) index
struct ZigZag {
    int nat[64];
    ZigZag()
    {
        int i = 0;
        for (int d = 0; d < 15; ++d) {
            int lo = d < 8 ? 0 : d - 7, hi = d < 8 ? d : 7;
            for (int k = lo; k <= hi; ++k) {
                int r = (d & 1) ? k : (hi + lo - k);
                nat[i++] = r * 8 + (d - r);
            }
        }
    }
};
inline const ZigZag kZZ;

// Canonical Huffman code (T.81 Annex C) of one DHT table, indexed by symbol.
struct HuffEnc {
    uint16_t code[256];
    uint8_t len[256];
    HuffEnc(const uint8_t bits[16], const uint8_t *vals) { huff::canonical_codes(bits, vals, code, len); }
};

// The four Annex K tables in the order [0 = DC luma, 1 = AC luma, 2 = DC chroma, 3 = AC chroma].
inline HuffEnc annex_k_table(int t)
{
    switch (t) {
    case 0: return HuffEnc(kDcLumaBits, kDcVals);
    case 1: return HuffEnc(kAcLumaBits, kAcLumaVals);
    case 2: return HuffEnc(kDcChromaBits, kDcVals);
    default: return HuffEnc(kAcChromaBits, kAcChromaVals);
    }
}

// IJG quality scaling of an Annex K table (natural order), clamped to 1..255.
inline void scaled_qt(const uint8_t base[64], int quality, uint8_t out_nat[64])
{
    int scale = quality < 50 ? 5000 / quality : 200 - 2 * quality;
    for (int i = 0; i < 64; ++i) {
        int t = (base[i] * scale + 50) / 100;
        out_nat[i] = (uint8_t)(t < 1 ? 1 : (t > 255 ? 255 : t));
    }
}

// cs[x][u] = C(u)/2 * cos((2x+1) u pi / 16): the FDCT basis both encoders multiply by
inline void fdct_cosines(double cs[8][8])
{
    for (int x = 0; x < 8; ++x)
        for (int u = 0; u < 8; ++u)
            cs[x][u] = (u == 0 ? std::sqrt(0.125) : 0.5) * std::cos((2 * x + 1) * u * M_PI / 16.0);
}

inline void put16(std::vector<uint8_t> &o, int v)
{
    o.push_back((uint8_t)(v >> 8));
    o.push_back((uint8_t)v);
}

// appends to a byte vector (the Out of the huff_opt.h writers)
struct VecOut {
    std::vector<uint8_t> &o;
    void put(uint32_t b) { o.push_back((uint8_t)b); }
};

inline void put_dht(std::vector<uint8_t> &o, int tc_th, const uint8_t bits[16], const uint8_t *vals)
{
    VecOut v{o};
    huff::put_dht(v, tc_th, bits, vals);
}

inline void put_dri(std::vector<uint8_t> &o, int dri)
{
    VecOut v{o};
    huff::put_dri(v, dri);
}

// The four Annex K tables as BITS / HUFFVAL, [0 = DC luma, 1 = AC luma, 2 = DC chroma, 3 = AC chroma]
inline const uint8_t *const kAnnexKBits[4] = {kDcLumaBits, kAcLumaBits, kDcChromaBits, kAcChromaBits};
inline const uint8_t *const kAnnexKVals[4] = {kDcVals, kAcLumaVals, kDcVals, kAcChromaVals};

// The encoder's quantiser ids: luma table 0 for component 0, chroma table 1 for components 1 and 2.
inline constexpr uint8_t kEncoderTq[3] = {0, 1, 1};

// The encoder's quantisers for `quality` in zig-zag order, by id ([0] luma, [1] chroma; [2], [3] unused, zeroed).
inline void encoder_qzz(int quality, uint8_t qzz[4][64])
{
    uint8_t qnat[2][64];
    scaled_qt(kLumaQ, quality, qnat[0]);
    scaled_qt(kChromaQ, quality, qnat[1]);
    std::memset(qzz, 0, 4 * 64);
    for (int t = 0; t < 2; ++t)
        for (int i = 0; i < 64; ++i)
            qzz[t][i] = qnat[t][kZZ.nat[i]];
}

// SOI, APP0 (JFIF 1.1), one DQT per quantiser id the components use (ascending), SOF0: the part of the header that does
// not depend on the Huffman tables.  tq: each component's quantiser id; qzz: the tables by id, zig-zag order.
inline void write_frame_prefix(std::vector<uint8_t> &o, int W, int H, int nc, const uint8_t tq[3], const uint8_t qzz[4][64])
{
    const uint8_t soi_app0[] = {0xFF, 0xD8, 0xFF, 0xE0, 0x00, 0x10, 'J',  'F',  'I',  'F',
                                0x00, 0x01, 0x01, 0x01, 0x00, 0x48, 0x00, 0x48, 0x00, 0x00};
    o.insert(o.end(), soi_app0, soi_app0 + sizeof soi_app0);
    for (int t = 0; t < 4; ++t) {
        bool used = false;
        for (int c = 0; c < nc; ++c)
            used |= tq[c] == t;
        if (!used)
            continue;
        o.push_back(0xFF);
        o.push_back(0xDB);
        put16(o, 67);
        o.push_back((uint8_t)t);
        o.insert(o.end(), qzz[t], qzz[t] + 64);
    }
    o.push_back(0xFF);
    o.push_back(0xC0);
    put16(o, 8 + 3 * nc);
    o.push_back(8);
    put16(o, H);
    put16(o, W);
    o.push_back((uint8_t)nc);
    for (int c = 0; c < nc; ++c) {
        o.push_back((uint8_t)(c + 1));
        o.push_back(0x11);
        o.push_back(tq[c]);
    }
}

// The prefix, then DHT 0x00, 0x10 [, 0x01, 0x11] with the given tables (Annex K by default) [, DRI when dri > 0]:
// everything up to the first SOS.
inline void write_frame_header(std::vector<uint8_t> &o, int W, int H, int nc, const uint8_t tq[3], const uint8_t qzz[4][64], int dri,
                               const uint8_t *const bits[4] = kAnnexKBits, const uint8_t *const vals[4] = kAnnexKVals)
{
    write_frame_prefix(o, W, H, nc, tq, qzz);
    for (int t = 0; t < (nc == 3 ? 4 : 2); ++t)
        put_dht(o, ((t & 1) << 4) | (t >> 1), bits[t], vals[t]);
    if (dri > 0)
        put_dri(o, dri);
}

// SOS of a scan of components c0..c1-1 (luma tables for component 0, chroma tables for the others)
inline void write_sos(std::vector<uint8_t> &o, int c0, int c1)
{
    VecOut v{o};
    huff::put_sos(v, c0, c1);
}

} // namespace jfif
} // namespace kpeg
#endif
