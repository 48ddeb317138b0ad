// encode_host.h -- host side of the GPU encoder's tables and container (host only; shared by csrc/encode.cu and
// the CPU replay in tests/emu/emu_encode.cpp).  Everything comes from jfif_write.h, the header the synthetic
// reference encoder writes its files with.
#ifndef KPEG_ENCODE_HOST_H
#define KPEG_ENCODE_HOST_H

#include <string.h>

#include <vector>

#include "encode_core.h"
#include "jfif_write.h"

namespace kpeg {
namespace enc {

inline void build_tables(int quality, EncTables *T)
{
    memset(T, 0, sizeof *T);
    jfif::fdct_cosines(T->cs);
    uint8_t qnat[2][64];
    jfif::scaled_qt(jfif::kLumaQ, quality, qnat[0]);
    jfif::scaled_qt(jfif::kChromaQ, quality, qnat[1]);
    for (int i = 0; i < 64; ++i) {
        T->nat[i] = (uint8_t)jfif::kZZ.nat[i];
        T->qzz[0][i] = qnat[0][jfif::kZZ.nat[i]];
        T->qzz[1][i] = qnat[1][jfif::kZZ.nat[i]];
    }
    for (int t = 0; t < 2; ++t) {
        const jfif::HuffEnc dc = jfif::annex_k_table(2 * t), ac = jfif::annex_k_table(2 * t + 1);
        for (int c = 0; c < 16; ++c) {
            T->dc_code[t][c] = dc.code[c];
            T->dc_len[t][c] = dc.len[c];
        }
        for (int s = 0; s < 256; ++s) {
            T->ac_code[t][s] = ac.code[s];
            T->ac_len[t][s] = ac.len[s];
        }
    }
}

// SOI .. SOF0: what comes before the Huffman tables (the host writes it in both modes)
inline std::vector<uint8_t> file_prefix(int width, int height, int ncomp, int quality)
{
    uint8_t qzz[4][64];
    jfif::encoder_qzz(quality, qzz);
    std::vector<uint8_t> o;
    jfif::write_frame_prefix(o, width, height, ncomp, jfif::kEncoderTq, qzz);
    return o;
}

// SOI .. SOS of the one interleaved scan with the Annex K tables (DRI when ri > 0): the prefix and the tail the
// optimised mode writes on the device (huff::put_header_tail) with its own tables
inline std::vector<uint8_t> file_header(int width, int height, int ncomp, int quality, int ri)
{
    std::vector<uint8_t> o = file_prefix(width, height, ncomp, quality);
    jfif::VecOut v{o};
    huff::put_header_tail(v, ncomp, jfif::kAnnexKBits, jfif::kAnnexKVals, ri);
    return o;
}

inline EncGeom geometry(int width, int height, int ncomp, int ri, uint32_t flags)
{
    EncGeom g = {};
    g.width = (uint32_t)width;
    g.height = (uint32_t)height;
    g.ncomp = (uint32_t)ncomp;
    g.mx = (g.width + 7u) / 8u;
    g.my = (g.height + 7u) / 8u;
    g.nmcu = (uint64_t)g.mx * g.my;
    g.nblk = g.nmcu * g.ncomp;
    g.ri = (uint32_t)ri;
    g.seg_mcus = ri > 0 ? (uint64_t)ri : g.nmcu;
    g.nseg = (g.nmcu + g.seg_mcus - 1) / g.seg_mcus;
    g.flags = flags;
    return g;
}

// Header + every block at max_block_bits + one padding byte per segment, all doubled by stuffing (every byte
// could be FF), + an RSTn marker between segments and EOI.  The Annex K header is the longest either mode writes.
inline uint64_t encode_bound(int width, int height, int ncomp, int quality, int ri, uint32_t flags = 0)
{
    const EncGeom g = geometry(width, height, ncomp, ri, flags);
    const uint64_t hdr = file_header(width, height, ncomp, quality, ri).size();
    const uint64_t unstuffed = (g.nblk * max_block_bits(flags) + 7u) / 8u + g.nseg;
    return hdr + 2u * unstuffed + 2u * (g.nseg - 1u) + 2u;
}

} // namespace enc
} // namespace kpeg
#endif
