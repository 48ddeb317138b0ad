// transcode_host.h -- host side of the lossless transcoder (kpeg_cuda_transcode): the output's geometry and header from
// the input's frame and the parameters.  Host only; shared by csrc/kpeg_cuda.cu and the CPU replay in
// tests/emu/emu_transcode.cpp.  The header is the encoder's (jfif_write.h), with the input's quantisers.
#ifndef KPEG_TRANSCODE_HOST_H
#define KPEG_TRANSCODE_HOST_H

#include <string.h>

#include <vector>

#include "encode_host.h"
#include "transcode_core.h"

namespace kpeg {
namespace tc {

// What the output needs to know about the input.
struct TcInput {
    uint32_t width, height, ncomp;
    uint8_t tq[3];        // quantiser id per component
    uint8_t qzz[4][64];   // quantisers by id, zig-zag order
    uint32_t restart;     // the input's restart interval (its first scan's DRI)
};

struct TcPlan {
    TcGeom g;
    uint8_t tq[3];
    uint8_t qzz[4][64]; // transposed (Q'[u][v] = Q[v][u]) by the transposing transforms
    int ri;             // output restart interval
};

// KPEG_OK, KPEG_ERR_ARG for bad parameters, KPEG_ERR_UNSUPPORTED when the transform's precondition fails.
inline int plan(const TcInput &in, const kpeg_transcode_params &p, TcPlan &out, const char **why)
{
    if (p.transform >= (uint32_t)NXFORM || p.restart_interval < -1 || p.restart_interval > 65535 ||
        (p.flags & ~KPEG_FLAG_OPTIMIZE_HUFFMAN) != 0u) {
        *why = "transcode parameters out of range";
        return KPEG_ERR_ARG;
    }
    if (!xform_allowed(p.transform, in.width, in.height)) {
        *why = "the transform would move a partial edge block (the image's size is not a multiple of 8 on its axis)";
        return KPEG_ERR_UNSUPPORTED;
    }
    const bool tr = transposes(p.transform);
    out.ri = p.restart_interval < 0 ? (int)in.restart : p.restart_interval;
    out.g.out = enc::geometry((int)(tr ? in.height : in.width), (int)(tr ? in.width : in.height), (int)in.ncomp, out.ri, p.flags);
    out.g.smx = (in.width + 7u) / 8u;
    out.g.smy = (in.height + 7u) / 8u;
    out.g.xform = p.transform;
    memcpy(out.tq, in.tq, sizeof out.tq);
    static constexpr XformTable T = make_xform_table();
    for (int t = 0; t < 4; ++t)
        for (int i = 0; i < 64; ++i)
            out.qzz[t][i] = in.qzz[t][tr ? T.e[KPEG_XFORM_TRANSPOSE][i] : i];
    return KPEG_OK;
}

// SOI .. SOF0 (optimised mode: the device writes the rest), or the whole header up to SOS with the Annex K tables.
inline std::vector<uint8_t> header(const TcPlan &pl, bool optimized)
{
    std::vector<uint8_t> o;
    const enc::EncGeom &g = pl.g.out;
    jfif::write_frame_prefix(o, (int)g.width, (int)g.height, (int)g.ncomp, pl.tq, pl.qzz);
    if (!optimized) {
        jfif::VecOut v{o};
        huff::put_header_tail(v, (int)g.ncomp, jfif::kAnnexKBits, jfif::kAnnexKVals, pl.ri);
    }
    return o;
}

// kpeg_encode_bound's derivation (encode_host.h) with this header: the range rules give the same per-block bound.
inline uint64_t bound(const TcPlan &pl)
{
    const enc::EncGeom &g = pl.g.out;
    const uint64_t unstuffed = (g.nblk * enc::max_block_bits(g.flags) + 7u) / 8u + g.nseg;
    return header(pl, false).size() + 2u * unstuffed + 2u * (g.nseg - 1u) + 2u;
}

} // namespace tc
} // namespace kpeg
#endif
