// tests/emu/emu_transcode.cpp -- TEST INFRASTRUCTURE: the GPU lossless transcoder (kpeg_cuda_transcode) replayed on the
// CPU from the same headers the sm_100a kernels and the host side are built from: the output's plan and header
// (transcode_host.h), TG's gather and range rules on swizzled, biased coefficient tiles (transcode_core.h), then the
// encoder's coded stages -- EH / EB with huff_opt.h's rule in optimised mode, E3..E5 (encode_core.h) -- in csrc/encode.cu's
// order.  The tiles are built here from given coefficients (the oracle's T.81 decode of the input), in K2's layout.
// Built on its own into libkpeg_emu_transcode.so (libkpeg_b200/_build.py: build_emu_transcode); nothing in the product
// calls it.
#include <stdint.h>
#include <string.h>

#include <algorithm>
#include <vector>

#include "encode_core.h"
#include "huff_opt.h"
#include "kpeg_cuda.h"
#include "transcode_host.h"

namespace {

using namespace kpeg;
using namespace kpeg::enc;

constexpr uint16_t BIAS = 0x8000u;

struct EmuHist {
    uint64_t *h;
    int t;
    void dc(int cat, int) { ++h[t * huff::NSYM + cat]; }
    void ac(int sym, int, int) { ++h[(t + 1) * huff::NSYM + sym]; }
    void zrl() { ++h[(t + 1) * huff::NSYM + 0xF0]; }
    void eob() { ++h[(t + 1) * huff::NSYM]; }
};

struct EmuWords {
    std::vector<uint32_t> &w;
    void store(uint64_t i, uint32_t v) { w[i] = v; }
    void orw(uint64_t i, uint32_t v) { w[i] |= v; }
};

struct EmuOut {
    uint8_t *p;
    uint64_t cap;
    void put(uint64_t i, uint32_t b)
    {
        if (i < cap)
            p[i] = (uint8_t)b;
    }
};

// K2's tile layout (kernels.cuh): value + COEF_BIAS, 16-byte chunk k of block b at chunk k ^ (b & 7)
uint16_t tile_at(const std::vector<uint16_t> &tiles, uint64_t b, int i) { return tiles[(b * 8u + ((unsigned)(i >> 3) ^ (b & 7u))) * 8u + (i & 7)]; }

} // namespace

extern "C" {

// coef: the input's coefficients [nblk][64] (MCU-interleaved, zig-zag, DC absolute); w, h, nc, tq[3], qzz[4][64],
// in_restart: the input's frame; restart, xform, flags: kpeg_transcode_params.  Returns 0, kpeg_cuda_transcode's error
// codes for bad parameters or preconditions, KPEG_ERR_UNSUPPORTED when TG's range flag is set, KPEG_ERR_NOMEM when the
// file does not fit cap (*len = its size).  info[0] = header bytes, [1] = unstuffed bytes, [2] = segments, [3] = bound.
int emu_transcode(const int16_t *coef, int w, int h, int nc, const uint8_t *tq, const uint8_t *qzz, int in_restart, int restart,
                  uint32_t xform, uint32_t flags, uint8_t *out, size_t cap, size_t *len, uint64_t *info)
{
    tc::TcInput in = {};
    in.width = (uint32_t)w;
    in.height = (uint32_t)h;
    in.ncomp = (uint32_t)nc;
    memcpy(in.tq, tq, 3);
    memcpy(in.qzz, qzz, sizeof in.qzz);
    in.restart = (uint32_t)in_restart;
    kpeg_transcode_params p = {restart, xform, flags};
    tc::TcPlan pl;
    const char *why = nullptr;
    const int prc = tc::plan(in, p, pl, &why);
    if (prc != KPEG_OK)
        return prc;
    const EncGeom &g = pl.g.out;
    // the decoder's tiles of the input (same block count: a transform moves blocks, it does not add any)
    std::vector<uint16_t> tiles(g.nblk * 64);
    for (uint64_t b = 0; b < g.nblk; ++b)
        for (int i = 0; i < 64; ++i)
            tiles[(b * 8u + ((unsigned)(i >> 3) ^ (b & 7u))) * 8u + (i & 7)] = (uint16_t)(coef[b * 64 + i] + BIAS);
    // TG: every output block's eight chunks from its source block's line, then the DC rule
    static constexpr tc::XformTable XT = tc::make_xform_table();
    std::vector<int16_t> oc(g.nblk * 64), dc(g.nblk);
    auto dc_of_out = [&](uint64_t ob) { return (int)(int16_t)(uint16_t)(tile_at(tiles, tc::source_index(pl.g, ob), 0) ^ BIAS); };
    bool ok = true;
    for (uint64_t ob = 0; ob < g.nblk; ++ob) {
        const uint64_t sb = tc::source_index(pl.g, ob);
        int16_t src[64];
        for (int i = 0; i < 64; ++i)
            src[i] = (int16_t)(uint16_t)(tile_at(tiles, sb, i) ^ BIAS);
        for (int k = 0; k < 8; ++k)
            ok = tc::gather_chunk(XT, xform, src, k, &oc[ob * 64 + 8 * k]) && ok;
        dc[ob] = oc[ob * 64];
        ok = tc::dc_in_range(pl.g, ob, dc[ob], dc_of_out) && ok;
    }
    info[3] = tc::bound(pl);
    if (!ok)
        return KPEG_ERR_UNSUPPORTED;
    auto diff_of = [&](uint64_t b) {
        const uint64_t m = b / g.ncomp;
        return dc[b] - (starts_segment(g, m) ? 0 : dc[b - g.ncomp]);
    };
    // EH / EB in optimised mode, else the Annex K codes
    EncTables T;
    build_tables(90, &T);
    std::vector<uint8_t> hdr = tc::header(pl, (flags & KPEG_FLAG_OPTIMIZE_HUFFMAN) != 0u);
    if (flags & KPEG_FLAG_OPTIMIZE_HUFFMAN) {
        std::vector<uint64_t> hist(4 * huff::NSYM, 0);
        for (uint64_t b = 0; b < g.nblk; ++b) {
            EmuHist v{hist.data(), b % g.ncomp ? 2 : 0};
            walk_block(diff_of(b), &oc[b * 64], v);
        }
        uint8_t bits[4][16] = {}, vals[4][256] = {};
        for (int t = 0; t < (nc == 3 ? 4 : 2); ++t) {
            huff::optimal_table(&hist[t * huff::NSYM], bits[t], vals[t]);
            uint16_t code[256];
            uint8_t ln[256];
            huff::canonical_codes(bits[t], vals[t], code, ln);
            if (t & 1) {
                memcpy(T.ac_code[t >> 1], code, sizeof code);
                memcpy(T.ac_len[t >> 1], ln, sizeof ln);
            } else {
                memcpy(T.dc_code[t >> 1], code, sizeof T.dc_code[0]);
                memcpy(T.dc_len[t >> 1], ln, sizeof T.dc_len[0]);
            }
        }
        jfif::VecOut o{hdr};
        const uint8_t *const bp[4] = {bits[0], bits[1], bits[2], bits[3]}, *const vp[4] = {vals[0], vals[1], vals[2], vals[3]};
        huff::put_header_tail(o, nc, bp, vp, pl.ri);
    }
    // E3
    std::vector<uint64_t> off(g.nblk + 1, 0);
    for (uint64_t b = 0; b < g.nblk; ++b) {
        BitCounter bc;
        code_block(T, b % g.ncomp ? 1 : 0, diff_of(b), &oc[b * 64], bc);
        off[b + 1] = off[b] + bc.n;
    }
    std::vector<uint64_t> seg_byte(g.nseg + 1, 0);
    for (uint64_t s = 0; s < g.nseg; ++s) {
        const uint64_t b0 = s * g.seg_mcus * g.ncomp, b1 = std::min<uint64_t>((s + 1) * g.seg_mcus, g.nmcu) * g.ncomp;
        seg_byte[s + 1] = seg_byte[s] + (off[b1] - off[b0] + 7) / 8;
    }
    const uint64_t N = seg_byte[g.nseg];
    // E4
    std::vector<uint32_t> words((N + 3) / 4 + 1, 0);
    EmuWords ew{words};
    for (uint64_t b = 0; b < g.nblk; ++b) {
        const uint64_t m = b / g.ncomp, s = m / g.seg_mcus;
        const uint64_t b0 = s * g.seg_mcus * g.ncomp, b1 = std::min<uint64_t>((s + 1) * g.seg_mcus, g.nmcu) * g.ncomp;
        BitEmitter<EmuWords> em(ew, seg_byte[s] * 8 + (off[b] - off[b0]));
        code_block(T, b % g.ncomp ? 1 : 0, diff_of(b), &oc[b * 64], em);
        if (b + 1 == b1) {
            const int pad = (int)((seg_byte[s + 1] - seg_byte[s]) * 8 - (off[b1] - off[b0]));
            if (pad)
                em.put((1u << pad) - 1u, pad);
        }
        em.finish();
    }
    // E5
    uint64_t ff = 0;
    for (uint64_t i = 0; i < N; ++i)
        ff += stream_byte(words.data(), i) == 0xFF;
    const uint64_t total = hdr.size() + N + ff + 2 * g.nseg;
    *len = total;
    info[0] = hdr.size();
    info[1] = N;
    info[2] = g.nseg;
    if (total > cap)
        return KPEG_ERR_NOMEM;
    memcpy(out, hdr.data(), hdr.size());
    EmuOut eo{out + hdr.size(), cap - hdr.size()};
    stuff_range(words.data(), seg_byte.data(), g.nseg, N, 0, N, 0, eo);
    return 0;
}

// The transform table (transcode_core.h): e[t][i] = source zig-zag index | 0x80 when negated
void emu_xform_table(uint8_t *out)
{
    static constexpr tc::XformTable XT = tc::make_xform_table();
    memcpy(out, XT.e, sizeof XT.e);
}

} // extern "C"
