// tests/emu/emu_encode_opt.cpp -- TEST INFRASTRUCTURE: the GPU encoder with optimised Huffman tables
// (KPEG_FLAG_OPTIMIZE_HUFFMAN) replayed on the CPU from the same host+device headers the sm_100a kernels are built from
// (encode_core.h, huff_opt.h, encode_host.h), in csrc/encode.cu's order: E1, E2, then EH (the symbol walk's histogram),
// EB (huff_opt.h's table rule, canonical codes into this encode's copy of the tables, the header tail after the host's
// prefix), then E3..E5 with those tables and the scan after the header.  E1..E5 themselves are replayed in their
// Annex K form, with the DC chain as a chunked map scan, by emu_encode.cpp; here the DC chain is the serial nudge.
// Built on its own into libkpeg_emu_encode_opt.so (libkpeg_b200/_build.py: build_emu_encode_opt); nothing in the
// product calls it.
#include <stdint.h>
#include <string.h>

#include <algorithm>
#include <vector>

#include "encode_core.h"
#include "encode_host.h"
#include "huff_opt.h"
#include "kpeg_cuda.h"

namespace {

using namespace kpeg::enc;

// EH's visitor without the warp aggregation: [4][257] counts in table order
struct EmuHist {
    uint64_t *h;
    int t;
    void dc(int cat, int) { ++h[t * kpeg::huff::NSYM + cat]; }
    void ac(int sym, int, int) { ++h[(t + 1) * kpeg::huff::NSYM + sym]; }
    void zrl() { ++h[(t + 1) * kpeg::huff::NSYM + 0xF0]; }
    void eob() { ++h[(t + 1) * kpeg::huff::NSYM]; }
};

struct EmuWords {
    std::vector<uint32_t> &w;
    uint32_t *clobbered;
    void store(uint64_t i, uint32_t v)
    {
        if (w[i] != 0)
            ++*clobbered; // a word the block owns was touched by another block
        w[i] = v;
    }
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

// EB: the tables of hist into T's code arrays, and the header (prefix + tail) into hdr
void build_optimised(const uint64_t *hist, int nc, int w, int h, int quality, int ri, EncTables &T, std::vector<uint8_t> &hdr)
{
    using namespace kpeg::huff;
    uint8_t bits[4][16] = {}, vals[4][256] = {};
    for (int t = 0; t < (nc == 3 ? 4 : 2); ++t) {
        optimal_table(&hist[t * NSYM], bits[t], vals[t]);
        uint16_t code[256];
        uint8_t len[256];
        canonical_codes(bits[t], vals[t], code, len);
        if (t & 1) {
            memcpy(T.ac_code[t >> 1], code, sizeof code);
            memcpy(T.ac_len[t >> 1], len, sizeof len);
        } else {
            memcpy(T.dc_code[t >> 1], code, sizeof T.dc_code[0]);
            memcpy(T.dc_len[t >> 1], len, sizeof T.dc_len[0]);
        }
    }
    hdr = file_prefix(w, h, nc, quality);
    kpeg::jfif::VecOut o{hdr};
    const uint8_t *const bp[4] = {bits[0], bits[1], bits[2], bits[3]}, *const vp[4] = {vals[0], vals[1], vals[2], vals[3]};
    put_header_tail(o, nc, bp, vp, ri);
}

} // namespace

extern "C" {

// The optimised-table GPU encode replayed on the CPU: pixels [h][w][ncomp] -> file bytes.  flags: KPEG_FLAG_REF_PARITY
// (KPEG_FLAG_OPTIMIZE_HUFFMAN is implied).  info[0] = words a block stored over another block's bits (must be 0),
// [1] = unstuffed bytes, [2] = segments, [3] = header bytes.  Returns 0, -1 on bad arguments, -4 when the file does not
// fit `cap` (*len = its size).
int emu_encode_opt(const uint8_t *pixels, int w, int h, int ncomp, int quality, int ri, uint32_t flags, uint8_t *out,
                   size_t cap, size_t *len, uint32_t *info)
{
    if (w < 1 || h < 1 || w > 65535 || h > 65535 || (ncomp != 1 && ncomp != 3) || quality < 1 || quality > 100 ||
        ri < 0 || ri > 65535)
        return -1;
    flags |= KPEG_FLAG_OPTIMIZE_HUFFMAN;
    EncTables T;
    build_tables(quality, &T);
    const EncGeom g = geometry(w, h, ncomp, ri, flags);
    const int nc = ncomp;
    // E1: FDCT + quantisation, per block
    std::vector<int16_t> coef(g.nblk * 64);
    std::vector<uint8_t> has_ac(g.nblk);
    for (uint64_t m = 0; m < g.nmcu; ++m) {
        const uint32_t bx = (uint32_t)(m % g.mx), by = (uint32_t)(m / g.mx);
        double blk[3][64], tmp[64];
        for (int r = 0; r < 8; ++r)
            for (int q = 0; q < 8; ++q) {
                const uint32_t y = std::min<uint32_t>(by * 8 + r, g.height - 1), x = std::min<uint32_t>(bx * 8 + q, g.width - 1);
                const uint8_t *s = pixels + ((size_t)y * g.width + x) * nc;
                if (nc == 1)
                    blk[0][r * 8 + q] = dsub(s[0], 128.0);
                else
                    rgb_to_ycc(s[0], s[1], s[2], &blk[0][r * 8 + q], &blk[1][r * 8 + q], &blk[2][r * 8 + q]);
            }
        for (int c = 0; c < nc; ++c) {
            for (int r = 0; r < 8; ++r)
                for (int v = 0; v < 8; ++v)
                    tmp[r * 8 + v] = fdct_row(&blk[c][r * 8], T.cs, v);
            int16_t *zz = &coef[(m * nc + c) * 64];
            for (int i = 0; i < 64; ++i)
                zz[i] = (int16_t)quantise(fdct_col(tmp, T.cs, T.nat[i] >> 3, T.nat[i] & 7), T.qzz[c ? 1 : 0][i], i == 0);
            for (int i = 1; i < 64; ++i)
                has_ac[m * nc + c] |= zz[i] != 0;
        }
    }
    // E2: DC nudge, the serial chain of each component
    std::vector<int16_t> dc(g.nblk);
    for (int c = 0; c < nc; ++c) {
        int prev = 0;
        for (uint64_t m = 0; m < g.nmcu; ++m) {
            const uint64_t b = m * nc + c;
            dc[b] = coef[b * 64];
            if (flags & KPEG_FLAG_REF_PARITY)
                prev = dc[b] = (int16_t)nudge_dc(dc[b], prev, has_ac[b] != 0, g.ri > 0 && starts_segment(g, m));
        }
    }
    auto diff_of = [&](uint64_t b) {
        const uint64_t m = b / nc;
        return dc[b] - (starts_segment(g, m) ? 0 : dc[b - nc]);
    };
    // EH, EB
    std::vector<uint64_t> hist(4 * kpeg::huff::NSYM, 0);
    for (uint64_t b = 0; b < g.nblk; ++b) {
        EmuHist v{hist.data(), b % nc ? 2 : 0};
        walk_block(diff_of(b), &coef[b * 64], v);
    }
    std::vector<uint8_t> hdr;
    build_optimised(hist.data(), nc, w, h, quality, ri, T, hdr);
    // E3: bit counts, their exclusive scan, segment lengths padded to bytes
    std::vector<uint64_t> off(g.nblk + 1, 0);
    for (uint64_t b = 0; b < g.nblk; ++b) {
        BitCounter bc;
        code_block(T, b % nc ? 1 : 0, diff_of(b), &coef[b * 64], bc);
        off[b + 1] = off[b] + bc.n;
    }
    std::vector<uint64_t> seg_byte(g.nseg + 1, 0);
    for (uint64_t s = 0; s < g.nseg; ++s) {
        const uint64_t b0 = s * g.seg_mcus * nc, b1 = std::min<uint64_t>((s + 1) * g.seg_mcus, g.nmcu) * nc;
        seg_byte[s + 1] = seg_byte[s] + (off[b1] - off[b0] + 7) / 8;
    }
    const uint64_t N = seg_byte[g.nseg];
    // E4: emission, blocks in reverse order (any order must give the same words)
    std::vector<uint32_t> words((N + 3) / 4 + 1, 0);
    uint32_t clobbered = 0;
    EmuWords ew{words, &clobbered};
    for (uint64_t b = g.nblk; b-- > 0;) {
        const uint64_t m = b / nc, s = m / g.seg_mcus;
        const uint64_t b0 = s * g.seg_mcus * nc, b1 = std::min<uint64_t>((s + 1) * g.seg_mcus, g.nmcu) * nc;
        BitEmitter<EmuWords> em(ew, seg_byte[s] * 8 + (off[b] - off[b0]));
        code_block(T, b % nc ? 1 : 0, diff_of(b), &coef[b * 64], em);
        if (b + 1 == b1) {
            const int pad = (int)((seg_byte[s + 1] - seg_byte[s]) * 8 - (off[b1] - off[b0]));
            if (pad)
                em.put((1u << pad) - 1u, pad);
        }
        em.finish();
    }
    // E5: stuffing after the header, tile by tile after a scan of the tiles' FF counts
    const uint64_t ntiles = (N + STUFF_TILE - 1) / STUFF_TILE;
    std::vector<uint64_t> tile_ff(ntiles + 1, 0);
    for (uint64_t t = 0; t < ntiles; ++t) {
        uint64_t k = 0;
        for (uint64_t i = t * STUFF_TILE; i < N && i < (t + 1) * STUFF_TILE; ++i)
            k += stream_byte(words.data(), i) == 0xFF;
        tile_ff[t + 1] = tile_ff[t] + k;
    }
    const uint64_t total = hdr.size() + N + tile_ff[ntiles] + 2 * g.nseg;
    *len = total;
    info[0] = clobbered;
    info[1] = (uint32_t)N;
    info[2] = (uint32_t)g.nseg;
    info[3] = (uint32_t)hdr.size();
    if (total > cap)
        return -4;
    memcpy(out, hdr.data(), hdr.size());
    EmuOut eo{out + hdr.size(), cap - hdr.size()};
    for (uint64_t t = 0; t < ntiles; ++t) {
        uint64_t ff = tile_ff[t];
        for (uint64_t th = 0; th < STUFF_THREADS; ++th) {
            const uint64_t i0 = std::min(N, t * STUFF_TILE + th * STUFF_BYTES_PER_THREAD);
            const uint64_t i1 = std::min(N, i0 + STUFF_BYTES_PER_THREAD);
            stuff_range(words.data(), seg_byte.data(), g.nseg, N, i0, i1, ff, eo);
            for (uint64_t i = i0; i < i1; ++i)
                ff += stream_byte(words.data(), i) == 0xFF;
        }
    }
    return 0;
}

// kpeg_encode_bound's arithmetic (encode_host.h) with flags
uint64_t emu_encode_bound_flags(int w, int h, int ncomp, int quality, int ri, uint32_t flags)
{
    return kpeg::enc::encode_bound(w, h, ncomp, quality, ri, flags);
}

// The optimal-table builder (huff_opt.h): freq[257] (entry 256 ignored) -> BITS, HUFFVAL; returns the symbol count
int emu_optimal_table(const uint64_t *freq, uint8_t *bits, uint8_t *vals) { return kpeg::huff::optimal_table(freq, bits, vals); }

} // extern "C"
