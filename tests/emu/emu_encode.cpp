// tests/emu/emu_encode.cpp -- TEST INFRASTRUCTURE: single-steps the GPU encoder's kernel logic on the CPU.  It
// includes the same host+device header the sm_100a encode kernels are built from (encode_core.h, with the host-side
// tables and header of encode_host.h) and replays E1..E5 of csrc/encode.cu in their order -- the DC chain as a
// chunked scan of map compositions, code emission with a check that no block stores over a word another block owns,
// stuffing tile by tile -- so the encoder's bytes can be checked against the host reference encoder without a GPU.
// Built on its own into libkpeg_emu_encode.so (libkpeg_b200/_build.py: build_emu_encode); nothing in the product
// calls it.
#include <stdint.h>
#include <string.h>

#include <algorithm>
#include <vector>

#include "encode_core.h"
#include "encode_host.h"
#include "kpeg_cuda.h"

// ---- encoder replay (encode_core.h, in the order csrc/encode.cu runs it) ----------------------------------

namespace {

// the 5-state map scan of one component's DC chain, cut into chunks of `chunk` blocks (0 = the serial nudge)
void emu_nudge_chain(const int16_t *raw, const uint8_t *has_ac, const uint8_t *first, uint64_t n, uint64_t chunk, int16_t *out)
{
    using namespace kpeg::enc;
    if (chunk == 0) {
        int prev = 0;
        for (uint64_t m = 0; m < n; ++m)
            prev = out[m] = (int16_t)nudge_dc(raw[m], prev, has_ac[m] != 0, first[m] != 0);
        return;
    }
    auto map_of = [&](uint64_t m) { return nudge_map(raw[m], m ? raw[m - 1] : 0, has_ac[m] != 0, first[m] != 0); };
    const uint64_t nchunks = (n + chunk - 1) / chunk;
    std::vector<uint32_t> agg(nchunks, MAP_IDENTITY);
    for (uint64_t c = 0; c < nchunks; ++c) // per-CTA reduction
        for (uint64_t m = c * chunk; m < n && m < (c + 1) * chunk; ++m)
            agg[c] = map_then(agg[c], map_of(m));
    uint32_t carry = MAP_IDENTITY; // spine: exclusive scan of the aggregates
    for (uint64_t c = 0; c < nchunks; ++c) {
        const uint32_t a = agg[c];
        agg[c] = carry;
        carry = map_then(carry, a);
    }
    for (uint64_t c = 0; c < nchunks; ++c) { // down-sweep
        uint32_t pre = agg[c];
        for (uint64_t m = c * chunk; m < n && m < (c + 1) * chunk; ++m) {
            const uint32_t mm = map_of(m);
            out[m] = (int16_t)(raw[m] + map_apply(mm, map_apply(pre, MAP_START)) - 2);
            pre = map_then(pre, mm);
        }
    }
}

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

} // namespace

extern "C" {

// Serial vs chunked DC chain (the map composition of the encoder's E2 scan).
void emu_nudge(const int16_t *raw, const uint8_t *has_ac, const uint8_t *first, uint64_t n, uint64_t chunk, int16_t *out)
{
    emu_nudge_chain(raw, has_ac, first, n, chunk, out);
}

// The whole GPU encode replayed on the CPU: pixels [h][w][ncomp] -> file bytes.  chunk: blocks per scan tile of the
// DC chain.  info[0] = words a block stored over another block's bits (must be 0), [1] = unstuffed bytes,
// [2] = segments.  Returns 0, -1 on bad arguments, -4 when the file does not fit `cap` (*len = its size).
int emu_encode(const uint8_t *pixels, int w, int h, int ncomp, int quality, int ri, uint32_t flags, uint64_t chunk,
               uint8_t *out, size_t cap, size_t *len, uint32_t *info)
{
    using namespace kpeg::enc;
    if (w < 1 || h < 1 || w > 65535 || h > 65535 || (ncomp != 1 && ncomp != 3) || quality < 1 || quality > 100 ||
        ri < 0 || ri > 65535)
        return -1;
    EncTables T;
    build_tables(quality, &T);
    const EncGeom g = geometry(w, h, ncomp, ri, flags);
    const int nc = ncomp;
    // E1: FDCT + quantisation, per block
    std::vector<int16_t> coef(g.nblk * 64);
    std::vector<int16_t> raw(g.nblk);
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
            raw[m * nc + c] = zz[0];
            for (int i = 1; i < 64; ++i)
                has_ac[m * nc + c] |= zz[i] != 0;
        }
    }
    // E2: DC nudge, one chain per component
    std::vector<int16_t> dc(raw);
    if (flags & KPEG_FLAG_REF_PARITY) {
        std::vector<int16_t> r(g.nmcu), o(g.nmcu);
        std::vector<uint8_t> a(g.nmcu), f(g.nmcu);
        for (int c = 0; c < nc; ++c) {
            for (uint64_t m = 0; m < g.nmcu; ++m) {
                r[m] = raw[m * nc + c];
                a[m] = has_ac[m * nc + c];
                f[m] = g.ri > 0 && starts_segment(g, m);
            }
            emu_nudge_chain(r.data(), a.data(), f.data(), g.nmcu, chunk ? chunk : 1, o.data());
            for (uint64_t m = 0; m < g.nmcu; ++m)
                dc[m * nc + c] = o[m];
        }
    }
    // E3: bit counts, their exclusive scan, segment lengths padded to bytes and their scan
    auto diff_of = [&](uint64_t b) {
        const uint64_t m = b / nc;
        return dc[b] - (starts_segment(g, m) ? 0 : dc[b - nc]);
    };
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
    // E5: stuffing, tile by tile after a scan of the tiles' FF counts
    const std::vector<uint8_t> hdr = file_header(w, h, ncomp, quality, ri);
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

// kpeg_encode_bound's arithmetic (encode_host.h), for the bound test
uint64_t emu_encode_bound(int w, int h, int ncomp, int quality, int ri) { return kpeg::enc::encode_bound(w, h, ncomp, quality, ri); }

} // extern "C"
