// synth_encoder.cpp -- deterministic synthetic baseline-JPEG encoder (see include/kpeg_synth.h).
//
// Host-only helper that produces the benchmark / parity inputs named in BASELINE.json.  Not part
// of the decode hot path and not derived from the reference's (non-functional) src/Encoder.cpp.
//
// Pipeline: integer pseudo-random pixel field -> JFIF RGB->YCbCr -> 8x8 FDCT (double) ->
// quantise (Annex K tables, IJG quality scaling) -> optional quirk-free DC nudge -> Huffman
// entropy coding (Annex K tables, or tables optimised for the image) with byte stuffing and optional DRI/RSTn.  Everything after the
// pixel field is kpeg_synth_encode_pixels, which takes any pixels: it is the byte-exact reference
// the GPU encoder (csrc/encode.cu) is tested against, so its arithmetic order is part of the
// contract (built with -ffp-contract=off; the tables come from csrc/jfif_write.h).

#include "kpeg_synth.h"

#include "jfif_write.h"

#include <algorithm>
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <thread>
#include <vector>

namespace {

using namespace kpeg::jfif;

// ---- content ------------------------------------------------------------------------------------

inline uint64_t mix64(uint64_t z)
{
    z += 0x9E3779B97F4A7C15ull;
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
    return z ^ (z >> 31);
}

// parabolic "sine": period 1024, range [-256, 256], integer only (no libm => bit-reproducible)
inline int wave(int t)
{
    t &= 1023;
    int u = t & 511;
    int w = (u * (512 - u)) >> 8;
    return (t & 512) ? -w : w;
}

struct Content {
    uint64_t seed;
    int amp;
    int ph[3][3];
    Content(uint64_t s, int a) : seed(s), amp(a)
    {
        for (int c = 0; c < 3; ++c)
            for (int k = 0; k < 3; ++k)
                ph[c][k] = (int)(mix64(seed * 0x100 + c * 16 + k) & 1023);
    }
    inline int at(int x, int y, int c) const
    {
        int v = 128;
        v += (wave(x * 3 + y * 5 + ph[c][0]) * 44) >> 8;
        v += (wave(x * 11 - y * 7 + ph[c][1]) * 18) >> 8;
        v += (wave((x >> 1) + (y >> 2) * 3 + ph[c][2]) * 30) >> 8;
        uint64_t h = mix64(seed ^ (((uint64_t)(uint32_t)y << 34) | ((uint64_t)(uint32_t)x << 2) | (uint64_t)c));
        int n = (int)(h & 255) + (int)((h >> 8) & 255) + (int)((h >> 16) & 255) + (int)((h >> 24) & 255) - 510;
        v += (n * amp) >> 8;
        return v < 0 ? 0 : (v > 255 ? 255 : v);
    }
};

// ---- entropy coder ------------------------------------------------------------------------------

struct BitWriter {
    std::vector<uint8_t> &out;
    uint64_t acc = 0;
    int n = 0;
    explicit BitWriter(std::vector<uint8_t> &o) : out(o) {}
    inline void put(uint32_t v, int bits)
    {
        acc = (acc << bits) | (v & ((1u << bits) - 1u));
        n += bits;
        while (n >= 8) {
            uint8_t b = (uint8_t)(acc >> (n - 8));
            out.push_back(b);
            if (b == 0xFF)
                out.push_back(0x00);
            n -= 8;
        }
    }
    inline void flush_ones()
    {
        if (n > 0)
            put((1u << (8 - n)) - 1u, 8 - n);
    }
};

inline int category(int v)
{
    int a = v < 0 ? -v : v, c = 0;
    while (a) {
        ++c;
        a >>= 1;
    }
    return c;
}

inline void put_value(BitWriter &bw, int v, int cat)
{
    if (cat)
        bw.put((uint32_t)(v < 0 ? v + (1 << cat) - 1 : v), cat);
}

struct Geometry {
    int W, H, nc_file, nc_content, mx, my;
    long nmcu;
};

bool check(const kpeg_synth_params *p)
{
    return p && p->width >= 1 && p->height >= 1 && p->width <= 65535 && p->height <= 65535 &&
           (p->file_components == 1 || p->file_components == 3) && p->quality >= 1 && p->quality <= 100 &&
           p->restart_interval >= 0 && p->restart_interval <= 65535;
}

Geometry geometry(const kpeg_synth_params *p)
{
    Geometry g;
    g.W = p->width;
    g.H = p->height;
    g.nc_file = p->file_components;
    g.nc_content = (p->file_components == 1 || (p->flags & KPEG_SYNTH_GRAY_CONTENT)) ? 1 : 3;
    g.mx = (g.W + 7) / 8;
    g.my = (g.H + 7) / 8;
    g.nmcu = (long)g.mx * g.my;
    return g;
}

int encode_coefficients(const kpeg_synth_coef_frame &f, const int16_t *coef, bool split, uint8_t **out, size_t *out_len);

// The coding path over a pixel buffer [H][W][nc_content].
int encode_pixels(const kpeg_synth_params *p, const uint8_t *px, uint8_t **out, size_t *out_len)
{
    const Geometry g = geometry(p);
    const int nc = g.nc_file;

    double cs[8][8]; // cs[x][u] = C(u)/2 * cos((2x+1) u pi / 16)
    fdct_cosines(cs);
    uint8_t qzz[4][64]; // the quantisers by id, zig-zag order
    encoder_qzz(p->quality, qzz);

    // quantised coefficients, [mcu][comp][zig-zag]
    std::vector<int16_t> coef;
    try {
        coef.assign((size_t)g.nmcu * nc * 64, 0);
    } catch (...) {
        return -2;
    }

    auto work = [&](int row0, int row1) {
        double blk[3][64], tmp[64];
        for (int by = row0; by < row1; ++by) {
            for (int bx = 0; bx < g.mx; ++bx) {
                for (int r = 0; r < 8; ++r) {
                    int y = std::min(by * 8 + r, g.H - 1);
                    for (int q = 0; q < 8; ++q) {
                        int x = std::min(bx * 8 + q, g.W - 1);
                        const uint8_t *s = px + ((size_t)y * g.W + x) * g.nc_content;
                        if (g.nc_content == 1) {
                            blk[0][r * 8 + q] = s[0] - 128.0;
                        } else {
                            double R = s[0], G = s[1], B = s[2];
                            blk[0][r * 8 + q] = 0.299 * R + 0.587 * G + 0.114 * B - 128.0;
                            blk[1][r * 8 + q] = -0.168736 * R - 0.331264 * G + 0.5 * B;
                            blk[2][r * 8 + q] = 0.5 * R - 0.418688 * G - 0.081312 * B;
                        }
                    }
                }
                size_t m = (size_t)by * g.mx + bx;
                for (int c = 0; c < g.nc_content; ++c) {
                    // rows then columns
                    for (int r = 0; r < 8; ++r)
                        for (int v = 0; v < 8; ++v) {
                            double s = 0;
                            for (int q = 0; q < 8; ++q)
                                s += blk[c][r * 8 + q] * cs[q][v];
                            tmp[r * 8 + v] = s;
                        }
                    int16_t *zz = &coef[(m * nc + c) * 64];
                    const uint8_t *qt = qzz[c ? 1 : 0];
                    for (int i = 0; i < 64; ++i) {
                        int u = kZZ.nat[i] >> 3, v = kZZ.nat[i] & 7;
                        double s = 0;
                        for (int r = 0; r < 8; ++r)
                            s += tmp[r * 8 + v] * cs[r][u];
                        long qv = std::lround(s / qt[i]);
                        long lim = i == 0 ? 2047 : 1023;
                        zz[i] = (int16_t)std::max(-lim, std::min(lim, qv));
                    }
                }
            }
        }
    };
    int nt = p->threads > 0 ? p->threads : (int)std::thread::hardware_concurrency();
    nt = std::max(1, std::min(nt, std::min(g.my, 64)));
    {
        std::vector<std::thread> th;
        for (int t = 0; t < nt; ++t)
            th.emplace_back(work, (int)((long)g.my * t / nt), (int)((long)g.my * (t + 1) / nt));
        for (auto &t : th)
            t.join();
    }

    const int ri = p->restart_interval;
    const bool emit_rst = ri > 0 && (p->flags & KPEG_SYNTH_EMIT_RESTART);
    if (p->flags & KPEG_SYNTH_QUIRK_FREE) {
        int prev[3] = {0, 0, 0};
        for (long m = 0; m < g.nmcu; ++m) {
            const bool first = ri > 0 && (m % ri) == 0;
            for (int c = 0; c < nc; ++c) {
                int16_t *zz = &coef[((size_t)m * nc + c) * 64];
                bool has_ac = false;
                for (int i = 1; i < 64 && !has_ac; ++i)
                    has_ac = zz[i] != 0;
                int dc = zz[0];
                if (has_ac) {
                    for (int step = 0; step < 8; ++step) {
                        int d = dc + ((step & 1) ? -((step + 1) / 2) : (step / 2));
                        if (d < -2047 || d > 2047)
                            continue;
                        if (d != prev[c] && !(first && d == 0)) {
                            dc = d;
                            break;
                        }
                    }
                }
                zz[0] = (int16_t)dc;
                prev[c] = dc;
            }
        }
    }

    kpeg_synth_coef_frame f = {};
    f.width = g.W;
    f.height = g.H;
    f.ncomp = nc;
    std::memcpy(f.tq, kEncoderTq, sizeof f.tq);
    std::memcpy(f.qt, qzz, sizeof f.qt);
    f.restart_interval = emit_rst ? ri : 0;
    f.flags = p->flags & KPEG_SYNTH_OPTIMIZE_HUFFMAN;
    return encode_coefficients(f, coef.data(), nc == 3 && (p->flags & KPEG_SYNTH_NON_INTERLEAVED), out, out_len);
}

// The baseline range rules: every DC difference (prediction per component, reset at every segment's first MCU) has
// category <= 11, every AC coefficient is within +-1023.  Beyond them no baseline Huffman table has a symbol.
bool codable(const kpeg_synth_coef_frame &f, const int16_t *coef, long nmcu)
{
    const int nc = f.ncomp, ri = f.restart_interval;
    int pred[3] = {0, 0, 0};
    for (long m = 0; m < nmcu; ++m) {
        if (ri > 0 && m % ri == 0)
            pred[0] = pred[1] = pred[2] = 0;
        for (int c = 0; c < nc; ++c) {
            const int16_t *zz = &coef[((size_t)m * nc + c) * 64];
            if (category(zz[0] - pred[c]) > 11)
                return false;
            pred[c] = zz[0];
            for (int i = 1; i < 64; ++i)
                if (zz[i] < -1023 || zz[i] > 1023)
                    return false;
        }
    }
    return true;
}

// The coding path from quantised coefficients [mcu][comp][zig-zag] (DC absolute): header, the scan (or, split, one scan
// per component), EOI.
int encode_coefficients(const kpeg_synth_coef_frame &f, const int16_t *coef, bool split, uint8_t **out, size_t *out_len)
{
    const int nc = f.ncomp, ri = f.restart_interval;
    const long nmcu = (long)((f.width + 7) / 8) * ((f.height + 7) / 8);
    if (!codable(f, coef, nmcu))
        return -1;
    std::vector<uint8_t> o;
    o.reserve((size_t)nmcu * nc * 24 + 1024);
    const bool emit_rst = ri > 0;
    // the Huffman tables: Annex K, or -- KPEG_SYNTH_OPTIMIZE_HUFFMAN -- optimal for this image's symbol counts, counted
    // below exactly as the coding loop further down codes the symbols
    const uint8_t *bits[4] = {kDcLumaBits, kAcLumaBits, kDcChromaBits, kAcChromaBits};
    const uint8_t *vals[4] = {kDcVals, kAcLumaVals, kDcVals, kAcChromaVals};
    uint8_t opt_bits[4][16], opt_vals[4][256];
    if (f.flags & KPEG_SYNTH_OPTIMIZE_HUFFMAN) {
        uint64_t freq[4][256] = {};
        int pred[3] = {0, 0, 0};
        for (long m = 0; m < nmcu; ++m) {
            if (emit_rst && m && (m % ri) == 0)
                pred[0] = pred[1] = pred[2] = 0;
            for (int c = 0; c < nc; ++c) {
                const int16_t *zz = &coef[((size_t)m * nc + c) * 64];
                uint64_t *fd = freq[c ? 2 : 0], *fa = freq[c ? 3 : 1];
                ++fd[category(zz[0] - pred[c])];
                pred[c] = zz[0];
                int run = 0;
                for (int i = 1; i < 64; ++i) {
                    if (zz[i] == 0) {
                        ++run;
                        continue;
                    }
                    for (; run > 15; run -= 16)
                        ++fa[0xF0];
                    ++fa[(run << 4) | category(zz[i])];
                    run = 0;
                }
                if (run)
                    ++fa[0x00];
            }
        }
        for (int t = 0; t < (nc == 3 ? 4 : 2); ++t) {
            kpeg::huff::optimal_table(freq[t], opt_bits[t], opt_vals[t]);
            bits[t] = opt_bits[t];
            vals[t] = opt_vals[t];
        }
    }
    write_frame_header(o, f.width, f.height, nc, f.tq, f.qt, ri, bits, vals);
    const HuffEnc dcL(bits[0], vals[0]), dcC(bits[2], vals[2]);
    const HuffEnc acL(bits[1], vals[1]), acC(bits[3], vals[3]);
    BitWriter bw(o);
    // one interleaved scan of all components, or -- KPEG_SYNTH_NON_INTERLEAVED -- one scan per component (T.81 A.2.3:
    // the MCU of a non-interleaved scan is one block, blocks in raster order; the restart interval counts those)
    for (int scan = 0; scan < (split ? nc : 1); ++scan) {
        const int c0 = split ? scan : 0, c1 = split ? scan + 1 : nc;
        write_sos(o, c0, c1);
        int pred[3] = {0, 0, 0};
        for (long m = 0; m < nmcu; ++m) {
            if (emit_rst && m && (m % ri) == 0) {
                bw.flush_ones();
                o.push_back(0xFF);
                o.push_back((uint8_t)(0xD0 + ((m / ri - 1) & 7)));
                pred[0] = pred[1] = pred[2] = 0;
            }
            for (int c = c0; c < c1; ++c) {
                const int16_t *zz = &coef[((size_t)m * nc + c) * 64];
                const HuffEnc &hd = c ? dcC : dcL, &ha = c ? acC : acL;
                int diff = zz[0] - pred[c];
                pred[c] = zz[0];
                int cat = category(diff);
                bw.put(hd.code[cat], hd.len[cat]);
                put_value(bw, diff, cat);
                int run = 0;
                for (int i = 1; i < 64; ++i) {
                    if (zz[i] == 0) {
                        ++run;
                        continue;
                    }
                    while (run > 15) {
                        bw.put(ha.code[0xF0], ha.len[0xF0]);
                        run -= 16;
                    }
                    cat = category(zz[i]);
                    int sym = (run << 4) | cat;
                    bw.put(ha.code[sym], ha.len[sym]);
                    put_value(bw, zz[i], cat);
                    run = 0;
                }
                if (run)
                    bw.put(ha.code[0x00], ha.len[0x00]);
            }
        }
        if (scan + 1 < (split ? nc : 1))
            bw.flush_ones(); // the next SOS marker starts on a byte boundary
    }
    bw.flush_ones();
    o.push_back(0xFF);
    o.push_back(0xD9);

    uint8_t *buf = (uint8_t *)std::malloc(o.size());
    if (!buf)
        return -2;
    std::memcpy(buf, o.data(), o.size());
    *out = buf;
    *out_len = o.size();
    return 0;
}

} // namespace

extern "C" int kpeg_synth_pixels(const kpeg_synth_params *p, uint8_t *dst)
{
    if (!check(p) || !dst)
        return -1;
    Geometry g = geometry(p);
    Content ct(p->seed, p->noise_amp > 0 ? p->noise_amp : 10);
    for (int y = 0; y < g.H; ++y)
        for (int x = 0; x < g.W; ++x)
            for (int c = 0; c < g.nc_content; ++c)
                dst[((size_t)y * g.W + x) * g.nc_content + c] = (uint8_t)ct.at(x, y, c);
    return 0;
}

extern "C" int kpeg_synth_encode_pixels(const kpeg_synth_params *p, const uint8_t *pixels, uint8_t **out, size_t *out_len)
{
    if (!check(p) || !pixels || !out || !out_len)
        return -1;
    return encode_pixels(p, pixels, out, out_len);
}

// generate the content (in parallel, rows split as the coding pass splits them), then encode it
extern "C" int kpeg_synth_encode(const kpeg_synth_params *p, uint8_t **out, size_t *out_len)
{
    if (!check(p) || !out || !out_len)
        return -1;
    const Geometry g = geometry(p);
    const Content ct(p->seed, p->noise_amp > 0 ? p->noise_amp : 10);
    std::vector<uint8_t> px;
    try {
        px.resize((size_t)g.W * g.H * g.nc_content);
    } catch (...) {
        return -2;
    }
    auto work = [&](int y0, int y1) {
        for (int y = y0; y < y1; ++y)
            for (int x = 0; x < g.W; ++x)
                for (int c = 0; c < g.nc_content; ++c)
                    px[((size_t)y * g.W + x) * g.nc_content + c] = (uint8_t)ct.at(x, y, c);
    };
    int nt = p->threads > 0 ? p->threads : (int)std::thread::hardware_concurrency();
    nt = std::max(1, std::min(nt, std::min(g.H, 64)));
    std::vector<std::thread> th;
    for (int t = 0; t < nt; ++t)
        th.emplace_back(work, (int)((long)g.H * t / nt), (int)((long)g.H * (t + 1) / nt));
    for (auto &t : th)
        t.join();
    return encode_pixels(p, px.data(), out, out_len);
}

extern "C" int kpeg_synth_encode_coefficients(const kpeg_synth_coef_frame *f, const int16_t *coef, uint8_t **out, size_t *out_len)
{
    if (!f || !coef || !out || !out_len || f->width < 1 || f->height < 1 || f->width > 65535 || f->height > 65535 ||
        (f->ncomp != 1 && f->ncomp != 3) || f->restart_interval < 0 || f->restart_interval > 65535 ||
        (f->flags & ~KPEG_SYNTH_OPTIMIZE_HUFFMAN) != 0u)
        return -1;
    for (int c = 0; c < f->ncomp; ++c)
        if (f->tq[c] > 3)
            return -1;
    return encode_coefficients(*f, coef, false, out, out_len);
}

extern "C" void kpeg_synth_free(uint8_t *buf) { std::free(buf); }
