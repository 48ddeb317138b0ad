// encode_core.h -- per-block logic of the GPU baseline-JPEG encoder (csrc/encode.cu), written as KPEG_HD
// functions so tests/emu/emu_encode.cpp (and, with optimised tables, emu_encode_opt.cpp) replays exactly what the
// kernels run.
//
// Exactness contract: the encoder writes byte for byte what kpeg_synth_encode_pixels (host/synth_encoder.cpp)
// writes for the same pixels and parameters.  So the double arithmetic below is one correctly rounded multiply
// or add at a time, in the synth's order (__dmul_rn / __dadd_rn on the device; the emulator and the synth are
// built with -ffp-contract=off), the cosines are the synth's own (host libm, uploaded), and the DC nudge that
// keeps a stream safe for the reference decoder's DC rule (SURVEY F1) is the synth's, restated as a map so it
// can be scanned in parallel.
#ifndef KPEG_ENCODE_CORE_H
#define KPEG_ENCODE_CORE_H

#include <math.h>
#include <stdint.h>

#include "kpeg_common.h"
#include "kpeg_cuda.h"

namespace kpeg {
namespace enc {

// Largest coded block: 22 DC bits (category <= 11, Annex K code <= 11 bits) + 63 AC positions of <= 26 bits each
// (code <= 16 bits + category <= 10).  With optimised tables (KPEG_FLAG_OPTIMIZE_HUFFMAN) every code may be 16 bits
// long: 27 DC bits + 63 x 26.  Derivation in include/kpeg_cuda.h, kpeg_encode_bound.
constexpr uint32_t MAX_BLOCK_BITS = 22u + 63u * 26u;
constexpr uint32_t MAX_BLOCK_BITS_OPT = 27u + 63u * 26u;

KPEG_HD uint32_t max_block_bits(uint32_t flags) { return (flags & KPEG_FLAG_OPTIMIZE_HUFFMAN) ? MAX_BLOCK_BITS_OPT : MAX_BLOCK_BITS; }

// Everything the kernels read; built on the host (encode_host.h) per quality and uploaded.
struct EncTables {
    double cs[8][8];         // cs[x][u] = C(u)/2 * cos((2x+1) u pi / 16), host libm
    uint16_t qzz[2][64];     // quantiser of zig-zag position i: [0] luma, [1] chroma
    uint8_t nat[64];         // zig-zag index -> natural index
    uint16_t dc_code[2][16]; // DC codes by category, [0] luma, [1] chroma (Annex K, or optimised per encode)
    uint8_t dc_len[2][16];
    uint16_t ac_code[2][256]; // AC codes by run/size symbol
    uint8_t ac_len[2][256];
};

KPEG_HD double dmul(double a, double b)
{
#if defined(__CUDA_ARCH__)
    return __dmul_rn(a, b);
#else
    return a * b;
#endif
}

KPEG_HD double dadd(double a, double b)
{
#if defined(__CUDA_ARCH__)
    return __dadd_rn(a, b);
#else
    return a + b;
#endif
}

KPEG_HD double dsub(double a, double b)
{
#if defined(__CUDA_ARCH__)
    return __dsub_rn(a, b);
#else
    return a - b;
#endif
}

// JFIF RGB -> level-shifted Y, Cb, Cr, in the synth's order of operations
KPEG_HD void rgb_to_ycc(double R, double G, double B, double *y, double *cb, double *cr)
{
    *y = dsub(dadd(dadd(dmul(0.299, R), dmul(0.587, G)), dmul(0.114, B)), 128.0);
    *cb = dadd(dsub(dmul(-0.168736, R), dmul(0.331264, G)), dmul(0.5, B));
    *cr = dsub(dsub(dmul(0.5, R), dmul(0.418688, G)), dmul(0.081312, B));
}

// row pass: sum_q row[q] * cs[q][v], q ascending from 0
KPEG_HD double fdct_row(const double *row, const double (*cs)[8], int v)
{
    double s = 0;
    for (int q = 0; q < 8; ++q)
        s = dadd(s, dmul(row[q], cs[q][v]));
    return s;
}

// column pass for output (u, v): sum_r tmp[r*8+v] * cs[r][u]
KPEG_HD double fdct_col(const double *tmp, const double (*cs)[8], int u, int v)
{
    double s = 0;
    for (int r = 0; r < 8; ++r)
        s = dadd(s, dmul(tmp[r * 8 + v], cs[r][u]));
    return s;
}

// lround(s / q) clamped to +-2047 (DC) or +-1023 (AC)
KPEG_HD int quantise(double s, int q, bool dc)
{
    const long long v = llround(s / (double)q);
    const long long lim = dc ? 2047 : 1023;
    return (int)(v < -lim ? -lim : (v > lim ? lim : v));
}

// ---- DC nudge (KPEG_FLAG_REF_PARITY) --------------------------------------------------------------
// The synth picks the first of dc, dc-1, dc+1, dc-2, dc+2, ... inside +-2047 that differs from the previous
// block's final DC (same component, chain NOT reset at restart boundaries) and, at a restart segment's first
// MCU, from 0; blocks without AC terms keep dc.  At most two values are excluded and the range cuts off at
// most one side, so the final DC is dc + o with o in -2..2.  As a function of the previous block's offset
// (state s = o_prev + 2) each block is a map {0..4} -> {0..4}, packed 3 bits per state; the chain of a
// component is the composition of its blocks' maps, which is associative: a parallel scan.
KPEG_HD int nudge_dc(int dc, int prev, bool has_ac, bool first)
{
    if (!has_ac)
        return dc;
    for (int step = 0; step < 8; ++step) {
        const int d = dc + ((step & 1) ? -((step + 1) / 2) : (step / 2));
        if (d < -2047 || d > 2047)
            continue;
        if (d != prev && !(first && d == 0))
            return d;
    }
    return dc;
}

constexpr uint32_t MAP_IDENTITY = 0u | (1u << 3) | (2u << 6) | (3u << 9) | (4u << 12);
constexpr int MAP_START = 2; // the chain starts from prev = 0: "previous raw DC" 0 with offset 0

// prev_raw: the previous block's DC before the nudge (0 for the first block of a chain)
KPEG_HD uint32_t nudge_map(int dc, int prev_raw, bool has_ac, bool first)
{
    uint32_t m = 0;
    for (int s = 0; s < 5; ++s)
        m |= (uint32_t)(nudge_dc(dc, prev_raw + s - 2, has_ac, first) - dc + 2) << (3 * s);
    return m;
}

KPEG_HD int map_apply(uint32_t m, int s) { return (int)((m >> (3 * s)) & 7u); }

// a first, then b
KPEG_HD uint32_t map_then(uint32_t a, uint32_t b)
{
    uint32_t r = 0;
    for (int s = 0; s < 5; ++s)
        r |= (uint32_t)map_apply(b, map_apply(a, s)) << (3 * s);
    return r;
}

// ---- entropy coding of one block ---------------------------------------------------------------------
KPEG_HD int category(int v)
{
    const uint32_t a = (uint32_t)(v < 0 ? -v : v);
#if defined(__CUDA_ARCH__)
    return 32 - __clz(a);
#else
    int c = 0;
    for (uint32_t x = a; x; x >>= 1)
        ++c;
    return c;
#endif
}

KPEG_HD uint32_t value_bits(int v, int cat) { return (uint32_t)(v < 0 ? v + (1 << cat) - 1 : v) & ((1u << cat) - 1u); }

// The one walk over a block's symbols, in stream order: v.dc(cat, diff), then per non-zero AC coefficient v.zrl() for
// every 16 zeros before it beyond 15 and v.ac(run/size symbol, cat, value), and v.eob() when the block ends in zeros.
// Code emission (E3, E4) and the symbol histogram (EH) are visitors of it, so they cannot disagree on the symbols.
// zz: the block's 64 zig-zag coefficients (zz[0] unused); diff: its DC difference.
template <class V>
KPEG_HD void walk_block(int diff, const int16_t *zz, V &v)
{
    v.dc(category(diff), diff);
    int run = 0;
    for (int i = 1; i < 64; ++i) {
        const int x = zz[i];
        if (x == 0) {
            ++run;
            continue;
        }
        while (run > 15) {
            v.zrl();
            run -= 16;
        }
        const int cat = category(x);
        v.ac((run << 4) | cat, cat, x);
        run = 0;
    }
    if (run)
        v.eob();
}

// The walk's visitor that codes with table pair t (0 luma, 1 chroma): sink.put(bits, n) with n <= 27 -- code and value
// bits together; a code is at most 16 bits with Annex K and with optimised tables alike, a DC value at most 11.
template <class Sink>
struct Coder {
    const EncTables &T;
    int t;
    Sink &sink;
    KPEG_HD void dc(int cat, int diff) { sink.put(((uint32_t)T.dc_code[t][cat] << cat) | value_bits(diff, cat), T.dc_len[t][cat] + cat); }
    KPEG_HD void ac(int sym, int cat, int x) { sink.put(((uint32_t)T.ac_code[t][sym] << cat) | value_bits(x, cat), T.ac_len[t][sym] + cat); }
    KPEG_HD void zrl() { sink.put(T.ac_code[t][0xF0], T.ac_len[t][0xF0]); }
    KPEG_HD void eob() { sink.put(T.ac_code[t][0x00], T.ac_len[t][0x00]); }
};

template <class Sink>
KPEG_HD void code_block(const EncTables &T, int t, int diff, const int16_t *zz, Sink &sink)
{
    Coder<Sink> c{T, t, sink};
    walk_block(diff, zz, c);
}

struct BitCounter {
    uint32_t n = 0;
    KPEG_HD void put(uint32_t, int bits) { n += (uint32_t)bits; }
};

// Writes bits MSB-first into a zeroed stream of big-endian 32-bit words from bit position `pos` on.  A word that
// lies wholly inside this writer's bits is stored; the first and last words, which it may share with the
// neighbouring blocks, are OR-ed in (Words::orw: atomicOr on the device).
template <class Words>
struct BitEmitter {
    Words &w;
    uint64_t idx;
    uint64_t acc = 0;
    int n;
    bool shared_first;
    KPEG_HD BitEmitter(Words &words, uint64_t pos) : w(words), idx(pos >> 5), n((int)(pos & 31u)), shared_first((pos & 31u) != 0) {}
    KPEG_HD void put(uint32_t v, int bits)
    {
        acc = (acc << bits) | v;
        n += bits;
        if (n >= 32) {
            n -= 32;
            const uint32_t word = (uint32_t)(acc >> n);
            acc &= (n ? ((1ull << n) - 1u) : 0ull);
            if (shared_first)
                w.orw(idx, word);
            else
                w.store(idx, word);
            shared_first = false;
            ++idx;
        }
    }
    KPEG_HD void finish()
    {
        if (n > 0)
            w.orw(idx, (uint32_t)(acc << (32 - n)));
    }
};

// ---- geometry ------------------------------------------------------------------------------------------
struct EncGeom {
    uint32_t width, height, ncomp;
    uint32_t mx, my;
    uint64_t nmcu, nblk;     // MCUs, blocks (nmcu * ncomp)
    uint32_t ri;             // restart interval in MCUs, 0 = none
    uint64_t nseg;           // restart segments (1 without restart interval)
    uint64_t seg_mcus;       // MCUs per segment
    uint32_t flags;
};

// DC prediction of block b: the block of the same component one MCU back, unless b's MCU starts a segment
KPEG_HD bool starts_segment(const EncGeom &g, uint64_t m) { return m % g.seg_mcus == 0; }

// Stuffing tiles (E5): bytes of the unstuffed stream per CTA
constexpr uint32_t STUFF_THREADS = 256;
constexpr uint32_t STUFF_BYTES_PER_THREAD = 16;
constexpr uint32_t STUFF_TILE = STUFF_THREADS * STUFF_BYTES_PER_THREAD;

KPEG_HD uint32_t stream_byte(const uint32_t *words, uint64_t i) { return (words[i >> 2] >> (24u - 8u * (uint32_t)(i & 3u))) & 0xFFu; }

// the segment holding unstuffed byte i: the last s with seg_byte[s] <= i
KPEG_HD uint64_t segment_of_byte(const uint64_t *seg_byte, uint64_t nseg, uint64_t i)
{
    uint64_t lo = 0, hi = nseg - 1;
    while (lo < hi) {
        const uint64_t mid = (lo + hi + 1) >> 1;
        if (seg_byte[mid] <= i)
            lo = mid;
        else
            hi = mid - 1;
    }
    return lo;
}

// Writes the stuffed form of unstuffed bytes [i0, i1): each byte at i + ff_before(i) + 2 * segment(i), a 00 after
// every FF, FF D0+(k&7) after the last byte of segment k (all but the last), FF D9 after the very last byte.
// Nothing at or past `cap` is written.
template <class Out>
KPEG_HD void stuff_range(const uint32_t *words, const uint64_t *seg_byte, uint64_t nseg, uint64_t N, uint64_t i0, uint64_t i1,
                         uint64_t ff_before, Out &out)
{
    if (i0 >= i1)
        return;
    uint64_t s = segment_of_byte(seg_byte, nseg, i0);
    for (uint64_t i = i0; i < i1; ++i) {
        while (seg_byte[s + 1] <= i)
            ++s;
        uint64_t p = i + ff_before + 2 * s;
        const uint32_t b = stream_byte(words, i);
        out.put(p++, b);
        if (b == 0xFFu) {
            out.put(p++, 0x00);
            ++ff_before;
        }
        if (i + 1 == seg_byte[s + 1]) {
            out.put(p++, 0xFF);
            out.put(p, i + 1 == N ? 0xD9u : 0xD0u + (uint32_t)(s & 7u));
        }
    }
}

} // namespace enc
} // namespace kpeg
#endif
