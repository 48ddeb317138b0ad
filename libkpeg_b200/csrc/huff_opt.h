// huff_opt.h -- optimised Huffman tables (ITU-T T.81 K.2, Figures K.1-K.3), canonical codes (T.81 C.2) and the part
// of a JPEG header that follows SOF0 (DHT, DRI, SOS), written as KPEG_HD code shared by the GPU encoder's table-build
// kernel (csrc/encode.cu, EB), the host header writer (jfif_write.h), the synthetic reference encoder and the CPU
// replay in tests/emu/emu_encode_opt.cpp.
//
// The table rule is libjpeg's jpeg_gen_optimal_table:
//   - a reserved symbol 256 gets frequency 1, so that no code is all ones;
//   - each step merges the two smallest non-zero frequencies (first the smaller, on a tie the larger symbol number);
//     the merged tree keeps the first one's slot, the second slot is emptied;
//   - a symbol's code length is its leaf depth; lengths over 16 are folded down as in Figure K.3, then one code of the
//     longest length (the reserved one) is removed;
//   - HUFFVAL lists the symbols 0..255 ordered by (unfolded length, symbol).
// Two deliberate differences: frequencies are 64-bit with no 10^9 sentinel (one table of a 65535 x 65535 image counts
// more than 2^32 symbols), and lengths are taken up to the deepest possible tree (256 levels), not libjpeg's 32.
#ifndef KPEG_HUFF_OPT_H
#define KPEG_HUFF_OPT_H

#include <stdint.h>

#include "kpeg_common.h"

namespace kpeg {
namespace huff {

constexpr int NSYM = 257;      // 256 symbols + the reserved one
constexpr int RESERVED = 256;
constexpr int MAX_DEPTH = 256; // deepest leaf of a tree with 257 leaves
constexpr int NNODE = 2 * NSYM - 1;

// merge order: a before b when a's frequency is smaller, on a tie when a's slot is larger
KPEG_HD bool merges_first(uint64_t fa, int a, uint64_t fb, int b) { return fa < fb || (fa == fb && a > b); }

// leaf depth of node s in a forest given as a parent array (-1 at the root)
KPEG_HD int leaf_depth(const int16_t *parent, int s)
{
    int d = 0;
    for (int n = parent[s]; n >= 0; n = parent[n])
        ++d;
    return d;
}

// Figure K.3: cnt[L] codes of length L for L = 0..max_depth (cnt[0..16] must exist even when max_depth < 16), folded
// to lengths <= 16; then the reserved code, one of the longest, is removed.  BITS[L-1] = cnt[L].
template <class Count>
KPEG_HD void fold_lengths(Count *cnt, int max_depth, uint8_t bits[16])
{
    for (int i = max_depth; i > 16; --i)
        while (cnt[i] > 0) {
            int j = i - 2;
            while (cnt[j] == 0)
                --j;
            cnt[i] -= 2;
            cnt[i - 1] += 1;
            cnt[j + 1] += 2;
            cnt[j] -= 1;
        }
    int i = 16;
    while (i > 0 && cnt[i] == 0)
        --i;
    if (i > 0)
        cnt[i] -= 1;
    for (int L = 1; L <= 16; ++L)
        bits[L - 1] = (uint8_t)cnt[L];
}

// T.81 C.2: the canonical code of every symbol of a DHT table; symbols not in it get length 0
KPEG_HD void canonical_codes(const uint8_t bits[16], const uint8_t *vals, uint16_t code[256], uint8_t len[256])
{
    for (int s = 0; s < 256; ++s) {
        code[s] = 0;
        len[s] = 0;
    }
    int c = 0, k = 0;
    for (int L = 1; L <= 16; ++L) {
        for (int i = 0; i < bits[L - 1]; ++i) {
            code[vals[k]] = (uint16_t)c++;
            len[vals[k]] = (uint8_t)L;
            ++k;
        }
        c <<= 1;
    }
}

// The whole rule, one thread (the reference; EB runs the same steps warp-parallel).  freq[0..255]: symbol counts
// (freq[256] is ignored: the reserved symbol always counts 1).  Returns the number of symbols in HUFFVAL.
KPEG_HD int optimal_table(const uint64_t *freq, uint8_t bits[16], uint8_t vals[256])
{
    uint64_t f[NSYM];
    int16_t parent[NNODE], node[NSYM];
    for (int s = 0; s < NSYM; ++s) {
        f[s] = s == RESERVED ? 1u : freq[s];
        node[s] = (int16_t)s;
    }
    for (int n = 0; n < NNODE; ++n)
        parent[n] = -1;
    for (int next = NSYM;; ++next) {
        int c1 = -1, c2 = -1;
        for (int s = 0; s < NSYM; ++s)
            if (f[s] && (c1 < 0 || merges_first(f[s], s, f[c1], c1)))
                c1 = s;
        for (int s = 0; s < NSYM; ++s)
            if (f[s] && s != c1 && (c2 < 0 || merges_first(f[s], s, f[c2], c2)))
                c2 = s;
        if (c2 < 0)
            break;
        f[c1] += f[c2];
        f[c2] = 0;
        parent[node[c1]] = parent[node[c2]] = (int16_t)next;
        node[c1] = (int16_t)next;
    }
    uint32_t cnt[MAX_DEPTH + 1] = {}, start[MAX_DEPTH + 2] = {};
    uint16_t depth[NSYM];
    int max_depth = 0;
    for (int s = 0; s < NSYM; ++s) {
        depth[s] = (uint16_t)((s == RESERVED || freq[s]) ? leaf_depth(parent, s) : 0);
        if (depth[s]) {
            ++cnt[depth[s]];
            max_depth = depth[s] > max_depth ? depth[s] : max_depth;
            if (s != RESERVED)
                ++start[depth[s] + 1];
        }
    }
    for (int d = 1; d <= MAX_DEPTH; ++d)
        start[d + 1] += start[d];
    int n = 0;
    for (int s = 0; s < 256; ++s)
        if (depth[s]) {
            vals[start[depth[s]]++] = (uint8_t)s;
            ++n;
        }
    fold_lengths(cnt, max_depth, bits);
    return n;
}

// ---- the header after SOF0 --------------------------------------------------------------------------------------
// Out: put(byte), appending; a host-only Out (jfif::VecOut) instantiates these on the host only.
#if defined(__CUDACC__)
#define KPEG_HD_OUT _Pragma("nv_exec_check_disable")
#else
#define KPEG_HD_OUT
#endif

KPEG_HD_OUT template <class Out>
KPEG_HD void put16(Out &o, uint32_t v)
{
    o.put((v >> 8) & 0xFFu);
    o.put(v & 0xFFu);
}

KPEG_HD_OUT template <class Out>
KPEG_HD void put_dht(Out &o, int tc_th, const uint8_t *bits, const uint8_t *vals)
{
    int n = 0;
    for (int i = 0; i < 16; ++i)
        n += bits[i];
    o.put(0xFF);
    o.put(0xC4);
    put16(o, 2 + 1 + 16 + n);
    o.put((uint32_t)tc_th);
    for (int i = 0; i < 16; ++i)
        o.put(bits[i]);
    for (int i = 0; i < n; ++i)
        o.put(vals[i]);
}

KPEG_HD_OUT template <class Out>
KPEG_HD void put_dri(Out &o, int ri)
{
    o.put(0xFF);
    o.put(0xDD);
    put16(o, 4);
    put16(o, (uint32_t)ri);
}

// SOS of a scan of components c0..c1-1 (luma tables for component 0, chroma tables for the others)
KPEG_HD_OUT template <class Out>
KPEG_HD void put_sos(Out &o, int c0, int c1)
{
    o.put(0xFF);
    o.put(0xDA);
    put16(o, 6 + 2 * (c1 - c0));
    o.put((uint32_t)(c1 - c0));
    for (int c = c0; c < c1; ++c) {
        o.put((uint32_t)(c + 1));
        o.put(c ? 0x11u : 0x00u);
    }
    o.put(0x00);
    o.put(0x3F);
    o.put(0x00);
}

// DHT 0x00, 0x10 [, 0x01, 0x11] [, DRI when ri > 0], SOS of the one interleaved scan.  Table t of bits / vals:
// 0 DC luma, 1 AC luma, 2 DC chroma, 3 AC chroma.
KPEG_HD_OUT template <class Out>
KPEG_HD void put_header_tail(Out &o, int nc, const uint8_t *const bits[4], const uint8_t *const vals[4], int ri)
{
    for (int t = 0; t < (nc == 3 ? 4 : 2); ++t)
        put_dht(o, ((t & 1) << 4) | (t >> 1), bits[t], vals[t]);
    if (ri > 0)
        put_dri(o, ri);
    put_sos(o, 0, nc);
}

} // namespace huff
} // namespace kpeg
#endif
