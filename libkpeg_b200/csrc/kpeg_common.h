// kpeg_common.h -- types shared by the CUDA kernels, the C-ABI host code and the CPU-side
// logic tests of the B200 baseline-JPEG decode path.
//
// Everything in the *_core.h headers is written as `KPEG_HD` (host + device) functions so the
// very same source that runs inside the sm_100a kernels can be single-stepped on the CPU by
// tests/ (tests/emu/) -- that is a test harness for the kernel logic, not a product code path:
// libkpeg_cuda.so contains no CPU decode.
#ifndef KPEG_COMMON_H
#define KPEG_COMMON_H

#include <stdint.h>

#if defined(__CUDACC__)
#define KPEG_HD __host__ __device__ __forceinline__
#define KPEG_D __device__ __forceinline__
#else
#define KPEG_HD inline
#endif

namespace kpeg {

// ---- Huffman lookup tables ---------------------------------------------------------------------
// One table per (component, DC/AC).  `fast` is indexed by the next LUT_BITS bits of the stream and
// resolves every code of length <= LUT_BITS in one shared-memory load; longer codes fall back to a
// canonical-code search over `bound` (T.81 Annex F.2.2.3 style), which the reference does by walking
// its tree bit by bit (HuffmanTree.cpp:164-193).
//
// fast entry (uint16): bits 0-4 TOTAL bits the symbol occupies (code length + magnitude bits, 1..27),
// bits 5-8 magnitude bits ("category"), bits 9-15 slot advance (number of zig-zag positions the
// symbol consumes: 1 for DC, run+1 for AC, 16 for ZRL, 64 for EOB -- the consumer clamps to the
// end of the block).  0 = not resolved.  The speculative passes only need the total and the advance.
#ifndef KPEG_LUT_BITS
#define KPEG_LUT_BITS 10
#endif
constexpr int LUT_BITS = KPEG_LUT_BITS;
constexpr int LUT_SIZE = 1 << LUT_BITS;
constexpr int SUB_BITS = 16 - LUT_BITS;   // a sub-table resolves the rest of a 16-bit window
constexpr int SUB_SIZE = 1 << SUB_BITS;
constexpr int LONG_CAP = LUT_BITS >= 10 ? 512 : 640; // second-level entries per table: 8 sub-tables of 64, or 5 of 128
// no code matches: "length" 17, no magnitude bits, and a slot advance no real symbol has (records carry the
// entry, so the expander recognises the pattern by it)
constexpr uint32_t ENTRY_ADV_INVALID = 127u;
constexpr uint32_t ENTRY_INVALID = 17u | (0u << 5) | (ENTRY_ADV_INVALID << 9);
constexpr int MAX_COMP = 3;
constexpr int MAX_LUTS = MAX_COMP * 2; // [comp*2 + (0=DC,1=AC)]

// Canonical description of one table (rare fallback + host-side construction).
struct HuffCanon {
    uint32_t bound[18];      // bound[L] = exclusive upper bound of the left-aligned 16-bit windows whose code has length <= L
    uint16_t first_code[18]; // first code value of length L
    uint16_t first_idx[18];  // index of its symbol
    uint8_t symbols[256];
    uint32_t is_ac;
    uint32_t pad_[3];
};

// What the entropy kernels keep in shared memory: a classic two-level table.  A first-level entry
// whose low five bits are zero is not a symbol: non-zero, it points at a 64-entry sub-table
// ((entry >> 5) - 1) indexed by stream bits 10..15, which resolves every code of up to 16 bits that
// starts with this 10-bit prefix in ONE more load (the Annex K AC tables need 5-6 sub-tables);
// zero, the prefix has no sub-table (more than LONG_CAP/64 long prefixes, or no code at all) and
// the canonical search decides.
struct LutSet {
    uint16_t fast[MAX_LUTS][LUT_SIZE];
    uint16_t longlut[MAX_LUTS][LONG_CAP];
    uint32_t long_n[MAX_LUTS]; // entries of longlut in use (multiple of 64)
    uint32_t pad_[2];
};
static_assert(sizeof(LutSet) % 16 == 0, "LutSet is copied to shared memory in 16-byte units");

// Symbol -> fast-table entry.  DC symbol: category = sym & 15, one slot.  AC symbol: run = sym >> 4,
// category = sym & 15; 0x00 (EOB) consumes the rest of the block, 0xF0 (ZRL) 16 slots
// (reference src/Decoder.cpp:706-803).
KPEG_HD uint32_t pack_entry(uint32_t len, uint32_t sym, bool is_ac)
{
    uint32_t size = sym & 15u;
    uint32_t adv = 1u;
    if (is_ac)
        adv = (sym == 0x00u) ? 64u : (sym >> 4) + 1u;
    return (len + size) | (size << 5) | (adv << 9);
}

// Device-side description of one decode job (one image, or a batch of same-plan images decoded as
// one concatenated stream).  Lives in global memory; kernels get a pointer.
struct DeviceTables {
    LutSet luts;
    HuffCanon canon[MAX_LUTS];
    float qscale[MAX_COMP][64]; // zig-zag order: quantiser * AAN prescale (fast IDCT path)
    // K3 stages the next two arrays in shared memory with one bulk copy each (16-byte aligned, contiguous):
    alignas(16) float qpair[MAX_COMP][64]; // qscale in the pair order of the packed transform: [2 p + h] = position pair_nat(p, h)
    alignas(16) float qdc[MAX_COMP][64];   // qpair with every AC entry zero: what a block that loses its AC terms (F1) multiplies by
    int32_t qint[MAX_COMP][64]; // zig-zag order: plain quantiser (exact path), MCU.cpp:110-112
    double cosd[8][8];          // cosd[x][u] = cos((2x+1)*u*pi/16) in double, host libm -- the factor of MCU.cpp:193
    float cc[8][8];             // (float)Cu*(float)Cv of MCU.cpp:190-193
};

// Geometry / stream description, passed by value to kernels.
struct JobGeom {
    uint32_t width, height;   // pixels per image
    uint32_t ncomp;           // 1 or 3
    uint32_t mcus_x, mcus_y;  // blocks per row / column (MCU == one 8x8 block per component)
    uint32_t mcus_per_image;
    uint32_t restart_interval; // MCUs, 0 = none
    uint32_t segs_per_image;   // restart intervals per image (1 if none)
    uint32_t nimages;
    uint32_t nseg;            // nimages * segs_per_image
    uint32_t total_blocks;    // nimages * mcus_per_image * ncomp
    uint32_t flags;           // KPEG_FLAG_*
    uint32_t sub_bits;        // bits per speculative subsequence (multiple of 32)
};

// ---- output geometry ------------------------------------------------------------------------------------------
// The decoded image of a plan: full size, or 1/2, 1/4, 1/8 of it (KPEG_FLAG_SCALE_* of kpeg_cuda.h: scale code in bits 2..3)
// rounded up as libjpeg's jdiv_round_up does.  Every buffer size, row placement and copy of the decode path goes
// through this one description.
constexpr uint32_t SCALE_FLAG_SHIFT = 2u, SCALE_FLAG_MASK = 12u;
KPEG_HD uint32_t scale_denom(uint32_t flags) { return 1u << ((flags & SCALE_FLAG_MASK) >> SCALE_FLAG_SHIFT); }

struct OutGeom {
    uint32_t width, height, ncomp; // of one output image
    uint32_t scale;                // 1, 2, 4 or 8
    KPEG_HD uint64_t row_bytes() const { return (uint64_t)width * ncomp; }
    KPEG_HD uint64_t bytes() const { return row_bytes() * height; } // one image; a batch holds its images back to back
    KPEG_HD uint32_t mcu_row(uint32_t r) const { return r * 8u / scale; } // output row where MCU row r begins
};

KPEG_HD OutGeom out_geom(uint32_t width, uint32_t height, uint32_t ncomp, uint32_t flags)
{
    const uint32_t s = scale_denom(flags);
    return OutGeom{(width + s - 1u) / s, (height + s - 1u) / s, ncomp, s};
}

// First absolute coefficient slot (block*64 + zig-zag index) of restart segment `seg`.
KPEG_HD uint32_t seg_slot_base(const JobGeom &g, uint32_t seg)
{
    if (seg >= g.nseg)
        return g.total_blocks * 64u;
    uint32_t img = seg / g.segs_per_image;
    uint32_t r = seg - img * g.segs_per_image;
    return (img * g.mcus_per_image + r * g.restart_interval) * g.ncomp * 64u;
}

KPEG_HD OutGeom out_geom(const JobGeom &g) { return out_geom(g.width, g.height, g.ncomp, g.flags); }

// ---- status word bits (device -> host) -----------------------------------------------------------
constexpr uint32_t ST_BAD_CODE = 1u;       // a bit pattern that is no Huffman code was consumed by the final decode
constexpr uint32_t ST_SLOT_OVERFLOW = 2u;  // a coefficient would land outside the image
constexpr uint32_t ST_SEG_MISMATCH = 4u;   // a restart interval did not hold the expected number of MCUs
constexpr uint32_t ST_BAD_MARKER = 8u;     // a marker other than RSTn inside the entropy-coded segment
constexpr uint32_t ST_EXIT_MISMATCH = 16u; // final decode left a subsequence in a different state than the relay recorded
constexpr uint32_t ST_SEG_COUNT = 32u;     // number of RSTn markers does not match the DRI interval
constexpr uint32_t ST_REC_OVERFLOW = 64u;   // a subsequence held more symbols than the record list has room for (-> Huffman final pass)

constexpr uint32_t ST_RELAY_TIMEOUT = 128u; // the relay loop's grid barrier gave up waiting (grid not co-resident): the host finishes the relay round by round


// Per-subsequence relay state: where the first symbol after the end of the subsequence starts and
// in which decoder state, plus how many coefficient slots were produced on the way.
struct alignas(16) SubState {
    uint32_t p;   // bit position (in the unstuffed stream) of the next symbol
    uint32_t n;   // slots produced since the entry of the subsequence, or since the last segment boundary crossed
    uint32_t cz;  // (component << 8) | zig-zag index of the next coefficient (0 = a DC symbol comes next)
    int32_t seg;  // index of the last segment boundary crossed inside the subsequence, -1 if none
};

} // namespace kpeg
#endif
