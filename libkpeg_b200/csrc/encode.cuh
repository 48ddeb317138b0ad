// encode.cuh -- launch interface of the GPU baseline-JPEG encoder (csrc/encode.cu), used by the C-ABI host code.
#ifndef KPEG_ENCODE_CUH
#define KPEG_ENCODE_CUH

#include <cuda_runtime.h>
#include <stddef.h>
#include <stdint.h>

#include "encode_core.h"
#include "transcode_core.h"

namespace kpeg {
namespace enc {

struct EncMeta {
    uint64_t unstuffed; // bytes of the unstuffed stream (segments padded to bytes)
    uint64_t scan_len;  // bytes written after the header: stuffed scan + RSTn markers + EOI
    uint64_t hdr_len;   // bytes of the header, where the scan starts (written by EB in optimised mode, else by E5)
    uint32_t range_fail; // transcode only: TG found a coefficient no baseline table codes (transcode_core.h)
    uint32_t pad;
};

// Device buffers of one encode (sizes: scratch_sizes).
struct EncBufs {
    const uint8_t *pixels;  // [height][width][ncomp]
    const EncTables *tables; // the cached per-quality tables (Annex K codes); never written
    EncTables *opt_tables;   // KPEG_FLAG_OPTIMIZE_HUFFMAN: this encode's copy with the optimised codes (EB)
    uint64_t *hist;          // KPEG_FLAG_OPTIMIZE_HUFFMAN: [4][257] symbol counts (EH), table order as in huff_opt.h
    int16_t *coef;          // [nblk][64] zig-zag
    int16_t *raw;           // [nblk] DC before the nudge
    int16_t *dc;            // [nblk] final DC (== raw without KPEG_FLAG_REF_PARITY)
    uint8_t *has_ac;        // [nblk]
    uint32_t *bits;         // [nblk]
    uint64_t *off;          // [nblk + 1] exclusive scan of bits
    uint64_t *seg_byte;     // [nseg + 1] byte offset of every segment in the unstuffed stream
    uint32_t *words;        // unstuffed stream, big-endian words
    void *agg;              // tile aggregates of the scans
    uint64_t *tile_ff;      // FF bytes per stuffing tile, then their exclusive scan
    EncMeta *meta;
    uint8_t *out;           // the file: the header (or, optimised, its prefix up to SOF0) is already there
    uint64_t out_cap;       // bytes writable at out
    uint64_t hdr_len;       // bytes already at out: the whole header, or the prefix in optimised mode
};

enum { BUF_COEF, BUF_RAW, BUF_DC, BUF_HAS_AC, BUF_BITS, BUF_OFF, BUF_SEG, BUF_WORDS, BUF_AGG, BUF_TILE_FF, BUF_COUNT };
// bytes each scratch buffer needs for an image of geometry g (words and tile_ff sized for the worst-case stream)
void scratch_sizes(const EncGeom &g, size_t sizes[BUF_COUNT]);

// Stage hooks for the caller's profiling events: called after each stage with a KPEG_T_* index.
typedef void (*StageMark)(void *user, int stage);

// Enqueues E1..E5 on `s` (with EH and EB between E2 and E3 in optimised mode).  Returns cudaSuccess or the first launch error.
cudaError_t launch_encode(const EncGeom &g, const EncBufs &b, cudaStream_t s, uint32_t *launches, StageMark mark, void *user);
// The stages after E2 (EH and EB in optimised mode, then E3..E5) on b.coef and the final DC values dc: what
// launch_encode runs after E1 / E2, and what the transcoder runs after TG.
cudaError_t launch_coded_stages(const EncGeom &g, const EncBufs &b, const int16_t *dc, cudaStream_t s, uint32_t *launches,
                                StageMark mark, void *user);

} // namespace enc

namespace tc {
// TG (transcode.cu): the decoder's coefficient tiles -> coef [nblk][64] and dc [nblk] of the output, moved by g.xform;
// *fail |= 1 when a value breaks the baseline range rules (zero it before).
void launch_gather(const TcGeom &g, const void *tiles, int16_t *coef, int16_t *dc, uint32_t *fail, cudaStream_t s, uint32_t *launches);
} // namespace tc
} // namespace kpeg
#endif
