/*
 * kpeg_synth.h -- deterministic synthetic baseline-JPEG encoder (host only, no CUDA).
 *
 * The reference's own encoder is non-functional (README.md:23; src/Encoder.cpp writes
 * "output.jpg" with 12.6 dB PSNR), so benchmark and parity inputs come from this committed
 * generator instead (BASELINE.json north_star).  It has no counterpart in the reference; the
 * only things it takes from it are the facts about which container layout the reference's
 * parser accepts (src/Decoder.cpp:53-75, SURVEY F7): segments are written in exactly the
 * order of misc/images/lena.jpg -- SOI, APP0(JFIF 1.1), DQT id0, DQT id1, SOF0, DHT 0x00,
 * 0x10, 0x01, 0x11, [DRI], SOS, scan, EOI -- with the ITU-T T.81 Annex K quantisation tables
 * (scaled by the usual IJG quality rule) and Annex K Huffman tables.
 *
 * "Twin" streams: two calls that differ only in KPEG_SYNTH_EMIT_RESTART, or only in
 * `file_components` (1 vs 3 with KPEG_SYNTH_GRAY_CONTENT), carry IDENTICAL quantised
 * coefficients.  The reference cannot parse DRI/RSTn or 1-component files (SURVEY F2,F3), so
 * the 3-component, marker-free twin is what it decodes while the GPU path decodes the other.
 * KPEG_SYNTH_QUIRK_FREE nudges DC values so that no block has "DC difference == 0 and a
 * non-zero AC coefficient" in EITHER twin (SURVEY F1,F4): such streams decode identically
 * with and without the reference's AC-dropping quirk.
 */
#ifndef KPEG_SYNTH_H
#define KPEG_SYNTH_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define KPEG_SYNTH_EMIT_RESTART 1u /* write DRI + RSTn (otherwise restart_interval only shapes the nudge) */
#define KPEG_SYNTH_GRAY_CONTENT 2u /* luminance-only content; chroma blocks (if any) are all zero */
#define KPEG_SYNTH_QUIRK_FREE 4u   /* see above */
#define KPEG_SYNTH_NON_INTERLEAVED 8u /* three-component files: one scan per component (T.81 A.2.3) instead of one interleaved scan */
/* Huffman tables optimised for the image's symbol counts (T.81 K.2 / K.3, the rule of KPEG_FLAG_OPTIMIZE_HUFFMAN in
 * include/kpeg_cuda.h) instead of the Annex K ones; the quantised coefficients do not change */
#define KPEG_SYNTH_OPTIMIZE_HUFFMAN 16u

typedef struct kpeg_synth_params {
    int32_t width, height;       /* pixels; any size >= 1 (edges are replicated to whole blocks) */
    int32_t file_components;     /* 1 or 3 */
    int32_t quality;             /* IJG quality 1..100 */
    int32_t restart_interval;    /* in MCUs, 0 = none */
    uint32_t flags;              /* KPEG_SYNTH_* */
    uint64_t seed;               /* content seed */
    int32_t noise_amp;           /* noise amplitude, 0 = default (10, sigma ~ 5.8 grey levels) */
    int32_t threads;             /* worker threads, 0 = hardware concurrency */
} kpeg_synth_params;

/* Encodes one image.  On success returns 0 and hands back a malloc'd buffer the caller must
 * release with kpeg_synth_free.  Returns -1 on bad parameters, -2 on allocation failure. */
int kpeg_synth_encode(const kpeg_synth_params *p, uint8_t **out, size_t *out_len);
void kpeg_synth_free(uint8_t *buf);

/* The same encoder over caller-supplied pixels: [height][width][file_components==1 or GRAY_CONTENT ? 1 : 3]
 * (interleaved R,G,B).  Uses width, height, file_components, quality, restart_interval, flags and threads; ignores
 * seed and noise_amp.  kpeg_synth_encode(p) == kpeg_synth_encode_pixels(p, kpeg_synth_pixels(p)) byte for byte.
 * With flags KPEG_SYNTH_QUIRK_FREE (or 0), plus KPEG_SYNTH_EMIT_RESTART when restart_interval > 0, this is the exact
 * file the GPU encoder (kpeg_cuda_encode, include/kpeg_cuda.h) writes with KPEG_FLAG_REF_PARITY (or 0); adding
 * KPEG_SYNTH_OPTIMIZE_HUFFMAN gives the file it writes with KPEG_FLAG_OPTIMIZE_HUFFMAN added. */
int kpeg_synth_encode_pixels(const kpeg_synth_params *p, const uint8_t *pixels, uint8_t **out, size_t *out_len);

/* The encoder's coding path over given quantised coefficients (what encode_pixels runs after the DC nudge):
 * coef is [nblk][64] int16, blocks MCU-interleaved (one block per component per MCU), zig-zag order, DC absolute.
 * Writes SOI, APP0, one DQT per quantiser id the components use (ascending, qt[id] in zig-zag order), SOF0 (ids 1..ncomp,
 * sampling 0x11, tq[c]), DHT (Annex K or, KPEG_SYNTH_OPTIMIZE_HUFFMAN, optimised), [DRI when restart_interval > 0], one
 * interleaved SOS, the scan with RSTn, EOI.  Returns -1 on bad parameters or when a DC difference has category > 11 or an
 * AC coefficient is outside +-1023 (no baseline table codes them), -2 on allocation failure.  The reference of the GPU
 * transcoder (kpeg_cuda_transcode). */
typedef struct kpeg_synth_coef_frame {
    int32_t width, height;    /* 1..65535 */
    int32_t ncomp;            /* 1 or 3 */
    uint8_t tq[3];            /* quantiser id (0..3) per component */
    uint8_t qt[4][64];        /* quantisers by id, zig-zag order (only the ids in tq are written) */
    int32_t restart_interval; /* MCUs, 0 = none */
    uint32_t flags;           /* 0 or KPEG_SYNTH_OPTIMIZE_HUFFMAN */
} kpeg_synth_coef_frame;
int kpeg_synth_encode_coefficients(const kpeg_synth_coef_frame *f, const int16_t *coef, uint8_t **out, size_t *out_len);

/* The source pixels the encoder compressed (before the lossy steps), for PSNR reporting.
 * dst is [height][width][file_components==1 or GRAY_CONTENT ? 1 : 3]. */
int kpeg_synth_pixels(const kpeg_synth_params *p, uint8_t *dst);

#ifdef __cplusplus
}
#endif
#endif
