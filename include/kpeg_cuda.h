/*
 * kpeg_cuda.h -- C ABI of the B200 (sm_100a) baseline-JPEG decode hot path, and of the GPU encoder (at the end).
 *
 * libKPEG has no plugin / FFI interface of its own: its hot path is reachable only through the
 * C++ class kpeg::JPEGDecoder (reference include/Decoder.hpp:26-128) and the `kpeg` CLI
 * (reference main.cpp:54-79).  This header is the thin boundary the drop-in JPEGDecoder in
 * libkpeg_b200/host/ calls; every entry point names the reference member(s) whose work it
 * replaces.  Plain pointers and sizes only, no C++ or torch types.  All file:line citations are
 * relative to /root/reference.
 *
 * There is NO CPU fallback behind this interface: every decode call runs the CUDA kernels in
 * libkpeg_b200/csrc/ and fails with KPEG_ERR_CUDA when no device is usable.
 */
#ifndef KPEG_CUDA_H
#define KPEG_CUDA_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* ---- return codes ------------------------------------------------------------------------ */
#define KPEG_OK 0
#define KPEG_ERR_FORMAT (-1)      /* malformed container      -> JPEGDecoder::ResultCode::ERROR     (Decoder.cpp:126-132) */
#define KPEG_ERR_UNSUPPORTED (-2) /* SOF1/SOF2/subsampling... -> JPEGDecoder::ResultCode::TERMINATE (Decoder.cpp:65-66,351-356) */
#define KPEG_ERR_STREAM (-3)      /* corrupt entropy-coded data (the reference hangs / reads out of bounds, Decoder.cpp:706-803) */
#define KPEG_ERR_NOMEM (-4)
#define KPEG_ERR_CUDA (-5)        /* no device / CUDA runtime failure (see kpeg_cuda_last_error) */
#define KPEG_ERR_ARG (-6)
#define KPEG_ERR_NOT_CONVERGED (-7) /* internal: speculative decode needed more fix-up rounds (retried automatically) */

/* ---- plan flags -------------------------------------------------------------------------- */
/* Reproduce MCU.cpp:97-104: a block whose DC *difference* is 0 loses its AC coefficients
 * (SURVEY F1).  ON for bit-exact parity with the reference; OFF for ITU-T T.81 behaviour. */
#define KPEG_FLAG_REF_PARITY 1u
/* Encode only (kpeg_encode_params.flags): code with Huffman tables optimised for the image (T.81 K.2) instead of the
 * Annex K ones.  The decode entry points ignore it. */
#define KPEG_FLAG_OPTIMIZE_HUFFMAN 2u
/* Decode only (kpeg_plan.flags and the `flags` argument of the file entry points): reduced-size output, what libjpeg's
 * scale_num / scale_denom = 1/2, 1/4, 1/8 (djpeg -scale 1/N) give.  The image comes out ceil(W/N) x ceil(H/N) (libjpeg's
 * jdiv_round_up), in the usual layouts.  The quantised coefficients are decoded exactly as at full size
 * (KPEG_FLAG_REF_PARITY still selects the DC-difference rule); only the reconstruction differs: per 8x8 block the
 * dequantised coefficients go through libjpeg-turbo's reduced IDCTs (jidctred.c: jpeg_idct_4x4, _2x2, _1x1; CONST_BITS 13,
 * PASS1_BITS 2, 64-bit products, the post-IDCT range-limit table indexed with & 1023, which wraps) and three components
 * through libjpeg's integer ycc_rgb_convert (SCALEBITS 16).  So at a reduced scale the colours are libjpeg's, not the
 * reference's float path; at full size (no scale bits) nothing changes.  kpeg_output_size gives the output size.
 * Encode and transcode reject these bits (KPEG_ERR_ARG). */
#define KPEG_FLAG_SCALE_1_2 4u
#define KPEG_FLAG_SCALE_1_4 8u
#define KPEG_FLAG_SCALE_1_8 12u
#define KPEG_FLAG_SCALE_MASK 12u

/* One Huffman table as it appears in a DHT segment (Types.hpp:116, Decoder.cpp:366-459). */
typedef struct kpeg_huff_spec {
    uint8_t counts[16];   /* number of codes of length 1..16 */
    uint8_t symbols[256]; /* symbols in order of increasing code length */
} kpeg_huff_spec;

/*
 * Everything the kernels need to know about one image, produced by the host-side container
 * parse (replaces the state JPEGDecoder accumulates in parseQuantizationTable / parseSOF0Segment /
 * parseHuffmanTable / parseSOSSegment, Decoder.cpp:230-530).  POD; caller-owned.
 */
typedef struct kpeg_plan {
    uint16_t width, height;     /* SOF0 X, Y (Decoder.cpp:301-364) */
    uint8_t ncomp;              /* 1 (T.81 extension, SURVEY F3) or 3; sampling is always 1x1 */
    uint8_t comp_tq[3];         /* quantisation-table id per component */
    uint8_t comp_td[3];         /* DC Huffman table id per component   */
    uint8_t comp_ta[3];         /* AC Huffman table id per component   */
    uint16_t restart_interval;  /* DRI value in MCUs, 0 = none (T.81 extension, SURVEY F2) */
    uint32_t flags;             /* KPEG_FLAG_* */
    uint8_t qt_present[4];
    uint8_t ht_present[2][4];
    uint16_t qt[4][64];         /* zig-zag (file) order, as Decoder.cpp:230-299 keeps them */
    kpeg_huff_spec ht[2][4];    /* [class 0=DC,1=AC][id] */
} kpeg_plan;

/* Stages timed with CUDA events on the decode stream while profiling is on. */
enum {
    KPEG_T_H2D = 0,        /* host -> device copy of the scan (host-pointer entry points only)            */
    KPEG_T_MEMSET,         /* zero-fill of bookkeeping, bit stream tail and coefficient buffer            */
    KPEG_T_UNSTUFF,        /* K0: unstuff_count + unstuff_scan + unstuff_write                            */
    KPEG_T_ENTROPY_COLD,   /* K1: speculative cold decode of every subsequence                            */
    KPEG_T_ENTROPY_RELAY,  /* K1: first relay round (every subsequence, emits symbol records)             */
    KPEG_T_ENTROPY_SCAN,   /* K1: segmented scan of slot counts and DC sums over the subsequences          */
    KPEG_T_ENTROPY_WRITE,  /* K2: record expansion + DC prediction -> coefficient tiles (or the Huffman final pass) */
    KPEG_T_DC_SCAN,        /* fallback only: DC prediction + tile conversion behind the Huffman final pass  */
    KPEG_T_IDCT,           /* K3: fused dequant + IDCT + colour + store, and the exact re-evaluation pass;
                              reduced-size decodes (KPEG_FLAG_SCALE_*): the reduced-size reconstruction kernel */
    KPEG_T_D2H,            /* device -> host copy of the pixels (host-pointer entry points only)          */
    KPEG_T_RELAY_SPARSE,   /* K1: later relay rounds (work list only) up to the fixed point               */
    KPEG_T_IDCT_PATCH,     /* (not used: the exact pass is timed with KPEG_T_IDCT)                         */
    KPEG_T_COUNT
};

/* Per-decode statistics.  Stage times are filled only while profiling is enabled
 * (kpeg_cuda_set_profiling); they are CUDA-event times on the decode stream, in milliseconds. */
typedef struct kpeg_stats {
    uint32_t width, height, ncomp; /* of the output image (the reduced size with KPEG_FLAG_SCALE_*; a crop's rectangle) */
    uint64_t scan_bytes;        /* stuffed entropy-coded bytes handed in                  */
    uint64_t unstuffed_bytes;   /* after FF00 / RSTn removal                              */
    uint32_t segments;          /* restart intervals found (1 when there is no DRI)       */
    uint32_t subsequences;      /* speculative decode units                               */
    uint32_t sync_rounds;       /* fix-up rounds that ran until the relay reached a fixed point */
    uint32_t exact_samples;     /* IDCT samples re-evaluated on the exact (reference-order) path */
    float ms[KPEG_T_COUNT];     /* per-stage CUDA-event time, indexed by KPEG_T_* */
    float ms_total;             /* first to last event of the call */
    uint32_t kernel_launches;   /* kernels launched for this decode */
} kpeg_stats;

typedef struct kpeg_ctx kpeg_ctx;

/* Host-only: bytes of the decoded image of `plan` (its dimensions, components and KPEG_FLAG_SCALE_* bits); *w / *h (either
 * may be NULL) receive the output width and height.  0 for a NULL plan or one with a zero dimension or 2 components.  Every
 * "width*height*ncomp" below means this size when scale bits are set; a batch holds its images back to back at it. */
size_t kpeg_output_size(const kpeg_plan *plan, uint32_t *w, uint32_t *h);

/* ---- host-side container parse (no CUDA) --------------------------------------------------
 * Replaces JPEGDecoder::decodeImageFile's marker loop + parseSegmentInfo + the parse* members
 * (Decoder.cpp:53-75,90-152,164-530,579-619).  T.81-correct superset of what the reference
 * accepts: unknown APPn/COM are skipped by length, DRI and Nf==1 are honoured.  On success
 * [*scan_off, *scan_off + *scan_len) is the entropy-coded segment (what scanImageData,
 * Decoder.cpp:532-577, would read: everything after the SOS header up to the EOI marker). */
int kpeg_parse_jfif(const uint8_t *file, size_t len, kpeg_plan *plan, size_t *scan_off, size_t *scan_len);

/* A frame with one scan PER component (T.81 A.2.3; the reference reads such SOS headers, Decoder.cpp:461-530, and then
 * decodes the first scan as if it were interleaved).  One kpeg_scan per SOS: `plan` is everything needed to decode THAT
 * scan on its own -- ncomp = its number of components (1 for a non-interleaved scan, with that component's selectors in
 * slot 0), the tables and restart interval in force at its SOS (they may be redefined between scans, T.81 B.2.3) --
 * comp[] the frame component behind each slot, [off, off + len) its entropy-coded segment inside the file.
 * kpeg_parse_jfif_scans accepts what kpeg_parse_jfif accepts (then *nscans == 1 and scans[0].plan == *frame) plus
 * three-component frames coded as three single-component scans in any order; *frame then holds the dimensions and,
 * in slots 0..2, the quantisers of components 0..2 (frame->restart_interval is 0: it is a per-scan property). */
typedef struct kpeg_scan {
    kpeg_plan plan;
    uint8_t comp[3];
    size_t off, len;
} kpeg_scan;
#define KPEG_MAX_SCANS 3
int kpeg_parse_jfif_scans(const uint8_t *file, size_t len, kpeg_plan *frame, kpeg_scan *scans, int max_scans, int *nscans);

/* ---- context ------------------------------------------------------------------------------ */
/* One context per (thread, device): owns eight lanes (a CUDA stream with its own device scratch and pinned
 * bookkeeping each), all grown on demand and reused across decodes.  Not thread-safe; use one context per thread. */
int kpeg_cuda_create(int device, kpeg_ctx **out);
void kpeg_cuda_destroy(kpeg_ctx *ctx);
const char *kpeg_cuda_last_error(const kpeg_ctx *ctx); /* never NULL */
int kpeg_cuda_device_count(void);
int kpeg_cuda_set_profiling(kpeg_ctx *ctx, int on);
/* Tuning knobs of the speculative entropy decode (0 = leave unchanged): bits per subsequence (a power of two, 64..1024,
 * or $KPEG_SUB_BITS; -1 = back to the default: chosen per job, 1024 for streams with long restart segments AND long blocks --
 * large high-quality images without restart markers -- and 512 otherwise) and the number of relay rounds issued up front when the cooperative
 * loop is unavailable (>= 2; default 8 or $KPEG_RELAY_ROUNDS; more are added automatically when needed). */
int kpeg_cuda_set_tuning(kpeg_ctx *ctx, int sub_bits, int relay_rounds);
/* The CUDA stream (cudaStream_t) all of this context's work is issued on. */
void *kpeg_cuda_stream(kpeg_ctx *ctx);

/* A process-wide pool of idle contexts: acquire hands out one for `device` (creating it when the pool has none),
 * release puts it back with its scratch memory intact.  What kpeg::JPEGDecoder uses, so that decoding file after
 * file (reference main.cpp:54-79 constructs a decoder per file) does not pay context creation every time.
 * Thread-safe.  kpeg_cuda_pool_clear destroys the idle contexts. */
int kpeg_cuda_acquire(int device, kpeg_ctx **out);
void kpeg_cuda_release(int device, kpeg_ctx *ctx);
void kpeg_cuda_pool_clear(void);

/* Pinned host memory for scan / pixel buffers (plain malloc'd memory also works, slower); pinned for every device.
 * kpeg_cuda_host_register pins memory the caller already owns (a frame shared between processes, say). */
void *kpeg_cuda_host_alloc(size_t bytes);
void kpeg_cuda_host_free(void *p);
int kpeg_cuda_host_register(void *p, size_t bytes);
void kpeg_cuda_host_unregister(void *p);
/* Device memory helpers for callers that keep data resident (bench, pipelines). */
void *kpeg_cuda_device_alloc(kpeg_ctx *ctx, size_t bytes);
void kpeg_cuda_device_free(kpeg_ctx *ctx, void *p);
int kpeg_cuda_memcpy_h2d(kpeg_ctx *ctx, void *dst, const void *src, size_t bytes);
int kpeg_cuda_memcpy_d2h(kpeg_ctx *ctx, void *dst, const void *src, size_t bytes);

/* ---- the hot path ------------------------------------------------------------------------- */
/*
 * Decode one entropy-coded segment to pixels.  Replaces JPEGDecoder::byteStuffScanData,
 * decodeScanData (Decoder.cpp:621-855), MCU::constructMCU / computeIDCT / performLevelShift /
 * convertYCbCrToRGB (MCU.cpp:64-279) and Image::createImageFromMCUs (Image.cpp:20-86).
 *
 *  scan, scan_len : HOST pointer to the stuffed entropy-coded bytes (may contain RSTn markers).
 *  pixels_out     : HOST buffer of width*height*ncomp bytes (kpeg_output_size); interleaved R,G,B rows top-down for
 *                   ncomp==3 (the payload Image::dumpRawData writes, Image.cpp:129-135), one gray
 *                   byte per pixel for ncomp==1.
 * Synchronous: returns after the pixels are in pixels_out.  An image of 64 MB of pixels or more whose restart interval is
 * a whole number of MCU rows is cut into bands that run on the context's lanes with their copies overlapping
 * ($KPEG_BANDS, default 4; 1 = one job).
 */
int kpeg_cuda_decode(kpeg_ctx *ctx, const kpeg_plan *plan, const uint8_t *scan, size_t scan_len,
                     uint8_t *pixels_out, kpeg_stats *stats);

/* Same, but `d_scan` and `d_pixels_out` are DEVICE pointers on the context's device; work is
 * enqueued on the context's stream and the call returns after the stream has drained and the
 * device-side status word has been checked. */
int kpeg_cuda_decode_device(kpeg_ctx *ctx, const kpeg_plan *plan, const uint8_t *d_scan, size_t scan_len,
                            uint8_t *d_pixels_out, kpeg_stats *stats);

/*
 * Batch of n images that share ONE plan (same dimensions, tables and restart interval -- the
 * case of BASELINE.json configs 4 and of repeated frames).  The scans are decoded as one
 * concatenated stream whose image boundaries are treated like restart boundaries, so the whole
 * batch costs one kernel sequence.  Host-pointer variant copies in/out through pinned staging.
 */
int kpeg_cuda_decode_batch(kpeg_ctx *ctx, const kpeg_plan *plan, int n, const uint8_t *const *scans,
                           const size_t *scan_lens, uint8_t *const *pixels_out, kpeg_stats *stats);
/* Device-resident batch: d_scans is ONE device buffer holding the n scans back to back,
 * scan_offsets[n+1] (host array) delimit them; d_pixels_out receives n images back to back. */
int kpeg_cuda_decode_batch_device(kpeg_ctx *ctx, const kpeg_plan *plan, int n, const uint8_t *d_scans,
                                  const uint64_t *scan_offsets, uint8_t *d_pixels_out, kpeg_stats *stats);
/* "Packed" batch stream = the n stuffed scans back to back, each FOLLOWED by one 2-byte RSTn marker
 * (FF D0+(i&7)).  kpeg_batch_pack builds it on the host; the *_packed_device entry decodes such a
 * stream that is already resident in device memory (no copies at all inside the call). */
size_t kpeg_batch_packed_size(int n, const size_t *scan_lens);
int kpeg_batch_pack(int n, const uint8_t *const *scans, const size_t *scan_lens, uint8_t *dst, size_t cap);
int kpeg_cuda_decode_batch_packed_device(kpeg_ctx *ctx, const kpeg_plan *plan, int n, const uint8_t *d_packed,
                                         size_t packed_len, uint8_t *d_pixels_out, kpeg_stats *stats);
/* Same, given the offsets of the n scans inside the packed stream (packed_offsets[n] = its length): the
 * batch is cut into up to four parts that run as concurrent jobs on the context's lanes (streams). */
int kpeg_cuda_decode_batch_packed_device_split(kpeg_ctx *ctx, const kpeg_plan *plan, int n, const uint8_t *d_packed,
                                               const uint64_t *packed_offsets, uint8_t *d_pixels_out, kpeg_stats *stats);

/* Deferred form: enqueue the batch and return at once; kpeg_cuda_wait completes everything submitted since the
 * last wait and returns the first failure (stats: accumulated over those batches).  Consecutive submissions
 * overlap on the device.  d_packed / d_pixels_out must stay valid until kpeg_cuda_wait returns.  Any other
 * decode call on the context completes pending submissions first. */
int kpeg_cuda_submit_batch_packed_device(kpeg_ctx *ctx, const kpeg_plan *plan, int n, const uint8_t *d_packed,
                                         const uint64_t *packed_offsets, uint8_t *d_pixels_out);
int kpeg_cuda_wait(kpeg_ctx *ctx, kpeg_stats *stats);
/* Deferred form of kpeg_cuda_decode_batch (host buffers, ideally pinned, in and out): returns once the copies
 * and kernels are enqueued; the pixels are valid after kpeg_cuda_wait.  scans[i] / pixels_out[i] must stay
 * valid and untouched until then (the pointer arrays themselves are read before the call returns). */
int kpeg_cuda_submit_batch(kpeg_ctx *ctx, const kpeg_plan *plan, int n, const uint8_t *const *scans,
                           const size_t *scan_lens, uint8_t *const *pixels_out);

/* The scans kpeg_parse_jfif_scans found, decoded to one frame (HOST buffers in and out, synchronous).  One interleaved
 * scan is kpeg_cuda_decode; three single-component scans are entropy-decoded one after another, each with its own
 * tables, into per-component coefficient tiles, which one small kernel interleaves into the MCU order K3 consumes --
 * from there on (dequantisation, IDCT, colour, store: MCU.cpp:110-279, Image.cpp:51-70) the path is the same.
 * frame->flags selects the parity mode for every scan. */
int kpeg_cuda_decode_scans(kpeg_ctx *ctx, const kpeg_plan *frame, const kpeg_scan *scans, int nscans, const uint8_t *file,
                           size_t file_len, uint8_t *pixels_out, kpeg_stats *stats);

/* Whole-file convenience used by the JPEGDecoder drop-in: parse (kpeg_parse_jfif_scans) + decode (kpeg_cuda_decode_scans).
 * pixels_out must hold width*height*ncomp bytes (query with kpeg_parse_jfif_scans first) -- cap is checked. */
int kpeg_cuda_decode_file(kpeg_ctx *ctx, const uint8_t *file, size_t len, uint32_t flags, uint8_t *pixels_out,
                          size_t cap, kpeg_plan *plan_out, kpeg_stats *stats);

/* n whole files of ANY mix of dimensions, tables and codings (what "decode this directory" needs; the reference
 * constructs one JPEGDecoder per file, main.cpp:54-79).  Parsed on the host; files whose plans are identical are decoded
 * together as one batch (kpeg_cuda_submit_batch: one kernel sequence per group), files coded one scan per component go
 * through kpeg_cuda_decode_scans.  pixels_out[i] must hold caps[i] >= width*height*ncomp bytes of file i (query with
 * kpeg_parse_jfif_scans).  results[i] (may be NULL) receives file i's own return code, plans_out[i] (may be NULL) its
 * frame plan; a bad file does not stop the others.  Returns KPEG_OK when every file decoded, else the first failure
 * (text: kpeg_cuda_last_error).  Host buffers (ideally pinned) in and out; synchronous. */
int kpeg_cuda_decode_files(kpeg_ctx *ctx, int n, const uint8_t *const *files, const size_t *lens, uint32_t flags,
                           uint8_t *const *pixels_out, const size_t *caps, kpeg_plan *plans_out, int *results, kpeg_stats *stats);

/* ---- crop decode ------------------------------------------------------------------------------------------------------
 * A rectangle of the output image: x, y, width, height in pixels of the image the same call without a crop would produce
 * (the full image, or the reduced one with KPEG_FLAG_SCALE_* bits, as libjpeg crops its scaled output).  The result is
 * byte for byte that output's rows y .. y+height-1, columns x .. x+width-1, written tightly packed (rows of
 * width*ncomp bytes); in both parity modes, at every scale.  The rectangle is exact: it is not widened to MCU boundaries
 * (djpeg -crop is).  An empty rectangle, or one that reaches past the output image, returns KPEG_ERR_ARG before any work
 * is enqueued.  The whole stream is still entropy-decoded (where each block begins depends on every symbol before it),
 * so corruption anywhere in it is KPEG_ERR_STREAM; only the strips of 32 MCUs that hold pixels of the rectangle are
 * expanded and reconstructed, and only the rectangle's bytes are written and copied.  kpeg_stats.width / height report
 * the rectangle (a batch: the first image's).  After a crop decode kpeg_cuda_read_coefficients returns
 * KPEG_ERR_UNSUPPORTED until the next decode without a crop on the context.  There are no tiled, deferred or
 * multi-file crop forms. */
typedef struct kpeg_crop {
    uint32_t x, y, width, height;
} kpeg_crop;

/* kpeg_cuda_decode, cropped: pixels_out is a HOST buffer of crop->width*crop->height*ncomp bytes.  One job on the
 * context's first lane (never cut into bands). */
int kpeg_cuda_decode_crop(kpeg_ctx *ctx, const kpeg_plan *plan, const uint8_t *scan, size_t scan_len, const kpeg_crop *crop,
                          uint8_t *pixels_out, kpeg_stats *stats);
/* kpeg_cuda_decode_device, cropped: DEVICE pointers in and out. */
int kpeg_cuda_decode_crop_device(kpeg_ctx *ctx, const kpeg_plan *plan, const uint8_t *d_scan, size_t scan_len,
                                 const kpeg_crop *crop, uint8_t *d_pixels_out, kpeg_stats *stats);
/* kpeg_cuda_decode_batch, cropped: image i's rectangle is crops[i], pixels_out[i] holds
 * crops[i].width*crops[i].height*ncomp bytes.  One kernel sequence per chunk, as kpeg_cuda_decode_batch. */
int kpeg_cuda_decode_batch_crop(kpeg_ctx *ctx, const kpeg_plan *plan, int n, const uint8_t *const *scans,
                                const size_t *scan_lens, const kpeg_crop *crops, uint8_t *const *pixels_out, kpeg_stats *stats);
/* kpeg_cuda_decode_file, cropped (frames coded one scan per component too): cap is checked against the crop's bytes. */
int kpeg_cuda_decode_file_crop(kpeg_ctx *ctx, const uint8_t *file, size_t len, uint32_t flags, const kpeg_crop *crop,
                               uint8_t *pixels_out, size_t cap, kpeg_plan *plan_out, kpeg_stats *stats);

/* Parity hook: the quantised coefficients of the LAST decode on this context, as the reference
 * holds them transiently inside MCU::constructMCU (MCU.cpp:93-108): [block][64] int16, blocks
 * MCU-interleaved (Y,Cb,Cr per MCU), zig-zag order, DC prediction already integrated.
 * `cap` is in int16 elements.  (After a decode that ran as several jobs -- a large restart-marked image cut into bands,
 * a batch cut into chunks -- these are the coefficients of the job that finished last.) */
int kpeg_cuda_read_coefficients(kpeg_ctx *ctx, int16_t *out, size_t cap);

/* Host-only: cut one restart-marked scan into `parts` bands of whole MCU rows; band b is the byte
 * range scan[out_begin[b], out_end[b]) and decodes as an image of the same width and tables whose
 * MCU rows are [out_row[b], out_row[b+1]).  This is how restart-interval tiles of a very large image
 * are spread over several GPUs (one context per GPU, no device-to-device traffic; the reference has
 * no tiling).  Needs a restart interval that is a whole number of MCU rows or divides one.
 * out_begin / out_end have `parts` entries, out_row has parts + 1. */
int kpeg_split_restart_bands(const uint8_t *scan, size_t len, const kpeg_plan *plan, int parts, uint64_t *out_begin,
                             uint64_t *out_end, uint32_t *out_row);

/* Host-only: the same kind of bands, cut at BYTE positions instead of given rows: band b begins at the first RSTn marker
 * at or after b/parts of the scan, and its rows follow from the number of restart markers it holds (counted by one host
 * thread per band) -- no single walk over all markers of a large scan; the bands' heights depend on the data.  Needs a
 * restart interval of whole MCU rows and at least two intervals per band (else KPEG_ERR_UNSUPPORTED: use
 * kpeg_split_restart_bands).  Same outputs as kpeg_split_restart_bands. */
int kpeg_split_restart_bands_by_bytes(const uint8_t *scan, size_t len, const kpeg_plan *plan, int parts, uint64_t *out_begin,
                                      uint64_t *out_end, uint32_t *out_row);

/* ---- one image over several GPUs (kpeg_tiled.cpp) ---------------------------------------------------------
 * The restart-interval tiles of one very large image, one band of whole MCU rows per listed device (a device may be
 * listed more than once), each band decoded by its own GPU straight into its rows of the caller's frame
 * pixels_out (ideally pinned: kpeg_cuda_host_alloc) -- the frame Image::createImageFromMCUs assembles
 * (Image.cpp:51-70), gathered on the host with no device-to-device traffic.  One host thread and one pooled context
 * per device.  An image whose restart interval does not line up with MCU rows (or has none) does not shard: it is
 * decoded whole on devices[0].  Errors: the return code; text in kpeg_tiled_last_error (per calling thread). */
int kpeg_cuda_decode_tiled(const int *devices, int ndev, const kpeg_plan *plan, const uint8_t *scan, size_t scan_len,
                           uint8_t *pixels_out, kpeg_stats *stats);
int kpeg_cuda_decode_file_tiled(const int *devices, int ndev, const uint8_t *file, size_t len, uint32_t flags,
                                uint8_t *pixels_out, size_t cap, kpeg_plan *plan_out, kpeg_stats *stats);
/* Same, the frame assembled in DEVICE memory of dst_device (d_frame: kpeg_output_size bytes there): every band
 * travels by one peer copy over NVLink (staged by the driver where there is no peer access), so a consumer on
 * dst_device never pays PCIe. */
int kpeg_cuda_decode_tiled_device(const int *devices, int ndev, const kpeg_plan *plan, const uint8_t *scan, size_t scan_len,
                                  int dst_device, uint8_t *d_frame, kpeg_stats *stats);
const char *kpeg_tiled_last_error(void);
/* One band of such a decode: host scan in, pixels to device memory d_dst of dst_device (this context's own device:
 * written in place by the kernels). */
int kpeg_cuda_decode_to_peer(kpeg_ctx *ctx, const kpeg_plan *plan, const uint8_t *scan, size_t scan_len, int dst_device,
                             uint8_t *d_dst, kpeg_stats *stats);

/* ---- output formats written on the GPU ------------------------------------------------------------------------
 * The file Image::dumpRawData writes (Image.cpp:108-140: P6 header, then R,G,B rows) assembled in device memory:
 * d_out[*ppm_off, *ppm_off + *ppm_len) holds it (ppm_off < 16 keeps the payload aligned for the kernels' vector
 * stores; d_out must be 16-byte aligned, cap >= 176 + 3*width*height of the output size: with KPEG_FLAG_SCALE_* the header
 * carries the reduced dimensions).  One-component images come out as R = G = B. */
int kpeg_cuda_decode_ppm_device(kpeg_ctx *ctx, const kpeg_plan *plan, const uint8_t *d_scan, size_t scan_len, uint8_t *d_out,
                                size_t cap, size_t *ppm_off, size_t *ppm_len, kpeg_stats *stats);
/* Interleaved R,G,B (the decode output) -> three planes [3][npixels], both in device memory. */
int kpeg_cuda_interleaved_to_planar(kpeg_ctx *ctx, const uint8_t *d_rgb, uint8_t *d_planes, size_t npixels);

/* Exact bytes of the PPM header Image::dumpRawData writes (Image.cpp:124-127); returns length. */
int kpeg_ppm_header(int width, int height, char *buf, size_t cap);

/* ---- encode: pixels -> baseline JPEG on the GPU (csrc/encode.cu) ----------------------------------------------
 * Baseline sequential, 8-bit, one component or three (4:4:4, JFIF YCbCr), ITU-T T.81 Annex K quantisation tables
 * scaled by the IJG quality rule, Annex K Huffman tables, optional restart interval (DRI + RSTn).  The file is byte
 * for byte what the synthetic reference encoder writes for the same pixels (kpeg_synth_encode_pixels,
 * include/kpeg_synth.h, with KPEG_SYNTH_QUIRK_FREE when flags has KPEG_FLAG_REF_PARITY, and KPEG_SYNTH_EMIT_RESTART
 * when restart_interval > 0): segments in lena's order, double-precision colour transform and FDCT, lround(s / q)
 * clamped to +-2047 (DC) / +-1023 (AC), edges replicated to whole blocks, 1-bit padding before every marker.
 * KPEG_FLAG_REF_PARITY nudges DC values (by at most 2) so that no block has a DC difference of 0 and AC terms: the
 * reference decoder drops the AC terms of such blocks (SURVEY F1), so only such a stream decodes to the same pixels
 * in both decode modes and in the reference.  Without it the quantisation is plain T.81. */
typedef struct kpeg_encode_params {
    uint16_t width, height;     /* 1..65535 */
    uint8_t ncomp;              /* 1 (gray) or 3 (interleaved R,G,B in; Y,Cb,Cr coded) */
    uint8_t quality;            /* IJG 1..100, Annex K tables */
    uint16_t restart_interval;  /* MCUs, 0 = none (no DRI) */
    uint32_t flags;             /* KPEG_FLAG_REF_PARITY: stream safe for the reference's DC rule (SURVEY F1);
                                   KPEG_FLAG_OPTIMIZE_HUFFMAN: optimised Huffman tables (below) */
} kpeg_encode_params;

/* KPEG_FLAG_OPTIMIZE_HUFFMAN: the same quantised coefficients, coded with the optimal tables for this image's symbol
 * counts (DC and AC luma: component 0; DC and AC chroma: components 1 and 2; counted after the DC nudge and with the DC
 * prediction reset at restart boundaries, as the symbols are coded).  The tables follow T.81 K.2 and the K.3 length
 * limit with libjpeg's jpeg_gen_optimal_table rule (reserved symbol 256 of frequency 1; merge the two smallest non-zero
 * frequencies, on a tie the larger symbol; fold lengths over 16; HUFFVAL by (length, symbol)), with 64-bit frequencies
 * and no depth limit before the fold.  Same segment order; the file is byte for byte what kpeg_synth_encode_pixels
 * writes with KPEG_SYNTH_OPTIMIZE_HUFFMAN added.  The histogram and the tables are built on the GPU, and the DHT, DRI
 * and SOS segments are written there too, so the call still needs no host round trip before the copy-out. */

/* Host only: the largest file kpeg_cuda_encode can write for these parameters (0 for bad parameters).
 * Per block at most 22 DC bits + 63 x 26 AC bits = 1660 bits with the Annex K tables, 27 + 63 x 26 = 1665 bits with
 * KPEG_FLAG_OPTIMIZE_HUFFMAN:
 *  - DC: an 8-bit block's DC coefficient is (1/8) * the sum of its 64 level-shifted samples, in [-1024, 1016] for Y and
 *    [-1020, 1020] for Cb / Cr even with quantiser 1, and the nudge moves it by 1 at most when only the previous
 *    value is excluded (0 is excluded only at a segment's first MCU, where the prediction is 0 and |diff| <= 1025):
 *    |difference| <= 1017 + 1025 = 2042 < 2048, category <= 11; the longest Annex K DC code of category 11 is the
 *    chroma one, 11 bits: 11 + 11 = 22 bits.  An optimised code is at most 16 bits: 16 + 11 = 27 bits.
 *  - AC: every coefficient is clamped to +-1023, category <= 10, and the longest code is 16 bits (Annex K and
 *    optimised alike): a non-zero coefficient costs <= 26 bits; a ZRL (<= 16 bits) stands for 16 positions and EOB
 *    (<= 16 bits) for at least one, so no position costs more than 26 bits: 63 x 26.
 *  - Header: an optimised DHT never holds more symbols than the Annex K one (12 DC, 162 AC), so the Annex K header
 *    bounds both.
 * Segments are padded to whole bytes (one byte each at most), every byte may be FF and be followed by a stuffed 00
 * (x 2), and there is one 2-byte RSTn between segments and the 2-byte EOI: bound = header + 2 * (ceil(blocks * bits / 8)
 * + segments) + 2 * segments. */
size_t kpeg_encode_bound(const kpeg_encode_params *p);
/* Encode host pixels ([height][width][ncomp], top-down) into the host buffer jpeg_out.  Synchronous.  When the file
 * is larger than cap: KPEG_ERR_NOMEM, *jpeg_len = the size it needs, nothing written to jpeg_out.  Bad parameters or
 * NULL pointers: KPEG_ERR_ARG (checked before the context is used).  stats: width/height/ncomp, scan_bytes (stuffed
 * scan bytes written), unstuffed_bytes, segments, kernel_launches; with profiling on, ms_total and the stage times:
 * ms[KPEG_T_H2D] / ms[KPEG_T_D2H] the copies, ms[KPEG_T_IDCT] the FDCT + quantisation, ms[KPEG_T_DC_SCAN] the DC nudge,
 * ms[KPEG_T_ENTROPY_SCAN] the symbol histogram and table build (KPEG_FLAG_OPTIMIZE_HUFFMAN only),
 * ms[KPEG_T_ENTROPY_WRITE] bit lengths, offsets and code emission, ms[KPEG_T_UNSTUFF] byte stuffing and markers. */
int kpeg_cuda_encode(kpeg_ctx *ctx, const kpeg_encode_params *p, const uint8_t *pixels, uint8_t *jpeg_out, size_t cap,
                     size_t *jpeg_len, kpeg_stats *stats);
/* Same with DEVICE buffers on the context's device: the file is assembled in d_out (header copied in, the scan written
 * right after it by the kernels; with KPEG_FLAG_OPTIMIZE_HUFFMAN only the part up to SOF0 is copied in and the rest of
 * the header is written by the kernels too).  When it is larger than cap: KPEG_ERR_NOMEM, *jpeg_len = the size it needs, and no
 * byte at or past d_out + cap has been written. */
int kpeg_cuda_encode_device(kpeg_ctx *ctx, const kpeg_encode_params *p, const uint8_t *d_pixels, uint8_t *d_out, size_t cap,
                            size_t *jpeg_len, kpeg_stats *stats);

/* ---- lossless transcode: baseline JPEG -> baseline JPEG on the GPU (csrc/transcode.cu) ---------------------------
 * Re-codes the quantised coefficients of a whole baseline file (anything kpeg_parse_jfif_scans accepts: one or three
 * components, 4:4:4, any DQT / DHT ids and contents, any restart interval, APPn / COM segments, three-component frames
 * coded one scan per component) with other Huffman tables, another restart interval or one of the eight lossless
 * transforms below, without going through pixels (what jpegtran does).  The output holds the SAME quantised coefficients
 * in the T.81 sense (no SURVEY F1 rule), moved by the transform, in the encoder's layout, so that a file
 * kpeg_cuda_encode wrote comes back byte for byte unchanged:
 *   SOI, APP0 (JFIF 1.1); one DQT per quantiser id the components use, ascending, with the input's values (transposed,
 *   Q'[u][v] = Q[v][u], by the transposing transforms); SOF0 with the output size, component ids 1..nc, sampling 0x11 and
 *   the input's Tq per component; DHT (Annex K, or with KPEG_FLAG_OPTIMIZE_HUFFMAN the tables of kpeg_cuda_encode's
 *   rule; the luma pair for component 0, the chroma pair for 1 and 2); [DRI]; one interleaved SOS and the scan; EOI.
 * APPn and COM segments are not copied.  The output is always JFIF (the decoder reads every three-component file as
 * YCbCr).  It is byte for byte what kpeg_synth_encode_coefficients (include/kpeg_synth.h) writes for the input's T.81
 * coefficients after the transform.
 *
 * Transforms (numbered as libjpeg's JXFORM_CODE; u is the vertical frequency, v the horizontal one).  A transform whose
 * flip would move a partial edge block gives KPEG_ERR_UNSUPPORTED (jpegtran -perfect):
 *   NONE        W x H                                    FLIP_H    W x H, needs W % 8 == 0, negates odd v
 *   FLIP_V      W x H, needs H % 8 == 0, negates odd u   TRANSPOSE H x W, F'[u][v] = F[v][u]
 *   TRANSVERSE  H x W, needs W, H % 8 == 0               ROT90     H x W (clockwise: transpose, then flip-h), needs H % 8 == 0
 *   ROT180      W x H, needs W, H % 8 == 0               ROT270    H x W (transpose, then flip-v), needs W % 8 == 0
 * Range rules: every DC difference in the output's block order and segmentation must have category <= 11, and every AC
 * coefficient must be within +-1023; else KPEG_ERR_UNSUPPORTED.  Files of 8-bit encoders satisfy both; a crafted file
 * whose absolute DC drifts past 2047 may not once it is re-segmented or transformed.  Under these rules a block costs
 * at most kpeg_encode_bound's 1660 bits (1665 optimised).
 *
 * Note on SURVEY F1: the coefficient identity is a T.81 statement.  With the restart interval and the orientation
 * unchanged the DC differences are unchanged too, and the output then also decodes to the input's pixels under
 * KPEG_FLAG_REF_PARITY; otherwise it may not, because the reference's F1 rule depends on the DC differences. */
#define KPEG_XFORM_NONE 0u
#define KPEG_XFORM_FLIP_H 1u
#define KPEG_XFORM_FLIP_V 2u
#define KPEG_XFORM_TRANSPOSE 3u
#define KPEG_XFORM_TRANSVERSE 4u
#define KPEG_XFORM_ROT90 5u
#define KPEG_XFORM_ROT180 6u
#define KPEG_XFORM_ROT270 7u
#define KPEG_TRANSCODE_KEEP_RESTART (-1)
typedef struct kpeg_transcode_params {
    int32_t restart_interval; /* output MCUs per interval: -1 = the input's (its first scan's DRI), 0 = none, 1..65535 */
    uint32_t transform;       /* KPEG_XFORM_* */
    uint32_t flags;           /* 0 or KPEG_FLAG_OPTIMIZE_HUFFMAN; anything else is KPEG_ERR_ARG */
} kpeg_transcode_params;
/* Host only: the largest file kpeg_cuda_transcode can write for this input and these parameters (kpeg_encode_bound's
 * derivation with up to three DQT segments in the header); 0 for a file the parser rejects, bad parameters or a
 * transform whose precondition fails. */
size_t kpeg_transcode_bound(const uint8_t *file, size_t len, const kpeg_transcode_params *p);
/* Host buffers in and out, synchronous.  When the file is larger than cap: KPEG_ERR_NOMEM, *out_len = the size it needs,
 * nothing written to out.  Errors: KPEG_ERR_FORMAT / KPEG_ERR_UNSUPPORTED for what the parser or the decoder rejects,
 * KPEG_ERR_STREAM for corrupt entropy data, KPEG_ERR_UNSUPPORTED for the transform preconditions and the range rules,
 * KPEG_ERR_ARG for bad parameters.  stats: the decode's stage slots as a decode fills them, and the whole re-encode
 * (gather, table build, bit lengths, emission, stuffing) in ms[KPEG_T_IDCT], the slot of a decode's reconstruction;
 * width / height / ncomp, scan_bytes, unstuffed_bytes and segments describe the output, subsequences and sync_rounds the
 * input's decode, kernel_launches both. */
int kpeg_cuda_transcode(kpeg_ctx *ctx, const uint8_t *file, size_t len, const kpeg_transcode_params *p, uint8_t *out,
                        size_t cap, size_t *out_len, kpeg_stats *stats);

#ifdef __cplusplus
}
#endif
#endif
