// kernels.cuh -- launch-side declarations of the sm_100a kernels (definitions in kernels.cu).
#ifndef KPEG_KERNELS_CUH
#define KPEG_KERNELS_CUH

#include <cuda_runtime.h>

#include "crop_geom.h"
#include "kpeg_common.h"

namespace kpeg {

constexpr int MAX_RELAY_ROUNDS = 64; // slots in DevMeta::changed

// DevMeta::changed slot of relay round r (r >= 1).  Rounds beyond the array reuse slots 2..63 (the
// host zeroes a slot before reusing it); 62 is even, so slot parity == round parity, which is what
// selects the ping-pong work list.
inline int relay_slot(int r) { return r < MAX_RELAY_ROUNDS ? r : 2 + ((r - 2) % (MAX_RELAY_ROUNDS - 2)); }

// Device-resident bookkeeping of one job; zeroed before every decode, read back once at the end.
struct DevMeta {
    uint32_t total_kept;   // unstuffed bytes
    uint32_t total_rst;    // RSTn markers found
    uint32_t total_bits;   // 8 * total_kept
    uint32_t nsub;         // subsequences actually used
    uint32_t status;       // ST_* bits
    uint32_t exact_samples; // IDCT samples re-evaluated in the reference's operation order (statistics)
    uint32_t colour_exact; // pixels whose colour took the double expression (statistics)
    uint32_t final_slot;   // absolute slot the last subsequence ended on
    uint32_t reserved_[2];
    uint32_t relay_rounds; // last relay round that ran (device-side round loop)
    uint32_t grid_bar;     // arrival counter of the relay loop's grid barrier
    uint32_t rec_alt_count; // private record areas handed out by the sparse relay rounds
    uint32_t changed[MAX_RELAY_ROUNDS];
};

struct UnstuffArgs {
    const uint8_t *scan; // stuffed entropy-coded bytes (device)
    uint32_t scan_len;
    uint32_t ntiles;
    uint32_t *tile_kept, *tile_rst;      // per-tile counts, then (after the scan kernel) exclusive offsets
    uint32_t *cls;                       // [ntiles * UNSTUFF_THREADS] per 16-byte chunk: keep mask | RSTn mask << 16
    uint8_t *words;                      // unstuffed stream as big-endian 32-bit words (byte address ^ 3)
    uint32_t *seg_bit;                   // [nseg + 2]
    uint32_t nseg;                       // expected number of segments
    DevMeta *meta;
};

constexpr int UNSTUFF_THREADS = 256;
constexpr int UNSTUFF_BYTES_PER_THREAD = 16;
constexpr int UNSTUFF_TILE = UNSTUFF_THREADS * UNSTUFF_BYTES_PER_THREAD;

struct EntropyArgs {
    const uint32_t *words;
    const uint32_t *seg_bit;
    const DeviceTables *tables;
    DevMeta *meta;
    SubState *state;      // [nsub_max] relay states X[i]
    uint32_t *worklist[2]; // [nsub_max] each: subsequences whose input changed in the previous relay round
    uint32_t *seg_hint;   // [nsub_max]
    uint32_t *start_slot; // [nsub_max] absolute slot at the entry of subsequence i
    uint2 *scan_tiles;    // [ceil(nsub_max / 1024)] per-tile aggregates / carries of the offset scan
    long long *scan_tiles_dcs; // the same for the packed DC sums
    long long *dcs;       // [nsub_max] packed sums of the DC differences each subsequence decoded (entropy_core.h, dcs_unpack)
    long long *dcpre;     // [nsub_max] ... scanned: the DC predictor values at the entry of every subsequence
    uint32_t *rec;        // symbol records, [group of 32 subsequences][rec_kmax][32] (nullptr = records off)
    uint32_t *nrec;       // [nsub_max] records per subsequence | (private area index + 1) << 10
    uint32_t *rec_alt;    // [rec_alt_cap][rec_kmax] private record areas of subsequences redone in sparse rounds
    uint32_t rec_alt_cap;
    uint32_t rec_kmax;
    int16_t *coef;        // [total_blocks][64]  (Huffman final pass only: records off)
    int16_t *dcdiff;      // [total_blocks]      (Huffman final pass only)
    uint32_t *strip_sub;  // [nstrips] subsequence in which the first slot of every K3 strip lies (written by the offset scan)
    uint32_t strip_slots; // coefficient slots per strip
    uint32_t nstrips;
    uint32_t nsub_max;
    JobGeom g;
};

constexpr int ENTROPY_THREADS = 128;

// ---- coefficient tiles: what K2 hands to K3 ------------------------------------------------------------------
// The quantised coefficients of a strip of IDCT_MCUS_PER_CTA consecutive MCUs (MCU-interleaved blocks: Y,Cb,Cr per
// MCU), DC prediction and the reference's DC-difference rule already applied, stored as the IMAGE OF K3's SHARED-MEMORY
// TILE: 16-bit values biased by COEF_BIAS (an empty slot is 0x8000), zig-zag order, one 128-byte line per block, and
// inside the line the 16-byte chunk k of block b at chunk position k ^ (b & 7).  Strips are whole multiples of eight
// blocks, so the swizzle is the same whether b counts from the strip or from the job.  K2 writes a tile with one bulk
// copy out of its shared memory, K3 reads it with one bulk copy into its own.
constexpr int IDCT_MCUS_PER_CTA = 32;
KPEG_HD uint32_t coef_tile_chunk(uint32_t block, uint32_t k) { return block * 8u + (k ^ (block & 7u)); } // in 16-byte chunks
KPEG_HD uint32_t coef_tile_byte(uint32_t slot) { return (slot * 2u) ^ ((slot >> 2) & 0x70u); }           // slot = block * 64 + zig-zag index

// K2 (k2_expand.cu): record expansion + DC prediction -> coefficient tiles
struct ExpandArgs {
    const uint32_t *rec;      // [group of 32 subsequences][rec_kmax][32]
    const uint32_t *nrec;     // [nsub]
    const uint32_t *rec_alt;  // private record areas (subsequences redone in sparse relay rounds)
    uint32_t rec_kmax;
    const uint32_t *start_slot; // [nsub]
    const uint32_t *strip_sub;  // [nstrips]
    const long long *dcpre;   // [nsub] packed DC predictor values at the entry of every subsequence (offset scan)
    void *tiles;              // [nstrips] tile images
    uint32_t nstrips;
    DevMeta *meta;
    JobGeom g;
    const uint32_t *strip_list; // crop decode: the strips to expand, sorted (nlisted of them); nullptr: every strip
    uint32_t nlisted;
};

// K3 (k3_fused.cu): dequantise + de-zigzag + IDCT + level shift + colour + store, from the coefficient tiles
struct IdctArgs {
    const void *tiles;        // [nstrips] tile images (K2, or tiles_from_matrix after the Huffman final pass)
    uint32_t nstrips;
    const DeviceTables *tables;
    uint8_t *pixels;          // [nimages][height][width][ncomp]
    uint4 *tie_rec;           // [nstrips][IDCT_TIE_LIST_CAP] records of the pixels inside the tie band (k3_fused.cu)
    uint32_t *tie_cnt;        // [nstrips] entries in use
    DevMeta *meta;
    JobGeom g;
};
constexpr int IDCT_TIE_LIST_CAP = 96; // a strip with more ties than this resolves them inside K3

// K3 of a crop decode (crop_geom.h): only the listed strips are reconstructed, and every store goes through crop[image].
// The kernels of a whole-image decode take the plain IdctArgs, so their code is the same as without crop decodes.
struct IdctCropArgs : IdctArgs {
    const uint32_t *strip_list = nullptr; // [nlisted], sorted
    uint32_t nlisted = 0;
    const CropWin *crop = nullptr;        // [nimages]; nullptr: no crop, every strip
};


void kernels_context_created();   // contexts of this process share the device: the cooperative relay loops of
void kernels_context_destroyed(); // all of them together must stay co-resident
void kernels_configure(int max_concurrent_jobs); // jobs (lanes) that may be on the device at the same time // per-device function attributes (call once after cudaSetDevice)
void launch_repack_scans(const uint8_t *stage, uint8_t *scan, const uint64_t *ends, uint32_t n, cudaStream_t s); // contiguous host scans -> packed batch
void launch_write_separators(uint8_t *scan, const uint64_t *ends, uint32_t n, cudaStream_t s); // RSTn after every scan of a packed batch
void launch_count_restart_markers(const uint8_t *scan, uint32_t len, uint32_t *count, cudaStream_t s); // *count += RSTn markers in scan[0, len)
void launch_gray_to_rgb(const uint8_t *gray, uint8_t *rgb, size_t npixels, cudaStream_t s);     // PPM payload of a one-component image
void launch_rgb_to_planar(const uint8_t *rgb, uint8_t *planes, size_t npixels, cudaStream_t s); // [3][H][W] planes
void launch_unstuff(const UnstuffArgs &a, uint32_t sub_bits, cudaStream_t s, uint32_t *launches);
void launch_entropy_cold(const EntropyArgs &a, cudaStream_t s, uint32_t *launches);
void launch_entropy_relay(const EntropyArgs &a, int round, cudaStream_t s, uint32_t *launches);
// rounds first..last (first >= 2) in ONE cooperative launch: a device-side loop with a grid barrier
// between rounds, stopping early at the fixed point; DevMeta::relay_rounds = last round that ran
// fails (nothing launched) when the driver refuses the cooperative launch; the caller then issues the rounds one by one
cudaError_t launch_entropy_relay_loop(const EntropyArgs &a, int first, int last, cudaStream_t s, uint32_t *launches);
void launch_entropy_scan(const EntropyArgs &a, cudaStream_t s, uint32_t *launches);
void launch_entropy_write(const EntropyArgs &a, cudaStream_t s, uint32_t *launches);  // Huffman final pass
// fallback only: DC prediction over the DC differences the Huffman final pass left (dcdiff -> dc), one CTA per restart segment
void launch_dc_integrate(const JobGeom &g, const int16_t *dcdiff, int16_t *dc, cudaStream_t s, uint32_t *launches);
void launch_expand(const ExpandArgs &a, cudaStream_t s, uint32_t *launches); // K2
// fallback (after the Huffman final pass + dc_integrate): plain coefficient matrix -> tile images
void launch_tiles_from_matrix(const JobGeom &g, const int16_t *coef, const int16_t *dc, void *tiles, cudaStream_t s, uint32_t *launches);
void launch_matrix_from_tiles(const void *tiles, int16_t *coef, uint32_t total_blocks, cudaStream_t s); // parity hook
// three one-component tile sets (one scan per component) -> the MCU-interleaved tiles K3 consumes
void launch_interleave_tiles(const void *t0, const void *t1, const void *t2, void *out, uint32_t nmcu_padded, cudaStream_t s,
                             uint32_t *launches);
// K3, or -- when a.g.flags has KPEG_FLAG_SCALE_* bits -- the reduced-size reconstruction (k3_scaled.cu) in its place
cudaError_t launch_idct(const IdctCropArgs &a, cudaStream_t s, uint32_t *launches);
cudaError_t launch_idct_scaled(const IdctCropArgs &a, cudaStream_t s, uint32_t *launches);
void k3_configure();                      // function attributes of the K3 kernels (called by kernels_configure)
uint32_t k3_strip_slots(uint32_t ncomp);  // coefficient slots one K3 strip covers

} // namespace kpeg
#endif
