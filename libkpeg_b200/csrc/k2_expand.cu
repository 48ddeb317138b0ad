// k2_expand.cu -- K2 of the B200 decode path: record expansion + DC prediction + the reference's DC-difference rule,
// one sm_100a kernel that turns K1's coefficient records into the coefficient tiles K3 consumes.
//
// What it replaces in the reference: MCU::constructMCU up to the dequantisation -- run-length expansion with the
// DC-difference quirk (src/MCU.cpp:93-104) and DC prediction (src/MCU.cpp:107-108).
//
// One CTA assembles the quantised coefficients of a strip of IDCT_MCUS_PER_CTA consecutive MCUs in shared memory and
// hands the finished tile to global memory with ONE bulk copy by the copy engine (cp.async.bulk.global.shared::cta,
// SASS UBLKCP).  The tile is written exactly as K3 wants it in ITS shared memory (16-bit values biased by COEF_BIAS,
// zig-zag order, 128-byte blocks with the 16-byte-chunk swizzle that makes K3's per-thread reads bank-conflict free), so
// K3 fetches it with one bulk copy in the other direction and no thread of either kernel spends an instruction on moving
// coefficients.
//
//   stage A  the strip's subsequences: strip_sub[] (which subsequence holds the strip's first slot), start_slot[] and
//            nrec[] come from the offset scan; empty tile
//   stage B  expansion.  Every record is (position, value) and self-contained, so the warps share the records k-major:
//            warp w takes records w*U .. w*U+U-1, then (w+NW)*U .., of 32 subsequences at a time -- a coalesced 128-byte
//            line per record index, all U loads in flight before the first value is used -- and drop the values into
//            the tile.  Kept deliberately light (about 40 registers, 12 KB of shared memory): the stage is a chain of
//            memory round trips, and what hides them is a dozen CTAs per SM.  (It used to be a stage of K3; there it
//            ran at K3's occupancy -- 80 registers, 8 CTAs of 3 warps -- and K3 spent half its time waiting on it.)
//   stage C  DC prediction: the predictors entering the strip = the predictors at the entry of the strip's first
//            subsequence (the offset scan's device-wide segmented prefix of the per-subsequence DC sums) + the DC
//            differences that subsequence decoded before the strip; a segmented warp scan over the strip's MCUs (reset
//            at restart intervals / image starts) does the rest.  Strips do not depend on one another.
//            Then MCU.cpp:97-104 (SURVEY F1): a block whose DC DIFFERENCE is 0 loses its AC terms.
//   stage D  tile -> global memory, one bulk copy
//
// All file:line citations are relative to /root/reference.
#include <cuda_runtime.h>
#include <stddef.h>
#include <stdint.h>

#include "entropy_core.h"
#include "kernels.cuh"
#include "kpeg_common.h"

namespace kpeg {

#ifndef KPEG_EXPAND_BATCH
#define KPEG_EXPAND_BATCH 16
#endif
constexpr int EXPAND_BATCH = KPEG_EXPAND_BATCH; // record loads in flight per lane
#ifndef KPEG_EXPAND_MIN_CTAS
#define KPEG_EXPAND_MIN_CTAS 12
#endif
constexpr int EXPAND_THREADS = 128;
#ifndef KPEG_EXPAND_PREFETCH_AHEAD
#define KPEG_EXPAND_PREFETCH_AHEAD 0
#endif
constexpr uint32_t EXPAND_PREFETCH_AHEAD = KPEG_EXPAND_PREFETCH_AHEAD; // strips ahead whose record lines are pulled into L2 (0 = off)
constexpr uint32_t EXPAND_PREFETCH_LINES = 112;                        // record indices per group of 32 subsequences
constexpr uint32_t BIAS2 = COEF_BIAS | (COEF_BIAS << 16);

__device__ __forceinline__ void st_shared_u16(uint32_t addr, uint32_t v)
{
    asm volatile("st.shared.u16 [%0], %1;" ::"r"(addr), "h"((uint16_t)v) : "memory");
}

template <int NC>
struct ExpandSmem {
    static constexpr int NB = IDCT_MCUS_PER_CTA * NC;
    uint4 coef[NB * 8]; // the tile image (coef_tile_byte)
    int32_t carry[4];   // DC predictors entering the strip
    uint32_t reset_slot; // slot of the last predictor restart at or before the strip's first MCU
    uint32_t mi0;        // MCU-in-image of the strip's first MCU
};

// LISTED (crop decode): CTA i expands strip a.strip_list[i]; the other strips' tiles are not written
template <int NC, bool LISTED>
__global__ void __launch_bounds__(EXPAND_THREADS, KPEG_EXPAND_MIN_CTAS) expand_kernel(ExpandArgs a)
{
    constexpr int NM = IDCT_MCUS_PER_CTA;
    constexpr int NB = NM * NC;
    constexpr int NW = EXPAND_THREADS / 32;
    constexpr uint32_t TILE_SLOTS = NB * 64u;
    __shared__ __align__(128) ExpandSmem<NC> sm;

    const int t = threadIdx.x;
    const uint32_t warp = (uint32_t)t >> 5, lane = (uint32_t)t & 31u;
    const uint32_t strip = LISTED ? __ldg(a.strip_list + blockIdx.x) : blockIdx.x;
    const uint32_t mcu0 = strip * NM, blk0 = mcu0 * NC;
    const uint32_t total_mcus = a.g.nimages * a.g.mcus_per_image;
    const uint32_t s0 = blk0 * 64u; // first slot of the strip; slots are < 2^32 (host_tables.h)

    // ---- stage A ---------------------------------------------------------------------------------------
    const uint32_t nsub = a.meta->nsub;
    const uint32_t first0 = min(__ldg(a.strip_sub + strip), nsub - 1u);
    const bool prefetch = LISTED ? blockIdx.x + EXPAND_PREFETCH_AHEAD < a.nlisted : strip + EXPAND_PREFETCH_AHEAD < a.nstrips;
    if (EXPAND_PREFETCH_AHEAD != 0u && prefetch) {
        // the record lines a strip that starts about one CTA lifetime from now will read: DRAM -> L2 now, so that its
        // batches wait for L2, not for DRAM.  (Which strip that is need not be exact.)
        const uint32_t ahead = LISTED ? __ldg(a.strip_list + blockIdx.x + EXPAND_PREFETCH_AHEAD) : strip + EXPAND_PREFETCH_AHEAD;
        const uint32_t fs = min(__ldg(a.strip_sub + ahead), nsub - 1u);
        const char *g0 = reinterpret_cast<const char *>(a.rec + ((size_t)(fs >> 5) * a.rec_kmax) * 32u);
        const uint32_t lines = min(a.rec_kmax, EXPAND_PREFETCH_LINES);
        for (uint32_t k = (uint32_t)t; k < 2u * lines; k += EXPAND_THREADS) {
            const uint32_t grp = k >= lines ? 1u : 0u; // the strip's subsequences usually straddle two groups of 32
            asm volatile("prefetch.global.L2 [%0];" ::"l"(g0 + ((size_t)grp * a.rec_kmax + (k - grp * lines)) * 128u));
        }
    }
    for (int i = t; i < NB * 8; i += EXPAND_THREADS)
        sm.coef[i] = make_uint4(BIAS2, BIAS2, BIAS2, BIAS2);
    if (t == 0) {
        const uint32_t img = mcu0 / a.g.mcus_per_image, mi = mcu0 - img * a.g.mcus_per_image;
        sm.mi0 = mi;
        // predictors restart at every restart interval and image (T.81 F.2.1.3.1)
        const uint32_t mreset = a.g.restart_interval ? mi - mi % a.g.restart_interval : 0u;
        sm.reset_slot = (img * a.g.mcus_per_image + mreset) * (uint32_t)NC * 64u;
        sm.carry[0] = sm.carry[1] = sm.carry[2] = 0;
    }
    __syncthreads();
    const uint32_t tile_addr = (uint32_t)__cvta_generic_to_shared(sm.coef);

    // ---- stage B: expansion of the records that fall into the strip ---------------------------------------
    // 32 subsequences at a time, one per lane -- or, with subsequences of 1024 bits (a strip then meets only ~14 of
    // them: more than half of the lanes would idle), 16 at a time with TWO lanes per subsequence, one taking its even
    // records, the other the odd ones.
    const bool pair = a.g.sub_bits >= 1024u;
    const uint32_t per_chunk = pair ? 16u : 32u, half = pair ? lane >> 4 : 0u, kstep = pair ? 2u : 1u;
    uint32_t first = first0;
    for (int chunk = 0; chunk < 256; ++chunk, first += per_chunk) { // a strip meets at most ~3 100 subsequences
        const uint32_t sub = first + (pair ? lane & 15u : lane);
        bool act = sub < nsub;
        const uint32_t ss = act ? __ldg(a.start_slot + sub) : 0xFFFFFFFFu;
        const uint32_t nr = act ? __ldg(a.nrec + sub) : 0u; // together with start_slot: one round trip, not two
        // the first subsequence begins at or before the strip's first slot, the others inside the strip -- or beyond it
        act = act && (ss <= s0 || ss - s0 < TILE_SLOTS);
        uint32_t n = 0, stride = 128u;
        const uint32_t *base = a.rec;
        if (act) {
            n = min(nr & 1023u, a.rec_kmax);
            if (nr >> 10) { // redone in a sparse relay round: private contiguous area
                base = a.rec_alt + (size_t)((nr >> 10) - 1u) * a.rec_kmax;
                stride = 4u;
            } else {
                base = a.rec + ((size_t)(sub >> 5) * a.rec_kmax) * 32u + (sub & 31u);
            }
        }
        // slot of record position 0 relative to the tile (may be "negative"); lanes without a subsequence get an
        // offset that keeps the out-of-range marker of the batched loads below out of range
        const uint32_t off0 = act ? (ss & ~63u) - s0 : TILE_SLOTS;
        // records this lane takes: all of them, or every other one starting at `half`
        const uint32_t mine = pair ? (n + 1u - half) >> 1 : n;
        const uint32_t nmax = __reduce_max_sync(0xffffffffu, mine);
        // A record index beyond the lane's count reads as position 0xFFFF, which falls outside every tile.
        const size_t rstride = (size_t)stride * kstep; // bytes between two records of this lane
        const char *bp = reinterpret_cast<const char *>(base) + (size_t)half * stride + (size_t)(warp * EXPAND_BATCH) * rstride;
        const size_t step = (size_t)(NW * EXPAND_BATCH) * rstride;
        for (uint32_t k0 = warp * EXPAND_BATCH; k0 < nmax; k0 += NW * EXPAND_BATCH, bp += step) {
            uint32_t r[EXPAND_BATCH];
#pragma unroll
            for (int u = 0; u < EXPAND_BATCH; ++u)
                r[u] = k0 + (uint32_t)u < mine ? __ldg(reinterpret_cast<const uint32_t *>(bp + (size_t)u * rstride)) : 0xFFFFFFFFu;
#pragma unroll
            for (int u = 0; u < EXPAND_BATCH; ++u) {
                const uint32_t off = off0 + record_pos(r[u]);
                if (off < TILE_SLOTS)
                    st_shared_u16(tile_addr + coef_tile_byte(off), r[u]);
            }
        }
        // the next subsequences matter only if the last one of these still begins inside the strip
        if (!__shfl_sync(0xffffffffu, act && sub + 1u < nsub ? 1 : 0, 31))
            break;
    }
    // ---- DC predictors entering the strip ------------------------------------------------------------------
    // = the predictors at the entry of the subsequence the strip's first slot lies in (from the offset scan, unless
    // they restart between that entry and the strip) + the DC differences that subsequence decoded before the strip
    // (its records at slot 0 of a block, between the last restart and the strip's first slot).  The last warp, lanes
    // over the records of that one subsequence; the lines were just read by the loop above.
    if (warp == NW - 1) {
        const uint32_t ss = __ldg(a.start_slot + first0);
        const uint32_t reset_slot = sm.reset_slot;
        int part[3] = {0, 0, 0};
        if (ss < s0 && reset_slot < s0) {
            const uint32_t nr = __ldg(a.nrec + first0);
            const uint32_t n = min(nr & 1023u, a.rec_kmax);
            const uint32_t *base = (nr >> 10) ? a.rec_alt + (size_t)((nr >> 10) - 1u) * a.rec_kmax
                                              : a.rec + ((size_t)(first0 >> 5) * a.rec_kmax) * 32u + (first0 & 31u);
            const uint32_t stride = (nr >> 10) ? 1u : 32u; // in records
            const uint32_t entry = ss & ~63u;
            for (uint32_t k = lane; k < n; k += 32u) {
                const uint32_t r = __ldg(base + (size_t)k * stride);
                const uint32_t at = entry + record_pos(r);
                if ((at & 63u) == 0u && at < s0 && at >= reset_slot) {
                    const uint32_t c = NC == 3 ? (at >> 6) % 3u : 0u;
                    const int v = record_value(r);
                    part[0] += c == 0u ? v : 0;
                    part[1] += c == 1u ? v : 0;
                    part[2] += c == 2u ? v : 0;
                }
            }
        }
#pragma unroll
        for (int c = 0; c < 3; ++c)
            part[c] = __reduce_add_sync(0xffffffffu, part[c]);
        if (lane == 0) {
            int pre[3] = {0, 0, 0};
            // no restart between the subsequence's entry and the strip.  An entry ON the restart slot (ss == reset_slot)
            // starts from zero: either the boundary was crossed at the very end of the subsequence before (its sums
            // are zero anyway) or the subsequence is entered in the padding bits BEFORE the boundary, and the prefix
            // it was handed still belongs to the interval that is ending
            if (ss > reset_slot && reset_slot < s0)
                dcs_unpack(a.dcpre[first0], pre);
            sm.carry[0] = pre[0] + part[0];
            sm.carry[1] = pre[1] + part[1];
            sm.carry[2] = pre[2] + part[2];
        }
    }
    __syncthreads();

    // ---- stage C: DC prediction, one thread per block (warp = component, lane = MCU) -------------------------
    if (t < NB) {
        const uint32_t comp = warp, ml = lane;
        const uint32_t bl = ml * NC + comp;
        const bool active = mcu0 + ml < total_mcus;
        const uint32_t dc_addr = tile_addr + bl * 128u + ((bl & 7u) << 4); // slot 0: chunk 0 of the block
        const uint32_t dcw = sm.coef[bl * 8u + (bl & 7u)].x;
        const int dcdiff = active ? (int)(dcw & 0xFFFFu) - (int)COEF_BIAS : 0;
        bool reset = false;
        if (active) {
            uint32_t mi = sm.mi0 + ml;
            if (mi >= a.g.mcus_per_image)
                mi %= a.g.mcus_per_image;
            reset = a.g.restart_interval ? (mi % a.g.restart_interval) == 0u : mi == 0u;
        }
        int v = dcdiff;
        uint32_t f = reset ? 1u : 0u;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const int ov = __shfl_up_sync(0xffffffffu, v, d);
            const uint32_t of = __shfl_up_sync(0xffffffffu, f, d);
            if ((int)ml >= d) {
                v = f ? v : v + ov;
                f |= of;
            }
        }
        const int dcv = (int)(short)(v + (f ? 0 : sm.carry[comp]));
        if (active) {
            if ((a.g.flags & 1u) && dcdiff == 0) { // MCU.cpp:97-104: the block keeps its DC value only
                sm.coef[bl * 8u + (bl & 7u)] = make_uint4((((uint32_t)dcv + COEF_BIAS) & 0xFFFFu) | (COEF_BIAS << 16), BIAS2, BIAS2, BIAS2);
#pragma unroll
                for (uint32_t k = 1; k < 8; ++k)
                    sm.coef[bl * 8u + (k ^ (bl & 7u))] = make_uint4(BIAS2, BIAS2, BIAS2, BIAS2);
            } else {
                st_shared_u16(dc_addr, (uint32_t)dcv + COEF_BIAS);
            }
        }
    }
    __syncthreads();

    // ---- stage D: the tile leaves by the copy engine ---------------------------------------------------------
    if (t == 0) {
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); // the threads' stores, before the bulk copy reads them
        char *dst = reinterpret_cast<char *>(a.tiles) + (size_t)strip * (NB * 128u);
        asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(dst), "r"(tile_addr), "r"((uint32_t)(NB * 128)) : "memory");
        asm volatile("cp.async.bulk.commit_group;" ::: "memory");
        asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); // shared memory may go once it has been read
    }
}

// ---- fallback: plain coefficient matrix -> tile images ---------------------------------------------------------
// Behind the Huffman final pass only (entropy_write leaves [block][64] int16 with the DC difference in slot 0, and
// dc_integrate_kernel the predicted DC values): apply the DC value and the F1 rule, bias, swizzle.  One thread per
// 16-byte chunk.
__global__ void __launch_bounds__(256) tiles_from_matrix_kernel(JobGeom g, const int16_t *coef, const int16_t *dc, uint4 *tiles,
                                                                uint32_t padded_blocks)
{
    const uint32_t i = blockIdx.x * 256u + threadIdx.x; // chunk index
    const uint32_t b = i >> 3, k = i & 7u;
    if (b >= padded_blocks)
        return;
    uint4 v = make_uint4(0, 0, 0, 0);
    if (b < g.total_blocks) {
        v = __ldg(reinterpret_cast<const uint4 *>(coef) + i);
        const int dcdiff = (int)__ldg(coef + (size_t)b * 64u);
        if ((g.flags & 1u) && dcdiff == 0)
            v = make_uint4(0, 0, 0, 0);
        if (k == 0u)
            v.x = (v.x & 0xFFFF0000u) | ((uint32_t)(uint16_t)__ldg(dc + b));
    }
    tiles[coef_tile_chunk(b, k)] = make_uint4(v.x ^ BIAS2, v.y ^ BIAS2, v.z ^ BIAS2, v.w ^ BIAS2);
}

// parity hook: tile images -> plain [block][64] int16 (what kpeg_cuda_read_coefficients returns)
__global__ void __launch_bounds__(256) matrix_from_tiles_kernel(const uint4 *tiles, uint4 *coef, uint32_t total_blocks)
{
    const uint32_t i = blockIdx.x * 256u + threadIdx.x;
    const uint32_t b = i >> 3, k = i & 7u;
    if (b >= total_blocks)
        return;
    const uint4 v = __ldg(tiles + coef_tile_chunk(b, k));
    coef[i] = make_uint4(v.x ^ BIAS2, v.y ^ BIAS2, v.z ^ BIAS2, v.w ^ BIAS2);
}

// ---- one scan per component (T.81 A.2.3) --------------------------------------------------------------------
// Every component was entropy-decoded as a one-component image of its own: its tiles hold block m of the component at
// block position m.  K3 wants the blocks of an MCU side by side (block m * 3 + c): one thread per 16-byte chunk.
__global__ void __launch_bounds__(256) interleave_tiles_kernel(const uint4 *t0, const uint4 *t1, const uint4 *t2, uint4 *out,
                                                               uint32_t nmcu_padded)
{
    const uint32_t i = blockIdx.x * 256u + threadIdx.x; // chunk index in the interleaved tiles
    const uint32_t gb = i >> 3, k = i & 7u;
    const uint32_t m = gb / 3u, c = gb - m * 3u;
    if (m >= nmcu_padded)
        return;
    const uint4 *src = c == 0u ? t0 : (c == 1u ? t1 : t2);
    out[coef_tile_chunk(gb, k)] = __ldg(src + coef_tile_chunk(m, k));
}

void launch_interleave_tiles(const void *t0, const void *t1, const void *t2, void *out, uint32_t nmcu_padded, cudaStream_t s,
                             uint32_t *launches)
{
    const uint32_t chunks = nmcu_padded * 3u * 8u;
    interleave_tiles_kernel<<<(chunks + 255u) / 256u, 256, 0, s>>>(reinterpret_cast<const uint4 *>(t0), reinterpret_cast<const uint4 *>(t1),
                                                                   reinterpret_cast<const uint4 *>(t2), reinterpret_cast<uint4 *>(out), nmcu_padded);
    ++*launches;
}

void launch_expand(const ExpandArgs &a, cudaStream_t s, uint32_t *launches)
{
    const uint32_t total_mcus = a.g.nimages * a.g.mcus_per_image;
    const uint32_t grid = (total_mcus + IDCT_MCUS_PER_CTA - 1) / IDCT_MCUS_PER_CTA;
    if (a.strip_list) {
        if (a.g.ncomp == 3)
            expand_kernel<3, true><<<a.nlisted, EXPAND_THREADS, 0, s>>>(a);
        else
            expand_kernel<1, true><<<a.nlisted, EXPAND_THREADS, 0, s>>>(a);
    } else if (a.g.ncomp == 3) {
        expand_kernel<3, false><<<grid, EXPAND_THREADS, 0, s>>>(a);
    } else {
        expand_kernel<1, false><<<grid, EXPAND_THREADS, 0, s>>>(a);
    }
    ++*launches;
}

void launch_tiles_from_matrix(const JobGeom &g, const int16_t *coef, const int16_t *dc, void *tiles, cudaStream_t s, uint32_t *launches)
{
    const uint32_t per = (uint32_t)IDCT_MCUS_PER_CTA * g.ncomp;
    const uint32_t padded = (g.total_blocks + per - 1u) / per * per;
    tiles_from_matrix_kernel<<<(padded * 8u + 255u) / 256u, 256, 0, s>>>(g, coef, dc, reinterpret_cast<uint4 *>(tiles), padded);
    ++*launches;
}

void launch_matrix_from_tiles(const void *tiles, int16_t *coef, uint32_t total_blocks, cudaStream_t s)
{
    matrix_from_tiles_kernel<<<(total_blocks * 8u + 255u) / 256u, 256, 0, s>>>(reinterpret_cast<const uint4 *>(tiles),
                                                                               reinterpret_cast<uint4 *>(coef), total_blocks);
}

} // namespace kpeg
