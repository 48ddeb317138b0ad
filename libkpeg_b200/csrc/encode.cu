// encode.cu -- sm_100a kernels of the baseline-JPEG encoder (C ABI: kpeg_cuda_encode*, kpeg_cuda.cu).
//
//   E1 enc_fdct_kernel     pixels -> level shift / colour transform -> 8x8 FDCT (FP64) -> quantised zig-zag int16
//   E2 DC nudge            KPEG_FLAG_REF_PARITY only: the synth's DC chain as a scan of 5-state maps (encode_core.h)
//   EH enc_hist_kernel     KPEG_FLAG_OPTIMIZE_HUFFMAN only: symbol counts per table (the walk E3 and E4 code)
//   EB enc_huff_build_kernel  KPEG_FLAG_OPTIMIZE_HUFFMAN only: one warp per table turns the counts into BITS / HUFFVAL
//                          (huff_opt.h), codes into this encode's copy of the tables, and DHT [DRI] SOS into the file
//   E3 bit lengths         per block, then a 64-bit exclusive scan (bit offsets) and a scan of the segments'
//                          byte-padded lengths
//   E4 enc_emit_kernel     every block writes its codes at its bit offset into a zeroed big-endian word stream
//   E5 stuffing            FF counts per tile, their scan, then the stream with 00 after every FF, RSTn between
//                          segments and EOI at the end, straight into the caller's buffer after the header
//
// Everything after E3's scans sizes itself from device memory (the stream length is not known on the host, nor, in
// optimised mode, the header length), with grid-stride loops over a grid sized for the worst-case stream, so one
// encode needs no host round trip.
#include <cuda_runtime.h>

#include <algorithm>

#include "encode.cuh"
#include "huff_opt.h"
#include "kpeg_cuda.h"

namespace kpeg {
namespace enc {
namespace {

constexpr int THREADS = 256;
constexpr int ITEMS = 8;
constexpr uint64_t SCAN_TILE = (uint64_t)THREADS * ITEMS;
constexpr int FDCT_MCUS = 8; // MCUs (one 64x8 pixel strip) per E1 CTA
constexpr uint32_t STREAM_GRID = 148u * 8u;

// ---- ordered block-wide exclusive scan for any associative (not necessarily commutative) operator ----------
template <class Op>
__device__ typename Op::T block_exclusive(typename Op::T x, const Op &op, typename Op::T *smem, typename Op::T *total)
{
    using T = typename Op::T;
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, nw = blockDim.x >> 5;
    T inc = x;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
        const T y = __shfl_up_sync(0xFFFFFFFFu, inc, d);
        if (lane >= d)
            inc = op.combine(y, inc);
    }
    if (lane == 31)
        smem[wid] = inc;
    __syncthreads();
    if (wid == 0) {
        T w = lane < nw ? smem[lane] : op.identity();
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const T y = __shfl_up_sync(0xFFFFFFFFu, w, d);
            if (lane >= d)
                w = op.combine(y, w);
        }
        smem[lane] = w;
    }
    __syncthreads();
    T ex = __shfl_up_sync(0xFFFFFFFFu, inc, 1);
    if (lane == 0)
        ex = op.identity();
    const T res = wid ? op.combine(smem[wid - 1], ex) : ex;
    *total = smem[nw - 1];
    __syncthreads();
    return res;
}

// ---- three-level scan (tile reduce, spine, down-sweep) over gridDim.y independent rows -----------------
// Op: T, identity(), combine(a, b) (a before b), load(row, i), store(row, i, exclusive prefix, item).
template <class Op>
__global__ void __launch_bounds__(THREADS) scan_reduce_kernel(Op op, uint64_t n, uint64_t ntiles, typename Op::T *agg)
{
    using T = typename Op::T;
    __shared__ T smem[32];
    const uint32_t row = blockIdx.y;
    for (uint64_t tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
        const uint64_t base = tile * SCAN_TILE + (uint64_t)threadIdx.x * ITEMS;
        T a = op.identity();
#pragma unroll
        for (int k = 0; k < ITEMS; ++k)
            if (base + k < n)
                a = op.combine(a, op.load(row, base + k));
        T tot;
        block_exclusive(a, op, smem, &tot);
        if (threadIdx.x == 0)
            agg[row * ntiles + tile] = tot;
    }
}

template <class Op>
__global__ void __launch_bounds__(THREADS) scan_spine_kernel(Op op, uint64_t ntiles, typename Op::T *agg)
{
    using T = typename Op::T;
    __shared__ T smem[32];
    T *a = agg + blockIdx.x * ntiles;
    const uint64_t per = (ntiles + THREADS - 1) / THREADS, t0 = threadIdx.x * per, t1 = min(t0 + per, ntiles);
    T x = op.identity();
    for (uint64_t t = t0; t < t1; ++t)
        x = op.combine(x, a[t]);
    T tot;
    T p = block_exclusive(x, op, smem, &tot);
    for (uint64_t t = t0; t < t1; ++t) {
        const T v = a[t];
        a[t] = p;
        p = op.combine(p, v);
    }
}

template <class Op>
__global__ void __launch_bounds__(THREADS) scan_down_kernel(Op op, uint64_t n, uint64_t ntiles, const typename Op::T *agg)
{
    using T = typename Op::T;
    __shared__ T smem[32];
    const uint32_t row = blockIdx.y;
    for (uint64_t tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
        const uint64_t base = tile * SCAN_TILE + (uint64_t)threadIdx.x * ITEMS;
        T v[ITEMS];
        T a = op.identity();
#pragma unroll
        for (int k = 0; k < ITEMS; ++k) {
            v[k] = base + k < n ? op.load(row, base + k) : op.identity();
            a = op.combine(a, v[k]);
        }
        T tot;
        T p = op.combine(agg[row * ntiles + tile], block_exclusive(a, op, smem, &tot));
#pragma unroll
        for (int k = 0; k < ITEMS; ++k)
            if (base + k < n) {
                op.store(row, base + k, p, v[k]);
                p = op.combine(p, v[k]);
            }
    }
}

template <class Op>
void run_scan(const Op &op, uint64_t n, uint32_t rows, typename Op::T *agg, cudaStream_t s, uint32_t *launches)
{
    const uint64_t ntiles = (n + SCAN_TILE - 1) / SCAN_TILE;
    const dim3 grid((unsigned)std::min<uint64_t>(ntiles, 65535u), rows);
    scan_reduce_kernel<Op><<<grid, THREADS, 0, s>>>(op, n, ntiles, agg);
    scan_spine_kernel<Op><<<rows, THREADS, 0, s>>>(op, ntiles, agg);
    scan_down_kernel<Op><<<grid, THREADS, 0, s>>>(op, n, ntiles, agg);
    *launches += 3;
}

// DC chain of component `row`: element m is MCU m's 5-state map; the store applies the prefix to the start state
struct NudgeOp {
    using T = uint32_t;
    const int16_t *raw;
    const uint8_t *has_ac;
    int16_t *dc;
    uint32_t nc;
    uint64_t seg_mcus;
    bool restart;
    __device__ T identity() const { return MAP_IDENTITY; }
    __device__ T combine(T a, T b) const { return map_then(a, b); }
    __device__ T load(uint32_t c, uint64_t m) const
    {
        const uint64_t b = m * nc + c;
        return nudge_map(raw[b], m ? raw[b - nc] : 0, has_ac[b] != 0, restart && m % seg_mcus == 0);
    }
    __device__ void store(uint32_t c, uint64_t m, T pre, T item) const
    {
        const uint64_t b = m * nc + c;
        dc[b] = (int16_t)(raw[b] + map_apply(item, map_apply(pre, MAP_START)) - 2);
    }
};

// bit offsets of the blocks: off[i] = sum of bits[0..i), off[n] = total
struct BitsOp {
    using T = unsigned long long;
    const uint32_t *bits;
    uint64_t *off;
    uint64_t n;
    __device__ T identity() const { return 0; }
    __device__ T combine(T a, T b) const { return a + b; }
    __device__ T load(uint32_t, uint64_t i) const { return bits[i]; }
    __device__ void store(uint32_t, uint64_t i, T pre, T item) const
    {
        off[i] = pre;
        if (i + 1 == n)
            off[n] = pre + item;
    }
};

// byte offsets of the restart segments, each padded to whole bytes: seg_byte[nseg] = unstuffed length
struct SegOp {
    using T = unsigned long long;
    const uint64_t *off;
    uint64_t *seg_byte;
    uint64_t nseg, seg_blocks, nblk;
    __device__ T identity() const { return 0; }
    __device__ T combine(T a, T b) const { return a + b; }
    __device__ T load(uint32_t, uint64_t s) const
    {
        const uint64_t b0 = s * seg_blocks, b1 = min(b0 + seg_blocks, nblk);
        return (off[b1] - off[b0] + 7u) >> 3;
    }
    __device__ void store(uint32_t, uint64_t s, T pre, T item) const
    {
        seg_byte[s] = pre;
        if (s + 1 == nseg)
            seg_byte[nseg] = pre + item;
    }
};

struct SumOp {
    using T = unsigned long long;
    __device__ T identity() const { return 0; }
    __device__ T combine(T a, T b) const { return a + b; }
};

// ---- E1 ------------------------------------------------------------------------------------------------
template <int NC>
__global__ void __launch_bounds__(THREADS) enc_fdct_kernel(EncGeom g, const uint8_t *__restrict__ px, const EncTables *__restrict__ T,
                                                           int16_t *__restrict__ coef, int16_t *__restrict__ raw, uint8_t *__restrict__ has_ac)
{
    constexpr int NB = NC * FDCT_MCUS;
    __shared__ double cs[8][8];
    __shared__ uint16_t qzz[2][64];
    __shared__ uint8_t nat[64];
    __shared__ uint8_t pix[8][64 * NC];
    __shared__ double blk[NB][64]; // block id = mcu * NC + component
    __shared__ double tmp[NB][64];
    __shared__ int nz[NB];
    const int tid = threadIdx.x;
    if (tid < 64) {
        cs[tid >> 3][tid & 7] = T->cs[tid >> 3][tid & 7];
        qzz[0][tid] = T->qzz[0][tid];
        qzz[1][tid] = T->qzz[1][tid];
        nat[tid] = T->nat[tid];
    }
    if (tid < NB)
        nz[tid] = 0;
    const uint32_t bx0 = blockIdx.x * FDCT_MCUS, by = blockIdx.y;
    const int nmcu = (int)min((uint32_t)FDCT_MCUS, g.mx - bx0);
    // the strip's pixel rows, edges replicated, through shared memory (RGB is interleaved)
    for (int idx = tid; idx < 8 * 64 * NC; idx += THREADS) {
        const int r = idx / (64 * NC), rem = idx - r * 64 * NC, q = rem / NC, c = rem - q * NC;
        const uint32_t y = min(by * 8u + r, g.height - 1u), x = min(bx0 * 8u + q, g.width - 1u);
        pix[r][rem] = px[((size_t)y * g.width + x) * NC + c];
    }
    __syncthreads();
    for (int p = tid; p < 8 * 8 * nmcu; p += THREADS) {
        const int r = p / (8 * nmcu), q = p - r * 8 * nmcu, m = q >> 3, e = r * 8 + (q & 7);
        if constexpr (NC == 1)
            blk[m][e] = dsub((double)pix[r][q], 128.0);
        else
            rgb_to_ycc(pix[r][3 * q], pix[r][3 * q + 1], pix[r][3 * q + 2], &blk[m * 3][e], &blk[m * 3 + 1][e], &blk[m * 3 + 2][e]);
    }
    __syncthreads();
    const int nout = nmcu * NC * 64;
    for (int o = tid; o < nout; o += THREADS) {
        const int b = o >> 6, r = (o >> 3) & 7, v = o & 7;
        tmp[b][r * 8 + v] = fdct_row(&blk[b][r * 8], cs, v);
    }
    __syncthreads();
    const uint64_t gb0 = ((uint64_t)by * g.mx + bx0) * NC;
    for (int o = tid; o < nout; o += THREADS) {
        const int b = o >> 6, i = o & 63, c = b % NC;
        const int val = quantise(fdct_col(tmp[b], cs, nat[i] >> 3, nat[i] & 7), qzz[c ? 1 : 0][i], i == 0);
        coef[(gb0 + b) * 64 + i] = (int16_t)val;
        if (i == 0)
            raw[gb0 + b] = (int16_t)val;
        else if (val)
            nz[b] = 1;
    }
    __syncthreads();
    if (tid < nmcu * NC)
        has_ac[gb0 + tid] = (uint8_t)nz[tid];
}

// ---- E3 / E4 ---------------------------------------------------------------------------------------------
__device__ __forceinline__ void load_tables(EncTables *dst, const EncTables *src)
{
    static_assert(sizeof(EncTables) % 8 == 0, "tables are staged in 8-byte words");
    const uint64_t *s = (const uint64_t *)src;
    uint64_t *d = (uint64_t *)dst;
    for (int i = threadIdx.x; i < (int)(sizeof(EncTables) / 8); i += blockDim.x)
        d[i] = s[i];
    __syncthreads();
}

__device__ __forceinline__ void load_block(const int16_t *src, int16_t zz[64])
{
    const int4 *s = (const int4 *)src;
#pragma unroll
    for (int k = 0; k < 8; ++k)
        ((int4 *)zz)[k] = s[k];
}

__device__ __forceinline__ int dc_diff(const EncGeom &g, const int16_t *dc, uint64_t b)
{
    const uint64_t m = b / g.ncomp;
    return dc[b] - (starts_segment(g, m) ? 0 : dc[b - g.ncomp]);
}

__global__ void __launch_bounds__(THREADS) enc_bits_kernel(EncGeom g, const EncTables *__restrict__ T_, const int16_t *__restrict__ coef,
                                                           const int16_t *__restrict__ dc, uint32_t *__restrict__ bits)
{
    __shared__ EncTables T;
    load_tables(&T, T_);
    const uint64_t b = (uint64_t)blockIdx.x * THREADS + threadIdx.x;
    if (b >= g.nblk)
        return;
    int16_t zz[64];
    load_block(coef + b * 64, zz);
    BitCounter bc;
    code_block(T, b % g.ncomp ? 1 : 0, dc_diff(g, dc, b), zz, bc);
    bits[b] = bc.n;
}

// ---- EH: symbol histogram ------------------------------------------------------------------------------------
constexpr uint32_t HIST_GRID = 148u * 4u; // CTAs (grid-stride): fewer global atomics when the per-CTA counts are flushed

// Counts into the CTA's [4][256] shared histogram.  EOB and the small categories are very hot bins, so the lanes of a
// warp that hit the same bin at the same time are folded into one shared atomic.
struct HistVisitor {
    uint32_t *h;
    int t; // DC table of the block's component (0 luma, 2 chroma); t + 1 is its AC table
    __device__ __forceinline__ void add(uint32_t bin)
    {
        const uint32_t m = __match_any_sync(__activemask(), bin);
        if ((threadIdx.x & 31u) == (uint32_t)(__ffs(m) - 1))
            atomicAdd(&h[bin], (uint32_t)__popc(m));
    }
    __device__ __forceinline__ void dc(int cat, int) { add((uint32_t)t * 256u + (uint32_t)cat); }
    __device__ __forceinline__ void ac(int sym, int, int) { add((uint32_t)(t + 1) * 256u + (uint32_t)sym); }
    __device__ __forceinline__ void zrl() { add((uint32_t)(t + 1) * 256u + 0xF0u); }
    __device__ __forceinline__ void eob() { add((uint32_t)(t + 1) * 256u); }
};

// hist: [4][257] uint64, zeroed on the stream before
__global__ void __launch_bounds__(THREADS) enc_hist_kernel(EncGeom g, const int16_t *__restrict__ coef, const int16_t *__restrict__ dc,
                                                           unsigned long long *__restrict__ hist)
{
    __shared__ uint32_t h[4 * 256];
    for (int i = threadIdx.x; i < 4 * 256; i += THREADS)
        h[i] = 0;
    __syncthreads();
    for (uint64_t b = (uint64_t)blockIdx.x * THREADS + threadIdx.x; b < g.nblk; b += (uint64_t)gridDim.x * THREADS) {
        int16_t zz[64];
        load_block(coef + b * 64, zz);
        HistVisitor v{h, b % g.ncomp ? 2 : 0};
        walk_block(dc_diff(g, dc, b), zz, v);
    }
    __syncthreads();
    for (int i = threadIdx.x; i < (g.ncomp == 3 ? 4 : 2) * 256; i += THREADS)
        if (h[i])
            atomicAdd(&hist[(i >> 8) * huff::NSYM + (i & 255)], (unsigned long long)h[i]);
}

// ---- EB: optimal tables, one warp per table ------------------------------------------------------------------------
constexpr int EB_PER_LANE = (huff::NSYM + 31) / 32; // slots lane + 32 j, j < 9

// Appends at out[pos], nothing at or past cap.
struct DevSeqOut {
    uint8_t *p;
    uint64_t pos, cap;
    __device__ void put(uint32_t b)
    {
        if (pos < cap)
            p[pos] = (uint8_t)b;
        ++pos;
    }
};

// The lane's first slot in merge order, skipping `skip`: (frequency, slot), slot -1 when it holds none.
__device__ __forceinline__ void lane_first(const uint64_t (&f)[EB_PER_LANE], int skip, uint64_t &bf, int &bs)
{
    const int lane = threadIdx.x & 31;
    bf = 0;
    bs = -1;
#pragma unroll
    for (int j = 0; j < EB_PER_LANE; ++j) {
        const int s = lane + 32 * j;
        if (f[j] && s != skip && (bs < 0 || huff::merges_first(f[j], s, bf, bs))) {
            bf = f[j];
            bs = s;
        }
    }
}

// The warp's first slot in merge order (lexicographic on (frequency, -slot)), -1 when no lane holds one.  Frequencies
// stay below 2^64 - 2^32 (they sum to the symbol count + 1), so ~0 in the high word means "none".
__device__ __forceinline__ int warp_first(uint64_t bf, int bs, uint64_t &f)
{
    const uint32_t hi = bs < 0 ? ~0u : (uint32_t)(bf >> 32);
    const uint32_t mh = __reduce_min_sync(0xFFFFFFFFu, hi);
    const uint32_t lo = bs >= 0 && hi == mh ? (uint32_t)bf : ~0u;
    const uint32_t ml = __reduce_min_sync(0xFFFFFFFFu, lo);
    f = ((uint64_t)mh << 32) | ml;
    return __reduce_max_sync(0xFFFFFFFFu, bs >= 0 && hi == mh && lo == ml ? bs : -1);
}

// One CTA of 32 * (2 or 4) threads.  Warp t builds table t (0 DC luma, 1 AC luma, 2 DC chroma, 3 AC chroma) from
// hist[t] with huff::optimal_table's rule: the merge loop keeps each lane's nine slots in registers and finds the two
// slots to merge with two warp-wide argmin reductions; code lengths are leaf depths of the parent array, lane-parallel;
// the K.3 fold runs on one lane; HUFFVAL is a counting sort by (length, symbol).  The codes go into Topt, a copy of the
// cached tables T_ (which stay untouched); then DHT [DRI] SOS are written at out[prefix_len..) and their end is the
// header length in meta.
__global__ void __launch_bounds__(128) enc_huff_build_kernel(EncGeom g, const unsigned long long *__restrict__ hist,
                                                             const EncTables *__restrict__ T_, EncTables *__restrict__ Topt,
                                                             uint8_t *__restrict__ out, uint64_t cap, uint64_t prefix_len,
                                                             EncMeta *__restrict__ meta)
{
    using namespace huff;
    __shared__ int16_t parent[4][NNODE];
    __shared__ int16_t node[4][NSYM];
    __shared__ uint32_t cnt[4][MAX_DEPTH + 1];   // codes by length, the reserved one included (then folded)
    __shared__ uint32_t start[4][MAX_DEPTH + 2]; // HUFFVAL position of the next symbol of each length
    __shared__ uint8_t bits[4][16];
    __shared__ uint8_t vals[4][256];
    __shared__ uint16_t code[4][256];
    __shared__ uint8_t len[4][256];
    {
        const uint64_t *src = (const uint64_t *)T_;
        uint64_t *dst = (uint64_t *)Topt;
        for (int i = threadIdx.x; i < (int)(sizeof(EncTables) / 8); i += blockDim.x)
            dst[i] = src[i];
    }
    const int t = threadIdx.x >> 5, lane = threadIdx.x & 31;
    for (int n = lane; n < NNODE; n += 32)
        parent[t][n] = -1;
    for (int s = lane; s < NSYM; s += 32)
        node[t][s] = (int16_t)s;
    for (int d = lane; d < MAX_DEPTH + 2; d += 32) {
        if (d <= MAX_DEPTH)
            cnt[t][d] = 0;
        start[t][d] = 0;
    }
    uint64_t f[EB_PER_LANE];
    uint32_t present = 0;
#pragma unroll
    for (int j = 0; j < EB_PER_LANE; ++j) {
        const int s = lane + 32 * j;
        f[j] = s < RESERVED ? hist[t * NSYM + s] : (s == RESERVED ? 1u : 0u);
        present |= (f[j] != 0 ? 1u : 0u) << j;
    }
    __syncthreads(); // Topt holds the copy before any warp writes its codes
    for (int next = NSYM;; ++next) {
        uint64_t bf, f1, f2;
        int bs;
        lane_first(f, -1, bf, bs);
        const int c1 = warp_first(bf, bs, f1);
        lane_first(f, c1, bf, bs);
        const int c2 = warp_first(bf, bs, f2);
        if (c2 < 0)
            break;
#pragma unroll
        for (int j = 0; j < EB_PER_LANE; ++j) {
            const int s = lane + 32 * j;
            if (s == c1)
                f[j] += f2;
            if (s == c2)
                f[j] = 0;
        }
        if (lane == 0) {
            parent[t][node[t][c1]] = parent[t][node[t][c2]] = (int16_t)next;
            node[t][c1] = (int16_t)next;
        }
    }
    __syncwarp();
    int dep[EB_PER_LANE];
    int dmax = 0;
#pragma unroll
    for (int j = 0; j < EB_PER_LANE; ++j) {
        const int s = lane + 32 * j;
        dep[j] = (present >> j) & 1u ? leaf_depth(parent[t], s) : 0;
        dmax = max(dmax, dep[j]);
        if (dep[j]) {
            atomicAdd(&cnt[t][dep[j]], 1u);
            if (s != RESERVED)
                atomicAdd(&start[t][dep[j] + 1], 1u);
        }
    }
    dmax = __reduce_max_sync(0xFFFFFFFFu, dmax);
    __syncwarp();
    if (lane == 0)
        for (int d = 1; d <= dmax; ++d)
            start[t][d + 1] += start[t][d];
    __syncwarp();
    // HUFFVAL: symbols 32 j .. 32 j + 31 in turn; lanes of equal length take consecutive places in lane order
#pragma unroll
    for (int j = 0; j < RESERVED / 32; ++j) {
        const int d = dep[j];
        const uint32_t m = __match_any_sync(0xFFFFFFFFu, d);
        if (d)
            vals[t][start[t][d] + __popc(m & ((1u << lane) - 1u))] = (uint8_t)(lane + 32 * j);
        __syncwarp();
        if (d && lane == __ffs(m) - 1)
            start[t][d] += __popc(m);
        __syncwarp();
    }
    if (lane == 0) {
        fold_lengths(cnt[t], dmax, bits[t]);
        canonical_codes(bits[t], vals[t], code[t], len[t]);
    }
    __syncwarp();
    if (t & 1) {
        for (int s = lane; s < 256; s += 32) {
            Topt->ac_code[t >> 1][s] = code[t][s];
            Topt->ac_len[t >> 1][s] = len[t][s];
        }
    } else if (lane < 16) {
        Topt->dc_code[t >> 1][lane] = code[t][lane];
        Topt->dc_len[t >> 1][lane] = len[t][lane];
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        DevSeqOut o{out, prefix_len, cap};
        const uint8_t *const bp[4] = {bits[0], bits[1], bits[2], bits[3]};
        const uint8_t *const vp[4] = {vals[0], vals[1], vals[2], vals[3]};
        put_header_tail(o, (int)g.ncomp, bp, vp, (int)g.ri);
        meta->hdr_len = o.pos;
    }
}

struct DevWords {
    uint32_t *w;
    __device__ void store(uint64_t i, uint32_t v) { w[i] = v; }
    __device__ void orw(uint64_t i, uint32_t v) { atomicOr(&w[i], v); }
};

__global__ void __launch_bounds__(THREADS) enc_zero_words_kernel(const uint64_t *__restrict__ total, uint32_t *__restrict__ words)
{
    const uint64_t nw = (*total + 3u) / 4u + 1u;
    for (uint64_t i = (uint64_t)blockIdx.x * THREADS + threadIdx.x; i < nw; i += (uint64_t)gridDim.x * THREADS)
        words[i] = 0;
}

__global__ void __launch_bounds__(THREADS) enc_emit_kernel(EncGeom g, const EncTables *__restrict__ T_, const int16_t *__restrict__ coef,
                                                           const int16_t *__restrict__ dc, const uint64_t *__restrict__ off,
                                                           const uint64_t *__restrict__ seg_byte, uint32_t *__restrict__ words)
{
    __shared__ EncTables T;
    load_tables(&T, T_);
    const uint64_t b = (uint64_t)blockIdx.x * THREADS + threadIdx.x;
    if (b >= g.nblk)
        return;
    const uint64_t m = b / g.ncomp, s = m / g.seg_mcus;
    const uint64_t b0 = s * g.seg_mcus * g.ncomp, b1 = min((s + 1) * g.seg_mcus, g.nmcu) * g.ncomp;
    int16_t zz[64];
    load_block(coef + b * 64, zz);
    DevWords dw{words};
    BitEmitter<DevWords> em(dw, seg_byte[s] * 8u + (off[b] - off[b0]));
    code_block(T, b % g.ncomp ? 1 : 0, dc_diff(g, dc, b), zz, em);
    if (b + 1 == b1) { // the segment's last block pads it to a byte boundary with 1-bits
        const int pad = (int)((seg_byte[s + 1] - seg_byte[s]) * 8u - (off[b1] - off[b0]));
        if (pad)
            em.put((1u << pad) - 1u, pad);
    }
    em.finish();
}

// ---- E5 ------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint64_t ff_count(const uint32_t *words, uint64_t i0, uint64_t i1)
{
    uint64_t k = 0;
    for (uint64_t i = i0; i < i1; ++i)
        k += stream_byte(words, i) == 0xFFu;
    return k;
}

__global__ void __launch_bounds__(STUFF_THREADS) enc_stuff_count_kernel(const uint64_t *__restrict__ seg_byte, uint64_t nseg,
                                                                       const uint32_t *__restrict__ words, uint64_t *__restrict__ tile_ff)
{
    __shared__ unsigned long long smem[32];
    const uint64_t N = seg_byte[nseg], ntiles = (N + STUFF_TILE - 1) / STUFF_TILE;
    const SumOp op;
    for (uint64_t t = blockIdx.x; t < ntiles; t += gridDim.x) {
        const uint64_t i0 = min(N, t * STUFF_TILE + (uint64_t)threadIdx.x * STUFF_BYTES_PER_THREAD);
        unsigned long long tot;
        block_exclusive((unsigned long long)ff_count(words, i0, min(N, i0 + STUFF_BYTES_PER_THREAD)), op, smem, &tot);
        if (threadIdx.x == 0)
            tile_ff[t] = tot;
    }
}

// one CTA: exclusive scan of the tiles' FF counts, and the length of what E5 writes
// host_hdr: the length of the header the host wrote (Annex K mode), 0 when EB wrote the header and its length
__global__ void __launch_bounds__(STUFF_THREADS) enc_stuff_spine_kernel(const uint64_t *__restrict__ seg_byte, uint64_t nseg,
                                                                       uint64_t *__restrict__ tile_ff, uint64_t host_hdr,
                                                                       EncMeta *__restrict__ meta)
{
    __shared__ unsigned long long smem[32];
    const uint64_t N = seg_byte[nseg], ntiles = (N + STUFF_TILE - 1) / STUFF_TILE;
    const SumOp op;
    const uint64_t per = (ntiles + STUFF_THREADS - 1) / STUFF_THREADS, t0 = threadIdx.x * per, t1 = min(t0 + per, ntiles);
    unsigned long long x = 0;
    for (uint64_t t = t0; t < t1; ++t)
        x += tile_ff[t];
    unsigned long long tot;
    unsigned long long p = block_exclusive(x, op, smem, &tot);
    for (uint64_t t = t0; t < t1; ++t) {
        const unsigned long long v = tile_ff[t];
        tile_ff[t] = p;
        p += v;
    }
    if (threadIdx.x == 0) {
        meta->unstuffed = N;
        meta->scan_len = N + tot + 2u * nseg; // RSTn between segments + EOI
        if (host_hdr)
            meta->hdr_len = host_hdr;
    }
}

struct DevOut {
    uint8_t *p;
    uint64_t cap;
    __device__ void put(uint64_t i, uint32_t b)
    {
        if (i < cap)
            p[i] = (uint8_t)b;
    }
};

__global__ void __launch_bounds__(STUFF_THREADS) enc_stuff_write_kernel(const uint64_t *__restrict__ seg_byte, uint64_t nseg,
                                                                       const uint32_t *__restrict__ words, const uint64_t *__restrict__ tile_ff,
                                                                       const EncMeta *__restrict__ meta, uint8_t *__restrict__ out, uint64_t cap)
{
    __shared__ unsigned long long smem[32];
    const uint64_t N = seg_byte[nseg], ntiles = (N + STUFF_TILE - 1) / STUFF_TILE;
    const SumOp op;
    const uint64_t hdr = meta->hdr_len; // the scan starts after the header
    DevOut o{out + hdr, cap > hdr ? cap - hdr : 0};
    for (uint64_t t = blockIdx.x; t < ntiles; t += gridDim.x) {
        const uint64_t i0 = min(N, t * STUFF_TILE + (uint64_t)threadIdx.x * STUFF_BYTES_PER_THREAD);
        const uint64_t i1 = min(N, i0 + STUFF_BYTES_PER_THREAD);
        unsigned long long tot;
        const unsigned long long before = tile_ff[t] + block_exclusive((unsigned long long)ff_count(words, i0, i1), op, smem, &tot);
        stuff_range(words, seg_byte, nseg, N, i0, i1, before, o);
    }
}

uint64_t unstuffed_bound(const EncGeom &g) { return (g.nblk * max_block_bits(g.flags) + 7u) / 8u + g.nseg; }

} // namespace

void scratch_sizes(const EncGeom &g, size_t sz[BUF_COUNT])
{
    const uint64_t ub = unstuffed_bound(g);
    const uint64_t tiles_blk = (g.nblk + SCAN_TILE - 1) / SCAN_TILE, tiles_seg = (g.nseg + SCAN_TILE - 1) / SCAN_TILE;
    const uint64_t tiles_map = g.ncomp * ((g.nmcu + SCAN_TILE - 1) / SCAN_TILE);
    sz[BUF_COEF] = g.nblk * 128u;
    sz[BUF_RAW] = sz[BUF_DC] = g.nblk * 2u;
    sz[BUF_HAS_AC] = g.nblk;
    sz[BUF_BITS] = g.nblk * 4u;
    sz[BUF_OFF] = (g.nblk + 1u) * 8u;
    sz[BUF_SEG] = (g.nseg + 1u) * 8u;
    sz[BUF_WORDS] = (ub / 4u + 2u) * 4u;
    sz[BUF_AGG] = std::max(std::max(tiles_blk, tiles_seg), tiles_map) * 8u + 8u;
    sz[BUF_TILE_FF] = (ub / STUFF_TILE + 2u) * 8u;
}

cudaError_t launch_encode(const EncGeom &g, const EncBufs &b, cudaStream_t s, uint32_t *launches, StageMark mark, void *user)
{
    // E1
    const dim3 fgrid((g.mx + FDCT_MCUS - 1) / FDCT_MCUS, g.my);
    if (g.ncomp == 3)
        enc_fdct_kernel<3><<<fgrid, THREADS, 0, s>>>(g, b.pixels, b.tables, b.coef, b.raw, b.has_ac);
    else
        enc_fdct_kernel<1><<<fgrid, THREADS, 0, s>>>(g, b.pixels, b.tables, b.coef, b.raw, b.has_ac);
    ++*launches;
    mark(user, KPEG_T_IDCT);
    // E2
    const int16_t *dc = b.raw;
    if (g.flags & KPEG_FLAG_REF_PARITY) {
        const NudgeOp op{b.raw, b.has_ac, b.dc, g.ncomp, g.seg_mcus, g.ri > 0};
        run_scan(op, g.nmcu, g.ncomp, (uint32_t *)b.agg, s, launches);
        dc = b.dc;
        mark(user, KPEG_T_DC_SCAN);
    }
    return launch_coded_stages(g, b, dc, s, launches, mark, user);
}

cudaError_t launch_coded_stages(const EncGeom &g, const EncBufs &b, const int16_t *dc, cudaStream_t s, uint32_t *launches, StageMark mark,
                                void *user)
{
    const unsigned bgrid = (unsigned)((g.nblk + THREADS - 1) / THREADS);
    // EH, EB: this image's tables, and the header after the host's prefix
    const EncTables *codes = b.tables;
    const bool opt = (g.flags & KPEG_FLAG_OPTIMIZE_HUFFMAN) != 0;
    if (opt) {
        cudaError_t e = cudaMemsetAsync(b.hist, 0, 4u * huff::NSYM * sizeof(uint64_t), s);
        if (e != cudaSuccess)
            return e;
        enc_hist_kernel<<<std::min(bgrid, HIST_GRID), THREADS, 0, s>>>(g, b.coef, dc, (unsigned long long *)b.hist);
        enc_huff_build_kernel<<<1, 32 * (g.ncomp == 3 ? 4 : 2), 0, s>>>(g, (const unsigned long long *)b.hist, b.tables, b.opt_tables,
                                                                          b.out, b.out_cap, b.hdr_len, b.meta);
        *launches += 2;
        codes = b.opt_tables;
        mark(user, KPEG_T_ENTROPY_SCAN);
    }
    // E3
    enc_bits_kernel<<<bgrid, THREADS, 0, s>>>(g, codes, b.coef, dc, b.bits);
    ++*launches;
    run_scan(BitsOp{b.bits, b.off, g.nblk}, g.nblk, 1, (unsigned long long *)b.agg, s, launches);
    run_scan(SegOp{b.off, b.seg_byte, g.nseg, g.seg_mcus * g.ncomp, g.nblk}, g.nseg, 1, (unsigned long long *)b.agg, s, launches);
    // E4
    const unsigned sgrid = (unsigned)std::min<uint64_t>(STREAM_GRID, unstuffed_bound(g) / STUFF_TILE + 1u);
    enc_zero_words_kernel<<<sgrid, THREADS, 0, s>>>(b.seg_byte + g.nseg, b.words);
    enc_emit_kernel<<<bgrid, THREADS, 0, s>>>(g, codes, b.coef, dc, b.off, b.seg_byte, b.words);
    *launches += 2;
    mark(user, KPEG_T_ENTROPY_WRITE);
    // E5
    enc_stuff_count_kernel<<<sgrid, STUFF_THREADS, 0, s>>>(b.seg_byte, g.nseg, b.words, b.tile_ff);
    enc_stuff_spine_kernel<<<1, STUFF_THREADS, 0, s>>>(b.seg_byte, g.nseg, b.tile_ff, opt ? 0u : b.hdr_len, b.meta);
    enc_stuff_write_kernel<<<sgrid, STUFF_THREADS, 0, s>>>(b.seg_byte, g.nseg, b.words, b.tile_ff, b.meta, b.out, b.out_cap);
    *launches += 3;
    mark(user, KPEG_T_UNSTUFF);
    return cudaGetLastError();
}

} // namespace enc
} // namespace kpeg
