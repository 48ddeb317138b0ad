// host_tables.h -- plan -> device tables / job geometry (host only, no CUDA).
//
// The only host arithmetic of the decode path: Huffman LUT construction (huff_lut.h), quantisers
// with the AAN prescale folded in, and the 64 double cosines + 64 float scale products the exact
// IDCT path needs, evaluated with the host libm exactly as the reference evaluates them
// (src/MCU.cpp:190-193).  Shared by kpeg_cuda.cu and the CPU logic tests (tests/emu).
#ifndef KPEG_HOST_TABLES_H
#define KPEG_HOST_TABLES_H

#include <math.h>
#include <string.h>

#include "huff_lut.h"
#include "idct_core.h"
#include "kpeg_common.h"
#include "kpeg_cuda.h"

namespace kpeg {

inline int build_device_tables(const kpeg_plan *pl, DeviceTables *T, const char **why)
{
    memset(T, 0, sizeof *T);
    static const ZigZagTables zz = make_zigzag_tables();
    for (unsigned c = 0; c < pl->ncomp; ++c) {
        const unsigned tq = pl->comp_tq[c], td = pl->comp_td[c], ta = pl->comp_ta[c];
        if (tq > 3 || td > 3 || ta > 3 || !pl->qt_present[tq] || !pl->ht_present[0][td] || !pl->ht_present[1][ta]) {
            *why = "plan references a table that was never defined";
            return KPEG_ERR_FORMAT;
        }
        if (build_huff_lut(pl->ht[0][td].counts, pl->ht[0][td].symbols, false, &T->luts, c * 2 + 0, &T->canon[c * 2 + 0]) ||
            build_huff_lut(pl->ht[1][ta].counts, pl->ht[1][ta].symbols, true, &T->luts, c * 2 + 1, &T->canon[c * 2 + 1])) {
            *why = "over-subscribed Huffman table";
            return KPEG_ERR_FORMAT;
        }
        for (int i = 0; i < 64; ++i) {
            const int nat = zz.zz2nat[i];
            const double s = aan_scale(nat >> 3) * aan_scale(nat & 7) / 8.0;
            T->qscale[c][i] = (float)((double)pl->qt[tq][i] * s);
            T->qint[c][i] = (int32_t)pl->qt[tq][i];
        }
        for (int j = 0; j < 64; ++j) {
            T->qpair[c][j] = T->qscale[c][zz.nat2zz[pair_nat(j >> 1, j & 1)]];
            T->qdc[c][j] = pair_nat(j >> 1, j & 1) == 0 ? T->qpair[c][j] : 0.0f;
        }
    }
    for (int x = 0; x < 8; ++x)
        for (int u = 0; u < 8; ++u)
            T->cosd[x][u] = cos((2 * x + 1) * u * M_PI / 16.0); // the expression of MCU.cpp:193
    for (int u = 0; u < 8; ++u)
        for (int v = 0; v < 8; ++v) {
            const float Cu = u == 0 ? 1.0 / sqrt(2.0) : 1.0; // MCU.cpp:190
            const float Cv = v == 0 ? 1.0 / sqrt(2.0) : 1.0; // MCU.cpp:191
            T->cc[u][v] = Cu * Cv;
        }
    return KPEG_OK;
}

// Records per subsequence the relay passes keep room for: 3/8 of its bits covers every table whose value-carrying
// symbols take at least 3 bits (code >= 2 bits + value >= 1 bit: all of Annex K); a stream that needs more sets
// ST_REC_OVERFLOW and is redone with the Huffman final pass.
inline uint32_t rec_kmax_of(uint32_t sub_bits) { return (sub_bits * 3u / 8u + 7u) & ~7u; }

// Whether the 1-bits that pad an interval before its RSTn marker (at most 7, T.81 F.1.2.3) can hold a whole DC symbol of
// the first component: its table has an all-ones code (it fills the code space, which T.81 C and libjpeg do not allow)
// whose length plus category is at most 7.  The decoder takes a symbol that fits before a boundary for data
// (entropy_core.h relay_run), so such padding would count as one more block.  That is harmless after the last MCU of
// a job, which is where a single image without restart markers has its only padding.
inline bool restart_padding_decodes(const kpeg_plan *pl)
{
    const unsigned td = pl->comp_td[0];
    if (td > 3 || !pl->ht_present[0][td])
        return false;
    const kpeg_huff_spec &h = pl->ht[0][td];
    uint32_t space = 0, nsym = 0; // code space in units of 2^-16
    int last_len = 0;
    for (int L = 1; L <= 16; ++L) {
        space += (uint32_t)h.counts[L - 1] << (16 - L);
        nsym += h.counts[L - 1];
        if (h.counts[L - 1])
            last_len = L;
    }
    if (space != (1u << 16) || nsym == 0 || nsym > 256)
        return false; // the last code is all ones only in a table that fills the code space
    return last_len + (h.symbols[nsym - 1] & 15) <= 7;
}

inline int make_job_geom(const kpeg_plan *pl, uint32_t nimages, uint32_t sub_bits, JobGeom *g, const char **why)
{
    if (pl->width == 0 || pl->height == 0 || (pl->ncomp != 1 && pl->ncomp != 3) || nimages == 0) {
        *why = "bad plan geometry";
        return KPEG_ERR_ARG;
    }
    g->width = pl->width;
    g->height = pl->height;
    g->ncomp = pl->ncomp;
    g->mcus_x = (pl->width + 7u) / 8u;
    g->mcus_y = (pl->height + 7u) / 8u;
    g->mcus_per_image = g->mcus_x * g->mcus_y;
    g->restart_interval = pl->restart_interval;
    g->segs_per_image = pl->restart_interval ? (g->mcus_per_image + pl->restart_interval - 1u) / pl->restart_interval : 1u;
    g->nimages = nimages;
    const uint64_t nseg = (uint64_t)nimages * g->segs_per_image;
    const uint64_t blocks = (uint64_t)nimages * g->mcus_per_image * g->ncomp;
    if (nseg >= (1ull << 31) || blocks * 64ull >= (1ull << 32)) {
        *why = "job too large for 32-bit slot indices; split the batch";
        return KPEG_ERR_ARG;
    }
    g->nseg = (uint32_t)nseg;
    g->total_blocks = (uint32_t)blocks;
    g->flags = pl->flags;
    g->sub_bits = sub_bits;
    return KPEG_OK;
}

} // namespace kpeg
#endif
