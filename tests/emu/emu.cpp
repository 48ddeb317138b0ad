// tests/emu/emu.cpp -- TEST INFRASTRUCTURE: single-steps the kernel logic of libkpeg_b200/csrc on
// the CPU.  It includes the very same host+device inline headers the sm_100a kernels are built
// from (unstuff_core.h, entropy_core.h, idct_core.h, host_tables.h) and replays, thread by
// thread, what kernels.cu does with them -- so the speculative-decode / relay / offset-scan logic
// and the two-tier IDCT + colour arithmetic can be checked against the oracle without a GPU.
// It is NOT linked into libkpeg_cuda.so and nothing in the product calls it.
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

#include <vector>

#include "entropy_core.h"
#include "host_tables.h"
#include "idct_core.h"
#include "kpeg_cuda.h"
#include "unstuff_core.h"

using namespace kpeg;

namespace {

// K0 replay: unstuff_count / unstuff_scan / unstuff_write in one sequential sweep.
void emu_unstuff(const uint8_t *scan, uint32_t len, uint32_t nseg, std::vector<uint8_t> &words,
                 std::vector<uint32_t> &seg_bit, uint32_t *total_bits, uint32_t *status)
{
    words.assign(((size_t)len + 3) / 4 * 4 + 32, 0);
    uint32_t pos = 0, ridx = 0, st = 0;
    std::vector<uint32_t> seg_pos;
    for (uint32_t base = 0; base < len; base += 16) {
        const ByteClass c = classify16(scan, len, base);
        if (c.bad)
            st |= ST_BAD_MARKER;
        for (int i = 0; i < 16; ++i) {
            if (c.rst & (1u << i)) {
                ++ridx;
                seg_pos.push_back(pos * 8u);
            }
            if (c.keep & (1u << i)) {
                words[pos ^ 3u] = (uint8_t)(c.b[i >> 2] >> (8 * (i & 3)));
                ++pos;
            }
        }
    }
    *total_bits = pos * 8u;
    seg_bit.assign((size_t)nseg + 2, *total_bits);
    seg_bit[0] = 0;
    seg_bit[nseg + 1] = 0xFFFFFFFFu;
    for (uint32_t r = 1; r <= ridx; ++r)
        if (r < nseg)
            seg_bit[r] = seg_pos[r - 1];
    if (ridx != nseg - 1 && ridx != nseg)
        st |= ST_SEG_COUNT;
    *status |= st;
}

uint32_t first_seg_at_or_after(const std::vector<uint32_t> &seg_bit, uint32_t nseg, uint32_t bit)
{
    uint32_t lo = 0, hi = nseg;
    while (lo < hi) {
        const uint32_t mid = (lo + hi) >> 1;
        if (seg_bit[mid] >= bit)
            hi = mid;
        else
            lo = mid + 1;
    }
    return lo;
}

} // namespace

extern "C" {

// info[0]=status, [1]=nsub, [2]=relay rounds until the fixed point, [3]=exact IDCT samples,
// [4]=exact colour pixels, [5]=total_bits, [6]=final_slot, [7]=record final pass == Huffman final pass,
// [8]=most records in one subsequence, [9]=subsequences with more records than the product keeps room for (rec_kmax_of:
// the device would redo the job with the Huffman final pass)
int emu_decode(const uint8_t *scan, size_t scan_len, const kpeg_plan *plan, uint32_t nimages, uint32_t sub_bits,
               int16_t *coef_out, uint8_t *pixels_out, uint32_t *info)
{
    JobGeom g;
    const char *why = nullptr;
    int rc = make_job_geom(plan, nimages, sub_bits, &g, &why);
    if (rc != KPEG_OK)
        return rc;
    DeviceTables *T = new DeviceTables;
    rc = build_device_tables(plan, T, &why);
    if (rc != KPEG_OK) {
        delete T;
        return rc;
    }
    uint32_t status = 0, total_bits = 0;
    std::vector<uint8_t> words;
    std::vector<uint32_t> seg_bit;
    emu_unstuff(scan, (uint32_t)scan_len, g.nseg, words, seg_bit, &total_bits, &status);
    uint32_t nsub = (total_bits + sub_bits - 1) / sub_bits;
    if (!nsub)
        nsub = 1;
    StreamView S{seg_bit.data(), total_bits};
    const PlainWords PW{(const uint32_t *)words.data()};
    const PlainLuts PL{&T->luts, T->canon};

    // K1 cold
    std::vector<SubState> X(nsub);
    std::vector<uint32_t> hint(nsub), used_p(nsub), used_cz(nsub);
    for (uint32_t sub = 0; sub < nsub; ++sub) {
        const uint32_t p0 = sub * sub_bits;
        const uint32_t end = std::min(p0 + sub_bits, total_bits);
        hint[sub] = g.nseg > 1 ? first_seg_at_or_after(seg_bit, g.nseg, p0) : (sub ? 1u : 0u);
        X[sub] = relay_span(PW, PL, S, g, end, p0, 0, 0, hint[sub]);
        used_p[sub] = p0;
        used_cz[sub] = 0;
    }
    // K1 relay (Jacobi-style rounds on a snapshot, like independent thread blocks would see it)
    uint32_t rounds = 0;
    for (;;) {
        uint32_t changed = 0;
        const std::vector<SubState> prev = X;
        for (uint32_t sub = 1; sub < nsub; ++sub) {
            const SubState in = prev[sub - 1];
            if (used_p[sub] == in.p && used_cz[sub] == (in.cz & CZ_STATE_MASK))
                continue;
            const uint32_t end = std::min((sub + 1) * sub_bits, total_bits);
            const SubState out = relay_span(PW, PL, S, g, end, in.p, (in.cz >> 8) & 3u, in.cz & 0xFF, hint[sub]);
            used_p[sub] = in.p;
            used_cz[sub] = in.cz & CZ_STATE_MASK;
            if (out.p != X[sub].p || out.cz != X[sub].cz || out.n != X[sub].n || out.seg != X[sub].seg) {
                X[sub] = out;
                ++changed;
            }
        }
        if (!changed)
            break;
        ++rounds;
        if (rounds > nsub + 2) {
            delete T;
            return KPEG_ERR_NOT_CONVERGED;
        }
    }
    // K1 scan
    std::vector<uint32_t> start(nsub);
    uint32_t f = 1, v = 0;
    for (uint32_t i = 0; i < nsub; ++i) {
        start[i] = v;
        const SubState st = X[i];
        if (st.seg >= 0) {
            f = 1;
            v = st.n + seg_slot_base(g, (uint32_t)st.seg);
        } else {
            v += st.n;
        }
    }
    (void)f;
    const uint32_t final_slot = v;
    // K1 write
    std::vector<int16_t> coef((size_t)g.total_blocks * 64, 0), dcdiff(g.total_blocks, 0), dc(g.total_blocks, 0);
    for (uint32_t sub = 0; sub < nsub; ++sub) {
        uint32_t p = 0, c = 0, z = 0;
        if (sub) {
            p = X[sub - 1].p;
            c = (X[sub - 1].cz >> 8) & 3u;
            z = X[sub - 1].cz & 0xFF;
        }
        const uint32_t slot = start[sub];
        uint32_t st = 0;
        if ((slot & 63u) != z || ((slot >> 6) % g.ncomp) != c)
            st |= ST_EXIT_MISMATCH;
        const uint32_t end = std::min((sub + 1) * sub_bits, total_bits);
        const SubState out = write_span(PW, PL, S, g, end, p, c, z, hint[sub], slot, coef.data(), dcdiff.data(), &st);
        if (out.p != X[sub].p || out.cz != (X[sub].cz & CZ_STATE_MASK))
            st |= ST_EXIT_MISMATCH;
        status |= st;
    }
    if (final_slot < g.total_blocks * 64u)
        status |= ST_SEG_MISMATCH;
    // Record flavour, as the product runs it: relay-style decode from the true entry states emitting one record per
    // value-carrying symbol (relay_run<true>), the checks of the offset scan's last phase (entropy_scan_apply_kernel),
    // then K3's expansion (k3_fused.cu stage B): every record is dropped at (entry block of its subsequence) * 64 +
    // position, no running state.  Must reproduce the Huffman final pass: coefficients, DC differences and verdict.
    uint32_t records_ok = 1;
    std::vector<int16_t> dc2; // DC values as K3 derives them (scan-based predictors); empty = not computed
    {
        struct HostRecorder {
            std::vector<uint32_t> *v;
            void emit(bool on, uint32_t, uint32_t w) const { if (on) v->push_back(w); }
        };
        std::vector<int16_t> coef2((size_t)g.total_blocks * 64, 0);
        const uint32_t total_slots = g.total_blocks * 64u;
        uint32_t st2 = 0, max_rec = 0, over_kmax = 0;
        std::vector<long long> dcs(nsub, 0), dcpre(nsub, 0); // K2 as a scan: per-subsequence DC sums and their segmented prefix
        std::vector<std::vector<uint32_t>> all_recs(nsub);
        for (uint32_t sub = 0; sub < nsub; ++sub) {
            uint32_t p = 0, c = 0, z = 0;
            if (sub) {
                p = X[sub - 1].p;
                c = (X[sub - 1].cz >> 8) & 3u;
                z = X[sub - 1].cz & 0xFF;
            }
            std::vector<uint32_t> recs;
            DecState d;
            dec_init(d, PW, S, p, c, z, hint[sub], 0);
            const uint32_t end = std::min((sub + 1) * sub_bits, total_bits);
            relay_run<true, true>(d, PW, PL, S, g, end, HostRecorder{&recs});
            const SubState out = relay_exit_state(d);
            dcs[sub] = d.dcs;
            all_recs[sub] = recs;
            if (d.nrec != recs.size())
                records_ok = 0;
            // the emitting decode ends in the state (and slot count) the relay's fixed point holds
            if (out.p != X[sub].p || ((out.cz ^ X[sub].cz) & CZ_STATE_MASK) || out.n != X[sub].n || out.seg != X[sub].seg)
                records_ok = 0;
            max_rec = std::max<uint32_t>(max_rec, d.nrec);
            over_kmax += d.nrec > rec_kmax_of(sub_bits) ? 1u : 0u;
            // entropy_scan_apply_kernel
            const uint32_t begin = start[sub], fin = sub + 1 < nsub ? start[sub + 1] : final_slot;
            st2 |= (out.cz & CZ_BAD_CODE) ? ST_BAD_CODE : 0u;
            st2 |= (out.cz & CZ_SLOT_OVERFLOW) ? ST_SLOT_OVERFLOW : 0u;
            st2 |= (out.cz & CZ_SEG_MISMATCH) ? ST_SEG_MISMATCH : 0u;
            const uint32_t reached = (begin & ~63u) + (out.cz >> CZ_POS_SHIFT);
            if (out.seg >= 0 && reached != fin && !((uint32_t)out.seg >= g.nseg && fin >= total_slots && reached >= total_slots))
                st2 |= ST_SEG_MISMATCH;
            if ((fin & 63u) != (out.cz & 63u) || ((fin >> 6) % g.ncomp) != ((out.cz >> 8) & 3u))
                st2 |= ST_EXIT_MISMATCH;
            // K3 stage B
            for (uint32_t r : recs) {
                const uint32_t at = (begin & ~63u) + record_pos(r);
                if (at < total_slots)
                    coef2[at] = (int16_t)record_value(r);
            }
        }
        if (final_slot < total_slots)
            st2 |= ST_SEG_MISMATCH;
        // entropy_scan_*: segmented prefix of the DC sums (reset wherever a subsequence crossed a boundary)
        {
            long long run = 0;
            for (uint32_t i = 0; i < nsub; ++i) {
                dcpre[i] = run;
                run = X[i].seg >= 0 ? dcs[i] : run + dcs[i];
            }
        }
        // K3 stages B/C (k3_fused.cu): the DC predictors entering every strip of 32 MCUs, from dcpre[] and the records of
        // the subsequence the strip's first slot lies in; then the segmented scan inside the strip.  Must give the
        // values the plain sequential prediction (K2 below) gives.
        if (status == 0 && st2 == 0) {
            dc2.assign(g.total_blocks, 0);
            const uint32_t nc = g.ncomp, total_mcus = g.nimages * g.mcus_per_image;
            const uint32_t sps = 32u * nc * 64u, nstrips = (total_mcus + 31u) / 32u;
            std::vector<uint32_t> strip_sub(nstrips, 0); // entropy_scan_apply_kernel: subsequence whose [begin, end) holds the strip's first slot
            for (uint32_t i = 0; i < nsub; ++i) {
                const uint32_t b = start[i], e = i + 1 < nsub ? start[i + 1] : final_slot;
                for (uint32_t s0i = (b + sps - 1u) / sps; e > b && s0i < nstrips && s0i * sps < e; ++s0i)
                    strip_sub[s0i] = i;
            }
            for (uint32_t strip = 0; strip < nstrips; ++strip) {
                const uint32_t mcu0 = strip * 32u, s0 = mcu0 * nc * 64u, first0 = strip_sub[strip];
                const uint32_t img = mcu0 / g.mcus_per_image, mi = mcu0 % g.mcus_per_image;
                const uint32_t mreset = g.restart_interval ? mi - mi % g.restart_interval : 0u;
                const uint32_t reset_slot = (img * g.mcus_per_image + mreset) * nc * 64u;
                const uint32_t ss = start[first0];
                int carry[3] = {0, 0, 0};
                if (ss > reset_slot && reset_slot < s0) // an entry ON the restart slot may still lie before the boundary (padding bits)
                    dcs_unpack(dcpre[first0], carry);
                if (ss < s0 && reset_slot < s0)
                    for (uint32_t r : all_recs[first0]) {
                        const uint32_t at = (ss & ~63u) + record_pos(r);
                        if ((at & 63u) == 0u && at < s0 && at >= reset_slot)
                            carry[(at >> 6) % nc] += record_value(r);
                    }
                int pred[3] = {carry[0], carry[1], carry[2]};
                for (uint32_t m = mcu0; m < std::min(mcu0 + 32u, total_mcus); ++m) {
                    const uint32_t mm = m % g.mcus_per_image;
                    if (g.restart_interval ? (mm % g.restart_interval) == 0 : mm == 0)
                        pred[0] = pred[1] = pred[2] = 0;
                    for (uint32_t c = 0; c < nc; ++c) {
                        pred[c] += coef2[((size_t)m * nc + c) * 64];
                        dc2[m * nc + c] = (int16_t)pred[c];
                    }
                }
            }
        }
        // the Huffman final pass keeps DC differences apart; the records put them into slot 0 of their blocks
        std::vector<int16_t> coef1 = coef;
        for (uint32_t b = 0; b < g.total_blocks; ++b)
            coef1[(size_t)b * 64] = dcdiff[b];
        if (status == 0 && (coef2 != coef1 || st2 != 0))
            records_ok = 0;
        if ((status != 0) != (st2 != 0)) // a stream one flavour rejects, the other must reject too
            records_ok = 0;
        if (info) {
            info[8] = max_rec;
            info[9] = over_kmax;
        }
    }
    // K2
    {
        int32_t pred[3] = {0, 0, 0};
        const uint32_t total_mcus = g.nimages * g.mcus_per_image;
        for (uint32_t m = 0; m < total_mcus; ++m) {
            const uint32_t mi = m % g.mcus_per_image;
            const bool reset = g.restart_interval ? (mi % g.restart_interval) == 0 : mi == 0;
            if (reset)
                pred[0] = pred[1] = pred[2] = 0;
            for (uint32_t c = 0; c < g.ncomp; ++c) {
                pred[c] += dcdiff[m * g.ncomp + c];
                dc[m * g.ncomp + c] = (int16_t)pred[c];
            }
        }
    }
    if (status == 0 && !dc2.empty() && dc2 != dc)
        records_ok = 0; // the scan-based predictors differ from the sequential prediction
    // merged coefficients (what kpeg_cuda_read_coefficients returns)
    std::vector<int16_t> merged((size_t)g.total_blocks * 64);
    for (uint32_t b = 0; b < g.total_blocks; ++b) {
        const bool drop = (g.flags & 1u) && dcdiff[b] == 0;
        merged[(size_t)b * 64] = dc[b];
        for (int i = 1; i < 64; ++i)
            merged[(size_t)b * 64 + i] = drop ? (int16_t)0 : coef[(size_t)b * 64 + i];
    }
    if (coef_out)
        memcpy(coef_out, merged.data(), merged.size() * 2);

    // K3 replay, block by block
    uint32_t exact = 0, colour_exact = 0;
    if (pixels_out) {
        static const ZigZagTables zz = make_zigzag_tables();
        const uint32_t nc = g.ncomp;
        const uint32_t total_mcus = g.nimages * g.mcus_per_image;
        for (uint32_t m = 0; m < total_mcus; ++m) {
            float samp[3][64];
            for (uint32_t c = 0; c < nc; ++c) {
                const int16_t *cz = &merged[((size_t)m * nc + c) * 64];
                float fb[64];
                for (int i = 0; i < 64; ++i)
                    fb[zz.zz2nat[i]] = (float)cz[i] * T->qscale[c][i];
                idct8x8_fast(fb);
                uint32_t A = 0;
                for (int i = 0; i < 64; ++i)
                    A += (uint32_t)abs((int)cz[i]) * (uint32_t)T->qint[c][i];
                const float thresh = 0.5f - tie_band((float)A);
                const float MAGIC = 12582912.0f;
                for (int s = 0; s < 64; ++s) {
                    volatile float t = fb[s] + MAGIC;
                    float r = t - MAGIC;
                    if (fabsf(fb[s] - r) > thresh) {
                        auto at = [&](int zi) { return (int)cz[zi]; };
                        r = (float)exact_sample(at, T->qint[c], T->cosd, T->cc, zz.nat2zz, s >> 3, s & 7);
                        ++exact;
                    }
                    samp[c][s] = r;
                }
            }
            const uint32_t img = m / g.mcus_per_image, mi = m % g.mcus_per_image;
            const uint32_t by = mi / g.mcus_x, bx = mi % g.mcus_x;
            uint8_t *base = pixels_out + (size_t)img * g.width * g.height * nc;
            for (int s = 0; s < 64; ++s) {
                const uint32_t y = by * 8 + (s >> 3), x = bx * 8 + (s & 7);
                if (y >= g.height || x >= g.width)
                    continue;
                uint8_t *o = base + ((size_t)y * g.width + x) * nc;
                if (nc == 3) {
                    int R, G, B;
                    if (!ycc_to_rgb_fast(samp[0][s], samp[1][s], samp[2][s], R, G, B)) {
                        ycc_to_rgb_exact((int)samp[0][s], (int)samp[1][s], (int)samp[2][s], R, G, B);
                        ++colour_exact;
                    }
                    o[0] = (uint8_t)clamp_u8(R);
                    o[1] = (uint8_t)clamp_u8(G);
                    o[2] = (uint8_t)clamp_u8(B);
                } else {
                    const float vv = fminf(fmaxf(samp[0][s] + 128.0f, 0.0f), 255.0f);
                    o[0] = (uint8_t)(int)vv;
                }
            }
        }
    }
    if (info) {
        info[0] = status;
        info[1] = nsub;
        info[2] = rounds;
        info[3] = exact;
        info[4] = colour_exact;
        info[5] = total_bits;
        info[6] = final_slot;
        info[7] = records_ok;
    }
    delete T;
    return KPEG_OK;
}

// idct_core.h widen_f32 on an array (tests: must equal the cast for zero and normal floats)
void emu_widen_f32(const float *in, double *out, size_t n)
{
    for (size_t i = 0; i < n; ++i)
        out[i] = widen_f32(in[i]);
}

// Two-tier colour conversion of one pixel (unshifted samples).  Returns 1 if the exact path ran.
int emu_colour(int y, int cb, int cr, int rgb[3])
{
    int R, G, B;
    if (ycc_to_rgb_fast((float)y, (float)cb, (float)cr, R, G, B)) {
        rgb[0] = clamp_u8(R);
        rgb[1] = clamp_u8(G);
        rgb[2] = clamp_u8(B);
        return 0;
    }
    ycc_to_rgb_exact(y, cb, cr, rgb[0], rgb[1], rgb[2]);
    return 1;
}

// Fast-path IDCT of one block, no tie handling: out[64] floats (unshifted), returns the tie band.
float emu_idct_fast(const int16_t zzc[64], const uint16_t qt[64], float out[64])
{
    static const ZigZagTables zz = make_zigzag_tables();
    float fb[64];
    for (int i = 0; i < 64; ++i) {
        const int nat = zz.zz2nat[i];
        const float qs = (float)((double)qt[i] * aan_scale(nat >> 3) * aan_scale(nat & 7) / 8.0);
        fb[nat] = (float)zzc[i] * qs;
    }
    idct8x8_fast(fb);
    uint32_t A = 0;
    for (int i = 0; i < 64; ++i)
        A += (uint32_t)abs((int)zzc[i]) * (uint32_t)qt[i];
    for (int s = 0; s < 64; ++s)
        out[s] = fb[s];
    return tie_band((float)A);
}

// Fast-path IDCT of one block as K3 sets it up (k3_fused.cu dequant_dezigzag): the prescaled quantisers of
// host_tables.h, and A accumulated in fp32 the way the kernel does it -- |prescaled coefficient| * aan_unscale, pair
// order, four partial sums for the AC terms, the DC term apart.  out[64] = fast samples (unshifted, natural order),
// *a_out = that A; returns the tie band the kernel derives from it.
float emu_idct_fast_k3(const int16_t zzc[64], const uint16_t qt[64], float out[64], float *a_out)
{
    static const ZigZagTables zz = make_zigzag_tables();
    float qscale[64], fb[64];
    for (int i = 0; i < 64; ++i) {
        const int nat = zz.zz2nat[i];
        const double s = aan_scale(nat >> 3) * aan_scale(nat & 7) / 8.0;
        qscale[i] = (float)((double)qt[i] * s);
        fb[nat] = (float)zzc[i] * qscale[i];
    }
    float A[4] = {0.0f, 0.0f, 0.0f, 0.0f}, dcterm = 0.0f;
    for (int p = 0; p < 32; ++p)
        for (int h = 0; h < 2; ++h) {
            const int n = pair_nat(p, h);
            const float f = fb[n]; // (float)c * qpair: the same product as the kernel's packed multiply
            if (n == 0)
                dcterm = fabsf(f) * aan_unscale(n);
            else
                A[2 * h + (p & 1)] = fmaf(fabsf(f), aan_unscale(n), A[2 * h + (p & 1)]);
        }
    const float a = ((A[0] + A[1]) + (A[2] + A[3])) + dcterm;
    idct8x8_fast(fb);
    for (int s = 0; s < 64; ++s)
        out[s] = fb[s];
    *a_out = a;
    return tie_band(a);
}

// Huffman LUT lookup of a left-aligned 32-bit window: returns the packed entry.
// mode 0: as the kernels do it (fast / long table / canonical); mode 1: canonical search only.
uint32_t emu_huff_lookup(const uint8_t counts[16], const uint8_t *symbols, int is_ac, uint32_t win, int mode)
{
    LutSet *L = new LutSet;
    HuffCanon canon;
    uint32_t e = 0xFFFFFFFFu;
    if (build_huff_lut(counts, symbols, is_ac != 0, L, 0, &canon) == 0) {
        if (mode == 1) {
            e = ENTRY_INVALID;
            const uint32_t w16 = win >> 16;
            for (int len = 1; len <= 16; ++len)
                if (w16 < canon.bound[len]) {
                    const uint32_t i = canon.first_idx[len] + ((w16 >> (16 - len)) - canon.first_code[len]);
                    e = pack_entry((uint32_t)len, canon.symbols[i & 255u], is_ac != 0);
                    break;
                }
        } else {
            const PlainLuts PL{L, &canon};
            e = PL.fast(0, win >> (32 - LUT_BITS));
            if ((e & 31u) == 0u)
                e = PL.slow(0, win, e);
        }
    }
    delete L;
    return e;
}

// The same lookup over n windows at once: out[i] = emu_huff_lookup(.., wins[i], mode).
void emu_huff_lookup_many(const uint8_t counts[16], const uint8_t *symbols, int is_ac, const uint32_t *wins, uint32_t n, int mode,
                          uint32_t *out)
{
    LutSet *L = new LutSet;
    HuffCanon canon;
    const bool ok = build_huff_lut(counts, symbols, is_ac != 0, L, 0, &canon) == 0;
    const PlainLuts PL{L, &canon};
    for (uint32_t i = 0; i < n; ++i) {
        const uint32_t win = wins[i];
        uint32_t e = 0xFFFFFFFFu;
        if (ok && mode == 1) {
            e = ENTRY_INVALID;
            const uint32_t w16 = win >> 16;
            for (int len = 1; len <= 16; ++len)
                if (w16 < canon.bound[len]) {
                    const uint32_t k = canon.first_idx[len] + ((w16 >> (16 - len)) - canon.first_code[len]);
                    e = pack_entry((uint32_t)len, canon.symbols[k & 255u], is_ac != 0);
                    break;
                }
        } else if (ok) {
            e = PL.fast(0, win >> (32 - LUT_BITS));
            if ((e & 31u) == 0u)
                e = PL.slow(0, win, e);
        }
        out[i] = e;
    }
    delete L;
}

// How the kernels' tables hold one Huffman table: *long_n = second-level entries in use, canonical[prefix] = 1 for
// every LUT_BITS-bit prefix that starts a longer code but got no sub-table (those codes take huff_slow_lookup).
// Returns the number of such prefixes, or -1 if the table does not build.
int emu_huff_layout(const uint8_t counts[16], const uint8_t *symbols, int is_ac, uint32_t *long_n, uint8_t *canonical)
{
    LutSet *L = new LutSet;
    HuffCanon canon;
    int n = -1;
    if (build_huff_lut(counts, symbols, is_ac != 0, L, 0, &canon) == 0) {
        n = 0;
        *long_n = L->long_n[0];
        for (uint32_t prefix = 0; prefix < (uint32_t)LUT_SIZE; ++prefix) {
            const bool longer = (prefix << (16 - LUT_BITS)) >= canon.bound[LUT_BITS] && (prefix << (16 - LUT_BITS)) < canon.bound[16];
            canonical[prefix] = longer && L->fast[0][prefix] == 0 ? 1u : 0u;
            n += canonical[prefix];
        }
    }
    delete L;
    return n;
}

// host_tables.h restart_padding_decodes: 1 if the job refuses restart intervals and batches for this plan
int emu_restart_padding_decodes(const kpeg_plan *plan) { return restart_padding_decodes(plan) ? 1 : 0; }

int emu_zigzag(int i) { return zigzag_to_natural(i); }

// Byte-parallel classification (classify16_swar) against the byte-wise one (classify16) on every whole
// 16-byte chunk of a buffer: returns the number of chunks whose keep / RSTn masks differ, *bad_differs says
// whether the "unexpected marker" verdict over the whole buffer differs.
uint32_t emu_classify_compare(const uint8_t *scan, uint32_t len, int *bad_differs)
{
    uint32_t mismatches = 0, bad_ref = 0, bad_swar = 0;
    for (uint32_t base = 0; base + 16u <= len; base += 16u) {
        const ByteClass c = classify16(scan, len, base);
        uint32_t b[4];
        memcpy(b, scan + base, 16);
        const uint32_t prev = base ? scan[base - 1] : 0u;
        const uint32_t next = base + 16u < len ? scan[base + 16] : 0xFFu;
        uint32_t keep, rst, bad;
        classify16_swar(b, prev, next, keep, rst, bad);
        if (keep != c.keep || rst != c.rst)
            ++mismatches;
        bad_ref |= c.bad;
        bad_swar |= bad;
    }
    if (bad_differs)
        *bad_differs = (bad_ref != 0) != (bad_swar != 0);
    return mismatches;
}

// The quantiser tables K3 stages by bulk copy (host_tables.h): qscale in zig-zag order, qpair / qdc in the pair
// order of the packed transform; pair_nat_out[2 p + h] = natural position of half h of pair p.
int emu_pair_tables(const kpeg_plan *plan, float *qscale_out, float *qpair_out, float *qdc_out, int *pair_nat_out)
{
    DeviceTables *T = new DeviceTables;
    const char *why = nullptr;
    const int rc = build_device_tables(plan, T, &why);
    if (rc == KPEG_OK) {
        memcpy(qscale_out, T->qscale, sizeof T->qscale);
        memcpy(qpair_out, T->qpair, sizeof T->qpair);
        memcpy(qdc_out, T->qdc, sizeof T->qdc);
        for (int j = 0; j < 64; ++j)
            pair_nat_out[j] = pair_nat(j >> 1, j & 1);
    }
    delete T;
    return rc;
}

} // extern "C"
