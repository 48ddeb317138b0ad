// emu_scaled.cpp -- CPU replay of idct_scaled_kernel (libkpeg_b200/csrc/k3_scaled.cu): the job geometry the host builds
// (make_job_geom), then strip by strip the kernel's stage 1 (one block at a time through idct_reduced.h's transform, into
// the strip's sample array) and stage 2 (every work item of the strip: strip_pixel, scaled_pixel_offset, ycc_rgb).
// Test infrastructure: the tests compare it with the C reference of ref_scaled.c and with the GPU.
#include <stdint.h>
#include <string.h>

#include <vector>

#include "host_tables.h"
#include "idct_reduced.h"

using namespace kpeg;

namespace {

// NM: MCUs per strip (IDCT_MCUS_PER_CTA of kernels.cuh, which needs the CUDA headers: the caller reads it from there)
template <int S>
void run(const JobGeom &g, uint32_t NM, const int16_t *coef, const int32_t (*q)[64], uint8_t *out)
{
    constexpr uint32_t K = 8 / S;
    const uint32_t NC = g.ncomp;
    const uint32_t total_mcus = g.nimages * g.mcus_per_image;
    const uint32_t nstrips = (total_mcus + NM - 1) / NM;
    const OutGeom o = out_geom(g);
    std::vector<uint8_t> samp((size_t)NC * NM * K * K);
    for (uint32_t strip = 0; strip < nstrips; ++strip) {
        const uint32_t mcu0 = strip * NM;
        for (uint32_t t = 0; t < NC * NM; ++t) { // stage 1: thread t = block (ml, comp)
            const uint32_t comp = t / NM, ml = t % NM, m = mcu0 + ml;
            if (m >= total_mcus)
                continue;
            const int16_t *blk = coef + ((size_t)m * NC + comp) * 64u;
            auto dq = [&](int zz) -> int32_t { return (int32_t)blk[zz] * q[comp][zz]; };
            red::idct_reduced<S>(dq, &samp[((size_t)comp * NM + ml) * K * K]);
        }
        for (uint32_t p = 0; p < NM * K * K; ++p) { // stage 2
            const red::StripPixel px = red::strip_pixel(p, K, NM);
            const uint32_t m = mcu0 + px.ml;
            if (m >= total_mcus)
                continue;
            const uint64_t off = red::scaled_pixel_offset(g, o, m, px.r, px.c);
            if (off == ~(uint64_t)0)
                continue;
            const uint32_t s = px.r * K + px.c;
            auto sample = [&](uint32_t c) { return (int)samp[((size_t)c * NM + px.ml) * K * K + s]; };
            if (NC == 3) {
                const uint32_t v = red::ycc_rgb(sample(0), sample(1), sample(2));
                out[off] = (uint8_t)v;
                out[off + 1] = (uint8_t)(v >> 8);
                out[off + 2] = (uint8_t)(v >> 16);
            } else {
                out[off] = (uint8_t)sample(0);
            }
        }
    }
}

} // namespace

extern "C" {

// coef: [nimages * blocks][64] zig-zag, MCU-interleaved (as K2's tiles hold them); qt: [ncomp][64] zig-zag;
// flags: KPEG_FLAG_SCALE_* (and anything else a plan may carry); strip_mcus: MCUs per strip, as the kernel is launched.
// out: kpeg_output_size bytes per image.
int emu_scaled_decode(const int16_t *coef, const uint16_t *qt, int width, int height, int ncomp, int nimages, uint32_t flags,
                      uint32_t strip_mcus, uint8_t *out)
{
    kpeg_plan pl;
    memset(&pl, 0, sizeof pl);
    pl.width = (uint16_t)width;
    pl.height = (uint16_t)height;
    pl.ncomp = (uint8_t)ncomp;
    pl.flags = flags;
    JobGeom g;
    const char *why = nullptr;
    if (strip_mcus == 0 || width < 1 || width > 65535 || height < 1 || height > 65535 || make_job_geom(&pl, (uint32_t)nimages, 512u, &g, &why) != KPEG_OK)
        return KPEG_ERR_ARG;
    int32_t q[3][64];
    for (int c = 0; c < ncomp; ++c)
        for (int i = 0; i < 64; ++i)
            q[c][i] = qt[c * 64 + i];
    switch (scale_denom(flags)) {
    case 2: run<2>(g, strip_mcus, coef, q, out); break;
    case 4: run<4>(g, strip_mcus, coef, q, out); break;
    case 8: run<8>(g, strip_mcus, coef, q, out); break;
    default: return KPEG_ERR_ARG;
    }
    return KPEG_OK;
}

// kpeg_common.h's output geometry, as the host uses it (kpeg_output_size and the row placement of bands)
int emu_out_geom(int width, int height, int ncomp, uint32_t flags, uint32_t *w, uint32_t *h, uint64_t *bytes)
{
    const OutGeom o = out_geom((uint32_t)width, (uint32_t)height, (uint32_t)ncomp, flags);
    *w = o.width;
    *h = o.height;
    *bytes = o.bytes();
    return (int)o.scale;
}

} // extern "C"
