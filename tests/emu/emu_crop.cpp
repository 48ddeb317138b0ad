// emu_crop.cpp -- the crop decode's geometry (libkpeg_b200/csrc/crop_geom.h) compiled for the host: the strip list the host
// uploads, and where every output pixel lands in the crop output, by the functions the kernels store through
// (crop_pixel_offset in idct_kernel, scaled_crop_offset in idct_scaled_kernel).  Test infrastructure: test_crop_host.py
// compares both with a numpy brute force.
#include <stdint.h>

#include <vector>

#include "crop_geom.h"
#include "idct_reduced.h"

using namespace kpeg;

namespace {

JobGeom geom(uint32_t w, uint32_t h, uint32_t ncomp, uint32_t flags, uint32_t nimages)
{
    JobGeom g = {};
    g.width = w;
    g.height = h;
    g.ncomp = ncomp;
    g.mcus_x = (w + 7u) / 8u;
    g.mcus_y = (h + 7u) / 8u;
    g.mcus_per_image = g.mcus_x * g.mcus_y;
    g.nimages = nimages;
    g.flags = flags;
    return g;
}

// rects: [nimages][4] = x, y, w, h; the crops lie back to back
std::vector<CropWin> windows(const JobGeom &g, const uint32_t *rects)
{
    std::vector<CropWin> wins(g.nimages);
    uint64_t off = 0;
    for (uint32_t i = 0; i < g.nimages; ++i) {
        wins[i] = CropWin{rects[4 * i], rects[4 * i + 1], rects[4 * i + 2], rects[4 * i + 3], off};
        off += (uint64_t)rects[4 * i + 2] * rects[4 * i + 3] * g.ncomp;
    }
    return wins;
}

} // namespace

extern "C" {

// the sorted strip list -> out[0, cap); returns its length
uint32_t emu_crop_strips(uint32_t w, uint32_t h, uint32_t ncomp, uint32_t flags, uint32_t nimages, const uint32_t *rects,
                         uint32_t strip_mcus, uint32_t *out, uint32_t cap)
{
    const JobGeom g = geom(w, h, ncomp, flags, nimages);
    const std::vector<CropWin> wins = windows(g, rects);
    const std::vector<uint32_t> list = crop_strip_list(g, wins.data(), strip_mcus);
    for (size_t i = 0; i < list.size() && i < cap; ++i)
        out[i] = list[i];
    return (uint32_t)list.size();
}

// out[img][oy][ox] (output image size) = byte offset of that pixel in the crop output, or -1 where it is skipped; every
// pixel of every MCU is visited as the kernels visit it: sample (r, c) of the K x K square of MCU m
void emu_crop_map(uint32_t w, uint32_t h, uint32_t ncomp, uint32_t flags, uint32_t nimages, const uint32_t *rects, int64_t *out)
{
    const JobGeom g = geom(w, h, ncomp, flags, nimages);
    const OutGeom o = out_geom(g);
    const std::vector<CropWin> wins = windows(g, rects);
    const uint32_t K = 8u / o.scale;
    for (uint32_t m = 0; m < g.nimages * g.mcus_per_image; ++m) {
        const uint32_t img = m / g.mcus_per_image, mi = m - img * g.mcus_per_image;
        const uint32_t by = mi / g.mcus_x, bx = mi - by * g.mcus_x;
        for (uint32_t r = 0; r < K; ++r)
            for (uint32_t c = 0; c < K; ++c) {
                const uint32_t ox = bx * K + c, oy = by * K + r;
                if (ox >= o.width || oy >= o.height)
                    continue; // beyond the ragged edge: no pixel of the output
                const uint64_t off = o.scale == 1 ? crop_pixel_offset(wins[img], ncomp, ox, oy)
                                                  : red::scaled_crop_offset(g, o, wins.data(), m, r, c);
                out[((uint64_t)img * o.height + oy) * o.width + ox] = off == CROP_SKIP ? -1 : (int64_t)off;
            }
    }
}

} // extern "C"
