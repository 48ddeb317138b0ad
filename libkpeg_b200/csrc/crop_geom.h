// crop_geom.h -- the geometry of a crop decode (kpeg_cuda_decode_crop*): which K3 strips hold pixels of the rectangles, and
// where an output pixel lands in the crop buffer.  KPEG_HD functions, so that the kernels and tests/emu/emu_crop.cpp compile
// the same source.
//
// A rectangle is given in the coordinates of the output image (out_geom: full size, or the reduced image of a
// KPEG_FLAG_SCALE_* decode).  The crop of image i is written row-major, rows of w * ncomp bytes, tightly packed, at byte
// `out_off` of the job's output; a batch's crops lie back to back.
#ifndef KPEG_CROP_GEOM_H
#define KPEG_CROP_GEOM_H

#include <stdint.h>

#include <vector>

#include "kpeg_common.h"

namespace kpeg {

struct CropWin {
    uint32_t x0, y0, w, h; // in output pixels
    uint64_t out_off;      // byte offset of this image's crop in the job's output
};

constexpr uint64_t CROP_SKIP = ~(uint64_t)0;

// byte offset of output pixel (ox, oy) of an image in the crop output, or CROP_SKIP when it lies outside the rectangle
KPEG_HD uint64_t crop_pixel_offset(const CropWin &c, uint32_t ncomp, uint32_t ox, uint32_t oy)
{
    if (ox - c.x0 >= c.w || oy - c.y0 >= c.h) // unsigned: also below x0 / y0
        return CROP_SKIP;
    return c.out_off + ((uint64_t)(oy - c.y0) * c.w + (ox - c.x0)) * ncomp;
}

// The MCUs whose output pixels meet the rectangle: block columns [bx0, bx1] of block rows [by0, by1].  An MCU covers output
// columns [bx K, bx K + K) and rows [by K, by K + K), K = 8 / scale (clipped at the image's edge).
struct CropMcus {
    uint32_t bx0, bx1, by0, by1;
};
KPEG_HD CropMcus crop_mcus(const CropWin &c, uint32_t scale)
{
    const uint32_t K = 8u / scale;
    return CropMcus{c.x0 / K, (c.x0 + c.w - 1u) / K, c.y0 / K, (c.y0 + c.h - 1u) / K};
}

// the window is a non-empty rectangle inside the output image o
KPEG_HD bool crop_fits(const OutGeom &o, uint32_t x, uint32_t y, uint32_t w, uint32_t h)
{
    return w != 0u && h != 0u && x < o.width && y < o.height && w <= o.width - x && h <= o.height - y;
}

// Host: the K3 strips (IDCT_MCUS_PER_CTA consecutive MCUs of the job, strip_mcus here) that hold at least one MCU meeting the
// rectangle of its image, sorted, each once (a strip that spans two images of a batch too).  wins[i] is image i's
// rectangle.  MCUs are visited in job order, so the strips come out non-decreasing.
inline std::vector<uint32_t> crop_strip_list(const JobGeom &g, const CropWin *wins, uint32_t strip_mcus)
{
    const uint32_t scale = out_geom(g).scale;
    std::vector<uint32_t> list;
    for (uint32_t img = 0; img < g.nimages; ++img) {
        const CropMcus m = crop_mcus(wins[img], scale);
        for (uint32_t by = m.by0; by <= m.by1; ++by) {
            const uint64_t row = (uint64_t)img * g.mcus_per_image + (uint64_t)by * g.mcus_x;
            const uint32_t s0 = (uint32_t)((row + m.bx0) / strip_mcus), s1 = (uint32_t)((row + m.bx1) / strip_mcus);
            for (uint32_t s = s0; s <= s1; ++s)
                if (list.empty() || list.back() != s)
                    list.push_back(s);
        }
    }
    return list;
}

} // namespace kpeg
#endif
