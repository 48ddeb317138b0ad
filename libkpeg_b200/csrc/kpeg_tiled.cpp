// kpeg_tiled.cpp -- multi-device entry points of the C ABI (include/kpeg_cuda.h): a process-wide pool of decode
// contexts, and the decode of ONE restart-marked image spread over several GPUs.
//
// The reference has no tiling and no devices; what has to come out is the frame Image::createImageFromMCUs assembles
// (reference src/Image.cpp:51-70: MCU (by, bx) covers pixel rows 8 by .. 8 by + 7) -- here every band of whole MCU rows
// is decoded by its own GPU straight into its rows of the caller's frame (a host gather; no device-to-device traffic),
// or into its rows of a frame on one GPU (peer copies over NVLink).  Host code only: everything CUDA goes through
// the single-device C ABI in kpeg_cuda.cu, one host thread per device.
#include <string.h>

#include <algorithm>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

#include "kpeg_common.h"
#include "kpeg_cuda.h"

namespace {

std::mutex g_pool_mutex;
std::vector<std::pair<int, kpeg_ctx *>> g_pool; // idle contexts: (device, context)

thread_local std::string t_tiled_err;

} // namespace

// ---- context pool -----------------------------------------------------------------------------------------
// Creating a context costs streams, pinned bookkeeping and, at its first decode, every scratch allocation; callers
// that decode one file per object (kpeg::JPEGDecoder) borrow a context instead and hand it back.
extern "C" int kpeg_cuda_acquire(int device, kpeg_ctx **out)
{
    if (!out)
        return KPEG_ERR_ARG;
    {
        std::lock_guard<std::mutex> lock(g_pool_mutex);
        for (size_t i = 0; i < g_pool.size(); ++i)
            if (g_pool[i].first == device) {
                *out = g_pool[i].second;
                g_pool.erase(g_pool.begin() + (long)i);
                return KPEG_OK;
            }
    }
    return kpeg_cuda_create(device, out);
}

extern "C" void kpeg_cuda_release(int device, kpeg_ctx *ctx)
{
    if (!ctx)
        return;
    std::lock_guard<std::mutex> lock(g_pool_mutex);
    g_pool.emplace_back(device, ctx);
}

extern "C" void kpeg_cuda_pool_clear(void)
{
    std::vector<std::pair<int, kpeg_ctx *>> idle;
    {
        std::lock_guard<std::mutex> lock(g_pool_mutex);
        idle.swap(g_pool);
    }
    for (auto &e : idle)
        kpeg_cuda_destroy(e.second);
}

extern "C" const char *kpeg_tiled_last_error(void) { return t_tiled_err.c_str(); }

// ---- one image over several devices ---------------------------------------------------------------------------
namespace {

struct BandJob {
    int device = 0;
    kpeg_plan plan;
    const uint8_t *scan = nullptr;
    size_t len = 0;
    uint32_t row0 = 0, rows = 0; // pixel rows of the full-size image
    size_t out_off = 0;         // where the band's output rows begin in the frame (reduced-size decodes: the reduced rows)
    int rc = KPEG_OK;
    std::string err;
    kpeg_stats stats;
};

// RSTn markers (FF D0 .. FF D7) in [p, end): inside entropy-coded data an FF is followed by 00, FF or a marker
uint64_t count_restart_markers(const uint8_t *p, const uint8_t *end)
{
    uint64_t n = 0;
    while (p + 1 < end) {
        const uint8_t *q = (const uint8_t *)memchr(p, 0xFF, (size_t)(end - 1 - p));
        if (!q)
            break;
        n += (q[1] & 0xF8u) == 0xD0u ? 1u : 0u;
        p = q + ((q[1] & 0xF8u) == 0xD0u ? 2 : 1);
    }
    return n;
}

} // namespace

// Host-only (include/kpeg_cuda.h): bands of whole MCU rows cut at BYTE positions.
extern "C" int kpeg_split_restart_bands_by_bytes(const uint8_t *scan, size_t len, const kpeg_plan *plan, int parts,
                                                 uint64_t *out_begin, uint64_t *out_end, uint32_t *out_row)
{
    if (!scan || !plan || parts < 1 || !out_begin || !out_end || !out_row)
        return KPEG_ERR_ARG;
    const uint32_t mx = ((uint32_t)plan->width + 7u) / 8u, my = ((uint32_t)plan->height + 7u) / 8u, ri = plan->restart_interval;
    if (parts < 2 || ri == 0 || ri % mx != 0 || my < (uint32_t)parts * (ri / mx) * 2u)
        return KPEG_ERR_UNSUPPORTED;
    const uint32_t rpi = ri / mx;
    out_begin[0] = 0;
    for (int k = 1; k < parts; ++k) {
        const uint8_t *p = scan + std::max<size_t>(len * (size_t)k / (size_t)parts, (size_t)out_begin[k - 1] + 1), *stop = scan + len, *cut = nullptr;
        while (p + 1 < stop) {
            const uint8_t *q = (const uint8_t *)memchr(p, 0xFF, (size_t)(stop - 1 - p));
            if (!q)
                break;
            if ((q[1] & 0xF8u) == 0xD0u) {
                cut = q;
                break;
            }
            p = q + 1;
        }
        if (!cut)
            return KPEG_ERR_UNSUPPORTED; // no marker left: fewer intervals than bands
        out_end[k - 1] = (uint64_t)(cut - scan);
        out_begin[k] = out_end[k - 1] + 2u;
    }
    out_end[parts - 1] = len;
    std::vector<uint64_t> markers((size_t)parts, 0);
    std::vector<std::thread> th;
    for (int k = 0; k + 1 < parts; ++k) // the last band holds whatever rows are left
        th.emplace_back([&, k] { markers[(size_t)k] = count_restart_markers(scan + out_begin[k], scan + out_end[k]); });
    for (auto &t : th)
        t.join();
    uint32_t row0 = 0;
    for (int k = 0; k < parts; ++k) {
        out_row[k] = row0;
        if (k + 1 < parts) {
            const uint64_t rows = (markers[(size_t)k] + 1u) * rpi;
            if (rows >= my - row0)
                return KPEG_ERR_STREAM; // more restart intervals than the frame has rows for
            row0 += (uint32_t)rows;
        }
    }
    out_row[parts] = my;
    return KPEG_OK;
}

namespace {

// Cut `scan` into one band per device; images without usable restart markers become one band on devices[0].
// Scans of 1 MB and more with a restart interval of whole MCU rows are cut at BYTE positions and the restart intervals
// of every band are counted by one host thread per band (kpeg_split_restart_bands_by_bytes); otherwise the cut points
// are found at given rows by ONE walk over all markers (kpeg_split_restart_bands: 12 ms for the 96 MB of a 16384x16384
// image, several times what a band then takes on its GPU).
int make_bands(const int *devices, int ndev, const kpeg_plan *plan, const uint8_t *scan, size_t len, std::vector<BandJob> &jobs)
{
    std::vector<uint64_t> b0((size_t)ndev), b1((size_t)ndev);
    std::vector<uint32_t> row((size_t)ndev + 1);
    int parts = ndev;
    int rc = KPEG_ERR_UNSUPPORTED;
    if (ndev > 1 && len >= ((size_t)1 << 20))
        rc = kpeg_split_restart_bands_by_bytes(scan, len, plan, ndev, b0.data(), b1.data(), row.data());
    if (rc == KPEG_ERR_UNSUPPORTED && ndev > 1)
        rc = kpeg_split_restart_bands(scan, len, plan, ndev, b0.data(), b1.data(), row.data());
    if (rc == KPEG_ERR_STREAM)
        return rc;
    if (rc != KPEG_OK) { // no restart interval that lines up with MCU rows: the image does not shard (DESIGN.md, "replicas only")
        parts = 1;
        b0[0] = 0;
        b1[0] = len;
        row[0] = 0;
        row[1] = ((uint32_t)plan->height + 7u) / 8u;
    }
    for (int k = 0; k < parts; ++k) {
        const uint32_t r0 = std::min<uint32_t>(row[(size_t)k] * 8u, plan->height), r1 = std::min<uint32_t>(row[(size_t)k + 1] * 8u, plan->height);
        if (r1 <= r0)
            continue; // more devices than MCU rows
        BandJob j;
        j.device = devices[k];
        j.plan = *plan;
        j.plan.height = (uint16_t)(r1 - r0);
        j.scan = scan + b0[(size_t)k];
        j.len = (size_t)(b1[(size_t)k] - b0[(size_t)k]);
        j.row0 = r0;
        j.rows = r1 - r0;
        const kpeg::OutGeom o = kpeg::out_geom(plan->width, plan->height, plan->ncomp, plan->flags);
        j.out_off = (size_t)o.mcu_row(row[(size_t)k]) * o.row_bytes();
        memset(&j.stats, 0, sizeof j.stats);
        jobs.push_back(j);
    }
    return KPEG_OK;
}

template <class F>
int run_bands(std::vector<BandJob> &jobs, F &&one)
{
    std::vector<std::thread> th;
    for (size_t k = 1; k < jobs.size(); ++k)
        th.emplace_back([&, k] { one(jobs[k]); });
    if (!jobs.empty())
        one(jobs[0]);
    for (auto &t : th)
        t.join();
    for (const BandJob &j : jobs)
        if (j.rc != KPEG_OK) {
            t_tiled_err = "device " + std::to_string(j.device) + ": " + j.err;
            return j.rc;
        }
    return KPEG_OK;
}

void sum_stats(const std::vector<BandJob> &jobs, const kpeg_plan *plan, kpeg_stats *stats)
{
    if (!stats)
        return;
    memset(stats, 0, sizeof *stats);
    const kpeg::OutGeom o = kpeg::out_geom(plan->width, plan->height, plan->ncomp, plan->flags);
    stats->width = o.width;
    stats->height = o.height;
    stats->ncomp = plan->ncomp;
    for (const BandJob &j : jobs) {
        stats->scan_bytes += j.stats.scan_bytes;
        stats->unstuffed_bytes += j.stats.unstuffed_bytes;
        stats->segments += j.stats.segments;
        stats->subsequences += j.stats.subsequences;
        stats->sync_rounds = std::max(stats->sync_rounds, j.stats.sync_rounds);
        stats->exact_samples += j.stats.exact_samples;
        stats->kernel_launches += j.stats.kernel_launches;
    }
}

} // namespace

extern "C" int kpeg_cuda_decode_tiled(const int *devices, int ndev, const kpeg_plan *plan, const uint8_t *scan, size_t scan_len,
                                      uint8_t *pixels_out, kpeg_stats *stats)
{
    if (!devices || ndev < 1 || !plan || !scan || !pixels_out)
        return KPEG_ERR_ARG;
    t_tiled_err.clear();
    std::vector<BandJob> jobs;
    const int src = make_bands(devices, ndev, plan, scan, scan_len, jobs);
    if (src != KPEG_OK) {
        t_tiled_err = "restart markers do not match the restart interval";
        return src;
    }
    const int rc = run_bands(jobs, [&](BandJob &j) {
        kpeg_ctx *ctx = nullptr;
        j.rc = kpeg_cuda_acquire(j.device, &ctx);
        if (j.rc != KPEG_OK) {
            j.err = "no usable CUDA device";
            return;
        }
        j.rc = kpeg_cuda_decode(ctx, &j.plan, j.scan, j.len, pixels_out + j.out_off, &j.stats);
        if (j.rc != KPEG_OK)
            j.err = kpeg_cuda_last_error(ctx);
        kpeg_cuda_release(j.device, ctx);
    });
    sum_stats(jobs, plan, stats);
    return rc;
}

// Same, the frame assembled in DEVICE memory of `dst_device` (d_frame: kpeg_output_size bytes, allocated by the
// caller on that device): every band is decoded on its own GPU and its rows travel by one peer copy (NVLink; staged
// through the host by the driver where peer access is unavailable).  A consumer on dst_device never pays PCIe.
extern "C" int kpeg_cuda_decode_tiled_device(const int *devices, int ndev, const kpeg_plan *plan, const uint8_t *scan,
                                             size_t scan_len, int dst_device, uint8_t *d_frame, kpeg_stats *stats)
{
    if (!devices || ndev < 1 || !plan || !scan || !d_frame)
        return KPEG_ERR_ARG;
    t_tiled_err.clear();
    std::vector<BandJob> jobs;
    const int src = make_bands(devices, ndev, plan, scan, scan_len, jobs);
    if (src != KPEG_OK) {
        t_tiled_err = "restart markers do not match the restart interval";
        return src;
    }
    const int rc = run_bands(jobs, [&](BandJob &j) {
        kpeg_ctx *ctx = nullptr;
        j.rc = kpeg_cuda_acquire(j.device, &ctx);
        if (j.rc != KPEG_OK) {
            j.err = "no usable CUDA device";
            return;
        }
        j.rc = kpeg_cuda_decode_to_peer(ctx, &j.plan, j.scan, j.len, dst_device, d_frame + j.out_off, &j.stats);
        if (j.rc != KPEG_OK)
            j.err = kpeg_cuda_last_error(ctx);
        kpeg_cuda_release(j.device, ctx);
    });
    sum_stats(jobs, plan, stats);
    return rc;
}

extern "C" int kpeg_cuda_decode_file_tiled(const int *devices, int ndev, const uint8_t *file, size_t len, uint32_t flags,
                                           uint8_t *pixels_out, size_t cap, kpeg_plan *plan_out, kpeg_stats *stats)
{
    if (!devices || ndev < 1 || !file || !pixels_out)
        return KPEG_ERR_ARG;
    kpeg_plan plan;
    size_t off = 0, slen = 0;
    const int prc = kpeg_parse_jfif(file, len, &plan, &off, &slen);
    if (prc != KPEG_OK) {
        t_tiled_err = prc == KPEG_ERR_UNSUPPORTED ? "unsupported JPEG coding" : "malformed JFIF container";
        return prc;
    }
    plan.flags = flags;
    if (plan_out)
        *plan_out = plan;
    if (kpeg_output_size(&plan, nullptr, nullptr) > cap) {
        t_tiled_err = "pixel buffer too small";
        return KPEG_ERR_ARG;
    }
    return kpeg_cuda_decode_tiled(devices, ndev, &plan, file + off, slen, pixels_out, stats);
}
