"""The crop decode on the CPU: its geometry (csrc/crop_geom.h, compiled into tests/emu/emu_crop.cpp) against a numpy brute
force, the ctypes mirror of kpeg_crop, the Python binding's checks of a crop tuple and the CLI's --crop parse error.
What the GPU has to produce is checked in test_gpu_crop.py."""
import ctypes as C
import re
import subprocess
from pathlib import Path

import numpy as np
import pytest

from libkpeg_b200 import api

ROOT = Path(__file__).resolve().parent.parent
EMU = ROOT / "tests" / "emu" / "libkpeg_emu_crop.so"
KPEG = ROOT / "libkpeg_b200" / "lib" / "kpeg"
SCALES = [1, 2, 4, 8]


def strip_mcus() -> int:
    text = (ROOT / "libkpeg_b200" / "csrc" / "kernels.cuh").read_text()
    return int(re.search(r"constexpr int IDCT_MCUS_PER_CTA = (\d+);", text).group(1))


@pytest.fixture(scope="module")
def emu():
    lib = C.CDLL(str(EMU))
    u32p, i64p = C.POINTER(C.c_uint32), C.POINTER(C.c_int64)
    lib.emu_crop_strips.restype = C.c_uint32
    lib.emu_crop_strips.argtypes = [C.c_uint32] * 5 + [u32p, C.c_uint32, u32p, C.c_uint32]
    lib.emu_crop_map.restype = None
    lib.emu_crop_map.argtypes = [C.c_uint32] * 5 + [u32p, i64p]
    return lib


def out_size(w, h, scale):
    return -(-w // scale), -(-h // scale)


def random_rect(rng, ow, oh):
    x, y = int(rng.integers(0, ow)), int(rng.integers(0, oh))
    kind = rng.integers(0, 4)
    if kind == 0:
        return (x, y, 1, 1)
    if kind == 1:
        return (0, 0, ow, oh)
    return (x, y, int(rng.integers(1, ow - x + 1)), int(rng.integers(1, oh - y + 1)))


def brute_strips(w, h, scale, rects, nm):
    ow, oh = out_size(w, h, scale)
    k = 8 // scale
    mx, my = -(-w // 8), -(-h // 8)
    strips = set()
    for img, (x, y, cw, ch) in enumerate(rects):
        for by in range(my):
            for bx in range(mx):
                x0, x1 = bx * k, min(bx * k + k, ow)
                y0, y1 = by * k, min(by * k + k, oh)
                if x0 < x + cw and x1 > x and y0 < y + ch and y1 > y:
                    strips.add((img * mx * my + by * mx + bx) // nm)
    return sorted(strips)


def brute_map(w, h, nc, scale, rects):
    ow, oh = out_size(w, h, scale)
    out = np.full((len(rects), oh, ow), -1, np.int64)
    off = 0
    for img, (x, y, cw, ch) in enumerate(rects):
        yy, xx = np.mgrid[0:ch, 0:cw]
        out[img, y:y + ch, x:x + cw] = off + (yy * cw + xx) * nc
        off += cw * ch * nc
    return out


def plans(seed=7, n=40):
    rng = np.random.default_rng(seed)
    sizes = [(8, 8), (1, 1), (17, 9), (203, 77), (300, 41), (64, 64), (257, 130), (33, 250), (1000, 24)]
    for i in range(n):
        w, h = sizes[i % len(sizes)] if i < len(sizes) else (int(rng.integers(1, 400)), int(rng.integers(1, 200)))
        yield w, h, (1, 3)[i % 2], SCALES[i % 4], 1 + i % 5, int(rng.integers(0, 2 ** 31))


@pytest.mark.parametrize("w,h,nc,scale,nimg,seed", list(plans()))
def test_geometry_matches_brute_force(emu, w, h, nc, scale, nimg, seed):
    rng = np.random.default_rng(seed)
    ow, oh = out_size(w, h, scale)
    rects = [random_rect(rng, ow, oh) for _ in range(nimg)]
    flat = (C.c_uint32 * (4 * nimg))(*[v for r in rects for v in r])
    flags = {1: 0, 2: api.KPEG_FLAG_SCALE_1_2, 4: api.KPEG_FLAG_SCALE_1_4, 8: api.KPEG_FLAG_SCALE_1_8}[scale]
    nm = strip_mcus()
    cap = nimg * (-(-w // 8)) * (-(-h // 8)) // nm + 2
    buf = (C.c_uint32 * cap)()
    n = emu.emu_crop_strips(w, h, nc, flags, nimg, flat, nm, buf, cap)
    assert list(buf[:n]) == brute_strips(w, h, scale, rects, nm), rects
    got = np.full((nimg, oh, ow), -7, np.int64)
    emu.emu_crop_map(w, h, nc, flags, nimg, flat, got.ctypes.data_as(C.POINTER(C.c_int64)))
    want = brute_map(w, h, nc, scale, rects)
    assert np.array_equal(got, want), rects
    inside = got[got >= 0]  # every crop pixel once, at a distinct offset inside the crops' bytes
    assert inside.size == sum(cw * ch for _, _, cw, ch in rects)
    assert np.unique(inside).size == inside.size and inside.max() < sum(cw * ch * nc for _, _, cw, ch in rects)


def test_4k_centre_crop_lists_one_strip_per_mcu_row(emu):
    """A 224 x 224 centre crop of 3840 x 2160: 28 MCU rows, each inside one strip (a 480-MCU row is 15 whole strips)."""
    rect = ((3840 - 224) // 2, (2160 - 224) // 2, 224, 224)
    flat = (C.c_uint32 * 4)(*rect)
    buf = (C.c_uint32 * 64)()
    n = emu.emu_crop_strips(3840, 2160, 3, 0, 1, flat, strip_mcus(), buf, 64)
    assert n == 28 and n == len(set(buf[:n]))


def test_crop_struct_matches_header():
    hdr = (ROOT / "include" / "kpeg_cuda.h").read_text()
    body = re.search(r"typedef struct kpeg_crop \{(.*?)\} kpeg_crop;", hdr, re.S).group(1)
    assert re.sub(r"\s+", " ", body).strip() == "uint32_t x, y, width, height;"
    assert C.sizeof(api.Crop) == 16 and [f for f, _ in api.Crop._fields_] == ["x", "y", "width", "height"]


@pytest.mark.parametrize("bad", [5, (1, 2, 3), (1, 2, 3, 4, 5), (0, 0, 0, 4), (0, 0, 4, 0), (-1, 0, 4, 4),
                                 (0, 0, 4.0, 4), ("0", 0, 4, 4), (True, 0, 4, 4), (0, 0, 1 << 32, 4)])
def test_python_rejects_malformed_crops(bad):
    with pytest.raises(ValueError):
        api.crop_struct(bad)
    plan = api.Plan()
    plan.width, plan.height, plan.ncomp = 16, 16, 3
    with pytest.raises(ValueError):  # before any C call: the decoder is never touched
        api.Decoder.decode_scan(None, plan, np.zeros(4, np.uint8), crop=bad)
    with pytest.raises(ValueError):
        api.Decoder.decode_batch(None, plan, [np.zeros(4, np.uint8)], crops=[bad])


def test_crop_shape():
    plan = api.Plan()
    plan.width, plan.height, plan.ncomp = 100, 50, 3
    assert api.crop_shape(plan, (3, 4, 10, 7)) == (7, 10, 3)
    plan.ncomp = 1
    assert api.crop_shape(plan, np.array([0, 0, 5, 2])) == (2, 5)


@pytest.mark.parametrize("arg", ["12x3+1", "0x3+1+1", "3x0+0+0", "axb+c+d", "12x3+1+2+", "-4x3+1+2", "12X3+1+2", ""])
def test_cli_rejects_malformed_crop(tmp_path, arg):
    """A malformed --crop prints the usage and fails before anything is decoded (no GPU needed)."""
    proc = subprocess.run([str(KPEG), "--quiet", "--crop", arg, "x.jpg"], cwd=tmp_path, capture_output=True, text=True)
    assert proc.returncode != 0
    assert "Malformed --crop" in proc.stdout and "--crop WxH+X+Y" in proc.stdout
    assert not (tmp_path / "x.ppm").exists()
