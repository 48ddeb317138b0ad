"""Reference, CPU replay and inputs of the reduced-size decode (KPEG_FLAG_SCALE_*), for test_scaled_host.py and
test_gpu_scaled.py.

The reference (emu/ref_scaled.c, restated from libjpeg-turbo's jidctred.c / jdmaster.c / jdcolor.c) reconstructs the
oracle's quantised coefficients -- either parity mode -- with the file's quantisers.  The replay (emu/emu_scaled.cpp)
runs the kernel's per-block and per-pixel code from libkpeg_b200/csrc/idct_reduced.h on the same coefficients."""
from __future__ import annotations

import ctypes as C
import functools
import io
from pathlib import Path

import numpy as np

import coef_fields as CF
import helpers as H
from libkpeg_b200.api import KPEG_FLAG_REF_PARITY, output_shape, parse_jfif_scans, scale_flags

EMU = Path(__file__).resolve().parent / "emu"
GOLDEN = Path(__file__).resolve().parent / "golden"
SCALES = (2, 4, 8)
# MCUs per strip of the reconstruction kernels (IDCT_MCUS_PER_CTA), read from the source the kernels are built from
STRIP_MCUS = int(CF._constexpr((Path(__file__).resolve().parent.parent / "libkpeg_b200" / "csrc" / "kernels.cuh").read_text(),
                               "IDCT_MCUS_PER_CTA"))


@functools.lru_cache(maxsize=None)
def _libs():
    from libkpeg_b200._build import build_emu_scaled
    build_emu_scaled()
    ref = C.CDLL(str(EMU / "libkpeg_ref_scaled.so"))
    ref.kpo_reconstruct_scaled.restype = C.c_int
    ref.kpo_reconstruct_scaled.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p]
    emu = C.CDLL(str(EMU / "libkpeg_emu_scaled.so"))
    emu.emu_scaled_decode.restype = C.c_int
    emu.emu_scaled_decode.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_uint32, C.c_uint32,
                                      C.c_void_p]
    emu.emu_out_geom.restype = C.c_int
    emu.emu_out_geom.argtypes = [C.c_int, C.c_int, C.c_int, C.c_uint32, C.POINTER(C.c_uint32), C.POINTER(C.c_uint32),
                                 C.POINTER(C.c_uint64)]
    return ref, emu


def frame_of(jpg: bytes):
    """-> (width, height, ncomp, [ncomp][64] zig-zag quantisers of the components) of an interleaved or per-component file"""
    frame, scans = parse_jfif_scans(jpg)
    nc = int(frame.ncomp)
    qt = np.zeros((nc, 64), np.uint16)
    for sc in scans:
        for j in range(sc.plan.ncomp):
            qt[int(sc.comp[j])] = list(sc.plan.qt[int(sc.plan.comp_tq[j])])
    return int(frame.width), int(frame.height), nc, qt


def shape(w: int, h: int, nc: int, scale: int):
    ow, oh = -(-w // scale), -(-h // scale)
    return (oh, ow, 3) if nc == 3 else (oh, ow)


def coefficients(jpg: bytes, parity: bool) -> np.ndarray:
    return np.ascontiguousarray(H.oracle_decode(jpg, parity=parity, want_pixels=False)["coef"], dtype=np.int16)


def reconstruct(coef: np.ndarray, qt: np.ndarray, w: int, h: int, nc: int, scale: int, nimages: int = 1) -> np.ndarray:
    """the C reference on given coefficients ([nimages * blocks][64]) -> nimages images back to back"""
    ref, _ = _libs()
    out = np.zeros((nimages,) + shape(w, h, nc, scale), np.uint8)
    coef = np.ascontiguousarray(coef, dtype=np.int16)
    qt = np.ascontiguousarray(qt, dtype=np.uint16)
    assert ref.kpo_reconstruct_scaled(coef.ctypes.data, qt.ctypes.data, w, h, nc, nimages, scale, out.ctypes.data) == 0
    return out if nimages > 1 else out[0]


def replay(coef: np.ndarray, qt: np.ndarray, w: int, h: int, nc: int, scale: int, nimages: int = 1, flags: int = 0) -> np.ndarray:
    """the CPU replay of the kernel on given coefficients"""
    _, emu = _libs()
    out = np.zeros((nimages,) + shape(w, h, nc, scale), np.uint8)
    coef = np.ascontiguousarray(coef, dtype=np.int16)
    qt = np.ascontiguousarray(qt, dtype=np.uint16)
    rc = emu.emu_scaled_decode(coef.ctypes.data, qt.ctypes.data, w, h, nc, nimages, scale_flags(flags, scale), STRIP_MCUS,
                               out.ctypes.data)
    assert rc == 0
    return out if nimages > 1 else out[0]


def reference(jpg: bytes, scale: int, parity: bool = False) -> np.ndarray:
    """The reduced-size image of a file: the oracle's coefficients (parity or T.81 mode) through the C reference."""
    w, h, nc, qt = frame_of(jpg)
    return reconstruct(coefficients(jpg, parity), qt, w, h, nc, scale)


def emu_decode(jpg: bytes, scale: int, parity: bool = False) -> np.ndarray:
    w, h, nc, qt = frame_of(jpg)
    return replay(coefficients(jpg, parity), qt, w, h, nc, scale)


def out_geom(w: int, h: int, nc: int, scale: int):
    """kpeg_common.h's OutGeom through the replay library -> (width, height, bytes)"""
    _, emu = _libs()
    ow, oh, nb = C.c_uint32(0), C.c_uint32(0), C.c_uint64(0)
    emu.emu_out_geom(w, h, nc, scale_flags(0, scale), C.byref(ow), C.byref(oh), C.byref(nb))
    return ow.value, oh.value, nb.value


# ---- inputs --------------------------------------------------------------------------------------------------------
def pil_jpeg(w: int, h: int, gray: bool, quality: int, seed: int, **kw) -> bytes:
    """A PIL (libjpeg-turbo) 4:4:4 / gray file of smooth content plus noise."""
    from PIL import Image
    rng = np.random.default_rng(seed)
    base = rng.random((h // 4 + 2, w // 4 + 2, 3)) * 255
    a = np.kron(base, np.ones((4, 4, 1)))[:h, :w] + rng.normal(0, float(rng.choice([2, 20, 60])), (h, w, 3))
    a = np.clip(a, 0, 255).astype(np.uint8)
    b = io.BytesIO()
    Image.fromarray(a[:, :, 0] if gray else a).save(b, "JPEG", quality=quality, subsampling=0, **kw)
    return b.getvalue()


def pil_files() -> list:
    """(name, bytes): PIL-written files -- sizes 1x1, smaller than the scale, ragged, with restart markers, optimised
    tables -- and lena."""
    out = []
    sizes = [(1, 1), (7, 9), (8, 8), (17, 23), (41, 70), (64, 37), (123, 45)]
    for i, (w, h) in enumerate(sizes):
        for gray in (False, True):
            for q in (20, 50, 75, 95, 100):
                if (i + q + gray) % 3 == 0 or (w, h) in ((1, 1), (7, 9)):
                    out.append((f"{w}x{h}{'g' if gray else ''}q{q}", pil_jpeg(w, h, gray, q, seed=i * 7 + q)))
    out.append(("opt-q85", pil_jpeg(97, 61, False, 85, seed=3, optimize=True)))
    out.append(("opt-gray-q60", pil_jpeg(50, 33, True, 60, seed=4, optimize=True)))
    out.append(("rst-q90", pil_jpeg(120, 72, False, 90, seed=5, restart_marker_blocks=3)))
    out.append(("rst-gray-q40", pil_jpeg(77, 40, True, 40, seed=6, restart_marker_blocks=1)))
    out.append(("lena", (GOLDEN / "lena.jpg").read_bytes()))
    return out


def pil_draft(jpg: bytes, scale: int) -> np.ndarray:
    """PIL's reduced-size decode (libjpeg's scale_denom).  Image.draft() derives the scale from a target size and
    cannot ask for 1/8 of an image narrower than 8 pixels, so this does what draft() does with the scale given."""
    from PIL import Image, ImageFile
    im = Image.open(io.BytesIO(jpg))
    w, h = im.size
    d, e, o, a = im.tile[0]
    e = (e[0], e[1], (e[2] - e[0] + scale - 1) // scale + e[0], (e[3] - e[1] + scale - 1) // scale + e[1])
    im._size = ((w + scale - 1) // scale, (h + scale - 1) // scale)
    im.tile = [ImageFile._Tile(d, e, o, a)]
    im.decoderconfig = (scale, 0)
    im.load()
    assert im.size == (-(-w // scale), -(-h // scale)), (im.size, w, h, scale)
    return np.asarray(im)


def field_files() -> list:
    """(name, bytes): the crafted coefficient fields (extreme DC and AC with quantisers of 255, colour lattices, DC-only
    fields), written with Annex K tables"""
    out = []
    for fam, w, h, nc in CF.cases():
        if fam in ("wide_and_huge", "colour_lattice", "dc_only"):
            for k, (_, jpg) in enumerate(CF.fields_and_files(fam, w, h, nc)):
                out.append((f"{fam}-{w}x{h}x{nc}-{k}", jpg))
    return out


@functools.lru_cache(maxsize=None)
def extreme_files() -> tuple:
    """Fields that drive the range-limit wrap and the 64-bit products of pass 2: every coefficient at its category
    limit (DC +-2047, AC +-1023) with quantisers of 255, in phase and with random signs."""
    import jpeg_writer as JW
    dc, ac = CF.annex_k_tables()
    rng = np.random.default_rng(77)
    out = []
    for nc, (w, h) in ((3, (40, 24)), (1, (33, 17))):
        nblk = ((w + 7) // 8) * ((h + 7) // 8) * nc
        coef = np.zeros((nblk, 64), np.int64)
        for b in range(nblk):
            kind = b % 4
            if kind == 0:
                coef[b] = np.concatenate([[2047], np.full(63, 1023)])
            elif kind == 1:
                coef[b] = -np.concatenate([[2047], np.full(63, 1023)])
            elif kind == 2:
                coef[b] = np.concatenate([[rng.choice([-2047, 2047])], rng.choice([-1023, 1023], size=63)])
            else:
                coef[b, 0] = rng.integers(-2047, 2048)
                coef[b, 1:] = rng.integers(-1023, 1024, size=63)
        # DC differences of more than 2047 are not codable: keep every DC within +-1023 of its predecessor's
        for c in range(nc):
            idx = np.arange(c, nblk, nc)
            for i in range(1, len(idx)):
                d = coef[idx[i], 0] - coef[idx[i - 1], 0]
                if abs(d) > 2047:
                    coef[idx[i], 0] = coef[idx[i - 1], 0] + np.sign(d) * 2047
        z = (0,) * nc
        qts = {c: [255] * 64 for c in range(nc)}
        jpg = JW.write_jpeg(coef, w, h, nc, qts, tq=tuple(range(nc)), dc_tables={0: dc}, ac_tables={0: ac}, td=z, ta=z)
        out.append((f"extreme-{w}x{h}x{nc}", jpg))
    return tuple(out)


PARITY_FLAGS = {True: KPEG_FLAG_REF_PARITY, False: 0}
__all__ = ["SCALES", "reference", "emu_decode", "reconstruct", "replay", "pil_files", "pil_draft", "field_files", "extreme_files",
           "output_shape", "frame_of", "shape", "out_geom", "coefficients", "PARITY_FLAGS"]
