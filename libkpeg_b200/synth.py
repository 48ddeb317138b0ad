"""ctypes binding of include/kpeg_synth.h -- the committed deterministic synthetic baseline-JPEG
encoder that produces benchmark and parity inputs (the reference's own encoder is non-functional,
reference README.md:23)."""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass
from pathlib import Path

import numpy as np

PKG = Path(__file__).resolve().parent

EMIT_RESTART = 1
GRAY_CONTENT = 2
QUIRK_FREE = 4
NON_INTERLEAVED = 8  # three-component files: one scan per component
OPTIMIZE_HUFFMAN = 16  # Huffman tables optimised for the image (the GPU encoder's KPEG_FLAG_OPTIMIZE_HUFFMAN)


class _Params(C.Structure):
    _fields_ = [("width", C.c_int32), ("height", C.c_int32), ("file_components", C.c_int32), ("quality", C.c_int32),
                ("restart_interval", C.c_int32), ("flags", C.c_uint32), ("seed", C.c_uint64), ("noise_amp", C.c_int32),
                ("threads", C.c_int32)]


@dataclass
class SynthParams:
    width: int
    height: int
    file_components: int = 3
    quality: int = 90
    restart_interval: int = 0
    flags: int = QUIRK_FREE
    seed: int = 0x6B706567
    noise_amp: int = 0
    threads: int = 0

    def _c(self) -> _Params:
        return _Params(self.width, self.height, self.file_components, self.quality, self.restart_interval, self.flags,
                       self.seed, self.noise_amp, self.threads)


class CoefFrame(C.Structure):
    """struct kpeg_synth_coef_frame"""
    _fields_ = [("width", C.c_int32), ("height", C.c_int32), ("ncomp", C.c_int32), ("tq", C.c_uint8 * 3),
                ("qt", (C.c_uint8 * 64) * 4), ("restart_interval", C.c_int32), ("flags", C.c_uint32)]


_lib = None


def _load():
    global _lib
    if _lib is None:
        path = PKG / "lib" / "libkpeg_synth.so"
        if not path.exists():
            from ._build import build_product
            build_product(("lib/libkpeg_synth.so",))
        lib = C.CDLL(str(path))
        lib.kpeg_synth_encode.restype = C.c_int
        lib.kpeg_synth_encode.argtypes = [C.POINTER(_Params), C.POINTER(C.POINTER(C.c_uint8)), C.POINTER(C.c_size_t)]
        lib.kpeg_synth_free.restype = None
        lib.kpeg_synth_free.argtypes = [C.POINTER(C.c_uint8)]
        lib.kpeg_synth_encode_pixels.restype = C.c_int
        lib.kpeg_synth_encode_pixels.argtypes = [C.POINTER(_Params), C.c_void_p, C.POINTER(C.POINTER(C.c_uint8)),
                                                 C.POINTER(C.c_size_t)]
        lib.kpeg_synth_encode_coefficients.restype = C.c_int
        lib.kpeg_synth_encode_coefficients.argtypes = [C.POINTER(CoefFrame), C.c_void_p, C.POINTER(C.POINTER(C.c_uint8)),
                                                       C.POINTER(C.c_size_t)]
        lib.kpeg_synth_pixels.restype = C.c_int
        lib.kpeg_synth_pixels.argtypes = [C.POINTER(_Params), C.c_void_p]
        _lib = lib
    return _lib


def synth_encode(p: SynthParams) -> np.ndarray:
    lib = _load()
    cp = p._c()
    out = C.POINTER(C.c_uint8)()
    n = C.c_size_t(0)
    rc = lib.kpeg_synth_encode(C.byref(cp), C.byref(out), C.byref(n))
    if rc != 0:
        raise RuntimeError(f"kpeg_synth_encode failed: {rc}")
    try:
        return np.ctypeslib.as_array(out, shape=(n.value,)).copy()
    finally:
        lib.kpeg_synth_free(out)


def synth_encode_pixels(p: SynthParams, pixels: np.ndarray) -> np.ndarray:
    """The synth's coding path over given pixels ([H][W][nc] uint8, nc = 1 or 3 as synth_pixels lays them out):
    the byte-exact reference of the GPU encoder.  seed and noise_amp are ignored."""
    lib = _load()
    nc = 1 if (p.file_components == 1 or (p.flags & GRAY_CONTENT)) else 3
    px = np.ascontiguousarray(pixels, dtype=np.uint8)
    if px.size != p.width * p.height * nc:
        raise ValueError(f"expected {p.height}x{p.width}x{nc} pixels, got shape {pixels.shape}")
    cp = p._c()
    out = C.POINTER(C.c_uint8)()
    n = C.c_size_t(0)
    rc = lib.kpeg_synth_encode_pixels(C.byref(cp), px.ctypes.data, C.byref(out), C.byref(n))
    if rc != 0:
        raise RuntimeError(f"kpeg_synth_encode_pixels failed: {rc}")
    try:
        return np.ctypeslib.as_array(out, shape=(n.value,)).copy()
    finally:
        lib.kpeg_synth_free(out)


def synth_pixels(p: SynthParams) -> np.ndarray:
    lib = _load()
    cp = p._c()
    nc = 1 if (p.file_components == 1 or (p.flags & GRAY_CONTENT)) else 3
    out = np.empty((p.height, p.width, nc), dtype=np.uint8)
    rc = lib.kpeg_synth_pixels(C.byref(cp), out.ctypes.data)
    if rc != 0:
        raise RuntimeError(f"kpeg_synth_pixels failed: {rc}")
    return out


def synth_encode_coefficients(width: int, height: int, coef: np.ndarray, tq, qt, restart_interval: int = 0,
                              optimize: bool = False) -> np.ndarray | None:
    """The synth's coding path over quantised coefficients (kpeg_synth_encode_coefficients): coef [nblk, 64] int16,
    MCU-interleaved, zig-zag, DC absolute; tq: each component's quantiser id; qt: {id: 64 values in zig-zag order}.
    The reference of the GPU transcoder.  None when a value breaks the baseline range rules."""
    lib = _load()
    nc = len(tq)
    f = CoefFrame()
    f.width, f.height, f.ncomp = width, height, nc
    for c, t in enumerate(tq):
        f.tq[c] = t
    for t, table in qt.items():
        for i, v in enumerate(table):
            f.qt[t][i] = int(v)
    f.restart_interval = restart_interval
    f.flags = OPTIMIZE_HUFFMAN if optimize else 0
    cf = np.ascontiguousarray(coef, dtype=np.int16)
    if cf.shape != (((width + 7) // 8) * ((height + 7) // 8) * nc, 64):
        raise ValueError(f"expected {((width + 7) // 8) * ((height + 7) // 8) * nc} blocks of 64, got {cf.shape}")
    out = C.POINTER(C.c_uint8)()
    n = C.c_size_t(0)
    rc = lib.kpeg_synth_encode_coefficients(C.byref(f), cf.ctypes.data, C.byref(out), C.byref(n))
    if rc == -1:
        return None
    if rc != 0:
        raise RuntimeError(f"kpeg_synth_encode_coefficients failed: {rc}")
    try:
        return np.ctypeslib.as_array(out, shape=(n.value,)).copy()
    finally:
        lib.kpeg_synth_free(out)
