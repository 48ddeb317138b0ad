"""Inputs and references of the encoder tests (test_encode_host.py on the CPU, test_gpu_encode.py on the GPU).

The byte-exact reference of the GPU encoder is the synthetic encoder's coding path over the same pixels
(kpeg_synth_encode_pixels) with QUIRK_FREE for the parity flag and EMIT_RESTART when there is a restart interval."""
from __future__ import annotations

import ctypes as C
from pathlib import Path

import numpy as np

import helpers as H
from libkpeg_b200.synth import EMIT_RESTART, QUIRK_FREE, SynthParams, synth_encode_pixels, synth_pixels

SIZES = [(1, 1), (7, 5), (61, 37), (1000, 600)]
QUALITIES = [1, 50, 95, 100]


def restart_intervals(width: int):
    return [0, 1, 7, (width + 7) // 8]  # none, every MCU, odd, one MCU row


def reference(pixels: np.ndarray, quality: int, restart_interval: int, parity: bool) -> bytes:
    h, w = pixels.shape[:2]
    nc = 1 if pixels.ndim == 2 else pixels.shape[2]
    flags = (QUIRK_FREE if parity else 0) | (EMIT_RESTART if restart_interval else 0)
    p = SynthParams(w, h, file_components=nc, quality=quality, restart_interval=restart_interval, flags=flags)
    return synth_encode_pixels(p, pixels.reshape(h, w, nc)).tobytes()


def synth_content(width: int, height: int, ncomp: int, seed: int = 7, noise_amp: int = 0) -> np.ndarray:
    px = synth_pixels(SynthParams(width, height, file_components=ncomp, seed=seed, noise_amp=noise_amp))
    return px if ncomp == 3 else px[..., 0]


def adversarial(width: int = 128, height: int = 96) -> dict:
    """name -> (pixels (H, W, 3) uint8, quality).  The cases where the DC chain, the code lengths or the stream size
    are at their extremes."""
    rng = np.random.default_rng(1234)
    y, x = np.mgrid[0:height, 0:width]
    flat = np.full((height, width, 3), 117, np.uint8)
    ripple = (flat.astype(np.int16) + np.where((x + y) % 2 == 0, 1, -1)[..., None]).astype(np.uint8)
    board = np.where(((x // 8) + (y // 8)) % 2 == 0, 255, 0).astype(np.uint8)
    pixel_board = np.where((x + y) % 2 == 0, 255, 0).astype(np.uint8)
    swing = np.stack([pixel_board, 255 - pixel_board, pixel_board], axis=-1)
    return {
        "constant": (flat, 90),                                            # every DC difference 0: the longest nudge chain
        "constant_ripple": (ripple, 100),                                  # +-1 AC terms under a constant DC
        "all_255": (np.full((height, width, 3), 255, np.uint8), 90),
        "all_0": (np.zeros((height, width, 3), np.uint8), 90),
        "block_checkerboard": (np.stack([board] * 3, axis=-1), 100),      # extreme DC steps
        "pixel_checkerboard": (np.ascontiguousarray(swing), 100),          # largest AC coefficients, longest codes
        "noise_q100": (rng.integers(0, 256, (height, width, 3), dtype=np.uint8), 100),
    }


_emu = None


def emu():
    """tests/emu/libkpeg_emu_encode.so: the CPU replay of the encode kernels (built on first use)."""
    global _emu
    if _emu is None:
        from libkpeg_b200._build import build_emu_encode
        build_emu_encode()
        lib = C.CDLL(str(Path(__file__).resolve().parent / "emu" / "libkpeg_emu_encode.so"))
        lib.emu_encode.restype = C.c_int
        lib.emu_encode.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_uint32, C.c_uint64,
                                   C.c_void_p, C.c_size_t, C.POINTER(C.c_size_t), C.c_void_p]
        lib.emu_encode_bound.restype = C.c_uint64
        lib.emu_encode_bound.argtypes = [C.c_int] * 5
        lib.emu_nudge.restype = None
        lib.emu_nudge.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint64, C.c_void_p]
        _emu = lib
    return _emu


def emu_encode(pixels: np.ndarray, quality: int, restart_interval: int, parity: bool, chunk: int = 7):
    """CPU replay of the GPU encoder (tests/emu/emu_encode.cpp) -> (bytes, info[3])."""
    lib = emu()
    px = np.ascontiguousarray(pixels, dtype=np.uint8)
    h, w = px.shape[:2]
    nc = 1 if px.ndim == 2 else px.shape[2]
    cap = int(lib.emu_encode_bound(w, h, nc, quality, restart_interval))
    out = np.zeros(cap, np.uint8)
    n = C.c_size_t(0)
    info = np.zeros(4, np.uint32)
    rc = lib.emu_encode(px.ctypes.data, w, h, nc, quality, restart_interval, 1 if parity else 0, chunk, out.ctypes.data,
                        cap, C.byref(n), info.ctypes.data)
    assert rc == 0, rc
    return out[:n.value].tobytes(), info


def psnr(a: np.ndarray, b: np.ndarray) -> float:
    mse = ((a.astype(np.float64) - b.astype(np.float64)) ** 2).mean()
    return float("inf") if mse == 0 else 10 * np.log10(255 ** 2 / mse)
