"""Reference and CPU replay of the encoder with optimised Huffman tables (KPEG_FLAG_OPTIMIZE_HUFFMAN), for
test_encode_optimize_host.py and test_gpu_encode_optimize.py.  The byte-exact reference is the synthetic encoder's coding
path (kpeg_synth_encode_pixels) with OPTIMIZE_HUFFMAN added to the flags encode_cases.reference uses."""
from __future__ import annotations

import ctypes as C
from pathlib import Path

import numpy as np

from libkpeg_b200.synth import EMIT_RESTART, OPTIMIZE_HUFFMAN, QUIRK_FREE, SynthParams, synth_encode_pixels


def reference(pixels: np.ndarray, quality: int, restart_interval: int, parity: bool) -> bytes:
    h, w = pixels.shape[:2]
    nc = 1 if pixels.ndim == 2 else pixels.shape[2]
    flags = OPTIMIZE_HUFFMAN | (QUIRK_FREE if parity else 0) | (EMIT_RESTART if restart_interval else 0)
    p = SynthParams(w, h, file_components=nc, quality=quality, restart_interval=restart_interval, flags=flags)
    return synth_encode_pixels(p, pixels.reshape(h, w, nc)).tobytes()


_emu = None


def emu():
    """tests/emu/libkpeg_emu_encode_opt.so: the CPU replay with optimised tables (built on first use)."""
    global _emu
    if _emu is None:
        from libkpeg_b200._build import build_emu_encode_opt
        build_emu_encode_opt()
        lib = C.CDLL(str(Path(__file__).resolve().parent / "emu" / "libkpeg_emu_encode_opt.so"))
        lib.emu_encode_opt.restype = C.c_int
        lib.emu_encode_opt.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_uint32,
                                       C.c_void_p, C.c_size_t, C.POINTER(C.c_size_t), C.c_void_p]
        lib.emu_encode_bound_flags.restype = C.c_uint64
        lib.emu_encode_bound_flags.argtypes = [C.c_int] * 5 + [C.c_uint32]
        lib.emu_optimal_table.restype = C.c_int
        lib.emu_optimal_table.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
        _emu = lib
    return _emu


def emu_encode(pixels: np.ndarray, quality: int, restart_interval: int, parity: bool):
    """CPU replay of the optimised-table GPU encode (tests/emu/emu_encode_opt.cpp) -> (bytes, info[4])."""
    lib = emu()
    px = np.ascontiguousarray(pixels, dtype=np.uint8)
    h, w = px.shape[:2]
    nc = 1 if px.ndim == 2 else px.shape[2]
    flags = 3 if parity else 2
    cap = int(lib.emu_encode_bound_flags(w, h, nc, quality, restart_interval, flags))
    out = np.zeros(cap, np.uint8)
    n = C.c_size_t(0)
    info = np.zeros(4, np.uint32)
    rc = lib.emu_encode_opt(px.ctypes.data, w, h, nc, quality, restart_interval, 1 if parity else 0, out.ctypes.data,
                            cap, C.byref(n), info.ctypes.data)
    assert rc == 0, rc
    return out[:n.value].tobytes(), info
