"""Reference, numpy transforms and CPU replay of the lossless transcoder (kpeg_cuda_transcode), for
test_transcode_host.py and test_gpu_transcode.py.

The reference is written independently of csrc/transcode_core.h: the oracle's T.81 coefficients of the input, moved by
a numpy transform on whole 8x8 frequency blocks, then coded by the synthetic encoder's coding path
(kpeg_synth_encode_coefficients)."""
from __future__ import annotations

import ctypes as C
from pathlib import Path

import numpy as np

import coef_fields as CF
import helpers as H
from coef_fields import ZZ_TO_NAT
from libkpeg_b200.api import parse_jfif_scans
from libkpeg_b200.synth import synth_encode_coefficients

UNSUPPORTED, ARG, NOMEM = -2, -6, -4
NAMES = ("none", "flip-h", "flip-v", "transpose", "transverse", "rot90", "rot180", "rot270")
TRANSPOSING = {3, 4, 5, 7}


def allowed(t: int, w: int, h: int) -> bool:
    """jpegtran -perfect: a flip of an axis needs whole blocks on it.  Axes flipped, in INPUT terms."""
    flips_x = t in (1, 4, 6, 7)  # the input's horizontal axis is reversed
    flips_y = t in (2, 4, 5, 6)
    return (not flips_x or w % 8 == 0) and (not flips_y or h % 8 == 0)


def transform_pixels(img: np.ndarray, t: int) -> np.ndarray:
    """What each transform does to an image, numpy's way (rows = y)."""
    return [lambda a: a, lambda a: a[:, ::-1], lambda a: a[::-1], lambda a: a.swapaxes(0, 1),
            lambda a: np.rot90(a, 2).swapaxes(0, 1), lambda a: np.rot90(a, -1), lambda a: np.rot90(a, 2),
            lambda a: np.rot90(a, 1)][t](img)


def transform_coefficients(coef: np.ndarray, w: int, h: int, nc: int, t: int):
    """[blocks][64] zig-zag, MCU-interleaved -> the same for the transformed image, and its (width, height).  Blocks are
    8x8 frequency arrays F[u][v] (u vertical): a horizontal flip reverses the block columns and negates odd v, a vertical
    flip reverses the block rows and negates odd u, a transpose swaps both the grid's axes and u with v."""
    mx, my = (w + 7) // 8, (h + 7) // 8
    nat = np.zeros((my * mx * nc, 64), dtype=np.int32)
    nat[:, ZZ_TO_NAT] = coef
    g = nat.reshape(my, mx, nc, 8, 8)
    sign = (-1) ** np.arange(8)

    def flip_h(a):
        return a[:, ::-1] * sign[None, None, None, None, :]

    def flip_v(a):
        return a[::-1] * sign[None, None, None, :, None]

    def transpose(a):
        return a.transpose(1, 0, 2, 4, 3)

    g = [lambda a: a, flip_h, flip_v, transpose, lambda a: flip_v(flip_h(transpose(a))), lambda a: flip_h(transpose(a)),
         lambda a: flip_v(flip_h(a)), lambda a: flip_v(transpose(a))][t](g)
    out = np.ascontiguousarray(g).reshape(-1, 64)[:, ZZ_TO_NAT].astype(np.int16)
    return out, (h, w) if t in TRANSPOSING else (w, h)


def transpose_qt(q) -> list:
    nat = np.zeros(64, dtype=np.int64)
    nat[ZZ_TO_NAT] = np.asarray(q)
    return [int(x) for x in nat.reshape(8, 8).T.ravel()[ZZ_TO_NAT]]


def frame_of(jpg: bytes):
    """-> (width, height, ncomp, tq per component, {id: zig-zag table}, restart interval of the first scan)"""
    frame, scans = parse_jfif_scans(jpg)
    nc = int(frame.ncomp)
    tq, qt = [0] * nc, {}
    for sc in scans:
        for j in range(sc.plan.ncomp):
            tid = int(sc.plan.comp_tq[j])
            tq[int(sc.comp[j])] = tid
            qt[tid] = [int(x) for x in sc.plan.qt[tid]]
    return int(frame.width), int(frame.height), nc, tq, qt, int(scans[0].plan.restart_interval)


def reference(jpg: bytes, restart: int = -1, transform: int = 0, optimize: bool = False):
    """The transcoded file, or UNSUPPORTED (precondition or range rules)."""
    w, h, nc, tq, qt, ri = frame_of(jpg)
    if not allowed(transform, w, h):
        return UNSUPPORTED
    coef = H.oracle_decode(jpg, parity=False, want_pixels=False)["coef"]
    oc, (ow, oh) = transform_coefficients(coef, w, h, nc, transform)
    if transform in TRANSPOSING:
        qt = {k: transpose_qt(v) for k, v in qt.items()}
    out = synth_encode_coefficients(ow, oh, oc, tq, qt, ri if restart < 0 else restart, optimize)
    return UNSUPPORTED if out is None else out.tobytes()


_emu = None


def emu():
    global _emu
    if _emu is None:
        from libkpeg_b200._build import build_emu_transcode
        build_emu_transcode()
        lib = C.CDLL(str(Path(__file__).resolve().parent / "emu" / "libkpeg_emu_transcode.so"))
        lib.emu_transcode.restype = C.c_int
        lib.emu_transcode.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.c_int,
                                      C.c_uint32, C.c_uint32, C.c_void_p, C.c_size_t, C.POINTER(C.c_size_t), C.c_void_p]
        lib.emu_xform_table.restype = None
        lib.emu_xform_table.argtypes = [C.c_void_p]
        _emu = lib
    return _emu


def emu_transcode(jpg: bytes, restart: int = -1, transform: int = 0, optimize: bool = False, cap: int | None = None):
    """CPU replay of the GPU transcoder -> (file bytes or error code, info[4] = header, unstuffed, segments, bound)."""
    lib = emu()
    w, h, nc, tq, qt, ri = frame_of(jpg)
    coef = np.ascontiguousarray(H.oracle_decode(jpg, parity=False, want_pixels=False)["coef"], dtype=np.int16)
    tqa = np.zeros(3, np.uint8)
    tqa[:nc] = tq
    qzz = np.zeros((4, 64), np.uint8)
    for k, v in qt.items():
        qzz[k] = v
    info = np.zeros(4, np.uint64)
    n = C.c_size_t(0)
    size = cap if cap is not None else 64 << 20
    out = np.zeros(max(size, 1), np.uint8)
    rc = lib.emu_transcode(coef.ctypes.data, w, h, nc, tqa.ctypes.data, qzz.ctypes.data, ri, restart, transform,
                           2 if optimize else 0, out.ctypes.data, size, C.byref(n), info.ctypes.data)
    if rc != 0:
        return rc, info
    return out[:n.value].tobytes(), info


def dc_drift_file() -> bytes:
    """One-component 64x16 file whose coded DC differences are all legal (each <= 2047) but whose absolute DC climbs
    past 2047 along the first block row: re-segmenting it (restart 1 resets the prediction to 0) or reordering its blocks
    makes a difference no baseline table codes."""
    mx, my = 8, 2
    coef = np.zeros((mx * my, 64), np.int16)
    dcs = [0, 1500, 3000, 4500, 6000, 7500, 9000, 10500]
    coef[:mx, 0] = dcs
    coef[mx:, 0] = dcs[::-1]  # the second row walks back down: raster order keeps every step at 1500
    return CF.encode(CF.Field("dc drift", 64, 16, 1, coef, [np.ones(64, np.int64)]))

