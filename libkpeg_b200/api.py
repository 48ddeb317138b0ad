"""ctypes binding of include/kpeg_cuda.h (the C ABI of the CUDA decode path).

Mirrors the reference's kpeg::JPEGDecoder life cycle (reference include/Decoder.hpp:40-60):
open -> decodeImageFile -> dumpRawData, plus the array-level entry points tests and bench need.
"""
from __future__ import annotations

import ctypes as C
import os
from pathlib import Path

import numpy as np

PKG = Path(__file__).resolve().parent
LIBDIR = PKG / "lib"

KPEG_OK = 0
KPEG_ERR_FORMAT, KPEG_ERR_UNSUPPORTED, KPEG_ERR_STREAM = -1, -2, -3
KPEG_ERR_NOMEM, KPEG_ERR_CUDA, KPEG_ERR_ARG, KPEG_ERR_NOT_CONVERGED = -4, -5, -6, -7
KPEG_FLAG_REF_PARITY = 1
KPEG_FLAG_OPTIMIZE_HUFFMAN = 2  # encode only: Huffman tables optimised for the image (T.81 K.2) instead of Annex K
# decode only: reduced-size output (libjpeg's scale 1/2, 1/4, 1/8 with its reduced IDCTs and integer colour)
KPEG_FLAG_SCALE_1_2, KPEG_FLAG_SCALE_1_4, KPEG_FLAG_SCALE_1_8, KPEG_FLAG_SCALE_MASK = 4, 8, 12, 12
_SCALE_FLAGS = {1: 0, 2: KPEG_FLAG_SCALE_1_2, 4: KPEG_FLAG_SCALE_1_4, 8: KPEG_FLAG_SCALE_1_8}
# lossless transforms of kpeg_cuda_transcode (numbered as libjpeg's JXFORM_CODE)
KPEG_XFORM_NONE, KPEG_XFORM_FLIP_H, KPEG_XFORM_FLIP_V, KPEG_XFORM_TRANSPOSE = 0, 1, 2, 3
KPEG_XFORM_TRANSVERSE, KPEG_XFORM_ROT90, KPEG_XFORM_ROT180, KPEG_XFORM_ROT270 = 4, 5, 6, 7
KPEG_TRANSCODE_KEEP_RESTART = -1
XFORM_NAMES = ("none", "flip-h", "flip-v", "transpose", "transverse", "rot90", "rot180", "rot270")

_ERR_NAMES = {
    -1: "KPEG_ERR_FORMAT", -2: "KPEG_ERR_UNSUPPORTED", -3: "KPEG_ERR_STREAM", -4: "KPEG_ERR_NOMEM",
    -5: "KPEG_ERR_CUDA", -6: "KPEG_ERR_ARG", -7: "KPEG_ERR_NOT_CONVERGED",
}


class KpegError(RuntimeError):
    def __init__(self, code: int, msg: str = ""):
        super().__init__(f"{_ERR_NAMES.get(code, code)}: {msg}")
        self.code = code


class HuffSpec(C.Structure):
    _fields_ = [("counts", C.c_uint8 * 16), ("symbols", C.c_uint8 * 256)]


class Plan(C.Structure):
    """struct kpeg_plan"""
    _fields_ = [
        ("width", C.c_uint16), ("height", C.c_uint16), ("ncomp", C.c_uint8),
        ("comp_tq", C.c_uint8 * 3), ("comp_td", C.c_uint8 * 3), ("comp_ta", C.c_uint8 * 3),
        ("restart_interval", C.c_uint16), ("flags", C.c_uint32),
        ("qt_present", C.c_uint8 * 4), ("ht_present", (C.c_uint8 * 4) * 2),
        ("qt", (C.c_uint16 * 64) * 4), ("ht", (HuffSpec * 4) * 2),
    ]


class Scan(C.Structure):
    """struct kpeg_scan: one SOS of a frame (kpeg_parse_jfif_scans)"""
    _fields_ = [("plan", Plan), ("comp", C.c_uint8 * 3), ("off", C.c_size_t), ("len", C.c_size_t)]


KPEG_MAX_SCANS = 3


class Stats(C.Structure):
    """struct kpeg_stats"""
    _fields_ = [
        ("width", C.c_uint32), ("height", C.c_uint32), ("ncomp", C.c_uint32),
        ("scan_bytes", C.c_uint64), ("unstuffed_bytes", C.c_uint64),
        ("segments", C.c_uint32), ("subsequences", C.c_uint32), ("sync_rounds", C.c_uint32),
        ("exact_samples", C.c_uint32),
        ("ms", C.c_float * 12), ("ms_total", C.c_float),
        ("kernel_launches", C.c_uint32),
    ]

    STAGES = ("h2d", "memset", "unstuff", "entropy_cold", "entropy_relay", "entropy_scan", "entropy_write", "dc_scan",
              "idct", "d2h", "relay_sparse", "idct_patch")

    def stage_ms(self) -> dict:
        return {name: float(self.ms[i]) for i, name in enumerate(self.STAGES)}

    def as_dict(self):
        d = {k: getattr(self, k) for k, _ in self._fields_ if k != "ms"}
        d["ms"] = self.stage_ms()
        return d


class EncodeParams(C.Structure):
    """struct kpeg_encode_params"""
    _fields_ = [("width", C.c_uint16), ("height", C.c_uint16), ("ncomp", C.c_uint8), ("quality", C.c_uint8),
                ("restart_interval", C.c_uint16), ("flags", C.c_uint32)]


class TranscodeParams(C.Structure):
    """struct kpeg_transcode_params"""
    _fields_ = [("restart_interval", C.c_int32), ("transform", C.c_uint32), ("flags", C.c_uint32)]


class Crop(C.Structure):
    """struct kpeg_crop: a rectangle of the output image (x, y, width, height in its pixels)"""
    _fields_ = [("x", C.c_uint32), ("y", C.c_uint32), ("width", C.c_uint32), ("height", C.c_uint32)]


# every symbol include/kpeg_cuda.h declares: (restype, argtypes)
_u8p = C.POINTER(C.c_uint8)
_vp = C.c_void_p
SYMBOLS = {
    "kpeg_parse_jfif": (C.c_int, [_vp, C.c_size_t, C.POINTER(Plan), C.POINTER(C.c_size_t), C.POINTER(C.c_size_t)]),
    "kpeg_parse_jfif_scans": (C.c_int, [_vp, C.c_size_t, C.POINTER(Plan), C.POINTER(Scan), C.c_int, C.POINTER(C.c_int)]),
    "kpeg_cuda_decode_scans": (C.c_int, [_vp, C.POINTER(Plan), C.POINTER(Scan), C.c_int, _vp, C.c_size_t, _vp, C.POINTER(Stats)]),
    "kpeg_cuda_decode_files": (C.c_int, [_vp, C.c_int, C.POINTER(_vp), C.POINTER(C.c_size_t), C.c_uint32, C.POINTER(_vp), C.POINTER(C.c_size_t),
                                         C.POINTER(Plan), C.POINTER(C.c_int), C.POINTER(Stats)]),
    "kpeg_output_size": (C.c_size_t, [C.POINTER(Plan), C.POINTER(C.c_uint32), C.POINTER(C.c_uint32)]),
    "kpeg_cuda_create": (C.c_int, [C.c_int, C.POINTER(_vp)]),
    "kpeg_cuda_destroy": (None, [_vp]),
    "kpeg_cuda_last_error": (C.c_char_p, [_vp]),
    "kpeg_cuda_device_count": (C.c_int, []),
    "kpeg_cuda_set_profiling": (C.c_int, [_vp, C.c_int]),
    "kpeg_cuda_set_tuning": (C.c_int, [_vp, C.c_int, C.c_int]),
    "kpeg_cuda_stream": (_vp, [_vp]),
    "kpeg_cuda_host_alloc": (_vp, [C.c_size_t]),
    "kpeg_cuda_host_free": (None, [_vp]),
    "kpeg_cuda_device_alloc": (_vp, [_vp, C.c_size_t]),
    "kpeg_cuda_device_free": (None, [_vp, _vp]),
    "kpeg_cuda_memcpy_h2d": (C.c_int, [_vp, _vp, _vp, C.c_size_t]),
    "kpeg_cuda_memcpy_d2h": (C.c_int, [_vp, _vp, _vp, C.c_size_t]),
    "kpeg_cuda_decode": (C.c_int, [_vp, C.POINTER(Plan), _vp, C.c_size_t, _vp, C.POINTER(Stats)]),
    "kpeg_cuda_decode_device": (C.c_int, [_vp, C.POINTER(Plan), _vp, C.c_size_t, _vp, C.POINTER(Stats)]),
    "kpeg_cuda_decode_crop": (C.c_int, [_vp, C.POINTER(Plan), _vp, C.c_size_t, C.POINTER(Crop), _vp, C.POINTER(Stats)]),
    "kpeg_cuda_decode_crop_device": (C.c_int, [_vp, C.POINTER(Plan), _vp, C.c_size_t, C.POINTER(Crop), _vp, C.POINTER(Stats)]),
    "kpeg_cuda_decode_batch_crop": (C.c_int, [_vp, C.POINTER(Plan), C.c_int, C.POINTER(_vp), C.POINTER(C.c_size_t),
                                              C.POINTER(Crop), C.POINTER(_vp), C.POINTER(Stats)]),
    "kpeg_cuda_decode_file_crop": (C.c_int, [_vp, _vp, C.c_size_t, C.c_uint32, C.POINTER(Crop), _vp, C.c_size_t,
                                             C.POINTER(Plan), C.POINTER(Stats)]),
    "kpeg_cuda_decode_batch": (C.c_int, [_vp, C.POINTER(Plan), C.c_int, C.POINTER(_vp), C.POINTER(C.c_size_t),
                                        C.POINTER(_vp), C.POINTER(Stats)]),
    "kpeg_cuda_decode_batch_device": (C.c_int, [_vp, C.POINTER(Plan), C.c_int, _vp, C.POINTER(C.c_uint64), _vp,
                                               C.POINTER(Stats)]),
    "kpeg_batch_packed_size": (C.c_size_t, [C.c_int, C.POINTER(C.c_size_t)]),
    "kpeg_batch_pack": (C.c_int, [C.c_int, C.POINTER(_vp), C.POINTER(C.c_size_t), _vp, C.c_size_t]),
    "kpeg_cuda_decode_batch_packed_device": (C.c_int, [_vp, C.POINTER(Plan), C.c_int, _vp, C.c_size_t, _vp,
                                                      C.POINTER(Stats)]),
    "kpeg_cuda_decode_batch_packed_device_split": (C.c_int, [_vp, C.POINTER(Plan), C.c_int, _vp, C.POINTER(C.c_uint64), _vp,
                                                            C.POINTER(Stats)]),
    "kpeg_cuda_submit_batch_packed_device": (C.c_int, [_vp, C.POINTER(Plan), C.c_int, _vp, C.POINTER(C.c_uint64), _vp]),
    "kpeg_cuda_wait": (C.c_int, [_vp, C.POINTER(Stats)]),
    "kpeg_cuda_submit_batch": (C.c_int, [_vp, C.POINTER(Plan), C.c_int, C.POINTER(_vp), C.POINTER(C.c_size_t),
                                        C.POINTER(_vp)]),
    "kpeg_cuda_decode_file": (C.c_int, [_vp, _vp, C.c_size_t, C.c_uint32, _vp, C.c_size_t, C.POINTER(Plan),
                                       C.POINTER(Stats)]),
    "kpeg_cuda_read_coefficients": (C.c_int, [_vp, _vp, C.c_size_t]),
    "kpeg_split_restart_bands": (C.c_int, [_vp, C.c_size_t, C.POINTER(Plan), C.c_int, C.POINTER(C.c_uint64),
                                          C.POINTER(C.c_uint64), C.POINTER(C.c_uint32)]),
    "kpeg_split_restart_bands_by_bytes": (C.c_int, [_vp, C.c_size_t, C.POINTER(Plan), C.c_int, C.POINTER(C.c_uint64),
                                          C.POINTER(C.c_uint64), C.POINTER(C.c_uint32)]),
    "kpeg_ppm_header": (C.c_int, [C.c_int, C.c_int, C.c_char_p, C.c_size_t]),
    "kpeg_cuda_acquire": (C.c_int, [C.c_int, C.POINTER(_vp)]),
    "kpeg_cuda_release": (None, [C.c_int, _vp]),
    "kpeg_cuda_pool_clear": (None, []),
    "kpeg_cuda_host_register": (C.c_int, [_vp, C.c_size_t]),
    "kpeg_cuda_host_unregister": (None, [_vp]),
    "kpeg_cuda_decode_tiled": (C.c_int, [C.POINTER(C.c_int), C.c_int, C.POINTER(Plan), _vp, C.c_size_t, _vp, C.POINTER(Stats)]),
    "kpeg_cuda_decode_file_tiled": (C.c_int, [C.POINTER(C.c_int), C.c_int, _vp, C.c_size_t, C.c_uint32, _vp, C.c_size_t,
                                             C.POINTER(Plan), C.POINTER(Stats)]),
    "kpeg_cuda_decode_tiled_device": (C.c_int, [C.POINTER(C.c_int), C.c_int, C.POINTER(Plan), _vp, C.c_size_t, C.c_int, _vp,
                                               C.POINTER(Stats)]),
    "kpeg_tiled_last_error": (C.c_char_p, []),
    "kpeg_cuda_decode_to_peer": (C.c_int, [_vp, C.POINTER(Plan), _vp, C.c_size_t, C.c_int, _vp, C.POINTER(Stats)]),
    "kpeg_cuda_decode_ppm_device": (C.c_int, [_vp, C.POINTER(Plan), _vp, C.c_size_t, _vp, C.c_size_t, C.POINTER(C.c_size_t),
                                             C.POINTER(C.c_size_t), C.POINTER(Stats)]),
    "kpeg_cuda_interleaved_to_planar": (C.c_int, [_vp, _vp, _vp, C.c_size_t]),
    "kpeg_encode_bound": (C.c_size_t, [C.POINTER(EncodeParams)]),
    "kpeg_cuda_encode": (C.c_int, [_vp, C.POINTER(EncodeParams), _vp, _vp, C.c_size_t, C.POINTER(C.c_size_t), C.POINTER(Stats)]),
    "kpeg_cuda_encode_device": (C.c_int, [_vp, C.POINTER(EncodeParams), _vp, _vp, C.c_size_t, C.POINTER(C.c_size_t),
                                         C.POINTER(Stats)]),
    "kpeg_transcode_bound": (C.c_size_t, [_vp, C.c_size_t, C.POINTER(TranscodeParams)]),
    "kpeg_cuda_transcode": (C.c_int, [_vp, _vp, C.c_size_t, C.POINTER(TranscodeParams), _vp, C.c_size_t, C.POINTER(C.c_size_t),
                                     C.POINTER(Stats)]),
}

_lib = None


def load_cuda_library() -> C.CDLL:
    """Load lib/libkpeg_cuda.so (built by `make -C libkpeg_b200` / __graft_entry__.build()).
    Fails loudly when it is missing: there is no other implementation to fall back to."""
    global _lib
    if _lib is not None:
        return _lib
    path = Path(os.environ.get("KPEG_CUDA_LIB", LIBDIR / "libkpeg_cuda.so"))
    if not path.exists():
        raise KpegError(KPEG_ERR_CUDA, f"{path} not built -- run `make -C {PKG}` (needs nvcc); "
                                       "libkpeg_b200 has no CPU fallback")
    lib = C.CDLL(str(path))
    for name, (res, args) in SYMBOLS.items():
        fn = getattr(lib, name)  # AttributeError if the library does not export a declared symbol
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def _ptr(a: np.ndarray) -> int:
    return a.ctypes.data


def parse_jfif(data: bytes | np.ndarray):
    """Host-side container parse -> (Plan, scan_offset, scan_len).  No CUDA involved."""
    lib = load_cuda_library()
    buf = np.frombuffer(data, dtype=np.uint8) if not isinstance(data, np.ndarray) else data
    plan = Plan()
    off, ln = C.c_size_t(0), C.c_size_t(0)
    rc = lib.kpeg_parse_jfif(_ptr(buf), buf.size, C.byref(plan), C.byref(off), C.byref(ln))
    if rc != KPEG_OK:
        raise KpegError(rc, "kpeg_parse_jfif")
    return plan, off.value, ln.value


def parse_jfif_scans(data: bytes | np.ndarray):
    """Container parse that also accepts frames coded one scan per component -> (frame Plan, [Scan, ...])."""
    lib = load_cuda_library()
    buf = np.frombuffer(data, dtype=np.uint8) if not isinstance(data, np.ndarray) else data
    frame = Plan()
    scans = (Scan * KPEG_MAX_SCANS)()
    n = C.c_int(0)
    rc = lib.kpeg_parse_jfif_scans(_ptr(buf), buf.size, C.byref(frame), scans, KPEG_MAX_SCANS, C.byref(n))
    if rc != KPEG_OK:
        raise KpegError(rc, "kpeg_parse_jfif_scans")
    return frame, [scans[i] for i in range(n.value)]


def scale_flags(flags: int, scale: int) -> int:
    """`flags` with its KPEG_FLAG_SCALE_* bits set for an output of 1/scale the size (scale 1, 2, 4 or 8)."""
    if scale not in _SCALE_FLAGS:
        raise ValueError(f"scale must be 1, 2, 4 or 8, not {scale!r}")
    return (flags & ~KPEG_FLAG_SCALE_MASK) | _SCALE_FLAGS[scale]


def _scaled_flags(flags: int, scale: int | None) -> int:
    """flags itself (scale None: its own KPEG_FLAG_SCALE_* bits decide), or flags asking for 1/scale the size"""
    return flags if scale is None else scale_flags(flags, scale)


def _scaled_plan(plan: Plan, scale: int | None) -> Plan:
    """plan itself (scale None: its own flags decide), or a copy whose flags ask for 1/scale the size"""
    if scale is None:
        return plan
    p = Plan.from_buffer_copy(plan)
    p.flags = scale_flags(p.flags, scale)
    return p


def output_shape(plan: Plan) -> tuple:
    """Shape of the decoded image of `plan` at the size its flags ask for (kpeg_output_size): (H, W, 3) or (H, W)."""
    w, h = C.c_uint32(0), C.c_uint32(0)
    if load_cuda_library().kpeg_output_size(C.byref(plan), C.byref(w), C.byref(h)) == 0:
        raise KpegError(KPEG_ERR_ARG, "kpeg_output_size: bad plan geometry")
    return (h.value, w.value, 3) if plan.ncomp == 3 else (h.value, w.value)


def crop_struct(crop) -> Crop:
    """(x, y, w, h) -> kpeg_crop.  ValueError for anything but four non-negative integers with w, h >= 1 (whether the
    rectangle lies inside the image is the decoder's check: KPEG_ERR_ARG)."""
    try:
        vals = tuple(crop)
    except TypeError:
        raise ValueError(f"crop must be (x, y, w, h), not {crop!r}") from None
    if len(vals) != 4 or not all(isinstance(v, (int, np.integer)) and not isinstance(v, bool) for v in vals):
        raise ValueError(f"crop must be four integers (x, y, w, h), not {crop!r}")
    x, y, w, h = (int(v) for v in vals)
    if x < 0 or y < 0 or w < 1 or h < 1 or max(x, y, w, h) >= 1 << 32:
        raise ValueError(f"crop (x, y, w, h) needs x, y >= 0 and w, h >= 1, not {crop!r}")
    return Crop(x, y, w, h)


def crop_shape(plan: Plan, crop) -> tuple:
    """Shape of the crop (x, y, w, h) of plan's decoded image: (h, w, 3) or (h, w), as output_shape."""
    c = crop_struct(crop)
    return (c.height, c.width, 3) if plan.ncomp == 3 else (c.height, c.width)


def ppm_header(width: int, height: int) -> bytes:
    lib = load_cuda_library()
    buf = C.create_string_buffer(256)
    n = lib.kpeg_ppm_header(width, height, buf, 256)
    return buf.raw[:n]


def encode_params(width: int, height: int, ncomp: int, quality: int = 90, restart_interval: int = 0,
                  flags: int = KPEG_FLAG_REF_PARITY) -> EncodeParams:
    """kpeg_encode_params, range-checked (ValueError) before the fields are narrowed to their C types."""
    if not (1 <= width <= 65535 and 1 <= height <= 65535 and ncomp in (1, 3) and 1 <= quality <= 100
            and 0 <= restart_interval <= 65535):
        raise ValueError(f"encode parameters out of range: {width}x{height}x{ncomp} q{quality} ri{restart_interval}")
    return EncodeParams(width, height, ncomp, quality, restart_interval, flags)


def encode_bound(width: int, height: int, ncomp: int, quality: int = 90, restart_interval: int = 0,
                 flags: int = KPEG_FLAG_REF_PARITY) -> int:
    """kpeg_encode_bound: the largest file the GPU encoder can write for these parameters (host only)."""
    p = encode_params(width, height, ncomp, quality, restart_interval, flags)
    return int(load_cuda_library().kpeg_encode_bound(C.byref(p)))


def transcode_params(restart_interval: int = KPEG_TRANSCODE_KEEP_RESTART, transform: int = KPEG_XFORM_NONE,
                     optimize: bool = False) -> TranscodeParams:
    """kpeg_transcode_params, range-checked (ValueError) before the fields are narrowed to their C types."""
    if not (-1 <= restart_interval <= 65535 and 0 <= transform <= 7):
        raise ValueError(f"transcode parameters out of range: restart {restart_interval}, transform {transform}")
    return TranscodeParams(restart_interval, transform, KPEG_FLAG_OPTIMIZE_HUFFMAN if optimize else 0)


def transcode_bound(data, restart_interval: int = KPEG_TRANSCODE_KEEP_RESTART, transform: int = KPEG_XFORM_NONE,
                    optimize: bool = False) -> int:
    """kpeg_transcode_bound: the largest file kpeg_cuda_transcode can write for this input (host only; 0 when the file,
    the parameters or the transform's precondition are rejected)."""
    buf = np.ascontiguousarray(np.frombuffer(data, dtype=np.uint8) if not isinstance(data, np.ndarray) else data)
    p = transcode_params(restart_interval, transform, optimize)
    return int(load_cuda_library().kpeg_transcode_bound(_ptr(buf), buf.size, C.byref(p)))


def _image_shape(pixels: np.ndarray):
    """(H, W, 3) or (H, W) / (H, W, 1) uint8 -> (height, width, ncomp)"""
    if pixels.dtype != np.uint8 or pixels.ndim not in (2, 3) or (pixels.ndim == 3 and pixels.shape[2] not in (1, 3)):
        raise ValueError("encode takes (H, W, 3) or (H, W) uint8 pixels")
    return pixels.shape[0], pixels.shape[1], 1 if pixels.ndim == 2 else pixels.shape[2]


class PinnedArray:
    """numpy view of cudaMallocHost memory obtained through the C ABI."""

    def __init__(self, nbytes: int):
        self._lib = load_cuda_library()
        self.ptr = self._lib.kpeg_cuda_host_alloc(max(nbytes, 1))
        if not self.ptr:
            raise KpegError(KPEG_ERR_NOMEM, "kpeg_cuda_host_alloc")
        self.nbytes = nbytes
        self.array = np.ctypeslib.as_array((C.c_uint8 * max(nbytes, 1)).from_address(self.ptr))[:nbytes]

    def free(self):
        if self.ptr:
            self.array = None
            self._lib.kpeg_cuda_host_free(self.ptr)
            self.ptr = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


class Decoder:
    """One CUDA decode context (kpeg_ctx).  `decode_file(bytes)` is the array-level equivalent of
    kpeg::JPEGDecoder::open + decodeImageFile (reference src/Decoder.cpp:30-45, 90-152); the result is
    the pixel payload Image::dumpRawData would write (src/Image.cpp:129-135)."""

    def __init__(self, device: int = 0, profiling: bool = False):
        self._lib = load_cuda_library()
        h = _vp()
        rc = self._lib.kpeg_cuda_create(device, C.byref(h))
        if rc != KPEG_OK:
            raise KpegError(rc, "kpeg_cuda_create: no usable CUDA device (there is no CPU fallback)")
        self._h = h
        self.device = device
        self.last_stats = Stats()
        self._pending = []
        if profiling:
            self.set_profiling(True)

    # -- housekeeping -----------------------------------------------------------------------
    def close(self):
        if getattr(self, "_h", None):
            self._lib.kpeg_cuda_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def _check(self, rc: int, what: str):
        if rc != KPEG_OK:
            raise KpegError(rc, f"{what}: {self._lib.kpeg_cuda_last_error(self._h).decode(errors='replace')}")

    def set_profiling(self, on: bool):
        self._check(self._lib.kpeg_cuda_set_profiling(self._h, int(on)), "set_profiling")

    def set_tuning(self, sub_bits: int = 0, relay_rounds: int = 0):
        self._check(self._lib.kpeg_cuda_set_tuning(self._h, sub_bits, relay_rounds), "set_tuning")

    @property
    def stream(self) -> int:
        return self._lib.kpeg_cuda_stream(self._h) or 0

    # -- decode -------------------------------------------------------------------------------
    def decode_file(self, data, flags: int = KPEG_FLAG_REF_PARITY, out: np.ndarray | None = None,
                    scale: int | None = None, crop=None) -> np.ndarray:
        """scale 1, 2, 4, 8: the image at 1/scale the size (sets the KPEG_FLAG_SCALE_* bits of flags; None: as flags has
        them).  crop (x, y, w, h): only that rectangle of the output image (kpeg_cuda_decode_file_crop)."""
        flags = _scaled_flags(flags, scale)
        c = None if crop is None else crop_struct(crop)
        buf = np.frombuffer(data, dtype=np.uint8) if not isinstance(data, np.ndarray) else data
        if c is not None:
            buf = np.ascontiguousarray(buf)
            frame, _ = parse_jfif_scans(buf)
            shape = crop_shape(frame, crop)
            if out is None:
                out = np.empty(shape, dtype=np.uint8)
            assert out.nbytes == int(np.prod(shape)) and out.flags.c_contiguous
            rc = self._lib.kpeg_cuda_decode_file_crop(self._h, _ptr(buf), buf.size, flags, C.byref(c), _ptr(out), out.nbytes,
                                                      None, C.byref(self.last_stats))
            self._check(rc, "kpeg_cuda_decode_file_crop")
            return out.reshape(shape)
        frame, scans = parse_jfif_scans(buf)
        if len(scans) == 1:
            plan = scans[0].plan
            plan.flags = flags
            return self.decode_scan(plan, buf[scans[0].off:scans[0].off + scans[0].len], out=out)
        # one scan per component: kpeg_cuda_decode_scans
        frame.flags = flags
        buf = np.ascontiguousarray(buf)
        shape = output_shape(frame)
        if out is None:
            out = np.empty(shape, dtype=np.uint8)
        assert out.nbytes == int(np.prod(shape)) and out.flags.c_contiguous
        arr = (Scan * len(scans))(*scans)
        rc = self._lib.kpeg_cuda_decode_scans(self._h, C.byref(frame), arr, len(scans), _ptr(buf), buf.size, _ptr(out),
                                              C.byref(self.last_stats))
        self._check(rc, "kpeg_cuda_decode_scans")
        return out.reshape(shape)

    def decode_files(self, files: list, flags: int = KPEG_FLAG_REF_PARITY, scale: int | None = None):
        """kpeg_cuda_decode_files: any mix of files in one call -> (list of images, or None where a file failed; list of
        per-file return codes).  Files with identical plans are decoded as one batch.  scale: as in decode_file."""
        flags = _scaled_flags(flags, scale)
        bufs = [np.ascontiguousarray(np.frombuffer(f, dtype=np.uint8) if not isinstance(f, np.ndarray) else f) for f in files]
        n = len(bufs)
        outs, shapes = [], []
        for b in bufs:
            try:
                frame, _ = parse_jfif_scans(b)
                frame.flags = flags
                shapes.append(output_shape(frame))
                outs.append(np.empty(int(np.prod(shapes[-1])), dtype=np.uint8))
            except KpegError:
                shapes.append(None)
                outs.append(np.empty(1, dtype=np.uint8))
        fp = (_vp * n)(*[_ptr(b) for b in bufs])
        fl = (C.c_size_t * n)(*[b.size for b in bufs])
        op = (_vp * n)(*[_ptr(o) for o in outs])
        oc = (C.c_size_t * n)(*[o.size for o in outs])
        res = (C.c_int * n)()
        self._lib.kpeg_cuda_decode_files(self._h, n, fp, fl, flags, op, oc, None, res, C.byref(self.last_stats))
        codes = [int(r) for r in res]
        return [o.reshape(sh) if (c == KPEG_OK and sh is not None) else None for o, sh, c in zip(outs, shapes, codes)], codes

    def decode_scan(self, plan: Plan, scan: np.ndarray, out: np.ndarray | None = None, scale: int | None = None,
                    crop=None) -> np.ndarray:
        """scale 1, 2, 4, 8 sets the plan's KPEG_FLAG_SCALE_* bits (None: as the plan has them).  crop (x, y, w, h): only
        that rectangle of the output image (kpeg_cuda_decode_crop)."""
        plan = _scaled_plan(plan, scale)
        c = None if crop is None else crop_struct(crop)
        scan = np.ascontiguousarray(scan, dtype=np.uint8)
        if c is not None:
            shape = crop_shape(plan, crop)
            if out is None:
                out = np.empty(shape, dtype=np.uint8)
            assert out.nbytes == int(np.prod(shape)) and out.flags.c_contiguous
            rc = self._lib.kpeg_cuda_decode_crop(self._h, C.byref(plan), _ptr(scan), scan.size, C.byref(c), _ptr(out),
                                                 C.byref(self.last_stats))
            self._check(rc, "kpeg_cuda_decode_crop")
            return out.reshape(shape)
        shape = output_shape(plan)
        if out is None:
            out = np.empty(shape, dtype=np.uint8)
        assert out.nbytes == int(np.prod(shape)) and out.flags.c_contiguous
        rc = self._lib.kpeg_cuda_decode(self._h, C.byref(plan), _ptr(scan), scan.size, _ptr(out),
                                        C.byref(self.last_stats))
        self._check(rc, "kpeg_cuda_decode")
        return out.reshape(shape)

    def decode_batch(self, plan: Plan, scans: list[np.ndarray], outs: list[np.ndarray] | None = None, scale: int | None = None,
                     crops: list | None = None):
        """crops: one rectangle (x, y, w, h) per image; image i's output is then that rectangle of it
        (kpeg_cuda_decode_batch_crop)."""
        plan = _scaled_plan(plan, scale)
        n = len(scans)
        if crops is not None:
            if len(crops) != n:
                raise ValueError(f"decode_batch: {n} scans but {len(crops)} crops")
            cs = [crop_struct(c) for c in crops]
        scans = [np.ascontiguousarray(s, dtype=np.uint8) for s in scans]
        if crops is not None:
            if outs is None:
                outs = [np.empty(crop_shape(plan, c), dtype=np.uint8) for c in crops]
            sp = (_vp * n)(*[_ptr(s) for s in scans])
            sl = (C.c_size_t * n)(*[s.size for s in scans])
            op = (_vp * n)(*[_ptr(o) for o in outs])
            rc = self._lib.kpeg_cuda_decode_batch_crop(self._h, C.byref(plan), n, sp, sl, (Crop * n)(*cs), op,
                                                       C.byref(self.last_stats))
            self._check(rc, "kpeg_cuda_decode_batch_crop")
            return outs
        shape = output_shape(plan)
        if outs is None:
            outs = [np.empty(shape, dtype=np.uint8) for _ in range(n)]
        sp = (_vp * n)(*[_ptr(s) for s in scans])
        sl = (C.c_size_t * n)(*[s.size for s in scans])
        op = (_vp * n)(*[_ptr(o) for o in outs])
        rc = self._lib.kpeg_cuda_decode_batch(self._h, C.byref(plan), n, sp, sl, op, C.byref(self.last_stats))
        self._check(rc, "kpeg_cuda_decode_batch")
        return outs

    def read_coefficients(self, nblocks: int) -> np.ndarray:
        out = np.empty((nblocks, 64), dtype=np.int16)
        self._check(self._lib.kpeg_cuda_read_coefficients(self._h, _ptr(out), out.size), "read_coefficients")
        return out

    # -- device-resident helpers (bench) ---------------------------------------------------------
    def device_alloc(self, nbytes: int) -> int:
        p = self._lib.kpeg_cuda_device_alloc(self._h, nbytes)
        if not p:
            raise KpegError(KPEG_ERR_NOMEM, "kpeg_cuda_device_alloc")
        return p

    def device_free(self, p: int):
        self._lib.kpeg_cuda_device_free(self._h, p)

    def h2d(self, dptr: int, src: np.ndarray):
        self._check(self._lib.kpeg_cuda_memcpy_h2d(self._h, dptr, _ptr(src), src.nbytes), "memcpy_h2d")

    def d2h(self, dst: np.ndarray, dptr: int):
        self._check(self._lib.kpeg_cuda_memcpy_d2h(self._h, _ptr(dst), dptr, dst.nbytes), "memcpy_d2h")

    def decode_device(self, plan: Plan, d_scan: int, scan_len: int, d_out: int, scale: int | None = None, crop=None):
        """d_out receives output_shape(plan) bytes (with scale: of the plan at that scale); with crop (x, y, w, h), the
        crop_shape(plan, crop) bytes of that rectangle (kpeg_cuda_decode_crop_device)."""
        plan = _scaled_plan(plan, scale)
        if crop is not None:
            c = crop_struct(crop)
            rc = self._lib.kpeg_cuda_decode_crop_device(self._h, C.byref(plan), d_scan, scan_len, C.byref(c), d_out,
                                                        C.byref(self.last_stats))
            self._check(rc, "kpeg_cuda_decode_crop_device")
            return
        rc = self._lib.kpeg_cuda_decode_device(self._h, C.byref(plan), d_scan, scan_len, d_out,
                                               C.byref(self.last_stats))
        self._check(rc, "kpeg_cuda_decode_device")

    def decode_batch_packed_device_split(self, plan: Plan, n: int, d_packed: int, offsets: np.ndarray, d_out: int):
        offsets = np.ascontiguousarray(offsets, dtype=np.uint64)
        rc = self._lib.kpeg_cuda_decode_batch_packed_device_split(
            self._h, C.byref(plan), n, d_packed, offsets.ctypes.data_as(C.POINTER(C.c_uint64)), d_out,
            C.byref(self.last_stats))
        self._check(rc, "kpeg_cuda_decode_batch_packed_device_split")

    def submit_batch_packed_device(self, plan: Plan, n: int, d_packed: int, offsets: np.ndarray, d_out: int):
        """Enqueue only (kpeg_cuda_submit_batch_packed_device); `wait()` completes and checks everything submitted."""
        offsets = np.ascontiguousarray(offsets, dtype=np.uint64)
        rc = self._lib.kpeg_cuda_submit_batch_packed_device(
            self._h, C.byref(plan), n, d_packed, offsets.ctypes.data_as(C.POINTER(C.c_uint64)), d_out)
        self._check(rc, "kpeg_cuda_submit_batch_packed_device")

    def submit_batch(self, plan: Plan, scans: list[np.ndarray], outs: list[np.ndarray]):
        """Enqueue only (kpeg_cuda_submit_batch, host buffers): `outs` are valid after `wait()`."""
        n = len(scans)
        for a in list(scans) + list(outs):
            if not (a.flags["C_CONTIGUOUS"] and a.dtype == np.uint8):
                raise ValueError("submit_batch needs contiguous uint8 arrays (they are used in place)")
        sp = (_vp * n)(*[_ptr(s) for s in scans])
        sl = (C.c_size_t * n)(*[s.size for s in scans])
        op = (_vp * n)(*[_ptr(o) for o in outs])
        self._pending.append((scans, outs))  # keep the buffers alive until wait()
        rc = self._lib.kpeg_cuda_submit_batch(self._h, C.byref(plan), n, sp, sl, op)
        self._check(rc, "kpeg_cuda_submit_batch")

    def prepare_batch(self, scans: list[np.ndarray], outs: list[np.ndarray]):
        """The pointer / length arrays kpeg_cuda_submit_batch takes, built once for buffers that are reused step after
        step (the marshalling of thousands of numpy arrays costs more than the call).  -> handle for submit_prepared."""
        n = len(scans)
        for a in list(scans) + list(outs):
            if not (a.flags["C_CONTIGUOUS"] and a.dtype == np.uint8):
                raise ValueError("prepare_batch needs contiguous uint8 arrays (they are used in place)")
        return (n, (_vp * n)(*[_ptr(s) for s in scans]), (C.c_size_t * n)(*[s.size for s in scans]),
                (_vp * n)(*[_ptr(o) for o in outs]), scans, outs)

    def submit_prepared(self, plan: Plan, handle):
        n, sp, sl, op, scans, outs = handle
        self._pending.append((scans, outs))
        self._check(self._lib.kpeg_cuda_submit_batch(self._h, C.byref(plan), n, sp, sl, op), "kpeg_cuda_submit_batch")

    def wait(self):
        rc = self._lib.kpeg_cuda_wait(self._h, C.byref(self.last_stats))
        self._pending.clear()
        self._check(rc, "kpeg_cuda_wait")

    def decode_ppm_device(self, plan: Plan, d_scan: int, scan_len: int, d_out: int, cap: int, scale: int | None = None):
        """GPU-side PPM writer (kpeg_cuda_decode_ppm_device) -> (offset, length) of the file inside d_out."""
        plan = _scaled_plan(plan, scale)
        off, ln = C.c_size_t(0), C.c_size_t(0)
        rc = self._lib.kpeg_cuda_decode_ppm_device(self._h, C.byref(plan), d_scan, scan_len, d_out, cap, C.byref(off),
                                                   C.byref(ln), C.byref(self.last_stats))
        self._check(rc, "kpeg_cuda_decode_ppm_device")
        return off.value, ln.value

    def interleaved_to_planar(self, d_rgb: int, d_planes: int, npixels: int):
        self._check(self._lib.kpeg_cuda_interleaved_to_planar(self._h, d_rgb, d_planes, npixels), "interleaved_to_planar")

    # -- encode ------------------------------------------------------------------------------------
    def encode(self, pixels: np.ndarray, quality: int = 90, restart_interval: int = 0,
               flags: int = KPEG_FLAG_REF_PARITY) -> np.ndarray:
        """Baseline JPEG of `pixels` ((H, W, 3) RGB or (H, W) gray uint8), encoded on the GPU (kpeg_cuda_encode).
        flags: KPEG_FLAG_REF_PARITY and / or KPEG_FLAG_OPTIMIZE_HUFFMAN (per-image Huffman tables: smaller files)."""
        h, w, nc = _image_shape(pixels)
        p = encode_params(w, h, nc, quality, restart_interval, flags)
        src = np.ascontiguousarray(pixels)
        out = np.empty(self._lib.kpeg_encode_bound(C.byref(p)), dtype=np.uint8)
        n = C.c_size_t(0)
        rc = self._lib.kpeg_cuda_encode(self._h, C.byref(p), _ptr(src), _ptr(out), out.size, C.byref(n),
                                        C.byref(self.last_stats))
        self._check(rc, "kpeg_cuda_encode")
        return out[:n.value].copy()

    def encode_device(self, d_pixels: int, width: int, height: int, ncomp: int, d_out: int, cap: int, quality: int = 90,
                      restart_interval: int = 0, flags: int = KPEG_FLAG_REF_PARITY) -> int:
        """kpeg_cuda_encode_device: device pixels in, the file assembled at d_out; returns its length.  A cap below it
        raises KpegError(KPEG_ERR_NOMEM) with the size needed in `.needed`."""
        p = encode_params(width, height, ncomp, quality, restart_interval, flags)
        n = C.c_size_t(0)
        rc = self._lib.kpeg_cuda_encode_device(self._h, C.byref(p), d_pixels, d_out, cap, C.byref(n),
                                               C.byref(self.last_stats))
        if rc == KPEG_ERR_NOMEM:
            err = KpegError(rc, f"kpeg_cuda_encode_device: {n.value} bytes needed, {cap} given")
            err.needed = n.value
            raise err
        self._check(rc, "kpeg_cuda_encode_device")
        return n.value

    # -- transcode ---------------------------------------------------------------------------------
    def transcode(self, data, restart_interval: int = KPEG_TRANSCODE_KEEP_RESTART, transform: int = KPEG_XFORM_NONE,
                  optimize: bool = False) -> bytes:
        """Lossless transcode on the GPU (kpeg_cuda_transcode): the same quantised coefficients, moved by `transform`
        (KPEG_XFORM_*), re-coded with another restart interval (-1 keeps the input's) and Annex K or, optimize, per-image
        Huffman tables."""
        buf = np.ascontiguousarray(np.frombuffer(data, dtype=np.uint8) if not isinstance(data, np.ndarray) else data)
        p = transcode_params(restart_interval, transform, optimize)
        cap = self._lib.kpeg_transcode_bound(_ptr(buf), buf.size, C.byref(p))
        out = np.empty(max(int(cap), 1), dtype=np.uint8)
        n = C.c_size_t(0)
        rc = self._lib.kpeg_cuda_transcode(self._h, _ptr(buf), buf.size, C.byref(p), _ptr(out), cap, C.byref(n),
                                           C.byref(self.last_stats))
        self._check(rc, "kpeg_cuda_transcode")
        return out[:n.value].tobytes()

    def transcode_into(self, data, out: np.ndarray, restart_interval: int = KPEG_TRANSCODE_KEEP_RESTART,
                       transform: int = KPEG_XFORM_NONE, optimize: bool = False) -> int:
        """kpeg_cuda_transcode into a caller's buffer (pinned for speed); returns the length.  A buffer below it raises
        KpegError(KPEG_ERR_NOMEM) with the size needed in `.needed`."""
        buf = np.ascontiguousarray(np.frombuffer(data, dtype=np.uint8) if not isinstance(data, np.ndarray) else data)
        p = transcode_params(restart_interval, transform, optimize)
        n = C.c_size_t(0)
        rc = self._lib.kpeg_cuda_transcode(self._h, _ptr(buf), buf.size, C.byref(p), _ptr(out), out.nbytes, C.byref(n),
                                           C.byref(self.last_stats))
        if rc == KPEG_ERR_NOMEM:
            err = KpegError(rc, f"kpeg_cuda_transcode: {n.value} bytes needed, {out.nbytes} given")
            err.needed = n.value
            raise err
        self._check(rc, "kpeg_cuda_transcode")
        return n.value

    def decode_batch_packed_device(self, plan: Plan, n: int, d_packed: int, packed_len: int, d_out: int):
        rc = self._lib.kpeg_cuda_decode_batch_packed_device(self._h, C.byref(plan), n, d_packed, packed_len, d_out,
                                                            C.byref(self.last_stats))
        self._check(rc, "kpeg_cuda_decode_batch_packed_device")


def decode_file_tiled(devices: list[int], data, flags: int = KPEG_FLAG_REF_PARITY, out: np.ndarray | None = None,
                      scale: int | None = None):
    """One image over several GPUs (kpeg_cuda_decode_file_tiled): restart-interval bands, one per listed device, each
    decoded into its rows of ONE host frame (scale: as in Decoder.decode_file).  Returns (pixels, Stats)."""
    lib = load_cuda_library()
    flags = _scaled_flags(flags, scale)
    buf = np.frombuffer(data, dtype=np.uint8) if not isinstance(data, np.ndarray) else data
    plan, _, _ = parse_jfif(buf)
    plan.flags = flags
    shape = output_shape(plan)
    if out is None:
        out = np.empty(shape, dtype=np.uint8)
    dv = (C.c_int * len(devices))(*devices)
    st = Stats()
    rc = lib.kpeg_cuda_decode_file_tiled(dv, len(devices), _ptr(buf), buf.size, flags, _ptr(out), out.nbytes, None, C.byref(st))
    if rc != KPEG_OK:
        raise KpegError(rc, f"kpeg_cuda_decode_file_tiled: {lib.kpeg_tiled_last_error().decode(errors='replace')}")
    return out.reshape(shape), st


def decode_tiled(devices: list[int], plan: Plan, scan: np.ndarray, out: np.ndarray) -> Stats:
    """kpeg_cuda_decode_tiled on an already parsed image: restart-interval bands of `scan`, one per listed device (a
    device may be listed several times: its bands then overlap their copies and kernels), into the rows of `out`."""
    lib = load_cuda_library()
    assert out.nbytes == int(np.prod(output_shape(plan))) and out.flags.c_contiguous and scan.flags.c_contiguous
    dv = (C.c_int * len(devices))(*devices)
    st = Stats()
    rc = lib.kpeg_cuda_decode_tiled(dv, len(devices), C.byref(plan), _ptr(scan), scan.size, _ptr(out), C.byref(st))
    if rc != KPEG_OK:
        raise KpegError(rc, f"kpeg_cuda_decode_tiled: {lib.kpeg_tiled_last_error().decode(errors='replace')}")
    return st


def packed_offsets(scans: list[np.ndarray]) -> np.ndarray:
    """Offsets of the scans inside the packed batch stream (each scan is followed by a 2-byte RSTn)."""
    off = np.zeros(len(scans) + 1, dtype=np.uint64)
    off[1:] = np.cumsum([int(s.size) + 2 for s in scans])
    return off


def pack_batch(scans: list[np.ndarray]) -> np.ndarray:
    """Host helper: the packed batch stream (scan, RSTn, scan, RSTn, ...) kpeg_batch_pack builds."""
    lib = load_cuda_library()
    n = len(scans)
    scans = [np.ascontiguousarray(s, dtype=np.uint8) for s in scans]
    sl = (C.c_size_t * n)(*[s.size for s in scans])
    total = lib.kpeg_batch_packed_size(n, sl)
    out = np.empty(total, dtype=np.uint8)
    sp = (_vp * n)(*[_ptr(s) for s in scans])
    rc = lib.kpeg_batch_pack(n, sp, sl, _ptr(out), out.size)
    if rc != KPEG_OK:
        raise KpegError(rc, "kpeg_batch_pack")
    return out
