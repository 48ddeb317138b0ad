"""Test-side bindings: the CPU oracle (oracle/_ref/libkpeg_oracle.so), the compiled unmodified
reference (oracle/_ref/kpeg_ref_quiet) and the CPU single-stepper of the kernel logic
(tests/emu/libkpeg_emu.so).  Only tests/, bench.py's cpu_baseline leg and __graft_entry__.smoke()
may touch oracle/ -- and only as the checker."""
from __future__ import annotations

import ctypes as C
import os
import shutil
import subprocess
import tempfile
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
ORACLE_DIR = ROOT / "oracle"
REF_BIN = ORACLE_DIR / "_ref" / "kpeg_ref_quiet"
GOLDEN = ROOT / "tests" / "golden"

KPO_FLAG_REF_PARITY = 1


class KpoImage(C.Structure):
    _fields_ = [("width", C.c_int32), ("height", C.c_int32), ("ncomp", C.c_int32), ("mcus_x", C.c_int32),
                ("mcus_y", C.c_int32), ("restart_interval", C.c_int32), ("nblocks", C.c_int64),
                ("scan_bytes", C.c_int64), ("coef", C.POINTER(C.c_int16)), ("pixels", C.POINTER(C.c_uint8))]


_oracle = None


def oracle():
    global _oracle
    if _oracle is None:
        so = ORACLE_DIR / "_ref" / "libkpeg_oracle.so"
        if not so.exists():
            subprocess.run(["make", "-C", str(ORACLE_DIR), "_ref/libkpeg_oracle.so"], check=True,
                           stdout=subprocess.DEVNULL)
        lib = C.CDLL(str(so))
        lib.kpo_decode.restype = C.c_int
        lib.kpo_decode.argtypes = [C.c_void_p, C.c_size_t, C.c_uint32, C.c_int, C.POINTER(KpoImage)]
        lib.kpo_free.argtypes = [C.POINTER(KpoImage)]
        lib.kpo_set_threads.argtypes = [C.c_int]
        lib.kpo_ppm_header.restype = C.c_int
        lib.kpo_ppm_header.argtypes = [C.c_int, C.c_int, C.c_char_p, C.c_size_t]
        lib.kpo_huff_codes.restype = C.c_int
        lib.kpo_huff_codes.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
        lib.kpo_huff_lookup.restype = C.c_int
        lib.kpo_huff_lookup.argtypes = [C.c_void_p, C.c_void_p, C.c_char_p]
        lib.kpo_extend.restype = C.c_int
        lib.kpo_extend.argtypes = [C.c_int, C.c_int]
        lib.kpo_zigzag_to_rc.argtypes = [C.c_int, C.POINTER(C.c_int), C.POINTER(C.c_int)]
        lib.kpo_idct8x8.argtypes = [C.c_void_p, C.c_void_p]
        lib.kpo_level_shift.restype = C.c_int
        lib.kpo_level_shift.argtypes = [C.c_float]
        lib.kpo_ycbcr_to_rgb.argtypes = [C.c_int, C.c_int, C.c_int, C.c_void_p]
        lib.kpo_block_to_samples.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
        _oracle = lib
    return _oracle


def oracle_decode(data, parity: bool = True, want_pixels: bool = True, threads: int | None = None):
    """-> dict(width, height, ncomp, coef [nblocks,64] int16, pixels [H,W,nc] uint8 or None)."""
    lib = oracle()
    buf = np.frombuffer(bytes(data), dtype=np.uint8) if not isinstance(data, np.ndarray) else data
    lib.kpo_set_threads(threads if threads else min(os.cpu_count() or 1, 32))
    img = KpoImage()
    rc = lib.kpo_decode(buf.ctypes.data, buf.size, KPO_FLAG_REF_PARITY if parity else 0, int(want_pixels), C.byref(img))
    if rc != 0:
        raise RuntimeError(f"kpo_decode rc={rc}")
    try:
        coef = np.ctypeslib.as_array(img.coef, shape=(img.nblocks, 64)).copy()
        pixels = None
        if want_pixels:
            shape = (img.height, img.width, 3) if img.ncomp == 3 else (img.height, img.width)
            pixels = np.ctypeslib.as_array(img.pixels, shape=shape).copy()
        return dict(width=img.width, height=img.height, ncomp=img.ncomp, coef=coef, pixels=pixels,
                    scan_bytes=img.scan_bytes, restart_interval=img.restart_interval)
    finally:
        lib.kpo_free(C.byref(img))


def have_reference_binary() -> bool:
    return REF_BIN.exists() and os.access(REF_BIN, os.X_OK)


def reference_decode(jpeg_bytes) -> bytes:
    """Run the compiled, unmodified reference (quiet-log twin) on one file in a scratch directory,
    one process per image (SURVEY F5).  Returns the PPM file bytes."""
    with tempfile.TemporaryDirectory() as td:
        p = Path(td) / "img.jpg"
        p.write_bytes(bytes(jpeg_bytes))
        subprocess.run([str(REF_BIN), str(p)], cwd=td, check=True, stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL,
                       timeout=1200)
        out = Path(td) / "img.ppm"
        if not out.exists():
            raise RuntimeError("reference produced no PPM (unsupported or malformed input)")
        return out.read_bytes()


def split_ppm(ppm: bytes):
    """-> (header bytes, payload ndarray [H,W,3])."""
    # P6\n#comment\nW H\n255\n
    lines = []
    pos = 0
    while len(lines) < 4:
        e = ppm.index(b"\n", pos)
        lines.append(ppm[pos:e])
        pos = e + 1
    w, h = map(int, lines[2].split())
    payload = np.frombuffer(ppm, dtype=np.uint8, count=w * h * 3, offset=pos).reshape(h, w, 3)
    return ppm[:pos], payload


_emu = None


def emu():
    global _emu
    if _emu is None:
        from libkpeg_b200._build import build_emu
        build_emu()
        lib = C.CDLL(str(ROOT / "tests" / "emu" / "libkpeg_emu.so"))
        lib.emu_decode.restype = C.c_int
        lib.emu_decode.argtypes = [C.c_void_p, C.c_size_t, C.c_void_p, C.c_uint32, C.c_uint32, C.c_void_p, C.c_void_p,
                                   C.c_void_p]
        lib.emu_colour.restype = C.c_int
        lib.emu_colour.argtypes = [C.c_int, C.c_int, C.c_int, C.c_void_p]
        lib.emu_idct_fast.restype = C.c_float
        lib.emu_idct_fast.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p]
        lib.emu_classify_compare.restype = C.c_uint32
        lib.emu_classify_compare.argtypes = [C.c_void_p, C.c_uint32, C.POINTER(C.c_int)]
        lib.emu_huff_lookup.restype = C.c_uint32
        lib.emu_huff_lookup.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_uint32, C.c_int]
        lib.emu_huff_lookup_many.restype = None
        lib.emu_huff_lookup_many.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_uint32, C.c_int, C.c_void_p]
        lib.emu_huff_layout.restype = C.c_int
        lib.emu_huff_layout.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.POINTER(C.c_uint32), C.c_void_p]
        lib.emu_restart_padding_decodes.restype = C.c_int
        lib.emu_restart_padding_decodes.argtypes = [C.c_void_p]
        lib.emu_zigzag.restype = C.c_int
        lib.emu_zigzag.argtypes = [C.c_int]
        lib.emu_pair_tables.restype = C.c_int
        lib.emu_pair_tables.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
        _emu = lib
    return _emu


def emu_decode(data, flags: int = 1, sub_bits: int = 512, want_pixels: bool = True, scans=None, plan=None):
    """CPU replay of the kernel pipeline on one file (or, with scans+plan, a packed batch)."""
    import libkpeg_b200 as K
    from libkpeg_b200.api import pack_batch
    lib = emu()
    if scans is None:
        buf = np.frombuffer(bytes(data), dtype=np.uint8) if not isinstance(data, np.ndarray) else data
        plan, off, ln = K.parse_jfif(buf)
        stream = np.ascontiguousarray(buf[off:off + ln])
        n = 1
    else:
        stream = pack_batch(scans)
        n = len(scans)
    plan.flags = flags
    nblocks = n * ((plan.width + 7) // 8) * ((plan.height + 7) // 8) * plan.ncomp
    coef = np.zeros((nblocks, 64), dtype=np.int16)
    shape = (n, plan.height, plan.width, plan.ncomp)
    pixels = np.zeros(shape, dtype=np.uint8) if want_pixels else None
    info = np.zeros(12, dtype=np.uint32)
    rc = lib.emu_decode(stream.ctypes.data, stream.size, C.addressof(plan), n, sub_bits, coef.ctypes.data,
                        pixels.ctypes.data if want_pixels else None, info.ctypes.data)
    if rc != 0:
        raise RuntimeError(f"emu_decode rc={rc}")
    if want_pixels:
        pixels = pixels[0] if scans is None else pixels
        if plan.ncomp == 1:
            pixels = pixels[..., 0]
    return dict(coef=coef, pixels=pixels, status=int(info[0]), nsub=int(info[1]), rounds=int(info[2]),
                exact=int(info[3]), colour_exact=int(info[4]), total_bits=int(info[5]), final_slot=int(info[6]),
                records_ok=bool(info[7]), max_records=int(info[8]), subs_over_kmax=int(info[9]), plan=plan)
