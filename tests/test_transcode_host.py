"""Lossless transcode (kpeg_cuda_transcode) on the CPU: the reference's self-consistency, the CPU replay of the GPU path
(tests/emu/emu_transcode.cpp) against the reference, the transform table against numpy on decoded pixels, the range
rules, parameters, the bound and the header layout."""
from __future__ import annotations

import ctypes as C
import io
import itertools

import numpy as np
import pytest

import coef_fields as CF
import helpers as H
import jpeg_writer as JW
import libkpeg_b200 as K
import transcode_cases as TC
from libkpeg_b200 import api
from libkpeg_b200.synth import (EMIT_RESTART, NON_INTERLEAVED, OPTIMIZE_HUFFMAN, QUIRK_FREE, SynthParams, synth_encode,
                                synth_encode_coefficients)


def synth(w, h, nc=3, q=90, ri=0, flags=0, seed=5):
    return synth_encode(SynthParams(w, h, file_components=nc, quality=q, restart_interval=ri,
                                    flags=flags | (EMIT_RESTART if ri else 0), seed=seed)).tobytes()


def with_app_segments(jpg: bytes) -> bytes:
    """APP1 (Exif-like) and COM segments inserted after APP0: the transcoder does not copy them."""
    app1 = b"\xff\xe1" + (2 + 14).to_bytes(2, "big") + b"Exif\0\0" + bytes(8)
    com = b"\xff\xfe" + (2 + 5).to_bytes(2, "big") + b"hello"
    return jpg[:20] + app1 + com + jpg[20:]


def pil_file(w, h, optimize):
    from PIL import Image
    rng = np.random.default_rng(w * 7 + h)
    img = (rng.random((h, w, 3)) * 60 + np.linspace(0, 190, w)[None, :, None]).astype(np.uint8)
    b = io.BytesIO()
    Image.fromarray(img).save(b, "JPEG", quality=88, subsampling=0, optimize=optimize)
    return b.getvalue()


def inputs():
    base = synth(40, 24, seed=9)
    cases = {
        "synth 64x48 q90": synth(64, 48),
        "synth 37x21 ragged q75 DRI 3": synth(37, 21, q=75, ri=3, seed=6),
        "synth gray 48x40 q95 opt": synth(48, 40, nc=1, q=95, flags=OPTIMIZE_HUFFMAN),
        "synth 24x16 one scan per component": synth(24, 16, flags=NON_INTERLEAVED),
        "distinct tables": JW.distinct_tables_variant(base, H.oracle_decode, K.parse_jfif),
        "APPn + COM": with_app_segments(synth(32, 24, seed=4)),
        "PIL 4:4:4": pil_file(48, 32, False),
        "PIL 4:4:4 optimize": pil_file(40, 24, True),
    }
    for fam in ("wide_and_huge", "dc_only"):
        for f in CF.build(fam, 128, 64, 3)[:1]:
            cases[f"coef field {fam}"] = CF.encode(f)
    return cases


INPUTS = inputs()


# ---- reference self-consistency -------------------------------------------------------------------------------------
@pytest.mark.parametrize("w,h,nc,q,ri,opt", [
    (64, 48, 3, 90, 0, False), (37, 21, 3, 75, 3, True), (17, 9, 1, 50, 0, False), (100, 61, 3, 95, 13, True),
    (8, 8, 1, 100, 1, True), (33, 40, 3, 30, 5, False)])
def test_reference_reproduces_the_encoders_files(w, h, nc, q, ri, opt):
    for flags in (0, QUIRK_FREE):
        jpg = synth(w, h, nc=nc, q=q, ri=ri, flags=flags | (OPTIMIZE_HUFFMAN if opt else 0))
        assert TC.reference(jpg, -1, 0, opt) == jpg


def test_encode_coefficients_rejects_uncodable_values():
    tq, qt = [0], {0: [1] * 64}
    coef = np.zeros((1, 64), np.int16)
    coef[0, 0] = 2048  # DC difference of category 12
    assert synth_encode_coefficients(8, 8, coef, tq, qt) is None
    coef[0, 0] = 2047
    assert synth_encode_coefficients(8, 8, coef, tq, qt) is not None
    coef[0, 5] = -1024  # AC beyond category 10
    assert synth_encode_coefficients(8, 8, coef, tq, qt) is None


# ---- the CPU replay of the GPU path against the reference ----------------------------------------------------------
@pytest.mark.parametrize("name", sorted(INPUTS))
def test_replay_matches_reference(name):
    jpg = INPUTS[name]
    for t, opt, ri in itertools.product(range(8), (False, True), (-1, 0, 2)):
        ref = TC.reference(jpg, ri, t, opt)
        got, info = TC.emu_transcode(jpg, ri, t, opt)
        assert got == ref, (name, TC.NAMES[t], opt, ri)
        if isinstance(ref, bytes):
            assert len(ref) <= int(info[3])
            assert K.transcode_bound(jpg, ri, t, opt) == int(info[3])


def test_replay_matches_reference_on_lena():
    jpg = (H.GOLDEN / "lena.jpg").read_bytes()
    for t, opt in itertools.product(range(8), (False, True)):
        ri = 64 if t % 2 else -1
        assert TC.emu_transcode(jpg, ri, t, opt)[0] == TC.reference(jpg, ri, t, opt), (TC.NAMES[t], opt)


# ---- the transform table against numpy, on decoded pixels -----------------------------------------------------------
@pytest.mark.parametrize("nc", [1, 3])
def test_transforms_against_numpy(nc):
    jpg = synth(48, 32, nc=nc, q=85, seed=21)
    src = H.oracle_decode(jpg, parity=False)["pixels"]
    worst = {}
    for t in range(8):
        out = TC.reference(jpg, -1, t)
        got = H.oracle_decode(out, parity=False)["pixels"]
        want = TC.transform_pixels(src, t)
        assert got.shape == want.shape, TC.NAMES[t]
        d = int(np.abs(got.astype(int) - want.astype(int)).max())
        worst[TC.NAMES[t]] = d
        if t in (0, 1, 2, 6):
            assert d == 0, (TC.NAMES[t], d)  # flips keep the IDCT's order of summation
        else:
            assert d <= 1, (TC.NAMES[t], d)  # a transpose reorders it: rounding may differ by one
    print("max |pixel difference| per transform:", worst)


def test_transform_table_is_numpys():
    """transcode_core.h's in-block table against the numpy transform of a block holding every position once."""
    tab = np.zeros((8, 64), np.uint8)
    TC.emu().emu_xform_table(tab.ctypes.data)
    blk = np.arange(1, 65, dtype=np.int16)[None, :]
    for t in range(8):
        moved, _ = TC.transform_coefficients(blk, 8, 8, 1, t)
        src = (tab[t] & 63).astype(int)
        sign = np.where(tab[t] & 0x80, -1, 1)
        assert np.array_equal(moved[0], sign * blk[0, src]), TC.NAMES[t]


# ---- range rules ------------------------------------------------------------------------------------------------------
def test_dc_drift_is_rejected_by_reference_and_replay():
    jpg = TC.dc_drift_file()
    coef = H.oracle_decode(jpg, parity=False, want_pixels=False)["coef"]
    assert coef[:, 0].max() > 2047  # absolute DC past 2047, every coded difference legal
    assert isinstance(TC.reference(jpg, -1, 0), bytes)
    assert TC.emu_transcode(jpg, -1, 0)[0] == TC.reference(jpg, -1, 0)
    for ri, t in ((1, 0), (0, 3), (0, 1), (-1, 2)):
        assert TC.reference(jpg, ri, t) == TC.UNSUPPORTED, (ri, t)
        assert TC.emu_transcode(jpg, ri, t)[0] == TC.UNSUPPORTED, (ri, t)


# ---- parameters, preconditions, bound, header ------------------------------------------------------------------------
def test_preconditions_table():
    for (w, h), t in itertools.product([(16, 16), (17, 16), (16, 17), (17, 17)], range(8)):
        jpg = synth(w, h, nc=1, seed=2)
        ok = TC.allowed(t, w, h)
        assert (K.transcode_bound(jpg, -1, t) > 0) == ok, (w, h, TC.NAMES[t])
        got, _ = TC.emu_transcode(jpg, -1, t)
        assert (got == TC.UNSUPPORTED) == (not ok), (w, h, TC.NAMES[t])
    expected = {1: "w", 2: "h", 4: "wh", 5: "h", 6: "wh", 7: "w"}  # the issue's table, axis by axis
    for t, need in expected.items():
        assert TC.allowed(t, 17, 16) == ("w" not in need) and TC.allowed(t, 16, 17) == ("h" not in need)


def test_bad_parameters():
    jpg = synth(16, 16)
    lib = api.load_cuda_library()
    buf = np.frombuffer(jpg, np.uint8)
    for p in (api.TranscodeParams(-2, 0, 0), api.TranscodeParams(65536, 0, 0), api.TranscodeParams(0, 8, 0),
              api.TranscodeParams(0, 0, 1), api.TranscodeParams(0, 0, 4)):
        assert lib.kpeg_transcode_bound(buf.ctypes.data, buf.size, C.byref(p)) == 0
        assert TC.emu().emu_transcode is not None
    assert lib.kpeg_transcode_bound(buf.ctypes.data, buf.size, None) == 0
    assert lib.kpeg_transcode_bound(buf.ctypes.data, 10, C.byref(api.TranscodeParams(0, 0, 0))) == 0
    with pytest.raises(ValueError):
        api.transcode_params(transform=9)


def test_bound_covers_worst_case_files():
    rng = np.random.default_rng(3)
    from libkpeg_b200.synth import synth_encode_pixels
    for nc, opt in ((3, False), (3, True), (1, True)):
        px = rng.integers(0, 256, size=(24, 40, nc) if nc == 3 else (24, 40), dtype=np.uint8)
        sp = SynthParams(40, 24, file_components=nc, quality=100, flags=OPTIMIZE_HUFFMAN if opt else 0)
        jpg = synth_encode_pixels(sp, px.reshape(24, 40, nc)).tobytes()
        for t, ri in ((0, 1), (5, 0), (6, 2)):
            out = TC.reference(jpg, ri, t, opt)
            assert isinstance(out, bytes) and len(out) <= K.transcode_bound(jpg, ri, t, opt)


def test_header_layout():
    jpg = JW.distinct_tables_variant(synth(16, 8, seed=3), H.oracle_decode, K.parse_jfif)
    out, _ = TC.emu_transcode(jpg, 1, 3, False)
    assert out[:20] == bytes.fromhex("ffd8ffe000104a46494600010101004800480000")
    frame, scans = api.parse_jfif_scans(out)
    assert (frame.width, frame.height, frame.ncomp) == (8, 16, 3) and len(scans) == 1
    assert list(scans[0].plan.comp_tq[:3]) == [2, 0, 1]
    assert scans[0].plan.restart_interval == 1
    # DQT ids ascending, the input's values transposed
    pos, ids = 2, []
    while out[pos + 1] != 0xC0:
        ln = int.from_bytes(out[pos + 2:pos + 4], "big")
        if out[pos + 1] == 0xDB:
            ids.append(out[pos + 4])
        pos += 2 + ln
    assert ids == [0, 1, 2]
    _, in_scans = api.parse_jfif_scans(jpg)
    for tid in range(3):
        assert list(scans[0].plan.qt[tid]) == TC.transpose_qt(list(in_scans[0].plan.qt[tid]))
    assert b"Exif" not in TC.emu_transcode(with_app_segments(synth(16, 16)), -1, 0)[0]


def test_struct_layout_matches_header():
    text = (H.ROOT / "include" / "kpeg_cuda.h").read_text()
    assert "int32_t restart_interval; /* output MCUs per interval" in text
    assert C.sizeof(api.TranscodeParams) == 12
    assert [f[0] for f in api.TranscodeParams._fields_] == ["restart_interval", "transform", "flags"]
    for i, name in enumerate(("NONE", "FLIP_H", "FLIP_V", "TRANSPOSE", "TRANSVERSE", "ROT90", "ROT180", "ROT270")):
        assert f"#define KPEG_XFORM_{name} {i}u" in text
        assert getattr(K, f"KPEG_XFORM_{name}") == i
    assert "#define KPEG_TRANSCODE_KEEP_RESTART (-1)" in text
