"""Lossless transcode on a B200 (kpeg_cuda_transcode): byte identity with the reference (transcode_cases.reference) on the
host test's inputs for every transform and both table modes, a 16384 x 16384 file there and back, identities with the
GPU encoder, coefficients and pixels of the output, the multi-GPU motivation (restart markers added, then a tiled
decode), errors, the CLI and a guard-mode run."""
import io
import itertools
import os
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest

import helpers as H
import libkpeg_b200 as K
import transcode_cases as TC
from libkpeg_b200 import api
from libkpeg_b200.synth import EMIT_RESTART, QUIRK_FREE, SynthParams, synth_encode, synth_pixels
from test_transcode_host import INPUTS, synth

pytestmark = pytest.mark.gpu
ROOT = Path(__file__).resolve().parent.parent
KPEG = ROOT / "libkpeg_b200" / "lib" / "kpeg"


@pytest.fixture(scope="module")
def dec():
    d = K.Decoder(device=0)
    yield d
    d.close()


def transcode_rc(dec, jpg, ri=-1, t=0, opt=False):
    try:
        return dec.transcode(jpg, ri, t, opt)
    except K.KpegError as e:
        return e.code


@pytest.mark.parametrize("name", sorted(INPUTS))
def test_bytes_equal_the_reference(dec, name):
    jpg = INPUTS[name]
    for t, opt, ri in itertools.product(range(8), (False, True), (-1, 0, 2)):
        assert transcode_rc(dec, jpg, ri, t, opt) == TC.reference(jpg, ri, t, opt), (name, TC.NAMES[t], opt, ri)


def test_lena_every_transform(dec, lena_jpg):
    for t, opt in itertools.product(range(8), (False, True)):
        assert dec.transcode(lena_jpg, 64, t, opt) == TC.reference(lena_jpg, 64, t, opt), (TC.NAMES[t], opt)


def test_16k_restart_markers_removed_and_added(dec):
    sp = SynthParams(16384, 16384, quality=85, restart_interval=2048, flags=QUIRK_FREE | EMIT_RESTART, seed=16)
    marked = synth_encode(sp).tobytes()
    sp.flags = QUIRK_FREE  # the twin: same coefficients, no DRI / RSTn
    plain = synth_encode(sp).tobytes()
    assert dec.transcode(marked, restart_interval=0) == plain
    assert dec.transcode(plain, restart_interval=2048) == marked


@pytest.mark.parametrize("nc", [1, 3])
def test_identities_with_the_encoder(dec, nc):
    px = synth_pixels(SynthParams(203, 97, file_components=nc, seed=7))
    px = px if nc == 3 else px[..., 0]
    for q in (50, 90):
        base = dec.encode(px, quality=q, flags=0).tobytes()
        assert dec.transcode(base) == base
        assert dec.transcode(base, restart_interval=5) == dec.encode(px, quality=q, restart_interval=5, flags=0).tobytes()
        assert dec.transcode(base, optimize=True) == dec.encode(px, quality=q, flags=K.KPEG_FLAG_OPTIMIZE_HUFFMAN).tobytes()
        r7 = dec.encode(px, quality=q, restart_interval=7, flags=0).tobytes()
        assert dec.transcode(r7) == r7


def test_coefficients_and_pixels(dec):
    from PIL import Image
    jpg = INPUTS["PIL 4:4:4"]
    w, h, nc, _, _, _ = TC.frame_of(jpg)
    src = H.oracle_decode(jpg, parity=False, want_pixels=False)["coef"]
    for t in range(8):
        out = dec.transcode(jpg, transform=t)
        got_px = dec.decode_file(out, flags=0)
        coef = dec.read_coefficients(src.shape[0])
        want, _ = TC.transform_coefficients(src, w, h, nc, t)
        assert np.array_equal(coef, want), TC.NAMES[t]
        if t == 0:
            a = np.asarray(Image.open(io.BytesIO(out)))
            b = np.asarray(Image.open(io.BytesIO(jpg)))
            assert np.array_equal(a, b)
            assert np.array_equal(got_px, dec.decode_file(jpg, flags=0))


def test_parity_pixels_kept_without_transform(dec, lena_jpg):
    for jpg in (lena_jpg, INPUTS["synth 37x21 ragged q75 DRI 3"], INPUTS["distinct tables"]):
        for opt in (False, True):
            out = dec.transcode(jpg, optimize=opt)
            assert np.array_equal(dec.decode_file(out), dec.decode_file(jpg))


def test_restart_markers_enable_the_tiled_decode(dec):
    sp = SynthParams(3840, 2160, quality=95, flags=QUIRK_FREE, seed=44)
    jpg = synth_encode(sp).tobytes()
    out = dec.transcode(jpg, restart_interval=3840 // 8)
    got, _ = api.decode_file_tiled([0, 0, 0, 0], out, flags=0)
    assert np.array_equal(got, dec.decode_file(jpg, flags=0))


def test_errors(dec):
    from PIL import Image
    img = np.asarray(synth_pixels(SynthParams(64, 48, seed=3)))
    for kw in (dict(progressive=True, subsampling=0), dict(subsampling=2)):
        b = io.BytesIO()
        Image.fromarray(img).save(b, "JPEG", quality=80, **kw)
        assert transcode_rc(dec, b.getvalue()) == K.api.KPEG_ERR_UNSUPPORTED, kw
    good = synth(64, 48, seed=8)
    _, off, ln = K.parse_jfif(good)
    bad = bytearray(good)
    bad[off + ln // 2:off + ln // 2 + 8] = b"\xff\xd3" * 4  # markers inside the scan
    assert transcode_rc(dec, bytes(bad)) == K.api.KPEG_ERR_STREAM
    ragged = synth(37, 21, seed=1)
    drift = TC.dc_drift_file()
    for jpg, t, ri in ((ragged, 1, -1), (ragged, 6, -1), (drift, 0, 1), (drift, 3, 0)):
        out = np.full(1 << 16, 0xAB, np.uint8)
        with pytest.raises(K.KpegError) as e:
            dec.transcode_into(jpg, out, ri, t)
        assert e.value.code == K.api.KPEG_ERR_UNSUPPORTED
        assert (out == 0xAB).all()
    # caps below the header and below the file
    full = dec.transcode(good, optimize=True)
    for cap in (10, 300, len(full) - 1):
        out = np.full(cap + 64, 0xAB, np.uint8)
        with pytest.raises(K.KpegError) as e:
            dec.transcode_into(good, out[:cap], optimize=True)
        assert e.value.code == K.api.KPEG_ERR_NOMEM and e.value.needed == len(full)
        assert (out == 0xAB).all()
    # the context still works
    assert dec.transcode(good) == TC.reference(good)
    px = synth_pixels(SynthParams(40, 24, seed=2))
    assert np.array_equal(dec.decode_file(dec.encode(px).tobytes()), H.oracle_decode(dec.encode(px).tobytes())["pixels"])


def test_cli(tmp_path, dec):
    jpg = synth(64, 48, seed=12)
    (tmp_path / "in.jpg").write_bytes(jpg)
    for t, name in enumerate(TC.NAMES):
        subprocess.run([str(KPEG), "--quiet", "--transform", name, "in.jpg", f"o{t}.jpg"], cwd=tmp_path, check=True)
        assert (tmp_path / f"o{t}.jpg").read_bytes() == TC.reference(jpg, -1, t), name
    subprocess.run([str(KPEG), "--quiet", "--optimize", "--restart", "4", "in.jpg", "opt.jpg"], cwd=tmp_path, check=True)
    assert (tmp_path / "opt.jpg").read_bytes() == TC.reference(jpg, 4, 0, True)
    (tmp_path / "bad.jpg").write_bytes(b"\xff\xd8\xff\xdb\x00")
    r = subprocess.run([str(KPEG), "--quiet", "bad.jpg", "x.jpg"], cwd=tmp_path, capture_output=True, text=True)
    assert r.returncode == 0 and not (tmp_path / "x.jpg").exists()
    assert "transcoding" in (tmp_path / "kpeg.log").read_text()
    px = synth_pixels(SynthParams(40, 24, seed=2))
    with open(tmp_path / "in.ppm", "wb") as f:
        f.write(b"P6\n40 24\n255\n" + px.tobytes())
    subprocess.run([str(KPEG), "--quiet", "in.ppm", "enc.jpg"], cwd=tmp_path, check=True)
    assert (tmp_path / "enc.jpg").read_bytes() == dec.encode(px).tobytes()


def test_guard_mode():
    code = ("import sys; sys.path[:0] = [%r, %r]\n" % (str(ROOT), str(ROOT / "tests")) +
            "import libkpeg_b200 as K, transcode_cases as TC\n"
            "from test_transcode_host import synth\n"
            "d = K.Decoder(0)\n"
            "for jpg in (synth(64, 48, ri=2), synth(24, 16, flags=8)):\n"
            "    for t, opt, ri in ((0, False, -1), (5, True, 0), (6, False, 3), (3, True, 1)):\n"
            "        assert d.transcode(jpg, ri, t, opt) == TC.reference(jpg, ri, t, opt)\n"
            "print('guard ok')\n")
    r = subprocess.run([sys.executable, "-c", code], env={**os.environ, "KPEG_GUARD": "1"}, capture_output=True, text=True)
    assert r.returncode == 0 and "guard ok" in r.stdout, r.stdout + r.stderr
