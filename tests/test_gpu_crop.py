"""The crop decode (kpeg_cuda_decode_crop*) on a B200: every crop equals the full decode of the same input with the same
flags, sliced, byte for byte -- in both parity modes, at every scale, for gray and colour, ragged sizes, restart intervals
and one scan per component, through every entry point (single, device, batch, file).  The crafted coefficient fields cut
by rectangles through their MCUs drive every pixel-writing path of K3 (stage-2 rows, colour-exact rewrites, tie records,
the in-kernel tie resolution, BLK_HUGE).  Also: guard bytes of the device output, the Huffman-final-pass fallback, errors
(bad rectangles, corruption outside the rectangle, read_coefficients after a crop), a guard-mode run and the CLI."""
import subprocess
from pathlib import Path

import numpy as np
import pytest

import coef_fields as CF
import libkpeg_b200 as K
import scaled_cases as SC
from libkpeg_b200 import api
from libkpeg_b200.synth import EMIT_RESTART, NON_INTERLEAVED, QUIRK_FREE, SynthParams, synth_encode

pytestmark = pytest.mark.gpu
ROOT = Path(__file__).resolve().parent.parent
KPEG = ROOT / "libkpeg_b200" / "lib" / "kpeg"
PARITIES = [True, False]
FLAGS = {True: api.KPEG_FLAG_REF_PARITY, False: 0}


def synth(w, h, q=90, ri=0, seed=1, flags=QUIRK_FREE):
    return synth_encode(SynthParams(w, h, quality=q, restart_interval=ri, seed=seed,
                                    flags=flags | (EMIT_RESTART if ri else 0))).tobytes()


LENA = (ROOT / "tests" / "golden" / "lena.jpg").read_bytes()
SYNTH = [("synth-ragged-dri", synth(203, 77, q=80, ri=7, seed=3)), ("synth-gray-dri", synth(301, 45, q=85, ri=5, seed=4)),
         ("synth-wide-dri-row", synth(530, 33, q=92, ri=67, seed=5)),
         ("synth-scan-per-comp", synth(120, 72, q=80, seed=6, flags=QUIRK_FREE | NON_INTERLEAVED))]
INPUTS = SC.pil_files() + SC.field_files()[::2] + list(SC.extreme_files()) + [("lena", LENA)] + SYNTH


def out_size(jpg, scale):
    frame, _ = api.parse_jfif_scans(np.frombuffer(jpg, np.uint8))
    return -(-frame.width // scale), -(-frame.height // scale), frame.ncomp


def rects(ow, oh, scale, seed=0, n_random=3):
    """the whole image, 1 x 1 at the four corners, odd offsets and widths, one across a strip boundary, one inside the
    last partial MCU, and a seeded random set"""
    k = 8 // scale
    out = [(0, 0, ow, oh), (0, 0, 1, 1), (ow - 1, 0, 1, 1), (0, oh - 1, 1, 1), (ow - 1, oh - 1, 1, 1)]
    x, y = min(3, ow - 1), min(5, oh - 1)
    out.append((x, y, max(1, min(13, ow - x)), max(1, min(7, oh - y))))
    sx = 32 * k  # first column of the second strip of an MCU row (when a row holds more than one strip)
    if ow > sx + 2:
        out.append((sx - 3, 0, min(11, ow - sx + 3), oh))
    else:  # narrow images: strips wrap rows, so a band of rows crosses a strip boundary
        x, y = min(1, ow - 1), min(1, oh - 1)
        out.append((x, y, ow - x, oh - y))
    lx, ly = (ow - 1) // k * k, (oh - 1) // k * k
    out.append((lx, ly, ow - lx, oh - ly))
    rng = np.random.default_rng(seed)
    for _ in range(n_random):
        x, y = int(rng.integers(0, ow)), int(rng.integers(0, oh))
        out.append((x, y, int(rng.integers(1, ow - x + 1)), int(rng.integers(1, oh - y + 1))))
    return out


def sliced(full, r):
    x, y, w, h = r
    return full[y:y + h, x:x + w]


def check(got, full, r, what):
    want = sliced(full, r)
    assert got.shape == want.shape and np.array_equal(got, want), f"{what} crop {r}: {int((got != want).sum())} bytes differ"


@pytest.mark.parametrize("parity", PARITIES, ids=["parity", "t81"])
@pytest.mark.parametrize("scale", SC.SCALES)
def test_file_crop_is_the_full_decode_sliced(decoder, scale, parity):
    for i, (name, jpg) in enumerate(INPUTS):
        full = decoder.decode_file(jpg, FLAGS[parity], scale=scale)
        ow, oh, _ = out_size(jpg, scale)
        for r in rects(ow, oh, scale, seed=i):
            got = decoder.decode_file(jpg, FLAGS[parity], scale=scale, crop=r)
            check(got, full, r, f"{name} 1/{scale}")
            assert (decoder.last_stats.width, decoder.last_stats.height) == (r[2], r[3])


def split(jpg):
    buf = np.frombuffer(jpg, np.uint8)
    plan, off, n = api.parse_jfif(buf)
    return plan, buf[off:off + n].copy()


@pytest.mark.parametrize("parity", PARITIES, ids=["parity", "t81"])
def test_single_device_and_guard_bytes(decoder, parity):
    guard = 256
    for i, (name, jpg) in enumerate([INPUTS[0], INPUTS[1], ("lena", LENA), SYNTH[0], SYNTH[1]]):
        plan, scan = split(jpg)
        plan.flags = FLAGS[parity]
        d_scan = decoder.device_alloc(scan.size + 64)
        decoder.h2d(d_scan, scan)
        for scale in SC.SCALES:
            full = decoder.decode_scan(plan, scan, scale=scale)
            ow, oh = full.shape[1], full.shape[0]
            for r in rects(ow, oh, scale, seed=100 + i):
                check(decoder.decode_scan(plan, scan, scale=scale, crop=r), full, r, f"single {name} 1/{scale}")
                nbytes = int(np.prod(api.crop_shape(plan, r)))
                d_out = decoder.device_alloc(nbytes + 2 * guard)
                pattern = np.full(nbytes + 2 * guard, 0xA5, np.uint8)
                decoder.h2d(d_out, pattern)
                decoder.decode_device(plan, d_scan, scan.size, d_out + guard, scale=scale, crop=r)
                back = np.empty(nbytes + 2 * guard, np.uint8)
                decoder.d2h(back, d_out)
                decoder.device_free(d_out)
                assert (back[:guard] == 0xA5).all() and (back[guard + nbytes:] == 0xA5).all(), f"device {name} {r}: guard bytes"
                check(back[guard:guard + nbytes].reshape(api.crop_shape(plan, r)), full, r, f"device {name} 1/{scale}")
        decoder.device_free(d_scan)


@pytest.mark.parametrize("parity", PARITIES, ids=["parity", "t81"])
@pytest.mark.parametrize("scale", SC.SCALES)
def test_batch_with_a_rectangle_per_image(decoder, scale, parity):
    """Same-plan images, each with its own rectangle -- the same image twice with two rectangles too; narrow images whose
    strips span two or three images (tie records and huge blocks on both sides of every boundary)."""
    groups = [[jpg for _, jpg in CF.narrow_batch()],
              [synth(203, 77, q=80, ri=7, seed=s) for s in (3, 3, 8, 9)],
              [synth(64, 40, q=95, seed=s, flags=QUIRK_FREE) for s in (1, 2, 3, 1)]]
    rng = np.random.default_rng(scale * 10 + parity)
    for jpgs in groups:
        plan, _ = split(jpgs[0])
        plan.flags = FLAGS[parity]
        scans = [split(j)[1] for j in jpgs]
        fulls = decoder.decode_batch(plan, scans, scale=scale)
        ow, oh = fulls[0].shape[1], fulls[0].shape[0]
        for _ in range(3):
            pool = rects(ow, oh, scale, seed=int(rng.integers(1 << 30)))
            crops = [pool[int(rng.integers(len(pool)))] for _ in scans]
            outs = decoder.decode_batch(plan, scans, scale=scale, crops=crops)
            for k, (got, full, r) in enumerate(zip(outs, fulls, crops)):
                check(got, full, r, f"batch image {k} 1/{scale}")
            assert (decoder.last_stats.width, decoder.last_stats.height) == crops[0][2:]


@pytest.mark.parametrize("parity", PARITIES, ids=["parity", "t81"])
@pytest.mark.parametrize("case", CF.cases(), ids=lambda c: f"{c[0]}-{c[1]}x{c[2]}x{c[3]}")
def test_k3_branches_are_windowed(decoder, case, parity):
    """Every pixel-writing path of K3, cut by rectangles through the MCUs that take it."""
    for k, (f, jpg) in enumerate(CF.fields_and_files(*case)):
        full = decoder.decode_file(jpg, FLAGS[parity])
        rs = rects(f.width, f.height, 1, seed=k, n_random=6)
        # rectangles whose edges pass through the middle of MCUs, at every MCU column of the first rows
        rs += [(bx * 8 + 3, 2, 5 + (bx % 3), min(f.height - 2, 13)) for bx in range(0, (f.width - 9) // 8, 3)]
        for r in rs:
            check(decoder.decode_file(jpg, FLAGS[parity], crop=r), full, r, f"{f.name}")


@pytest.mark.parametrize("parity", PARITIES, ids=["parity", "t81"])
def test_4k_workload(decoder, parity):
    jpg = synth_encode(SynthParams(3840, 2160, quality=95)).tobytes()
    full = decoder.decode_file(jpg, FLAGS[parity])
    for r in [((3840 - 224) // 2, (2160 - 224) // 2, 224, 224), (960, 540, 1920, 1080), (0, 1000, 3840, 8), (3839, 2159, 1, 1)]:
        check(decoder.decode_file(jpg, FLAGS[parity], crop=r), full, r, "4K q95")
    for scale in (2, 8):
        fs = decoder.decode_file(jpg, FLAGS[parity], scale=scale)
        r = (fs.shape[1] // 2 - 50, fs.shape[0] // 2 - 30, 101, 61)
        check(decoder.decode_file(jpg, FLAGS[parity], scale=scale, crop=r), fs, r, f"4K q95 1/{scale}")


def test_huffman_final_pass_fallback(monkeypatch, decoder):
    monkeypatch.setenv("KPEG_NO_RECORDS", "1")
    dec = K.Decoder(device=0)
    monkeypatch.delenv("KPEG_NO_RECORDS")
    try:
        for i, (name, jpg) in enumerate([("lena", LENA)] + SYNTH + SC.field_files()[:4]):
            for parity in PARITIES:
                for scale in SC.SCALES:
                    full = decoder.decode_file(jpg, FLAGS[parity], scale=scale)
                    ow, oh, _ = out_size(jpg, scale)
                    for r in rects(ow, oh, scale, seed=i):
                        check(dec.decode_file(jpg, FLAGS[parity], scale=scale, crop=r), full, r, f"no-records {name} 1/{scale}")
    finally:
        dec.close()


def test_bad_rectangles_leave_the_output_untouched(decoder):
    jpg = SYNTH[0][1]
    plan, scan = split(jpg)
    d_scan = decoder.device_alloc(scan.size + 64)
    decoder.h2d(d_scan, scan)
    for scale in SC.SCALES:
        ow, oh = -(-plan.width // scale), -(-plan.height // scale)
        for r in [(ow, 0, 1, 1), (0, oh, 1, 1), (ow - 3, 0, 4, 1), (0, oh - 1, 1, 2), (0, 0, ow + 1, oh)]:
            out = np.full(api.crop_shape(plan, r), 0x5A, np.uint8)
            for call in (lambda: decoder.decode_scan(plan, scan, scale=scale, crop=r, out=out),
                         lambda: decoder.decode_file(jpg, 0, scale=scale, crop=r, out=out),
                         lambda: decoder.decode_batch(plan, [scan, scan], scale=scale, crops=[(0, 0, 1, 1), r],
                                                      outs=[np.zeros((1, 1, 3), np.uint8), out])):
                with pytest.raises(api.KpegError) as e:
                    call()
                assert e.value.code == api.KPEG_ERR_ARG, r
                assert (out == 0x5A).all(), r
            d_out = decoder.device_alloc(out.nbytes)
            decoder.h2d(d_out, out)
            with pytest.raises(api.KpegError) as e:
                decoder.decode_device(plan, d_scan, scan.size, d_out, scale=scale, crop=r)
            assert e.value.code == api.KPEG_ERR_ARG
            back = np.empty_like(out)
            decoder.d2h(back, d_out)
            decoder.device_free(d_out)
            assert (back == 0x5A).all(), r
    decoder.device_free(d_scan)


def test_corruption_outside_the_rectangle_is_reported(decoder):
    """The whole stream is entropy-decoded: a marker that is no RSTn near the end of the scan fails a crop of the top-left
    corner as it fails the full decode."""
    for name, jpg in [SYNTH[0], ("synth-no-dri", synth(256, 128, q=90, seed=12))]:
        plan, scan = split(jpg)
        bad = scan.copy()
        at = bad.size - 20
        bad[at:at + 2] = [0xFF, 0xC4]
        with pytest.raises(api.KpegError) as e:
            decoder.decode_scan(plan, bad)
        assert e.value.code == api.KPEG_ERR_STREAM
        with pytest.raises(api.KpegError) as e:
            decoder.decode_scan(plan, bad, crop=(0, 0, 8, 8))
        assert e.value.code == api.KPEG_ERR_STREAM, name
        full = decoder.decode_scan(plan, scan)  # and the context is fine afterwards
        check(decoder.decode_scan(plan, scan, crop=(0, 0, 8, 8)), full, (0, 0, 8, 8), name)


def test_read_coefficients_after_a_crop(decoder):
    for jpg in (LENA, SYNTH[3][1]):
        full = decoder.decode_file(jpg)
        frame, _ = api.parse_jfif_scans(np.frombuffer(jpg, np.uint8))
        nblocks = (-(-frame.width // 8)) * (-(-frame.height // 8)) * frame.ncomp
        coef = decoder.read_coefficients(nblocks)
        decoder.decode_file(jpg, crop=(1, 1, 5, 5))
        with pytest.raises(api.KpegError) as e:
            decoder.read_coefficients(nblocks)
        assert e.value.code == api.KPEG_ERR_UNSUPPORTED
        assert np.array_equal(decoder.decode_file(jpg), full)
        assert np.array_equal(decoder.read_coefficients(nblocks), coef)


def test_guard_mode(monkeypatch):
    monkeypatch.setenv("KPEG_GUARD", "1")
    dec = K.Decoder(device=0)
    monkeypatch.delenv("KPEG_GUARD")
    try:
        for i, (name, jpg) in enumerate([("lena", LENA)] + SYNTH + list(SC.extreme_files())):
            for scale in SC.SCALES:
                full = dec.decode_file(jpg, scale=scale)
                ow, oh, _ = out_size(jpg, scale)
                for r in rects(ow, oh, scale, seed=i, n_random=1):
                    check(dec.decode_file(jpg, scale=scale, crop=r), full, r, f"guard {name} 1/{scale}")
        plan, scan = split(SYNTH[0][1])
        fulls = dec.decode_batch(plan, [scan] * 3)
        crops = [(0, 0, 1, 1), (5, 6, 100, 40), (202, 76, 1, 1)]
        for got, full, r in zip(dec.decode_batch(plan, [scan] * 3, crops=crops), fulls, crops):
            check(got, full, r, "guard batch")
    finally:
        dec.close()


@pytest.mark.parametrize("scale", [1, 2, 8])
def test_cli_crop(decoder, tmp_path, scale):
    for name, jpg in [("lena", LENA), SYNTH[1], SYNTH[3]]:
        src = tmp_path / f"{name}.jpg"
        src.write_bytes(jpg)
        ow, oh, nc = out_size(jpg, scale)
        r = (min(7, ow - 1), min(3, oh - 1), max(1, min(50, ow - 7)), max(1, min(21, oh - 3)))
        cmd = [str(KPEG), "--quiet", "--crop", f"{r[2]}x{r[3]}+{r[0]}+{r[1]}", str(src)]
        if scale != 1:
            cmd[2:2] = ["--scale", f"1/{scale}"]
        subprocess.run(cmd, cwd=tmp_path, check=True, capture_output=True)
        ppm = (tmp_path / f"{name}.ppm").read_bytes()
        hdr = api.ppm_header(r[2], r[3])
        assert ppm[:len(hdr)] == hdr
        got = np.frombuffer(ppm[len(hdr):], np.uint8).reshape(r[3], r[2], 3)
        want = decoder.decode_file(jpg, scale=scale, crop=r)
        if want.ndim == 2:
            want = np.repeat(want[:, :, None], 3, axis=2)
        assert np.array_equal(got, want), f"{name} 1/{scale}"
