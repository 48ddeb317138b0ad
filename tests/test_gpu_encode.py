"""The GPU encoder (kpeg_cuda_encode / _device, Decoder.encode, the kpeg CLI's encode mode) on a B200: byte identity
with the synthetic reference encoder's coding path over the same pixels, adversarial inputs, round trips through the
GPU decoder and the oracle, the two entry points, one context for both directions, and the CLI."""
import hashlib
import io
import itertools
import subprocess
from pathlib import Path

import numpy as np
import pytest

import encode_cases as EC
import helpers as H
import libkpeg_b200 as K
from libkpeg_b200 import api

pytestmark = pytest.mark.gpu
ROOT = Path(__file__).resolve().parent.parent
KPEG = ROOT / "libkpeg_b200" / "lib" / "kpeg"


@pytest.fixture(scope="module")
def dec():
    d = K.Decoder(device=0)
    yield d
    d.close()


def flags(parity):
    return K.KPEG_FLAG_REF_PARITY if parity else 0


@pytest.mark.parametrize("w,h", EC.SIZES)
@pytest.mark.parametrize("nc", [1, 3])
def test_bytes_equal_the_reference(dec, w, h, nc):
    px = EC.synth_content(w, h, nc, seed=w + 2 * h, noise_amp=0 if w < 100 else 30)
    for q, ri, parity in itertools.product(EC.QUALITIES, EC.restart_intervals(w), [True, False]):
        got = dec.encode(px, quality=q, restart_interval=ri, flags=flags(parity)).tobytes()
        assert got == EC.reference(px, q, ri, parity), (q, ri, parity)
        st = dec.last_stats
        assert st.scan_bytes + 2 < len(got) and st.segments == (1 if ri == 0 else -(-((w + 7) // 8) * ((h + 7) // 8) // ri))


@pytest.mark.parametrize("w,h,q,ri", [(1921, 1081, 90, 0), (1921, 1081, 75, 241), (3840, 2160, 95, 0), (3840, 2160, 95, 16)])
def test_bytes_equal_the_reference_large(dec, w, h, q, ri):
    px = EC.synth_content(w, h, 3, seed=w)
    for parity in (True, False):
        assert dec.encode(px, quality=q, restart_interval=ri, flags=flags(parity)).tobytes() == EC.reference(px, q, ri, parity)


@pytest.mark.parametrize("name", sorted(EC.adversarial()))
def test_adversarial_pixels(dec, name):
    px, q = EC.adversarial()[name]
    h, w = px.shape[:2]
    for ri, parity in itertools.product([0, 1, 5], [True, False]):
        got = dec.encode(px, quality=q, restart_interval=ri, flags=flags(parity)).tobytes()
        assert got == EC.reference(px, q, ri, parity), (ri, parity)
        assert len(got) <= K.encode_bound(w, h, 3, q, ri)


def test_noise_q100_fits_the_bound(dec):
    px = np.random.default_rng(9).integers(0, 256, (1080, 1920, 3), dtype=np.uint8)
    for ri in (0, 1):
        got = dec.encode(px, quality=100, restart_interval=ri).tobytes()
        assert got == EC.reference(px, 100, ri, True)
        assert len(got) <= K.encode_bound(1920, 1080, 3, 100, ri)


def test_scan_beyond_2_pow_32_bits(dec):
    """64-bit bit offsets: a 16384 x 16384 noise frame at q100 has a scan of more than 2^32 bits."""
    px = np.random.default_rng(11).integers(0, 256, (16384, 16384, 3), dtype=np.uint8)
    got = dec.encode(px, quality=100, restart_interval=0)
    assert dec.last_stats.unstuffed_bytes * 8 > 2 ** 32
    ref = EC.reference(px, 100, 0, True)
    assert hashlib.sha256(got.tobytes()).hexdigest() == hashlib.sha256(ref).hexdigest()


def test_round_trip(dec):
    PIL = pytest.importorskip("PIL.Image")
    for (w, h), nc, q, ri in [((256, 192), 3, 95, 0), ((61, 37), 3, 50, 7), ((200, 120), 1, 90, 25), ((1000, 600), 3, 95, 125)]:
        px = EC.synth_content(w, h, nc, seed=q)
        for parity in (True, False):
            jpg = dec.encode(px, quality=q, restart_interval=ri, flags=flags(parity)).tobytes()
            for mode in (True, False):
                ref = H.oracle_decode(jpg, parity=mode)
                got = dec.decode_file(jpg, flags=flags(mode))
                assert np.array_equal(dec.read_coefficients(ref["coef"].shape[0]), ref["coef"])
                assert np.array_equal(got, ref["pixels"])
            if parity:  # the nudged stream decodes the same in both modes
                assert np.array_equal(H.oracle_decode(jpg, parity=True)["pixels"], H.oracle_decode(jpg, parity=False)["pixels"])
            if q == 95:
                assert EC.psnr(H.oracle_decode(jpg, parity=True)["pixels"], px) > 35.0
            ext = np.asarray(PIL.open(io.BytesIO(jpg)).convert("RGB" if nc == 3 else "L")).astype(np.int16)
            assert np.abs(H.oracle_decode(jpg, parity=False)["pixels"].astype(np.int16) - ext).max() <= 6


def test_device_entry_point_and_cap(dec):
    w, h = 333, 221
    px = EC.synth_content(w, h, 3, seed=3)
    want = dec.encode(px, quality=88, restart_interval=9).tobytes()
    cap = K.encode_bound(w, h, 3, 88, 9)
    d_px, d_out = dec.device_alloc(px.nbytes), dec.device_alloc(cap + 4096)
    try:
        dec.h2d(d_px, px)
        n = dec.encode_device(d_px, w, h, 3, d_out, cap, quality=88, restart_interval=9)
        got = np.empty(n, np.uint8)
        dec.d2h(got, d_out)
        assert got.tobytes() == want
        for small in (len(want) - 1, len(want) // 2, 100, 0):
            canary = np.full(cap + 4096, 0xA5, np.uint8)
            dec.h2d(d_out, canary)
            with pytest.raises(K.KpegError) as e:
                dec.encode_device(d_px, w, h, 3, d_out, small, quality=88, restart_interval=9)
            assert e.value.code == api.KPEG_ERR_NOMEM and e.value.needed == len(want)
            back = np.empty(cap + 4096, np.uint8)
            dec.d2h(back, d_out)
            assert (back[small:] == 0xA5).all(), "bytes written past cap"
            assert back[:small].tobytes() == want[:small]
        # host entry point: too small a buffer
        lib = K.load_cuda_library()
        p = api.encode_params(w, h, 3, 88, 9)
        out = np.full(len(want) + 64, 0xA5, np.uint8)
        import ctypes as C
        ln = C.c_size_t(0)
        rc = lib.kpeg_cuda_encode(dec._h, C.byref(p), px.ctypes.data, out.ctypes.data, len(want) - 1, C.byref(ln), None)
        assert rc == api.KPEG_ERR_NOMEM and ln.value == len(want) and (out == 0xA5).all()
    finally:
        dec.device_free(d_px)
        dec.device_free(d_out)


def test_one_context_for_both_directions():
    sizes = [(64, 48), (320, 200), (1000, 600), (1921, 1081)]
    with K.Decoder(device=0) as mixed:
        seen = []
        for (w, h) in sizes:
            px = EC.synth_content(w, h, 3, seed=w)
            jpg = mixed.encode(px, quality=90, restart_interval=w // 8).tobytes()
            a = mixed.decode_file(jpg)
            b = mixed.decode_file(EC.reference(px, 80, 0, True))
            jpg2 = mixed.encode(a, quality=70).tobytes()
            seen.append((jpg, a, b, jpg2))
    with K.Decoder(device=0) as fresh:
        for (w, h), (jpg, a, b, jpg2) in zip(sizes, seen):
            px = EC.synth_content(w, h, 3, seed=w)
            assert fresh.encode(px, quality=90, restart_interval=w // 8).tobytes() == jpg
            assert np.array_equal(fresh.decode_file(jpg), a)
            assert np.array_equal(fresh.decode_file(EC.reference(px, 80, 0, True)), b)
            assert fresh.encode(a, quality=70).tobytes() == jpg2


def write_pnm(path, px):
    h, w = px.shape[:2]
    magic = b"P6" if px.ndim == 3 else b"P5"
    path.write_bytes(magic + b"\n# written by a test\n" + f"{w} {h}\n255\n".encode() + px.tobytes())


def test_cli_encode(tmp_path, dec):
    px = EC.synth_content(203, 97, 3, seed=4)
    write_pnm(tmp_path / "in.ppm", px)
    r = subprocess.run([str(KPEG), "--quiet", "in.ppm", "out.jpg"], cwd=tmp_path, capture_output=True, text=True)
    assert r.returncode == 0
    jpg = (tmp_path / "out.jpg").read_bytes()
    assert jpg == dec.encode(px, quality=90).tobytes()
    r = subprocess.run([str(KPEG), "--quiet", "out.jpg"], cwd=tmp_path, capture_output=True, text=True)
    assert r.returncode == 0
    _, payload = H.split_ppm((tmp_path / "out.ppm").read_bytes())
    assert np.array_equal(payload, H.oracle_decode(jpg, parity=True)["pixels"])
    # options, P5
    gray = EC.synth_content(64, 40, 1, seed=5)
    write_pnm(tmp_path / "g.pgm", gray)
    subprocess.run([str(KPEG), "--quiet", "--quality", "75", "--restart", "3", "--t81", "g.pgm", "g.jpg"], cwd=tmp_path, check=True)
    g = (tmp_path / "g.jpg").read_bytes()
    assert g == EC.reference(gray, 75, 3, False) and K.parse_jfif(g)[0].ncomp == 1
    # malformed input: logged, exit 0, no file
    (tmp_path / "bad.ppm").write_bytes(b"P6\n10 10\n255\n" + bytes(20))
    r = subprocess.run([str(KPEG), "bad.ppm", "bad.jpg"], cwd=tmp_path, capture_output=True, text=True)
    assert r.returncode == 0 and "truncated" in r.stdout and not (tmp_path / "bad.jpg").exists()
