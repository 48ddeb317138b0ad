"""The GPU encoder with optimised Huffman tables (KPEG_FLAG_OPTIMIZE_HUFFMAN) on a B200: byte identity with the
reference encoder (KPEG_SYNTH_OPTIMIZE_HUFFMAN), round trips through the GPU decoder, the oracle and PIL, smaller files
than the Annex K twin, one context mixing both table kinds, the device entry point with its cap, and `kpeg --optimize`."""
import itertools
import io
import subprocess
from pathlib import Path

import numpy as np
import pytest

import encode_cases as EC
import encode_opt_cases as EO
import helpers as H
import libkpeg_b200 as K
from libkpeg_b200 import api

pytestmark = pytest.mark.gpu
ROOT = Path(__file__).resolve().parent.parent
KPEG = ROOT / "libkpeg_b200" / "lib" / "kpeg"
OPT = K.KPEG_FLAG_OPTIMIZE_HUFFMAN


@pytest.fixture(scope="module")
def dec():
    d = K.Decoder(device=0)
    yield d
    d.close()


def flags(parity, optimize=True):
    return (K.KPEG_FLAG_REF_PARITY if parity else 0) | (OPT if optimize else 0)


@pytest.mark.parametrize("w,h", EC.SIZES)
@pytest.mark.parametrize("nc", [1, 3])
def test_bytes_equal_the_reference(dec, w, h, nc):
    px = EC.synth_content(w, h, nc, seed=w + 3 * h, noise_amp=0 if w < 100 else 30)
    for q, ri, parity in itertools.product(EC.QUALITIES, EC.restart_intervals(w), [True, False]):
        got = dec.encode(px, quality=q, restart_interval=ri, flags=flags(parity)).tobytes()
        assert got == EO.reference(px, q, ri, parity), (q, ri, parity)
        assert len(got) <= K.encode_bound(w, h, nc, q, ri, flags=flags(parity))
        assert dec.last_stats.scan_bytes + 2 < len(got)


@pytest.mark.parametrize("w,h,q,ri", [(1921, 1081, 90, 0), (1921, 1081, 75, 241), (3840, 2160, 95, 0), (3840, 2160, 95, 16)])
def test_bytes_equal_the_reference_large(dec, w, h, q, ri):
    px = EC.synth_content(w, h, 3, seed=w + 1)
    for parity in (True, False):
        got = dec.encode(px, quality=q, restart_interval=ri, flags=flags(parity)).tobytes()
        assert got == EO.reference(px, q, ri, parity)


@pytest.mark.parametrize("name", sorted(EC.adversarial()) + ["flat_gray", "flat_rgb"])
def test_adversarial_and_flat_frames(dec, name):
    """Flat frames give single-symbol tables (1-bit codes); the adversarial ones the longest codes and DC chains."""
    if name == "flat_gray":
        px, q = np.full((40, 72), 200, np.uint8), 75
    elif name == "flat_rgb":
        px, q = np.full((48, 64, 3), (10, 200, 90), np.uint8), 90
    else:
        px, q = EC.adversarial()[name]
    h, w = px.shape[:2]
    nc = 1 if px.ndim == 2 else 3
    for ri, parity in itertools.product([0, 1, 5], [True, False]):
        got = dec.encode(px, quality=q, restart_interval=ri, flags=flags(parity)).tobytes()
        assert got == EO.reference(px, q, ri, parity), (ri, parity)
        assert len(got) <= K.encode_bound(w, h, nc, q, ri, flags=flags(parity))


def test_noise_q100_fits_the_bound(dec):
    px = np.random.default_rng(19).integers(0, 256, (1080, 1920, 3), dtype=np.uint8)
    for ri in (0, 1):
        got = dec.encode(px, quality=100, restart_interval=ri, flags=flags(True)).tobytes()
        assert got == EO.reference(px, 100, ri, True)
        assert len(got) <= K.encode_bound(1920, 1080, 3, 100, ri, flags=flags(True))


def test_round_trip(dec):
    PIL = pytest.importorskip("PIL.Image")
    for (w, h), nc, q, ri in [((256, 192), 3, 95, 0), ((61, 37), 3, 50, 7), ((200, 120), 1, 90, 25), ((1000, 600), 3, 95, 125)]:
        px = EC.synth_content(w, h, nc, seed=q + 1)
        for parity in (True, False):
            jpg = dec.encode(px, quality=q, restart_interval=ri, flags=flags(parity)).tobytes()
            twin = dec.encode(px, quality=q, restart_interval=ri, flags=flags(parity, optimize=False)).tobytes()
            for mode in (True, False):
                ref = H.oracle_decode(jpg, parity=mode)
                got = dec.decode_file(jpg, flags=K.KPEG_FLAG_REF_PARITY if mode else 0)
                assert np.array_equal(dec.read_coefficients(ref["coef"].shape[0]), ref["coef"])
                assert np.array_equal(got, ref["pixels"])
                assert np.array_equal(got, H.oracle_decode(twin, parity=mode)["pixels"]), "pixels of the Annex K twin"
            ext = np.asarray(PIL.open(io.BytesIO(jpg)).convert("RGB" if nc == 3 else "L")).astype(np.int16)
            assert np.abs(H.oracle_decode(jpg, parity=False)["pixels"].astype(np.int16) - ext).max() <= 6


@pytest.mark.parametrize("w,h", [(1000, 600), (3840, 2160)])
def test_optimised_files_are_smaller(dec, w, h):
    px = EC.synth_content(w, h, 3, seed=w)
    ratios = {}
    for q in (50, 75, 90, 95):
        opt = dec.encode(px, quality=q, flags=flags(True))
        ak = dec.encode(px, quality=q, flags=flags(True, optimize=False))
        assert opt.size < ak.size, q
        ratios[q] = round(opt.size / ak.size, 4)
    print(f"\n{w}x{h} optimised / Annex K size: {ratios}")


def test_one_context_both_table_kinds():
    """Annex K and optimised encodes interleaved at the same and at different qualities, with decodes between them: a
    fresh context reproduces every file (the per-encode tables never leak into the per-quality cache)."""
    jobs = [((320, 200), 90, 0, OPT), ((320, 200), 90, 0, 0), ((640, 360), 90, 7, OPT), ((640, 360), 60, 7, 0),
            ((64, 48), 60, 0, OPT), ((64, 48), 60, 0, 0), ((1000, 600), 95, 0, OPT), ((1000, 600), 90, 0, 0)]
    with K.Decoder(device=0) as mixed:
        seen = []
        for (w, h), q, ri, f in jobs:
            px = EC.synth_content(w, h, 3, seed=w + q)
            jpg = mixed.encode(px, quality=q, restart_interval=ri, flags=K.KPEG_FLAG_REF_PARITY | f).tobytes()
            seen.append((jpg, mixed.decode_file(jpg)))
    with K.Decoder(device=0) as fresh:
        for ((w, h), q, ri, f), (jpg, pixels) in zip(jobs, seen):
            px = EC.synth_content(w, h, 3, seed=w + q)
            assert jpg == (EO.reference(px, q, ri, True) if f else EC.reference(px, q, ri, True))
            assert fresh.encode(px, quality=q, restart_interval=ri, flags=K.KPEG_FLAG_REF_PARITY | f).tobytes() == jpg
            assert np.array_equal(fresh.decode_file(jpg), pixels)


def test_device_entry_point_and_cap(dec):
    w, h, q, ri = 333, 221, 88, 9
    px = EC.synth_content(w, h, 3, seed=3)
    f = flags(True)
    want = dec.encode(px, quality=q, restart_interval=ri, flags=f).tobytes()
    assert want == EO.reference(px, q, ri, True)
    prefix = want.index(b"\xff\xc4")  # the host writes up to SOF0, the device the rest
    sos_end = want.index(b"\xff\xda") + 2 + 6 + 2 * 3
    cap = K.encode_bound(w, h, 3, q, ri, flags=f)
    d_px, d_out = dec.device_alloc(px.nbytes), dec.device_alloc(cap + 4096)
    try:
        dec.h2d(d_px, px)
        n = dec.encode_device(d_px, w, h, 3, d_out, cap, quality=q, restart_interval=ri, flags=f)
        got = np.empty(n, np.uint8)
        dec.d2h(got, d_out)
        assert got.tobytes() == want
        for small in (len(want) - 1, len(want) // 2, sos_end, sos_end - 1, prefix + 7, prefix, prefix - 3, 100, 1, 0):
            canary = np.full(cap + 4096, 0xA5, np.uint8)
            dec.h2d(d_out, canary)
            with pytest.raises(K.KpegError) as e:
                dec.encode_device(d_px, w, h, 3, d_out, small, quality=q, restart_interval=ri, flags=f)
            assert e.value.code == api.KPEG_ERR_NOMEM and e.value.needed == len(want)
            back = np.empty(cap + 4096, np.uint8)
            dec.d2h(back, d_out)
            assert (back[small:] == 0xA5).all(), f"bytes written past cap {small}"
            assert back[:small].tobytes() == want[:small]
        import ctypes as C
        lib = K.load_cuda_library()
        p = api.encode_params(w, h, 3, q, ri, f)
        out = np.full(len(want) + 64, 0xA5, np.uint8)
        ln = C.c_size_t(0)
        rc = lib.kpeg_cuda_encode(dec._h, C.byref(p), px.ctypes.data, out.ctypes.data, len(want) - 1, C.byref(ln), None)
        assert rc == api.KPEG_ERR_NOMEM and ln.value == len(want) and (out == 0xA5).all()
        rc = lib.kpeg_cuda_encode(dec._h, C.byref(p), px.ctypes.data, out.ctypes.data, len(want), C.byref(ln), None)
        assert rc == api.KPEG_OK and out[:len(want)].tobytes() == want and (out[len(want):] == 0xA5).all()
    finally:
        dec.device_free(d_px)
        dec.device_free(d_out)


def test_stats_of_the_optimised_mode(dec):
    px = EC.synth_content(640, 480, 3, seed=2)
    dec.set_profiling(True)
    try:
        dec.encode(px, quality=90, flags=flags(True, optimize=False))
        plain = dec.last_stats.kernel_launches
        assert dec.last_stats.ms[5] == 0.0  # KPEG_T_ENTROPY_SCAN: not used without the flag
        dec.encode(px, quality=90, flags=flags(True))
        assert dec.last_stats.kernel_launches == plain + 2
        assert dec.last_stats.ms[5] > 0.0
    finally:
        dec.set_profiling(False)


def write_pnm(path, px):
    h, w = px.shape[:2]
    magic = b"P6" if px.ndim == 3 else b"P5"
    path.write_bytes(magic + b"\n" + f"{w} {h}\n255\n".encode() + px.tobytes())


def test_cli_optimize(tmp_path, dec):
    px = EC.synth_content(203, 97, 3, seed=4)
    write_pnm(tmp_path / "in.ppm", px)
    r = subprocess.run([str(KPEG), "--quiet", "--optimize", "in.ppm", "out.jpg"], cwd=tmp_path, capture_output=True, text=True)
    assert r.returncode == 0
    jpg = (tmp_path / "out.jpg").read_bytes()
    assert jpg == dec.encode(px, quality=90, flags=K.KPEG_FLAG_REF_PARITY | OPT).tobytes()
    r = subprocess.run([str(KPEG), "--quiet", "out.jpg"], cwd=tmp_path, capture_output=True, text=True)
    assert r.returncode == 0
    _, payload = H.split_ppm((tmp_path / "out.ppm").read_bytes())
    assert np.array_equal(payload, H.oracle_decode(jpg, parity=True)["pixels"])
    gray = EC.synth_content(64, 40, 1, seed=5)
    write_pnm(tmp_path / "g.pgm", gray)
    subprocess.run([str(KPEG), "--quiet", "--optimize", "--quality", "75", "--restart", "3", "--t81", "g.pgm", "g.jpg"],
                   cwd=tmp_path, check=True)
    assert (tmp_path / "g.jpg").read_bytes() == EO.reference(gray, 75, 3, False)
