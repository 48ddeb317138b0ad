"""The encoder without a GPU: the C ABI's struct and argument checks, kpeg_encode_bound, the synth's pixel entry point
(the byte-exact reference), and the CPU replay of the encode kernels' logic (tests/emu/emu_encode.cpp) against that
reference -- including the parallel scan of the DC nudge chain in arbitrary chunkings."""
import ctypes as C
import itertools
import subprocess
from pathlib import Path

import numpy as np
import pytest

import encode_cases as EC
import libkpeg_b200 as K
from libkpeg_b200 import api
from libkpeg_b200.synth import EMIT_RESTART, QUIRK_FREE, SynthParams, synth_encode, synth_encode_pixels, synth_pixels

ROOT = Path(__file__).resolve().parent.parent


def test_encode_params_layout_matches_the_header(tmp_path):
    fields = [f for f, _ in api.EncodeParams._fields_]
    offs = "".join(f'printf(" %zu", offsetof(kpeg_encode_params, {f}));' for f in fields)
    src = ('#include <stdio.h>\n#include <stddef.h>\n#include "kpeg_cuda.h"\n'
           f'int main(){{printf("%zu", sizeof(kpeg_encode_params));{offs}printf("\\n");return 0;}}\n')
    exe = tmp_path / "enc_sizeof"
    subprocess.run(["gcc", "-x", "c", "-", f"-I{ROOT / 'include'}", "-o", str(exe)], input=src.encode(), check=True)
    got = list(map(int, subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.split()))
    assert got == [C.sizeof(api.EncodeParams)] + [getattr(api.EncodeParams, f).offset for f in fields]


def test_argument_checks_need_no_context():
    lib = K.load_cuda_library()
    ok = api.EncodeParams(16, 16, 3, 90, 0, 1)
    n = C.c_size_t(0)
    buf = np.zeros(16, np.uint8)
    assert lib.kpeg_encode_bound(None) == 0
    assert lib.kpeg_cuda_encode(None, C.byref(ok), buf.ctypes.data, buf.ctypes.data, 16, C.byref(n), None) == api.KPEG_ERR_ARG
    assert lib.kpeg_cuda_encode_device(None, C.byref(ok), 1, 1, 16, C.byref(n), None) == api.KPEG_ERR_ARG
    for bad in [api.EncodeParams(0, 16, 3, 90, 0, 1), api.EncodeParams(16, 0, 3, 90, 0, 1), api.EncodeParams(16, 16, 2, 90, 0, 1),
                api.EncodeParams(16, 16, 3, 0, 0, 1), api.EncodeParams(16, 16, 3, 101, 0, 1), api.EncodeParams(16, 16, 3, 90, 0, 8)]:
        assert lib.kpeg_encode_bound(C.byref(bad)) == 0
        assert lib.kpeg_cuda_encode(None, C.byref(bad), buf.ctypes.data, buf.ctypes.data, 16, C.byref(n), None) == api.KPEG_ERR_ARG
    with pytest.raises(ValueError):
        K.encode_bound(70000, 16, 3)


@pytest.mark.parametrize("w,h", EC.SIZES)
@pytest.mark.parametrize("nc", [1, 3])
def test_synth_encode_is_encode_pixels_of_synth_pixels(w, h, nc):
    for q, ri, quirk, amp in itertools.product(EC.QUALITIES, [0, 1, 7], [0, QUIRK_FREE], [0, 200]):
        if w * h > 10000 and (q, ri) not in ((95, 0), (50, 7), (100, 1)):
            continue  # the large size on a few combinations
        p = SynthParams(w, h, file_components=nc, quality=q, restart_interval=ri, flags=quirk | EMIT_RESTART,
                        noise_amp=amp, seed=w + q)
        ref = synth_encode(p)
        assert np.array_equal(synth_encode_pixels(p, synth_pixels(p)), ref), (q, ri, quirk, amp)
        # seed and noise_amp only shape the content
        p2 = SynthParams(**{**p.__dict__, "seed": 1, "noise_amp": 3})
        assert np.array_equal(synth_encode_pixels(p2, synth_pixels(p)), ref)


@pytest.mark.parametrize("w,h", EC.SIZES)
@pytest.mark.parametrize("nc", [1, 3])
def test_cpu_replay_matches_the_reference(w, h, nc):
    px = EC.synth_content(w, h, nc, seed=w * 3 + h, noise_amp=0 if w < 100 else 30)
    for q, ri, parity in itertools.product(EC.QUALITIES, EC.restart_intervals(w), [True, False]):
        if w * h > 10000 and q not in (50, 100):
            continue
        got, info = EC.emu_encode(px, q, ri, parity, chunk=1 + (q + ri) % 29)
        assert info[0] == 0, "a block overwrote a word another block owns"
        assert got == EC.reference(px, q, ri, parity), (q, ri, parity)


@pytest.mark.parametrize("name", sorted(EC.adversarial()))
@pytest.mark.parametrize("ri", [0, 5])
def test_cpu_replay_adversarial(name, ri):
    px, q = EC.adversarial()[name]
    for parity in (True, False):
        got, info = EC.emu_encode(px, q, ri, parity, chunk=13)
        assert info[0] == 0
        assert got == EC.reference(px, q, ri, parity)
        assert len(got) <= K.encode_bound(px.shape[1], px.shape[0], 3, q, ri)


def test_bound_covers_the_worst_streams():
    """Noise and full-swing pixel checkerboards at q100, with a restart marker after every MCU: the bound holds with
    room to spare, and it is what the emulator's arithmetic says."""
    rng = np.random.default_rng(5)
    worst = 0.0
    for px in [rng.integers(0, 256, (64, 64, 3), dtype=np.uint8), EC.adversarial(64, 64)["pixel_checkerboard"][0],
               rng.integers(0, 256, (33, 17), dtype=np.uint8)]:
        h, w = px.shape[:2]
        nc = 1 if px.ndim == 2 else 3
        for ri in (0, 1):
            got, _ = EC.emu_encode(px, 100, ri, True)
            bound = K.encode_bound(w, h, nc, 100, ri)
            assert bound == EC.emu().emu_encode_bound(w, h, nc, 100, ri)
            assert len(got) <= bound
            worst = max(worst, len(got) / bound)
    assert worst < 0.5


def chain(n, rng, kind):
    if kind == "flat":  # constant DC with AC terms everywhere: every block depends on the one before
        raw = np.full(n, 37, np.int16)
        ac = np.ones(n, np.uint8)
    elif kind == "edges":  # DC at the clamp, runs of equal values, and blocks without AC terms
        raw = rng.choice(np.array([-2047, -2046, -1, 0, 1, 2046, 2047], np.int16), n)
        ac = (rng.random(n) < 0.8).astype(np.uint8)
    else:
        raw = rng.integers(-3, 4, n).astype(np.int16)
        ac = (rng.random(n) < 0.9).astype(np.uint8)
    return raw, ac


@pytest.mark.parametrize("kind", ["flat", "edges", "small"])
def test_map_scan_equals_the_serial_nudge(kind):
    lib = EC.emu()
    rng = np.random.default_rng({"flat": 1, "edges": 2, "small": 3}[kind])
    n = 129600 if kind == "flat" else 20000
    raw, ac = chain(n, rng, kind)
    for ri in (0, 1, 3, 480):
        first = np.zeros(n, np.uint8) if ri == 0 else (np.arange(n) % ri == 0).astype(np.uint8)
        serial = np.zeros(n, np.int16)
        lib.emu_nudge(raw.ctypes.data, ac.ctypes.data, first.ctypes.data, n, 0, serial.ctypes.data)
        assert (np.abs(serial.astype(np.int32) - raw) <= 2).all()
        if kind == "flat":
            assert (serial != raw).any()
        for chunk in (1, 2, 7, 32, 2048, 4093, n + 5):
            scanned = np.zeros(n, np.int16)
            lib.emu_nudge(raw.ctypes.data, ac.ctypes.data, first.ctypes.data, n, chunk, scanned.ctypes.data)
            assert np.array_equal(scanned, serial), (ri, chunk)
