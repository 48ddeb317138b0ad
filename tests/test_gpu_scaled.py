"""The reduced-size decode (KPEG_FLAG_SCALE_*) on a B200: byte identity with the C reference of scaled_cases.py at 1/2,
1/4 and 1/8 in both parity modes through every decode entry point (single, device, batches plain / packed / split /
deferred, one scan per component, decode_file, decode_files, the PPM writer, tiled over devices [0, 0], a banded large
image), the Huffman-final-pass fallback, the 4K q95 workload, PIL's draft() on PIL files, full-size decodes unchanged,
errors, a guard-mode run and the CLI."""
import os
import subprocess
import sys
from pathlib import Path

import numpy as np
import pytest

import libkpeg_b200 as K
import scaled_cases as SC
from libkpeg_b200 import api
from libkpeg_b200.synth import EMIT_RESTART, NON_INTERLEAVED, QUIRK_FREE, SynthParams, synth_encode

pytestmark = pytest.mark.gpu
ROOT = Path(__file__).resolve().parent.parent
KPEG = ROOT / "libkpeg_b200" / "lib" / "kpeg"
PARITIES = [True, False]
FLAGS = {True: api.KPEG_FLAG_REF_PARITY, False: 0}


@pytest.fixture(scope="module")
def dec():
    d = K.Decoder(device=0)
    yield d
    d.close()


def synth(w, h, q=90, ri=0, seed=1, flags=QUIRK_FREE):
    return synth_encode(SynthParams(w, h, quality=q, restart_interval=ri, seed=seed,
                                    flags=flags | (EMIT_RESTART if ri else 0))).tobytes()


INPUTS = SC.pil_files() + SC.field_files()[::3] + list(SC.extreme_files()) + [
    ("synth-ragged-dri", synth(203, 77, q=80, ri=7, seed=3)), ("synth-96x50", synth(96, 50, seed=4))]


@pytest.mark.parametrize("parity", PARITIES, ids=["parity", "t81"])
@pytest.mark.parametrize("scale", SC.SCALES)
def test_single_and_file_decode_match_reference(dec, scale, parity):
    for name, jpg in INPUTS:
        ref = SC.reference(jpg, scale, parity)
        got = dec.decode_file(jpg, FLAGS[parity], scale=scale)
        assert got.shape == ref.shape and np.array_equal(got, ref), f"{name} 1/{scale}"
        st = dec.last_stats
        assert (st.height, st.width) == ref.shape[:2], name


@pytest.mark.parametrize("scale", SC.SCALES)
def test_pil_draft_equality(dec, scale):
    for name, jpg in SC.pil_files():
        assert np.array_equal(dec.decode_file(jpg, 0, scale=scale), SC.pil_draft(jpg, scale)), f"{name} 1/{scale}"


@pytest.mark.parametrize("parity", PARITIES, ids=["parity", "t81"])
def test_device_and_ppm_writer(dec, parity):
    for name, jpg in [INPUTS[0], INPUTS[5], INPUTS[-2], INPUTS[-1]]:
        plan, off, ln = api.parse_jfif(jpg)
        plan.flags = FLAGS[parity]
        scan = np.frombuffer(jpg, np.uint8)[off:off + ln].copy()
        d_scan = dec.device_alloc(ln + 64)
        dec.h2d(d_scan, scan)
        for scale in SC.SCALES:
            ref = SC.reference(jpg, scale, parity)
            d_out = dec.device_alloc(ref.nbytes * 3 + 256)
            dec.decode_device(plan, d_scan, ln, d_out, scale=scale)
            got = np.empty(ref.nbytes, np.uint8)
            dec.d2h(got, d_out)
            assert np.array_equal(got.reshape(ref.shape), ref), f"device {name} 1/{scale}"
            cap = ref.shape[0] * ref.shape[1] * 3 + 176
            po, pl = dec.decode_ppm_device(plan, d_scan, ln, d_out, cap, scale=scale)
            ppm = np.empty(po + pl, np.uint8)
            dec.d2h(ppm, d_out)
            hdr = api.ppm_header(ref.shape[1], ref.shape[0])
            rgb = ref if ref.ndim == 3 else np.repeat(ref[:, :, None], 3, axis=2)
            assert ppm[po:po + len(hdr)].tobytes() == hdr, name
            assert np.array_equal(ppm[po + len(hdr):], rgb.reshape(-1)), f"ppm {name} 1/{scale}"
            dec.device_free(d_out)
        dec.device_free(d_scan)


def _same_plan_batch(n=6, w=70, h=45, q=85):
    jpgs = [synth(w, h, q=q, seed=100 + i) for i in range(n)]
    plan, _, _ = api.parse_jfif(jpgs[0])
    scans = []
    for j in jpgs:
        _, off, ln = api.parse_jfif(j)
        scans.append(np.frombuffer(j, np.uint8)[off:off + ln].copy())
    return jpgs, plan, scans


@pytest.mark.parametrize("parity", PARITIES, ids=["parity", "t81"])
@pytest.mark.parametrize("scale", SC.SCALES)
def test_batches(dec, scale, parity):
    jpgs, plan, scans = _same_plan_batch()
    plan.flags = FLAGS[parity]
    refs = [SC.reference(j, scale, parity) for j in jpgs]
    n, one = len(jpgs), refs[0].nbytes
    # host batch (a submission and its wait)
    outs = dec.decode_batch(plan, scans, scale=scale)
    assert all(np.array_equal(o, r) for o, r in zip(outs, refs)), "decode_batch"
    # device: packed, split, deferred, unpacked
    packed = api.pack_batch(scans)
    offs = api.packed_offsets(scans)
    d_in = dec.device_alloc(packed.size + 64)
    dec.h2d(d_in, packed)
    d_out = dec.device_alloc(one * n + 64)
    sp = api._scaled_plan(plan, scale)
    got = np.empty(one * n, np.uint8)
    for how in ("packed", "split", "deferred", "unpacked"):
        if how == "packed":
            dec.decode_batch_packed_device(sp, n, d_in, packed.size, d_out)
        elif how == "split":
            dec.decode_batch_packed_device_split(sp, n, d_in, offs, d_out)
        elif how == "deferred":
            dec.submit_batch_packed_device(sp, n, d_in, offs, d_out)
            dec.wait()
        else:
            raw = np.concatenate(scans)
            d_raw = dec.device_alloc(raw.size + 64)
            dec.h2d(d_raw, raw)
            so = np.zeros(n + 1, np.uint64)
            so[1:] = np.cumsum([s.size for s in scans])
            dec._check(dec._lib.kpeg_cuda_decode_batch_device(dec._h, api.C.byref(sp), n, d_raw,
                                                              so.ctypes.data_as(api.C.POINTER(api.C.c_uint64)), d_out,
                                                              api.C.byref(dec.last_stats)), "decode_batch_device")
            dec.device_free(d_raw)
        dec.d2h(got, d_out)
        for k in range(n):
            assert np.array_equal(got[k * one:(k + 1) * one].reshape(refs[k].shape), refs[k]), f"{how} image {k} 1/{scale}"
    dec.device_free(d_in)
    dec.device_free(d_out)
    # deferred host submission into one frame buffer (one copy per chunk)
    frame = np.empty(one * n, np.uint8)
    dec.submit_batch(sp, scans, [frame[k * one:(k + 1) * one] for k in range(n)])
    dec.wait()
    assert all(np.array_equal(frame[k * one:(k + 1) * one].reshape(refs[k].shape), refs[k]) for k in range(n))


@pytest.mark.parametrize("parity", PARITIES, ids=["parity", "t81"])
def test_one_scan_per_component_and_decode_files(dec, parity):
    ni = synth(120, 72, q=80, seed=12, flags=QUIRK_FREE | NON_INTERLEAVED)
    mix = [ni, synth(64, 40, seed=13), synth(64, 40, seed=14), SC.pil_files()[3][1], (SC.GOLDEN / "lena.jpg").read_bytes()]
    for scale in SC.SCALES:
        assert np.array_equal(dec.decode_file(ni, FLAGS[parity], scale=scale), SC.reference(ni, scale, parity)), f"scans 1/{scale}"
        imgs, codes = dec.decode_files(mix, FLAGS[parity], scale=scale)
        assert codes == [0] * len(mix)
        for k, (img, jpg) in enumerate(zip(imgs, mix)):
            assert np.array_equal(img, SC.reference(jpg, scale, parity)), f"decode_files #{k} 1/{scale}"


def _big(side_w, side_h, q):
    return synth(side_w, side_h, q=q, ri=(side_w + 7) // 8, seed=21)


@pytest.mark.parametrize("scale", SC.SCALES)
def test_tiled_and_banded(dec, scale):
    """A restart-marked 4K file over devices [0, 0] (bands at the reduced rows), and a 5000 x 4600 image (69 MB at full
    size: the decode is cut into bands on the context's lanes whatever the scale)."""
    jpg4k = _big(3840, 2160, 90)
    for parity in PARITIES:
        ref = SC.reference(jpg4k, scale, parity)
        got, st = api.decode_file_tiled([0, 0], jpg4k, FLAGS[parity], scale=scale)
        assert np.array_equal(got, ref) and (st.height, st.width) == ref.shape[:2], f"tiled 1/{scale}"
    big = _big(5000, 4600, 85)
    ref = SC.reference(big, scale, True)
    got = dec.decode_file(big, api.KPEG_FLAG_REF_PARITY, scale=scale)
    assert np.array_equal(got, ref), f"banded 1/{scale}"
    assert (dec.last_stats.height, dec.last_stats.width) == ref.shape[:2]


def test_baseline_4k_q95_workload(dec):
    jpgs = [synth_encode(SynthParams(3840, 2160, quality=95, seed=0xB200 + i, flags=QUIRK_FREE)).tobytes() for i in range(2)]
    plan, _, _ = api.parse_jfif(jpgs[0])
    scans = []
    for j in jpgs:
        _, off, ln = api.parse_jfif(j)
        scans.append(np.frombuffer(j, np.uint8)[off:off + ln].copy())
    for parity in PARITIES:
        plan.flags = FLAGS[parity]
        for scale in SC.SCALES:
            outs = dec.decode_batch(plan, scans, scale=scale)
            for o, j in zip(outs, jpgs):
                assert np.array_equal(o, SC.reference(j, scale, parity)), f"4K q95 1/{scale} parity={parity}"


def test_huffman_final_pass_fallback(monkeypatch):
    monkeypatch.setenv("KPEG_NO_RECORDS", "1")
    d = K.Decoder(device=0)
    try:
        for name, jpg in INPUTS[::4]:
            for scale in SC.SCALES:
                assert np.array_equal(d.decode_file(jpg, scale=scale), SC.reference(jpg, scale, True)), f"{name} 1/{scale}"
    finally:
        d.close()


def test_full_size_unchanged(dec):
    """No scale bits, or scale=1: today's decode, the same launches; a reduced decode has one launch fewer (one
    reconstruction kernel instead of K3 and its patch pass)."""
    for name, jpg in INPUTS[::5]:
        a = dec.decode_file(jpg)
        la = dec.last_stats.kernel_launches
        b = dec.decode_file(jpg, scale=1)
        assert np.array_equal(a, b) and dec.last_stats.kernel_launches == la, name
        dec.decode_file(jpg, scale=2)
        assert dec.last_stats.kernel_launches == la - 1, name


def test_errors(dec):
    good = synth(64, 48, seed=8)
    _, off, ln = api.parse_jfif(good)
    bad = bytearray(good)
    bad[off + ln // 2:off + ln // 2 + 8] = b"\xff\xd3" * 4  # markers inside the scan
    for scale in SC.SCALES:
        with pytest.raises(K.KpegError) as e:
            dec.decode_file(bytes(bad), scale=scale)
        assert e.value.code == api.KPEG_ERR_STREAM
    good = synth(64, 48, seed=32)
    buf = np.frombuffer(good, np.uint8)
    for scale in SC.SCALES:
        need = int(np.prod(SC.shape(64, 48, 3, scale)))
        out = np.full(need + 16, 0x5A, np.uint8)
        rc = dec._lib.kpeg_cuda_decode_file(dec._h, buf.ctypes.data, buf.size, api.scale_flags(1, scale), out.ctypes.data,
                                            need - 1, None, None)
        assert rc == api.KPEG_ERR_ARG and (out == 0x5A).all()
        rc = dec._lib.kpeg_cuda_decode_file(dec._h, buf.ctypes.data, buf.size, api.scale_flags(1, scale), out.ctypes.data,
                                            need, None, None)
        assert rc == 0 and (out[need:] == 0x5A).all()


def test_guard_mode_run():
    code = ("import sys; sys.path[:0] = [%r, %r]\n"
            "import numpy as np, libkpeg_b200 as K, scaled_cases as SC\n"
            "d = K.Decoder(0)\n"
            "for name, jpg in SC.pil_files()[::4]:\n"
            "    for s in SC.SCALES:\n"
            "        assert np.array_equal(d.decode_file(jpg, scale=s), SC.reference(jpg, s, True)), name\n"
            "print('ok')\n") % (str(ROOT), str(ROOT / "tests"))
    r = subprocess.run([sys.executable, "-c", code], env={**os.environ, "KPEG_GUARD": "1"}, capture_output=True, text=True,
                       timeout=600)
    assert r.returncode == 0 and "ok" in r.stdout, r.stdout + r.stderr


@pytest.mark.parametrize("extra", [[], ["--t81"], ["--devices", "0,0"]], ids=["parity", "t81", "devices"])
def test_cli_scale(tmp_path, extra):
    jpg = _big(640, 480, 90)
    (tmp_path / "pic.jpg").write_bytes(jpg)
    parity = "--t81" not in extra
    for s in SC.SCALES:
        r = subprocess.run([str(KPEG), "--quiet", *extra, "--scale", f"1/{s}", "pic.jpg"], cwd=tmp_path, capture_output=True,
                           text=True, timeout=300)
        assert r.returncode == 0, r.stdout + r.stderr
        ref = SC.reference(jpg, s, parity)
        want = api.ppm_header(ref.shape[1], ref.shape[0]) + ref.tobytes()
        assert (tmp_path / "pic.ppm").read_bytes() == want, f"1/{s} {extra}"
    # 1/1 is the full-size decode of the drop-in decoder
    subprocess.run([str(KPEG), "--quiet", "--scale", "1/1", "pic.jpg"], cwd=tmp_path, check=True, timeout=300)
    full = (tmp_path / "pic.ppm").read_bytes()
    subprocess.run([str(KPEG), "--quiet", "pic.jpg"], cwd=tmp_path, check=True, timeout=300)
    assert (tmp_path / "pic.ppm").read_bytes() == full and len(full) > 640 * 480 * 3
