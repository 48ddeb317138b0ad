"""K3's reconstruction branches on the GPU, each driven on purpose by a crafted coefficient field (tests/coef_fields.py):
the DC-only shortcut, the fast transform and its tie band, tie records and the in-kernel resolution of a strip with
more ties than its list, the three colour modes, BLK_HUGE MCUs, byte stores of ragged rows, images narrower than a
strip.  Coefficients and pixels must equal the oracle's bit for bit, in both parity modes."""
import numpy as np
import pytest

import coef_fields as CF
import helpers as H
import libkpeg_b200 as K

pytestmark = pytest.mark.gpu


def decode_and_compare(dec, f, jpg, parity):
    got = dec.decode_file(jpg, flags=K.KPEG_FLAG_REF_PARITY if parity else 0)
    ref = H.oracle_decode(jpg, parity=parity)
    coef = dec.read_coefficients(ref["coef"].shape[0])
    assert np.array_equal(coef, ref["coef"]), f"{f.name}: coefficients differ from the oracle"
    bad = got != ref["pixels"]
    if f.ncomp == 3:
        bad = bad.any(axis=-1)
    if bad.any():
        ys, xs = np.nonzero(bad)
        mcus = sorted({int(y // 8 * f.mcus_x + x // 8) for y, x in zip(ys, xs)})
        pytest.fail(f"{f.name} {f.width}x{f.height}x{f.ncomp} parity={parity}: {int(bad.sum())} pixels differ, "
                    f"MCUs {mcus[:12]}")
    return got


@pytest.mark.parametrize("parity", [True, False], ids=["parity", "t81"])
@pytest.mark.parametrize("case", CF.cases(), ids=lambda c: f"{c[0]}-{c[1]}x{c[2]}x{c[3]}")
def test_family(decoder, case, parity):
    for (f, jpg), facts in zip(CF.fields_and_files(*case), CF.facts_of(*case)):
        decode_and_compare(decoder, f, jpg, parity)
        if facts["ties"].sum() > 0:  # tied samples in blocks that are neither DC-only nor huge
            assert decoder.last_stats.exact_samples > 0, f"{f.name}: no sample took the exact path"


def test_narrow_images_batch(decoder):
    """Strips that span two or three images (mcu_origin's division path, the pixel index of a tie record), with huge
    and tied blocks on both sides of every image boundary."""
    fields = CF.narrow_batch()
    plan, _, _ = K.parse_jfif(np.frombuffer(fields[0][1], dtype=np.uint8))
    scans = []
    for _, jpg in fields:
        buf = np.frombuffer(jpg, dtype=np.uint8)
        _, off, n = K.parse_jfif(buf)
        scans.append(buf[off:off + n])
    for parity in (True, False):
        plan.flags = K.KPEG_FLAG_REF_PARITY if parity else 0
        outs = decoder.decode_batch(plan, scans)
        assert decoder.last_stats.exact_samples > 0
        for (f, jpg), got in zip(fields, outs):
            ref = H.oracle_decode(jpg, parity=parity)
            assert np.array_equal(got, ref["pixels"]), f"{f.name} parity={parity}"


TUNING_CASES = [("exact_ties", 250, 44, 3), ("wide_and_huge", 124, 60, 3), ("exact_ties", 124, 60, 1)]


def test_subsequence_size_does_not_matter_to_k3():
    dec = K.Decoder(device=0)
    try:
        dec.set_tuning(sub_bits=64)
        for case in TUNING_CASES:
            for f, jpg in CF.fields_and_files(*case):
                decode_and_compare(dec, f, jpg, parity=True)
    finally:
        dec.close()


def test_huffman_final_pass_does_not_matter_to_k3(monkeypatch):
    monkeypatch.setenv("KPEG_NO_RECORDS", "1")
    dec = K.Decoder(device=0)
    monkeypatch.delenv("KPEG_NO_RECORDS")
    try:
        for case in TUNING_CASES:
            for f, jpg in CF.fields_and_files(*case):
                decode_and_compare(dec, f, jpg, parity=True)
    finally:
        dec.close()
