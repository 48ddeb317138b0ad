"""The reduced-size decode (KPEG_FLAG_SCALE_*) on the CPU: the C reference restated from libjpeg against PIL's draft()
decode, the CPU replay of the kernel's arithmetic (csrc/idct_reduced.h) against the reference, the output geometry and
kpeg_output_size.  What the GPU has to match is checked in test_gpu_scaled.py."""
import numpy as np
import pytest

import scaled_cases as SC
from libkpeg_b200 import api

PIL_FILES = SC.pil_files()


@pytest.mark.parametrize("scale", SC.SCALES)
@pytest.mark.parametrize("name,jpg", PIL_FILES, ids=[n for n, _ in PIL_FILES])
def test_reference_matches_pil_draft(name, jpg, scale):
    """PIL-written 4:4:4 and gray files, T.81 coefficients: byte for byte what libjpeg-turbo's scaled decode gives."""
    ref = SC.reference(jpg, scale, parity=False)
    pil = SC.pil_draft(jpg, scale)
    assert ref.shape == pil.shape
    assert np.array_equal(ref, pil), f"{name} 1/{scale}: {int((ref != pil).sum())} bytes differ"


@pytest.mark.parametrize("scale", SC.SCALES)
@pytest.mark.parametrize("parity", [True, False], ids=["parity", "t81"])
def test_replay_matches_reference_on_pil_files(parity, scale):
    for name, jpg in PIL_FILES:
        assert np.array_equal(SC.emu_decode(jpg, scale, parity), SC.reference(jpg, scale, parity)), f"{name} 1/{scale}"


FIELDS = SC.field_files() + list(SC.extreme_files())


@pytest.mark.parametrize("scale", SC.SCALES)
@pytest.mark.parametrize("name,jpg", FIELDS, ids=[n for n, _ in FIELDS])
def test_replay_matches_reference_on_crafted_fields(name, jpg, scale):
    for parity in (True, False):
        ref = SC.reference(jpg, scale, parity)
        assert np.array_equal(SC.emu_decode(jpg, scale, parity), ref), f"{name} 1/{scale} parity={parity}"


def test_extreme_fields_reach_the_wrap_and_64_bit_products():
    """The extreme fields are what they claim: dequantised coefficients of 2047 x 255, and pass-2 sums of the 4x4
    transform beyond 32 bits -- and samples whose range-limit index lies in the wrapping part of the table."""
    for name, jpg in SC.extreme_files():
        w, h, nc, qt = SC.frame_of(jpg)
        coef = SC.coefficients(jpg, parity=False).astype(np.int64)
        dq = coef * qt[np.arange(coef.shape[0]) % nc].astype(np.int64)
        assert np.abs(dq).max() == 2047 * 255, name
        # pass 1 of jpeg_idct_4x4 on the in-phase block (all +), then pass 2's largest term, in exact integers
        nat = np.zeros(64, np.int64)
        nat[SC.CF.ZZ_TO_NAT] = dq[0]
        ws0 = (nat.reshape(8, 8)[0, 0] << 14)  # tmp0 of column 0 alone already needs 35 bits
        assert abs(int(ws0)) > 2 ** 31, name
    # the reference's output on them differs from a clamping range limit (the table wraps)
    name, jpg = SC.extreme_files()[0]
    w, h, nc, qt = SC.frame_of(jpg)
    got = SC.reference(jpg, 8)
    coef = SC.coefficients(jpg, parity=False).astype(np.int64)
    y = (coef[0::nc, 0] * 255 + 4) >> 3  # 1/8: DESCALE(dq_dc, 3) per block, before the range limit
    assert (np.abs(y) > 127).any() and ((np.abs(y) % 1024) >= 128).any(), "no sample reaches the clamping part of the table"


@pytest.mark.parametrize("scale", SC.SCALES)
def test_where_pil_agrees_on_extreme_fields(scale):
    """The contract on crafted extremes is the C reference.  PIL's libjpeg-turbo is a SIMD build whose reduced IDCTs use
    16-bit lanes, so it may differ there: record it, assert only that the reference is deterministic and the replay agrees."""
    agree = {}
    for name, jpg in SC.extreme_files():
        ref = SC.reference(jpg, scale)
        pil = SC.pil_draft(jpg, scale)
        agree[name] = bool(np.array_equal(ref, pil))
        assert np.array_equal(SC.reference(jpg, scale), ref)
        assert np.array_equal(SC.emu_decode(jpg, scale), ref)
    print(f"1/{scale}: PIL draft() equal to the reference on extreme fields: {agree}")


def test_replay_places_batches_back_to_back():
    """n images of one geometry decoded as one job land one after another at the reduced size."""
    jpgs = [SC.pil_jpeg(37, 21, False, 80, seed=s) for s in range(3)]
    w, h, nc, qt = SC.frame_of(jpgs[0])
    coef = np.concatenate([SC.coefficients(j, False) for j in jpgs])
    for scale in SC.SCALES:
        got = SC.replay(coef, qt, w, h, nc, scale, nimages=3)
        for k, j in enumerate(jpgs):
            assert np.array_equal(got[k], SC.reconstruct(SC.coefficients(j, False), SC.frame_of(j)[3], w, h, nc, scale))


def test_output_size_for_every_size_and_scale():
    """kpeg_output_size and the geometry the kernels use: ceil(W / N) x ceil(H / N) (libjpeg's jdiv_round_up)."""
    lib = api.load_cuda_library()
    plan = api.Plan()
    for nc in (1, 3):
        plan.ncomp = nc
        for s, flag in ((1, 0), (2, api.KPEG_FLAG_SCALE_1_2), (4, api.KPEG_FLAG_SCALE_1_4), (8, api.KPEG_FLAG_SCALE_1_8)):
            for w in range(1, 41):
                for h in range(1, 41):
                    plan.width, plan.height, plan.flags = w, h, flag | api.KPEG_FLAG_REF_PARITY
                    ow, oh = api.C.c_uint32(0), api.C.c_uint32(0)
                    n = lib.kpeg_output_size(api.C.byref(plan), api.C.byref(ow), api.C.byref(oh))
                    ew, eh = -(-w // s), -(-h // s)
                    assert (ow.value, oh.value, n) == (ew, eh, ew * eh * nc), (w, h, nc, s)
                    if s > 1:
                        assert SC.out_geom(w, h, nc, s) == (ew, eh, ew * eh * nc)
                    assert api.output_shape(plan) == ((eh, ew, 3) if nc == 3 else (eh, ew))
    plan.width = 0
    assert lib.kpeg_output_size(api.C.byref(plan), None, None) == 0
    plan.width, plan.ncomp = 8, 2
    assert lib.kpeg_output_size(api.C.byref(plan), None, None) == 0
    assert lib.kpeg_output_size(None, None, None) == 0


def test_scale_keyword_and_flags():
    assert api.scale_flags(api.KPEG_FLAG_REF_PARITY, 4) == api.KPEG_FLAG_REF_PARITY | api.KPEG_FLAG_SCALE_1_4
    assert api.scale_flags(api.KPEG_FLAG_SCALE_1_8 | 1, 1) == 1
    for bad in (0, 3, 16, "2"):
        with pytest.raises(ValueError):
            api.scale_flags(0, bad)


def test_encode_and_transcode_reject_scale_bits():
    """The scale bits are decode-only: the encoder's and the transcoder's host-side checks refuse them."""
    lib = api.load_cuda_library()
    for flag in (api.KPEG_FLAG_SCALE_1_2, api.KPEG_FLAG_SCALE_1_8):
        p = api.EncodeParams(16, 16, 3, 90, 0, flag)
        assert lib.kpeg_encode_bound(api.C.byref(p)) == 0
        tp = api.TranscodeParams(-1, 0, flag)
        jpg = np.frombuffer((SC.GOLDEN / "lena.jpg").read_bytes(), np.uint8)
        assert lib.kpeg_transcode_bound(jpg.ctypes.data, jpg.size, api.C.byref(tp)) == 0
