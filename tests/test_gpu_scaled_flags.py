"""The Python file entry points take the reduced size either from `scale=` or from KPEG_FLAG_SCALE_* bits already in
`flags`: with scale left at None the bits decide, so decode_file(jpg, flags=KPEG_FLAG_SCALE_1_2) is a 1/2 decode, as
decode_scan / decode_batch / decode_device keep the bits of their plan."""
import numpy as np
import pytest

import libkpeg_b200 as K
import scaled_cases as SC
from libkpeg_b200 import api
from libkpeg_b200.synth import EMIT_RESTART, QUIRK_FREE, SynthParams, synth_encode

SCALE_BITS = {2: api.KPEG_FLAG_SCALE_1_2, 4: api.KPEG_FLAG_SCALE_1_4, 8: api.KPEG_FLAG_SCALE_1_8}


def test_scale_none_keeps_the_bits_of_flags():
    for s, bits in SCALE_BITS.items():
        f = api.KPEG_FLAG_REF_PARITY | bits
        assert api._scaled_flags(f, None) == f
        assert api._scaled_flags(f, 1) == api.KPEG_FLAG_REF_PARITY
        assert api._scaled_flags(api.KPEG_FLAG_REF_PARITY, s) == f


@pytest.mark.gpu
def test_file_entry_points_honour_scale_bits_in_flags():
    jpg = dict(SC.pil_files())["opt-q85"]  # 97 x 61
    big = synth_encode(SynthParams(640, 480, quality=90, restart_interval=80, seed=5, flags=QUIRK_FREE | EMIT_RESTART)).tobytes()
    with K.Decoder(0) as dec:
        for s, bits in SCALE_BITS.items():
            for parity, pf in ((True, api.KPEG_FLAG_REF_PARITY), (False, 0)):
                ref = SC.reference(jpg, s, parity)
                assert np.array_equal(dec.decode_file(jpg, pf | bits), ref), f"decode_file 1/{s}"
                imgs, codes = dec.decode_files([jpg, big], pf | bits)
                assert codes == [0, 0] and np.array_equal(imgs[0], ref), f"decode_files 1/{s}"
                assert np.array_equal(imgs[1], SC.reference(big, s, parity)), f"decode_files 1/{s}"
                got, _ = api.decode_file_tiled([0, 0], big, pf | bits)
                assert np.array_equal(got, SC.reference(big, s, parity)), f"decode_file_tiled 1/{s}"
            # an explicit scale overrides the bits
            assert dec.decode_file(jpg, api.KPEG_FLAG_REF_PARITY | bits, scale=1).shape[:2] == (61, 97)
