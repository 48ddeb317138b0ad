"""K1 (entropy decode) on the GPU with crafted Huffman tables and streams (tests/huffman_cases.py): the canonical search,
record overflow and its rerun with the Huffman final pass, a table that turns records off, relay chains far longer than
the device loop, code-length edges, and tables that fill the code space.  Coefficients and pixels must equal the
oracle's bit for bit, in both parity modes, at subsequence sizes 64, 512 and 1024, through decode_file, decode_batch
and decode_files; the stats show that each family took its path.  Plans whose restart padding decodes as a symbol are
refused by every entry point that would meet such padding, and decode where there is none."""
import numpy as np
import pytest

import helpers as H
import huffman_cases as HC
import libkpeg_b200 as K
from libkpeg_b200.api import KPEG_ERR_UNSUPPORTED, KPEG_OK

pytestmark = pytest.mark.gpu

SUB_BITS = (64, 512, 1024)
PARITY = (True, False)


def _flags(parity):
    return K.KPEG_FLAG_REF_PARITY if parity else 0


def _decoder(monkeypatch, sub_bits, **env):
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    dec = K.Decoder(device=0)
    for k in env:
        monkeypatch.delenv(k)
    dec.set_tuning(sub_bits=sub_bits)
    return dec


@pytest.fixture(scope="module")
def contexts():
    """{(sub_bits, records): Decoder}; records False = a KPEG_NO_RECORDS=1 context (Huffman final pass)."""
    mp = pytest.MonkeyPatch()
    out = {}
    try:
        for sb in SUB_BITS:
            out[(sb, True)] = _decoder(mp, sb)
            out[(sb, False)] = _decoder(mp, sb, KPEG_NO_RECORDS="1")
        yield out
    finally:
        for d in out.values():
            d.close()
        mp.undo()


def _check(dec, jpg, parity, what):
    got = dec.decode_file(jpg, flags=_flags(parity))
    ref = H.oracle_decode(jpg, parity=parity)
    coef = dec.read_coefficients(ref["coef"].shape[0])
    assert np.array_equal(coef, ref["coef"]), f"{what}: coefficients differ from the oracle"
    assert np.array_equal(got, ref["pixels"]), f"{what}: {int((got != ref['pixels']).sum())} pixel values differ"
    return dec.last_stats


@pytest.mark.parametrize("case", HC.CASES, ids=lambda c: c.name)
def test_decode_file(contexts, case):
    jpg, _ = HC.build(case)
    T = HC.thresholds()
    for sb in SUB_BITS:
        for parity in PARITY:
            what = f"{case.name} sub_bits={sb} parity={parity}"
            st = _check(contexts[(sb, True)], jpg, parity, what)
            launches, rounds = st.kernel_launches, st.sync_rounds
            st0 = _check(contexts[(sb, False)], jpg, parity, what + " (Huffman final pass)")
            if case.family == "slow_sync":
                assert rounds > T["MAX_RELAY_ROUNDS"] - 2 and st0.sync_rounds > T["MAX_RELAY_ROUNDS"] - 2, (what, rounds)
            if case.family == "record_overflow":  # the record pass, then the rerun with the Huffman final pass
                assert launches > st0.kernel_launches, (what, launches, st0.kernel_launches)
            if case.family == "records_off":  # the Huffman final pass straight away
                assert launches == st0.kernel_launches, (what, launches, st0.kernel_launches)


@pytest.mark.parametrize("case", [c for c in HC.CASES if c.family != "all_ones_padding"], ids=lambda c: c.name)
def test_decode_batch_and_files(contexts, case):
    """Several files of one plan as one batch (RSTn between the images) and through decode_files.  (all_ones_padding:
    test_all_ones_padding_without_restarts.)"""
    files = HC.batch(case)
    plan, scans = HC.scans_of(files)
    for sb in (64, 512):
        dec = contexts[(sb, True)]
        for parity in PARITY:
            refs = [H.oracle_decode(f, parity=parity)["pixels"] for f in files]
            plan.flags = _flags(parity)
            outs = dec.decode_batch(plan, scans)
            for k, (got, ref) in enumerate(zip(outs, refs)):
                assert np.array_equal(got, ref), f"{case.name} sub_bits={sb} parity={parity}: batch image {k}"
            imgs, codes = dec.decode_files(files, flags=_flags(parity))
            assert codes == [KPEG_OK] * len(files), (case.name, codes)
            for k, (got, ref) in enumerate(zip(imgs, refs)):
                assert np.array_equal(got, ref), f"{case.name} sub_bits={sb} parity={parity}: decode_files image {k}"


def _unsupported(fn):
    with pytest.raises(K.KpegError) as e:
        fn()
    assert e.value.code == KPEG_ERR_UNSUPPORTED, str(e.value)


@pytest.mark.parametrize("case", HC.REFUSED_CASES, ids=lambda c: c.name)
def test_all_ones_padding_is_refused(decoder, case):
    """Restart padding that decodes as a DC symbol: every entry point refuses the file (one scan per component and the
    transcoder included) instead of returning a wrong image."""
    files = HC.batch(case)
    _unsupported(lambda: decoder.decode_file(files[0]))
    _unsupported(lambda: decoder.transcode(files[0]))
    imgs, codes = decoder.decode_files(files)
    assert codes == [KPEG_ERR_UNSUPPORTED] * len(files) and imgs == [None] * len(files)
    if case.interleaved:
        plan, scans = HC.scans_of(files)
        _unsupported(lambda: decoder.decode_batch(plan, scans))
        _unsupported(lambda: decoder.decode_batch(plan, scans[:1]))


@pytest.mark.parametrize("case", [c for c in HC.CASES if c.family == "all_ones_padding"], ids=lambda c: c.name)
def test_all_ones_padding_without_restarts(decoder, case):
    """The same tables without restart markers: one image decodes bit-exact (test_decode_file) and transcodes
    losslessly; a batch of them has image boundaries and is refused; decode_files decodes them one job each, also
    next to a refused file and an ordinary one."""
    files = HC.batch(case)
    plan, scans = HC.scans_of(files)
    _unsupported(lambda: decoder.decode_batch(plan, scans))
    refused = HC.build(HC.REFUSED_CASES[0])[0]
    other = HC.build(HC.CASES[0])[0]
    mixed = files + [refused, other]
    imgs, codes = decoder.decode_files(mixed)
    assert codes == [KPEG_OK] * len(files) + [KPEG_ERR_UNSUPPORTED, KPEG_OK], codes
    for k, f in enumerate(files + [None, other]):
        if f is not None:
            assert np.array_equal(imgs[k], H.oracle_decode(f, parity=True)["pixels"]), f"decode_files image {k}"
    out = decoder.transcode(files[0])
    assert np.array_equal(H.oracle_decode(out, parity=False, want_pixels=False)["coef"],
                          H.oracle_decode(files[0], parity=False, want_pixels=False)["coef"])


def test_guard_mode_over_all_families(monkeypatch):
    """KPEG_GUARD=1: the guard bytes around every device buffer survive every family (record overflow reruns, host
    relay rounds, the Huffman final pass) and the refusals."""
    dec = _decoder(monkeypatch, 64, KPEG_GUARD="1")
    try:
        for case in HC.CASES:
            _check(dec, HC.build(case)[0], True, f"{case.name} (guard)")
        for case in HC.REFUSED_CASES:
            _unsupported(lambda: dec.decode_file(HC.build(case)[0]))
    finally:
        dec.close()
