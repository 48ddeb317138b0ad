"""K1 (entropy decode) on crafted Huffman tables and streams (tests/huffman_cases.py), on the CPU: the kernels' two-level
lookup against the canonical search and the oracle's tree walk for every 16-bit window, the replay of the kernel logic
(tests/emu, the same entropy_core.h) against the oracle at four subsequence sizes in both parity modes, and for every
family a witness that its stream reaches the path it is there for."""
import ctypes as C

import numpy as np
import pytest

import helpers as H
import huffman_cases as HC
import jpeg_writer as JW
import libkpeg_b200 as K

SUB_BITS = (64, 96, 512, 1024)


def _tables(case):
    """Every distinct (is_ac, (counts, symbols)) the case's file defines."""
    dct, act, *_ = HC._component_tables(case)
    out = {}
    for is_ac, tabs in ((0, dct), (1, act)):
        for t in tabs.values():
            out[(is_ac, tuple(t[0]), tuple(t[1]))] = (is_ac, t)
    return list(out.values())


ALL_TABLES = {}
for _case in HC.CASES + HC.REFUSED_CASES:
    for _is_ac, _t in _tables(_case):
        ALL_TABLES.setdefault(f"{_case.family}-{'ac' if _is_ac else 'dc'}{len(ALL_TABLES)}", (_is_ac, _t))


def _arrays(t):
    counts = np.array(t[0], dtype=np.uint8)
    syms = np.zeros(256, dtype=np.uint8)
    syms[:len(t[1])] = t[1]
    return counts, syms


def _expected_entry(length, sym, is_ac):
    """kpeg_common.h pack_entry, restated: total bits | category << 5 | slot advance << 9."""
    size = sym & 15
    adv = (64 if sym == 0 else (sym >> 4) + 1) if is_ac else 1
    return (length + size) | (size << 5) | (adv << 9)


@pytest.mark.parametrize("name", sorted(ALL_TABLES))
def test_lookup_every_window(name):
    """The kernel lookup (first level, sub-tables, canonical search), the canonical search alone and the oracle's
    tree walk (HuffmanTree::contains) give the same symbol and length for every 16-bit window."""
    is_ac, t = ALL_TABLES[name]
    counts, syms = _arrays(t)
    o = H.oracle()
    # the oracle's answer for every window: its codes (each a complete code, no shorter prefix one) spread over the
    # windows they start
    codes = np.zeros(256, dtype=np.uint16)
    lens = np.zeros(256, dtype=np.uint8)
    n = o.kpo_huff_codes(counts.ctypes.data, syms.ctypes.data, codes.ctypes.data, lens.ctypes.data)
    assert n == len(t[1])
    want = np.full(65536, 17 | (127 << 9), dtype=np.uint32)  # ENTRY_INVALID: no code starts the window
    for i in range(n):
        L, code = int(lens[i]), int(codes[i])
        bits = format(code, "b").zfill(L)
        assert o.kpo_huff_lookup(counts.ctypes.data, syms.ctypes.data, bits.encode()) == t[1][i]
        for k in range(1, L):
            assert o.kpo_huff_lookup(counts.ctypes.data, syms.ctypes.data, bits[:k].encode()) == -1
        want[code << (16 - L):(code + 1) << (16 - L)] = _expected_entry(L, t[1][i], is_ac)
    rng = np.random.default_rng(7)
    wins = ((np.arange(65536, dtype=np.uint64) << 16) | rng.integers(0, 65536, 65536).astype(np.uint64)).astype(np.uint32)
    emu = H.emu()
    for mode in (0, 1):
        got = np.zeros(65536, dtype=np.uint32)
        emu.emu_huff_lookup_many(counts.ctypes.data, syms.ctypes.data, is_ac, wins.ctypes.data, 65536, mode, got.ctypes.data)
        bad = np.nonzero(got != want)[0]
        assert bad.size == 0, f"mode {mode}: {bad.size} windows differ, first {int(bad[0]):016b}"


def test_canonical_search_layout():
    """The canonical_search AC table has more long prefixes than the second-level table holds; the emulator's view of
    the kernel tables (long_n, the prefixes left to the search) agrees with the count from the codes."""
    T = HC.thresholds()
    t = HC.canonical_ac()
    counts, syms = _arrays(t)
    longs = HC.long_prefixes(t)
    cap = T["LONG_CAP"] // T["SUB_SIZE"]
    assert len(longs) > cap
    long_n = C.c_uint32()
    canonical = np.zeros(1 << T["LUT_BITS"], dtype=np.uint8)
    n = H.emu().emu_huff_layout(counts.ctypes.data, syms.ctypes.data, 1, C.byref(long_n), canonical.ctypes.data)
    assert long_n.value == T["LONG_CAP"]
    assert n == len(longs) - cap
    assert set(np.nonzero(canonical)[0]) == set(sorted(longs)[cap:])


@pytest.mark.parametrize("case", HC.CASES, ids=lambda c: c.name)
def test_replay_equals_oracle(case):
    jpg, _ = HC.build(case)
    for parity in (True, False):
        ref = H.oracle_decode(jpg, parity=parity)
        for sb in SUB_BITS:
            e = H.emu_decode(jpg, flags=1 if parity else 0, sub_bits=sb)
            assert e["status"] == 0, f"sub_bits {sb} parity={parity}: status {e['status']:#x}"
            assert e["records_ok"], f"sub_bits {sb}: the record flavour differs from the Huffman final pass"
            assert np.array_equal(e["coef"], ref["coef"]), f"sub_bits {sb} parity={parity}: coefficients differ"
            assert np.array_equal(e["pixels"], ref["pixels"]), f"sub_bits {sb} parity={parity}: pixels differ"


def _family_cases(family):
    return [c for c in HC.CASES if c.family == family]


def test_witness_canonical_search():
    for case in _family_cases("canonical_search"):
        assert HC.facts(case)["canonical_prefixes_used"] > 0, case.name


@pytest.mark.parametrize("sb", SUB_BITS)
def test_witness_record_overflow(sb):
    kmax = HC.rec_kmax(sb)
    for case in _family_cases("record_overflow"):
        assert HC.facts(case)["max_records"][sb] > kmax, case.name
        e = H.emu_decode(HC.build(case)[0], sub_bits=sb, want_pixels=False)
        assert e["max_records"] > kmax and e["subs_over_kmax"] > 0, case.name


def test_witness_records_off():
    for case in _family_cases("records_off"):
        f = HC.facts(case)
        assert f["declared_max_category"] > 11 >= f["used_max_category"], case.name


@pytest.mark.parametrize("sb", SUB_BITS)
def test_witness_slow_sync(sb):
    """No speculative decode synchronises: the relay takes one round per subsequence, more than the device loop runs."""
    T = HC.thresholds()
    for case in _family_cases("slow_sync"):
        e = H.emu_decode(HC.build(case)[0], sub_bits=sb, want_pixels=False)
        assert e["rounds"] == e["nsub"] - 1 > T["MAX_RELAY_ROUNDS"] - 2, case.name
        assert e["nsub"] <= 2000, case.name  # the GPU runs about nsub / 2 host iterations


def test_witness_code_length_edges():
    lb = HC.thresholds()["LUT_BITS"]
    for case in _family_cases("code_length_edges"):
        f = HC.facts(case)
        assert {1, lb, lb + 1, 16} <= f["code_lengths"], case.name
        assert f["s27_cross64"], case.name  # a 27-bit symbol across a 64-bit subsequence (and word) boundary
        if case.restart == "none":
            assert f["offsets27"] == set(range(32)), case.name


@pytest.mark.parametrize("family", ["complete", "reserved"])
def test_witness_complete_vs_reserved(family):
    """The complete table's all-ones code plus its category is one bit longer than the longest padding; the other
    table has none.  Neither is refused, and both decode with restart markers (test_replay_equals_oracle)."""
    for case in _family_cases(family):
        f = HC.facts(case)
        assert case.restart != "none"
        for a in f["all_ones"]:
            assert (a is not None and a[0] + (a[1] & 15) == 8) if family == "complete" else a is None, case.name
        plan, _, _ = K.parse_jfif(HC.build(case)[0])
        assert H.emu().emu_restart_padding_decodes(C.addressof(plan)) == 0, case.name


def test_all_ones_padding_rule():
    """A DC table whose all-ones code fits in the padding: the plan is marked (the product refuses restart intervals and
    batches for it), and the replay shows why -- with restart markers the padding decodes as one more block.  One image
    without restart markers decodes (test_replay_equals_oracle)."""
    for case in HC.REFUSED_CASES + tuple(_family_cases("all_ones_padding")):
        jpg, _ = HC.build(case)
        frame, scans = K.api.parse_jfif_scans(np.frombuffer(jpg, dtype=np.uint8))
        for sc in scans:
            assert H.emu().emu_restart_padding_decodes(C.addressof(sc.plan)) == 1, case.name
        if case.interleaved and case.restart != "none":
            ref = H.oracle_decode(jpg, parity=True)
            e = H.emu_decode(jpg, sub_bits=512, want_pixels=False)
            assert e["status"] != 0 or not np.array_equal(e["coef"], ref["coef"]), case.name


@pytest.mark.parametrize("length,category,refused", [(1, 0, True), (3, 4, True), (4, 3, True), (4, 4, False),
                                                     (7, 0, True), (8, 0, False)])
def test_all_ones_rule_boundary(length, category, refused):
    """restart_padding_decodes marks exactly the full DC tables whose all-ones code and category fit in 7 bits."""
    pool = [s for s in range(16) if s != category]
    pairs = [(L, pool[L - 1]) for L in range(1, length + 1)] + [(length, category)]  # the last code is all ones
    full = HC.table(pairs)
    assert HC.kraft(full) == 1.0 and HC.all_ones_symbol(full) == (length, category)
    reserved = HC.table(pairs[:-1] + [(length + 1, category)])
    assert HC.all_ones_symbol(reserved) is None
    for t, want in ((full, refused), (reserved, False)):
        jpg = JW.write_jpeg(np.zeros((4, 64), dtype=np.int16), 16, 16, 1, {0: [1] * 64}, (0,), {0: t},
                            {0: HC.SMALL_AC}, (0,), (0,))
        plan, _, _ = K.parse_jfif(jpg)
        assert H.emu().emu_restart_padding_decodes(C.addressof(plan)) == int(want), (length, category)
