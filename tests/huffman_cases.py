"""TEST INFRASTRUCTURE: crafted Huffman tables and the streams that drive the entropy decoder (K1) down its rare paths.
Every common encoder writes Annex K tables or libjpeg-style optimised ones; these families do not:

  canonical_search      an AC table with more ten-bit prefixes of long codes than the second-level table holds: the
                        rest take the canonical search (entropy_core.h huff_slow_lookup)
  record_overflow       value symbols of two bits (a 1-bit code, +-1): a subsequence holds more records than rec_kmax,
                        the device redoes the job with the Huffman final pass
  records_off           a DHT that declares categories 12..15 (never used): the job takes the Huffman final pass
  slow_sync             one 1-bit code per table and an all-zero scan: no speculative decode ever synchronises, the
                        relay needs one round per subsequence
  code_length_edges     codes of 1, LUT_BITS, LUT_BITS + 1 and 16 bits; 27-bit DC symbols (16-bit code, category 11)
                        at every bit offset mod 32
  all_ones_padding      tables of two 1-bit codes: the padding before a restart marker decodes as symbols
  complete / reserved   a DC table that fills the code space (all-ones code one bit too long to fit in the padding)
                        against one that leaves the all-ones code free

Layouts: one and three components (three: a table pair and a quantiser of its own per component, ids other than
0/1/1), restart intervals of 1, 7 and one MCU row.  The thresholds come from the source text, and each family states
what in its stream crosses them (facts), so a changed constant fails the tests instead of quietly testing nothing."""
from __future__ import annotations

import functools
import re
import zlib
from dataclasses import dataclass
from pathlib import Path

import numpy as np

import jpeg_writer as JW

CSRC = Path(__file__).resolve().parent.parent / "libkpeg_b200" / "csrc"


# ---- thresholds, from the source text ------------------------------------------------------------
def _c_expr(expr: str) -> str:
    expr = re.sub(r"\b(\d+)u\b", r"\1", expr)  # 7u -> 7
    expr = expr.replace("/", "//")  # unsigned division
    m = re.fullmatch(r"\s*(.+?)\s*\?\s*(.+?)\s*:\s*(.+?)\s*", expr)  # a ? b : c
    return f"({m.group(2)}) if ({m.group(1)}) else ({m.group(3)})" if m else expr


def _constexpr(text: str, name: str, env: dict) -> int:
    m = re.search(rf"constexpr\s+\w+\s+{name}\s*=\s*([^;]+);", text)
    assert m, f"{name} not found"
    return int(eval(_c_expr(m.group(1)), {"__builtins__": {}}, env))  # noqa: S307 -- constants of our own sources


@functools.lru_cache(maxsize=None)
def thresholds() -> dict:
    common = (CSRC / "kpeg_common.h").read_text()
    m = re.search(r"#define\s+KPEG_LUT_BITS\s+(\d+)", common)
    assert m, "KPEG_LUT_BITS not found"
    t = {"KPEG_LUT_BITS": int(m.group(1))}
    for name in ("LUT_BITS", "SUB_BITS", "SUB_SIZE", "LONG_CAP"):
        t[name] = _constexpr(common, name, t)
    t["MAX_RELAY_ROUNDS"] = _constexpr((CSRC / "kernels.cuh").read_text(), "MAX_RELAY_ROUNDS", t)
    m = re.search(r"rec_kmax_of\(uint32_t sub_bits\)\s*\{\s*return\s+([^;]+);", (CSRC / "host_tables.h").read_text())
    assert m, "rec_kmax_of not found"
    t["rec_kmax_expr"] = _c_expr(m.group(1))
    return t


def rec_kmax(sub_bits: int) -> int:
    return int(eval(thresholds()["rec_kmax_expr"], {"__builtins__": {}}, {"sub_bits": sub_bits}))  # noqa: S307


# ---- tables --------------------------------------------------------------------------------------
def table(pairs):
    """[(code length, symbol), ...] in canonical order -> (counts[16], symbols)."""
    pairs = sorted(pairs, key=lambda p: p[0])
    counts = [0] * 16
    for length, _ in pairs:
        counts[length - 1] += 1
    return counts, [s for _, s in pairs]


def kraft(tab) -> float:
    return sum(n * 2.0 ** -(L + 1) for L, n in enumerate(tab[0]))


def all_ones_symbol(tab):
    """(length, symbol) of the table's all-ones code, or None (T.81 C reserves it; a full code space does not)."""
    counts, syms = tab
    if kraft(tab) != 1.0:
        return None
    return max(L + 1 for L in range(16) if counts[L]), syms[int(sum(counts)) - 1]


def long_prefixes(tab) -> set:
    """LUT_BITS-bit prefixes that start a code longer than LUT_BITS."""
    lb = thresholds()["LUT_BITS"]
    return {code >> (L - lb) for code, L in JW.canonical_codes(*tab).values() if L > lb}


def _annex_k():
    import coef_fields as CF
    return CF.annex_k_tables()


SLOW_DC = table([(1, 0x00)])  # '0': category 0; '1' is no code
SLOW_AC = table([(1, 0x02)])  # '0': run 0, category 2 -- with the value -3 ('00') the scan is all zero bits
ALL_ONES_DC = table([(1, 0x00), (1, 0x01)])  # '1' (category 1) is a code
ALL_ONES_AC = table([(1, 0x00), (1, 0x01)])
COMPLETE_DC = table([(1, 0), (2, 1), (3, 2), (4, 3), (4, 4)])  # all-ones '1111' + 4 value bits: 8 > 7 padding bits
RESERVED_DC = table([(1, 0), (2, 1), (3, 2), (4, 3), (5, 4)])
SMALL_AC = table([(2, 0x00), (2, 0x01), (3, 0x02), (3, 0x11), (4, 0x21), (4, 0x12), (4, 0x31), (5, 0x03), (5, 0xF0)])
OVERFLOW_AC = table([(1, 0x01), (2, 0x00), (4, 0x02), (4, 0x11), (4, 0x21), (4, 0xF0)])
EDGE_DC = table([(1, 0), (2, 1), (3, 2), (4, 3), (5, 4), (6, 5), (7, 6), (8, 7), (9, 8), (10, 9), (11, 10), (16, 11)])
EDGE_AC = table([(1, 0x01), (2, 0x00), (3, 0x02), (4, 0x11), (5, 0xF0), (10, 0x03), (11, 0x21), (16, 0x0A), (16, 0x31),
                 (16, 0x4A)])


def canonical_ac():
    short = [0x00, 0x01, 0x02, 0x11, 0xF0]
    longs = [(r << 4) | s for r in range(16) for s in range(1, 7) if ((r << 4) | s) not in short]
    return table([(L, s) for L, s in zip((1, 2, 3, 4, 5), short)] + [(11, s) for s in longs[:63]] +
                 [(12, s) for s in longs[63:65]])


def records_off_dc():
    """Annex K's luminance DC table and four 12-bit codes for categories 12..15."""
    dc, _ = _annex_k()
    lengths = [L + 1 for L in range(16) for _ in range(int(dc[0][L]))]
    return table(list(zip(lengths, dc[1])) + [(12, 12), (12, 13), (12, 14), (12, 15)])


# ---- coefficient fields --------------------------------------------------------------------------
def _dc_diffs(rng, n, cats):
    """n DC differences with categories drawn from `cats`; signs keep the running value inside +-2047."""
    out, pred = np.zeros(n, dtype=np.int64), 0
    for i in range(n):
        s = int(rng.choice(cats))
        v = int(rng.integers(1 << (s - 1), 1 << s)) if s else 0
        sign = -1 if pred > 0 else (1 if pred < 0 else int(rng.choice([-1, 1])))
        out[i] = sign * v
        pred += out[i]
    return out


def _ac_from_symbols(rng, syms, target):
    """One block's AC coefficients from run/size symbols drawn from `syms` until zig-zag index `target`."""
    blk = np.zeros(64, dtype=np.int64)
    z = 1
    while z <= target:
        sym = int(rng.choice(syms))
        r, s = sym >> 4, sym & 15
        if z + r > 63:
            break
        z += r
        blk[z] = int(rng.integers(1 << (s - 1), 1 << s)) * int(rng.choice([-1, 1]))
        z += 1
    return blk


def _value_syms(ac):
    return [s for s in ac[1][:int(sum(ac[0]))] if s & 15]


def gen_blocks(family, rng, nb, dc, ac):
    """[nb][64] zig-zag blocks of one component (DC as differences in column 0) for the family's tables."""
    out = np.zeros((nb, 64), dtype=np.int64)
    vs = _value_syms(ac)
    dc_cats = sorted({s & 15 for s in dc[1][:int(sum(dc[0]))] if (s & 15) <= 11})
    if family == "slow_sync":
        out[:, 1:] = -3
        return out
    if family == "code_length_edges":
        out[:, 0] = _dc_diffs(rng, nb, [11] * 6 + dc_cats)
        for b in range(nb):
            k = int(rng.integers(0, 8))  # +-1 coefficients of 2 bits each: walks the offsets of the next DC symbol
            out[b, 1:1 + k] = rng.choice([-1, 1], size=k)
            if rng.random() < 0.3:
                out[b, 1:] = _ac_from_symbols(rng, vs, int(rng.integers(1, 40)))[1:]
        return out
    out[:, 0] = _dc_diffs(rng, nb, dc_cats)
    codes = JW.canonical_codes(*ac)
    longs = [s for s in vs if codes[s][1] > thresholds()["LUT_BITS"]]
    for b in range(nb):
        if family == "record_overflow" and rng.random() < 0.7:
            out[b, 1:] = rng.choice([-1, 1], size=63)
        elif family == "all_ones_padding":
            k = int(rng.integers(0, 64))
            out[b, 1:1 + k] = rng.choice([-1, 1], size=k)
        elif family == "canonical_search":
            out[b, 1:] = _ac_from_symbols(rng, longs * 4 + vs, int(rng.integers(8, 60)))[1:]
        else:
            out[b, 1:] = _ac_from_symbols(rng, vs, int(rng.integers(0, 50)))[1:]
    return out


def _integrate(diffs, restart):
    """DC differences -> DC values, predictors reset every `restart` MCUs (0: never)."""
    vals, pred = np.zeros_like(diffs), 0
    for m, d in enumerate(diffs):
        if restart and m % restart == 0:
            pred = 0
        pred += int(d)
        vals[m] = pred
    return vals


# ---- cases ---------------------------------------------------------------------------------------
FAMILY_TABLES = {
    "canonical_search": lambda: (_annex_k()[0], canonical_ac()),
    "record_overflow": lambda: (_annex_k()[0], OVERFLOW_AC),
    "records_off": lambda: (records_off_dc(), _annex_k()[1]),
    "slow_sync": lambda: (SLOW_DC, SLOW_AC),
    "code_length_edges": lambda: (EDGE_DC, EDGE_AC),
    "all_ones_padding": lambda: (ALL_ONES_DC, ALL_ONES_AC),
    "complete": lambda: (COMPLETE_DC, SMALL_AC),
    "reserved": lambda: (RESERVED_DC, SMALL_AC),
}
FAMILIES = tuple(FAMILY_TABLES)


@dataclass(frozen=True)
class Case:
    family: str
    width: int
    height: int
    ncomp: int
    restart: str = "none"  # "none", "1", "7", "row"
    interleaved: bool = True

    @property
    def name(self):
        return (f"{self.family}-{self.width}x{self.height}x{self.ncomp}-ri_{self.restart}"
                + ("" if self.interleaved else "-scans"))

    def restart_interval(self):
        return {"none": 0, "1": 1, "7": 7, "row": (self.width + 7) // 8}[self.restart]


CASES = (
    Case("canonical_search", 256, 128, 1),
    Case("canonical_search", 120, 64, 3, "row"),
    Case("canonical_search", 96, 56, 3, "7"),
    Case("record_overflow", 256, 128, 1),
    Case("record_overflow", 96, 64, 3, "1"),
    Case("record_overflow", 200, 64, 1, "row"),
    Case("records_off", 128, 128, 1),
    Case("records_off", 96, 64, 3, "7"),
    Case("slow_sync", 256, 128, 1),
    Case("slow_sync", 128, 64, 3),
    Case("code_length_edges", 256, 128, 1),
    Case("code_length_edges", 104, 64, 3, "row"),
    Case("code_length_edges", 128, 64, 1, "1"),
    Case("all_ones_padding", 256, 64, 1),
    Case("all_ones_padding", 96, 48, 3),
    Case("complete", 128, 64, 1, "1"),
    Case("complete", 96, 56, 3, "7"),
    Case("complete", 120, 48, 3, "row"),
    Case("reserved", 128, 64, 1, "1"),
    Case("reserved", 96, 56, 3, "row"),
)

# the same tables with restart markers / as a batch: refused (host_tables.h restart_padding_decodes)
REFUSED_CASES = (
    Case("all_ones_padding", 64, 16, 1, "1"),
    Case("all_ones_padding", 128, 32, 1, "7"),
    Case("all_ones_padding", 96, 48, 3, "row"),
    Case("all_ones_padding", 96, 48, 3, "1", interleaved=False),
)


def _component_tables(case: Case):
    """(dc_tables, ac_tables, td, ta, qts, tq): one component uses ids 0/0; three use a pair of their own each (DC ids
    1, 0, 2; AC ids 2, 0, 1 -- AC tables with symbols of equal length shuffled) and quantisers 2, 0, 1."""
    dc, ac = FAMILY_TABLES[case.family]()
    q = [1] + [1 + (i % 3) for i in range(1, 64)]
    if case.ncomp == 1:
        return {0: dc}, {0: ac}, (0,), (0,), {0: q}, (0,)
    td, ta = (1, 0, 2), (2, 0, 1)
    acs = [ac, JW.permuted_table(*ac, seed=5), JW.permuted_table(*ac, seed=6)]
    qts = {2: q, 0: [1] + [2] * 63, 1: [1] + [1 + (i % 5) for i in range(1, 64)]}
    return ({td[c]: dc for c in range(3)}, {ta[c]: acs[c] for c in range(3)}, td, ta, qts, (2, 0, 1))


@functools.lru_cache(maxsize=None)
def build(case: Case, seed: int = 0):
    """-> (jpeg bytes, marks: [(bit, component, is_ac, symbol, code length, category)] of every scan)."""
    dct, act, td, ta, qts, tq = _component_tables(case)
    rng = np.random.default_rng([zlib.crc32(case.name.encode()), seed])
    nmcu = ((case.width + 7) // 8) * ((case.height + 7) // 8)
    ri = case.restart_interval()
    coef = np.zeros((nmcu * case.ncomp, 64), dtype=np.int64)
    for c in range(case.ncomp):
        blocks = gen_blocks(case.family, rng, nmcu, dct[td[c]], act[ta[c]])
        blocks[:, 0] = _integrate(blocks[:, 0], ri)
        coef[c::case.ncomp] = blocks
    marks = []
    jpg = JW.write_jpeg(coef, case.width, case.height, case.ncomp, qts, tq, dct, act, td, ta, comp_ids=(7, 3, 9),
                        interleaved=case.interleaved, restart_interval=ri, marks=marks)
    return jpg, tuple(marks)


def batch(case: Case, n: int = 3):
    """n files of one plan (same tables, size and interval), different content."""
    return [build(case, seed)[0] for seed in range(n)]


def scans_of(files):
    import libkpeg_b200 as K
    plan, scans = None, []
    for jpg in files:
        buf = np.frombuffer(jpg, dtype=np.uint8)
        plan, off, n = K.parse_jfif(buf)
        scans.append(buf[off:off + n])
    return plan, scans


# ---- what a stream contains, against the thresholds -----------------------------------------------------
def facts(case: Case) -> dict:
    """What the stream holds, from the writer's marks (no decoder involved)."""
    T = thresholds()
    jpg, marks = build(case)
    dct, act, td, ta, _, _ = _component_tables(case)
    f = {}
    codes = [(JW.canonical_codes(*dct[td[c]]), JW.canonical_codes(*act[ta[c]])) for c in range(case.ncomp)]
    lengths = {L for (_, _, _, _, L, _) in marks}
    f["code_lengths"] = lengths
    f["bits"] = max(b + L + s for b, _, _, _, L, s in marks)
    # canonical search: prefixes past the second-level table's capacity that the stream uses
    lb, cap = T["LUT_BITS"], T["LONG_CAP"] // T["SUB_SIZE"]
    used = set()
    for _, c, is_ac, sym, L, _ in marks:
        if L > lb:
            code = codes[c][is_ac][sym][0]
            tab = act[ta[c]] if is_ac else dct[td[c]]
            ranked = sorted(long_prefixes(tab))
            if ranked.index(code >> (L - lb)) >= cap:
                used.add((c, is_ac, code >> (L - lb)))
    f["canonical_prefixes_used"] = len(used)
    # value symbols (records) per window of sub_bits bits, most of any window
    starts = np.array([b for b, _, _, _, _, s in marks if s], dtype=np.int64)
    f["max_records"] = {sb: int(np.bincount(starts // sb).max()) if starts.size else 0 for sb in (64, 96, 512, 1024)}
    # 27-bit symbols: offsets mod 32, and whether one crosses a 64-bit subsequence boundary
    s27 = [b for b, _, _, _, L, s in marks if L + s == 27]
    f["offsets27"] = {b % 32 for b in s27}
    f["s27_cross64"] = any(b // 64 != (b + 26) // 64 for b in s27)
    f["all_ones"] = [all_ones_symbol(dct[td[c]]) for c in range(case.ncomp)]
    f["declared_max_category"] = max(s & 15 for tabs in (dct, act) for t in tabs.values() for s in t[1][:int(sum(t[0]))])
    f["used_max_category"] = max(s for *_, s in marks)
    return f
