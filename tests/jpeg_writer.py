"""TEST INFRASTRUCTURE: a small pure-Python baseline-JPEG entropy coder.  It re-encodes a field of quantised
coefficients ([blocks][64], MCU-interleaved, zig-zag order, DC values integrated -- what the oracle returns) with
ANY assignment of quantiser / Huffman tables to components, so the tests can build files the committed C++
generator does not produce: three distinct quantiser tables, a Huffman table pair of its own for every component,
table ids in another order than the 0/1/1 of every common encoder, non-interleaved (one scan per component) files.
Only for small images: it is a Python loop per coefficient."""
from __future__ import annotations

import numpy as np


def canonical_codes(counts, symbols):
    """T.81 Annex C: symbol -> (code, length)."""
    out, code, k = {}, 0, 0
    for length in range(1, 17):
        for _ in range(int(counts[length - 1])):
            out[int(symbols[k])] = (code, length)
            code += 1
            k += 1
        code <<= 1
    return out


def permuted_table(counts, symbols, seed):
    """A different valid table with the same code lengths: symbols of equal code length shuffled."""
    rng = np.random.default_rng(seed)
    symbols = [int(s) for s in symbols[:int(sum(counts))]]
    out, k = [], 0
    for length in range(16):
        grp = symbols[k:k + int(counts[length])]
        k += int(counts[length])
        out += [grp[i] for i in rng.permutation(len(grp))]
    return list(int(c) for c in counts), out


class BitWriter:
    """bits: bits written so far, padding included -- the bit position in the scan once stuffed bytes and markers are
    taken out."""

    def __init__(self):
        self.out = bytearray()
        self.acc = 0
        self.n = 0
        self.bits = 0

    def put(self, code, length):
        self.acc = (self.acc << length) | (code & ((1 << length) - 1))
        self.n += length
        self.bits += length
        while self.n >= 8:
            b = (self.acc >> (self.n - 8)) & 0xFF
            self.out.append(b)
            if b == 0xFF:
                self.out.append(0x00)
            self.n -= 8
        self.acc &= (1 << self.n) - 1

    def flush(self):
        if self.n:
            self.put((1 << (8 - self.n)) - 1, 8 - self.n)

    def marker(self, m):
        """Pad to a byte with 1-bits (T.81 F.1.2.3) and write marker 0xFF m (RSTn)."""
        self.flush()
        self.out += bytes([0xFF, m])


def _category(v):
    return int(abs(int(v))).bit_length()


def _magnitude_bits(v, cat):
    v = int(v)
    return v if v >= 0 else v + (1 << cat) - 1


def encode_blocks(bw, blocks, dc_codes, ac_codes, pred, marks=None):
    """blocks: iterable of (component, int16[64]); pred: running DC predictors (list, updated in place).
    marks: a list that gets (bw.bits, component, is_ac, symbol, code length, category) of every symbol written."""
    def put(c, is_ac, sym, size):
        code = (ac_codes if is_ac else dc_codes)[c][sym]
        if marks is not None:
            marks.append((bw.bits, c, is_ac, sym, code[1], size))
        bw.put(*code)

    for c, blk in blocks:
        diff = int(blk[0]) - pred[c]
        pred[c] = int(blk[0])
        cat = _category(diff)
        put(c, False, cat, cat)
        if cat:
            bw.put(_magnitude_bits(diff, cat), cat)
        run = 0
        last = 0
        nz = np.nonzero(blk[1:])[0]
        last = int(nz[-1]) + 1 if nz.size else 0
        for z in range(1, last + 1):
            v = int(blk[z])
            if v == 0:
                run += 1
                continue
            while run > 15:
                put(c, True, 0xF0, 0)
                run -= 16
            cat = _category(v)
            put(c, True, (run << 4) | cat, cat)
            bw.put(_magnitude_bits(v, cat), cat)
            run = 0
        if last < 63:
            put(c, True, 0x00, 0)


def _seg(marker, payload):
    return bytes([0xFF, marker]) + (len(payload) + 2).to_bytes(2, "big") + bytes(payload)


def write_jpeg(coef, width, height, ncomp, qts, tq, dc_tables, ac_tables, td, ta, comp_ids=(1, 2, 3),
               interleaved=True, extra_segments=b"", scan_order=None, redefine=None, restart_interval=0, marks=None):
    """coef [blocks][64] (MCU-interleaved, zig-zag, DC integrated).  qts: {id: 64 values (zig-zag)};
    dc_tables / ac_tables: {id: (counts[16], symbols)}; tq / td / ta: table id per component.
    restart_interval: MCUs per interval (a DRI segment, RSTn markers after every interval, predictors reset, T.81
    F.1.2.3 / F.2.1.3.1); marks: see encode_blocks (bit positions count from the start of the scan they are in).
    Non-interleaved files only: scan_order = the components in the order their scans are written (default 0, 1, 2);
    redefine = {component: (dc_tables, ac_tables, td, ta)}: DHT segments written right before that component's scan
    (they REPLACE tables of the same id, T.81 B.2.4.2) and the selectors that scan uses."""
    coef = np.asarray(coef, dtype=np.int16).reshape(-1, 64)
    mx, my = (width + 7) // 8, (height + 7) // 8
    assert coef.shape[0] == mx * my * ncomp
    out = bytearray(b"\xff\xd8")
    out += _seg(0xE0, b"JFIF\0\x01\x01\0\0\x01\0\x01\0\0")
    out += extra_segments
    for qid, q in qts.items():
        out += _seg(0xDB, bytes([qid]) + bytes(int(x) for x in q))
    sof = bytes([8]) + height.to_bytes(2, "big") + width.to_bytes(2, "big") + bytes([ncomp])
    for c in range(ncomp):
        sof += bytes([comp_ids[c], 0x11, tq[c]])
    out += _seg(0xC0, sof)
    if restart_interval:
        out += _seg(0xDD, int(restart_interval).to_bytes(2, "big"))
    for cls, tabs in ((0, dc_tables), (1, ac_tables)):
        for tid, (counts, symbols) in tabs.items():
            n = int(sum(counts))
            out += _seg(0xC4, bytes([(cls << 4) | tid]) + bytes(int(x) for x in counts) + bytes(int(s) for s in symbols[:n]))
    dc_codes = [canonical_codes(*dc_tables[td[c]]) for c in range(ncomp)]
    ac_codes = [canonical_codes(*ac_tables[ta[c]]) for c in range(ncomp)]
    scans = [list(range(ncomp))] if interleaved else [[c] for c in (scan_order or range(ncomp))]
    td, ta = list(td), list(ta)
    for comps in scans:
        if redefine and not interleaved and comps[0] in redefine:
            c = comps[0]
            new_dc, new_ac, td[c], ta[c] = redefine[c]
            for cls, tabs in ((0, new_dc), (1, new_ac)):
                for tid, (counts, symbols) in tabs.items():
                    n = int(sum(counts))
                    out += _seg(0xC4, bytes([(cls << 4) | tid]) + bytes(int(x) for x in counts) + bytes(int(s) for s in symbols[:n]))
            dc_codes[c] = canonical_codes(*new_dc[td[c]]) if td[c] in new_dc else canonical_codes(*dc_tables[td[c]])
            ac_codes[c] = canonical_codes(*new_ac[ta[c]]) if ta[c] in new_ac else canonical_codes(*ac_tables[ta[c]])
        sos = bytes([len(comps)])
        for c in comps:
            sos += bytes([comp_ids[c], (td[c] << 4) | ta[c]])
        sos += bytes([0, 63, 0])
        out += _seg(0xDA, sos)
        bw = BitWriter()
        pred = [0] * ncomp
        nmcu = mx * my
        step = restart_interval or nmcu
        for i, m0 in enumerate(range(0, nmcu, step)):
            if m0:
                bw.marker(0xD0 + (i - 1) % 8)
                pred = [0] * ncomp
            encode_blocks(bw, ((c, coef[m * ncomp + c]) for m in range(m0, min(m0 + step, nmcu)) for c in comps), dc_codes,
                          ac_codes, pred, marks)
        bw.flush()
        out += bw.out
    out += b"\xff\xd9"
    return bytes(out)


def tables_of(plan):
    """{(class, id): (counts, symbols)} of a parsed plan (libkpeg_b200.api.Plan)."""
    out = {}
    for cls in range(2):
        for tid in range(4):
            if plan.ht_present[cls][tid]:
                h = plan.ht[cls][tid]
                counts = [int(x) for x in h.counts]
                out[(cls, tid)] = (counts, [int(s) for s in h.symbols[:sum(counts)]])
    return out


def distinct_tables_variant(jpg, oracle_decode, parse_jfif, seed=1):
    """Re-encode `jpg` (3-component 4:4:4) with three distinct quantiser tables (ids 2, 0, 1 for Y, Cb, Cr), a DC and
    an AC Huffman table of its own for every component (ids Y 1/2, Cb 0/0, Cr 2/1: none of them the 0/1/1 mapping)
    and component ids 7, 3, 9.  The coefficients are kept; the quantisers differ, so the pixels do."""
    plan, _, _ = parse_jfif(jpg)
    ref = oracle_decode(jpg, parity=False, want_pixels=False)
    t = tables_of(plan)
    dc_l, ac_l, dc_c, ac_c = t[(0, 0)], t[(1, 0)], t[(0, 1)], t[(1, 1)]
    qy = [int(x) for x in plan.qt[0]]
    qc = [int(x) for x in plan.qt[1]]
    qts = {2: qy, 0: qc, 1: [min(255, x + 1 + (i % 3)) for i, x in enumerate(qc)]}
    dc_tables = {1: dc_l, 0: dc_c, 2: permuted_table(*dc_c, seed=seed)}
    ac_tables = {2: ac_l, 0: ac_c, 1: permuted_table(*ac_l, seed=seed + 1)}
    return write_jpeg(ref["coef"], plan.width, plan.height, 3, qts, tq=(2, 0, 1), dc_tables=dc_tables,
                      ac_tables=ac_tables, td=(1, 0, 2), ta=(2, 0, 1), comp_ids=(7, 3, 9))
