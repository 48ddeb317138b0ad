"""Optimised Huffman tables (KPEG_FLAG_OPTIMIZE_HUFFMAN) without a GPU: the table builder of csrc/huff_opt.h against an
independent Python implementation of T.81 Figures K.1-K.3 and against libjpeg-turbo's own optimised files, the CPU
replay of EH, EB and the device-written header against the reference encoder (KPEG_SYNTH_OPTIMIZE_HUFFMAN), coefficient
twins, the argument checks and the bound, and a pin on the synthetic encoder's output without the new flag."""
import ctypes as C
import hashlib
import io
import itertools

import numpy as np
import pytest

import encode_cases as EC
import encode_opt_cases as EO
import helpers as H
import libkpeg_b200 as K
from libkpeg_b200 import api
from libkpeg_b200.synth import OPTIMIZE_HUFFMAN, SynthParams, synth_encode

# ---- an independent builder, straight from T.81 Figures K.1 (code sizes), K.2 (BITS) and K.3 (length limit) -------
def py_optimal_table(freq):
    """freq: 256 counts -> (BITS [16], HUFFVAL, folded: whether a length over 16 was folded).  Figure K.1 with the
    reserved symbol 256 of frequency 1 and ties going to the larger symbol number; codesize via the OTHERS chains."""
    f = [int(x) for x in freq] + [1]
    codesize, others = [0] * 257, [-1] * 257
    while True:
        v1 = min((x for x in f if x), default=None)
        c1 = max(i for i in range(257) if f[i] == v1) if v1 is not None else -1
        rest = [f[i] for i in range(257) if f[i] and i != c1]
        if not rest:
            break
        v2 = min(rest)
        c2 = max(i for i in range(257) if f[i] == v2 and i != c1)
        f[c1] += f[c2]
        f[c2] = 0
        codesize[c1] += 1
        while others[c1] >= 0:
            c1 = others[c1]
            codesize[c1] += 1
        others[c1] = c2
        codesize[c2] += 1
        while others[c2] >= 0:
            c2 = others[c2]
            codesize[c2] += 1
    bits = [0] * 258
    for i in range(257):
        if codesize[i]:
            bits[codesize[i]] += 1
    folded = any(bits[17:])
    for i in range(257, 16, -1):  # Figure K.3
        while bits[i] > 0:
            j = i - 2
            while bits[j] == 0:
                j -= 1
            bits[i] -= 2
            bits[i - 1] += 1
            bits[j + 1] += 2
            bits[j] -= 1
    i = 16
    while i > 0 and bits[i] == 0:
        i -= 1
    if i > 0:
        bits[i] -= 1
    huffval = [s for L in range(1, 258) for s in range(256) if codesize[s] == L]
    return bits[1:17], huffval, folded


def c_optimal_table(freq):
    f = np.zeros(257, np.uint64)
    f[:256] = np.asarray(freq, dtype=np.uint64)
    bits, vals = np.zeros(16, np.uint8), np.zeros(256, np.uint8)
    n = EO.emu().emu_optimal_table(f.ctypes.data, bits.ctypes.data, vals.ctypes.data)
    return list(bits), list(vals[:n])


def code_lengths(bits, vals):
    """symbol -> length of the canonical code BITS / HUFFVAL give it"""
    lens, k = {}, 0
    for L in range(1, 17):
        for _ in range(bits[L - 1]):
            lens[vals[k]] = L
            k += 1
    return lens


def annex_k_lengths(t):
    """the Annex K code lengths of table t, read back from a reference file"""
    plan, _, _ = K.parse_jfif(EC.reference(np.zeros((8, 8, 3), np.uint8), 50, 0, False))
    spec = plan.ht[t & 1][t >> 1]
    return code_lengths(list(spec.counts), list(spec.symbols))


def check_invariants(freq, bits, vals, folded, annex_t=None):
    lens = code_lengths(bits, vals)
    used = [s for s in range(256) if freq[s]]
    assert sorted(lens) == used, "HUFFVAL holds exactly the symbols that occur"
    assert all(1 <= L <= 16 for L in lens.values())
    assert sum(2.0 ** -L for L in lens.values()) < 1.0, "Kraft sum below 1: no code is all ones"
    assert [(lens[s], s) for s in vals] == sorted((lens[s], s) for s in vals) or folded, "HUFFVAL by (length, symbol)"
    if annex_t is not None and not folded:
        ak = annex_k_lengths(annex_t)
        if all(s in ak for s in used):
            assert sum(int(freq[s]) * lens[s] for s in used) <= sum(int(freq[s]) * ak[s] for s in used) + 15


def fib(n, start=1):
    a, b, out = start, start, []
    for _ in range(n):
        out.append(a)
        a, b = b, a + b
    return out


def histograms():
    rng = np.random.default_rng(2024)
    cases = {}
    for k in range(6):
        h = np.zeros(256, np.uint64)
        nz = rng.choice(256, size=int(rng.integers(2, 200)), replace=False)
        h[nz] = rng.integers(1, 10 ** (k + 1), nz.size).astype(np.uint64)
        cases[f"random{k}"] = h
    cases["dc_like"] = np.array([900, 3000, 2500, 1800, 1200, 700, 300, 90, 20, 3, 1, 1] + [0] * 244, np.uint64)
    cases["equal_16"] = np.array([5] * 16 + [0] * 240, np.uint64)
    cases["equal_162"] = np.array([7] * 162 + [0] * 94, np.uint64)
    cases["equal_256"] = np.full(256, 3, np.uint64)
    cases["single"] = np.array([0] * 17 + [123456] + [0] * 238, np.uint64)
    cases["single_zero"] = np.array([1] + [0] * 255, np.uint64)
    cases["all_256_random"] = rng.integers(1, 1000, 256).astype(np.uint64)
    f40 = np.zeros(256, np.uint64)
    f40[rng.choice(256, 40, replace=False)] = fib(40)
    cases["fib40"] = f40
    f90 = np.zeros(256, np.uint64)
    f90[np.arange(90) * 2] = fib(90)  # depths far beyond 32, sums near 2^63
    cases["fib90"] = f90
    big = np.zeros(256, np.uint64)
    big[:100] = rng.integers(2 ** 32, 2 ** 40, 100).astype(np.uint64)
    big[100:110] = [1, 1, 2, 3, 5, 8, 13, 21, 34, 55]
    cases["above_2_pow_32"] = big
    return cases


@pytest.mark.parametrize("name", sorted(histograms()))
def test_builder_matches_figures_k1_to_k3(name):
    freq = histograms()[name]
    bits, vals = c_optimal_table(freq)
    pb, pv, folded = py_optimal_table(freq)
    assert bits == pb and vals == pv
    if name in ("fib40", "fib90"):
        assert folded
    check_invariants(freq, bits, vals, folded)


def symbol_histograms(coef, ncomp, restart_interval=0):
    """[4][256] symbol counts of zig-zag coefficients [blocks][64] (DC absolute, blocks MCU-interleaved), counted as
    T.81 F.1.2 codes them: table order DC luma, AC luma, DC chroma, AC chroma."""
    hist = np.zeros((4, 256), np.uint64)
    coef = np.asarray(coef, np.int64)
    nb = coef.shape[0]
    comp = np.arange(nb) % ncomp
    mcu = np.arange(nb) // ncomp
    prev = np.zeros(nb, np.int64)
    for c in range(ncomp):
        idx = np.nonzero(comp == c)[0]
        dc = coef[idx, 0]
        p = np.concatenate([[0], dc[:-1]])
        if restart_interval:
            p[mcu[idx] % restart_interval == 0] = 0
        prev[idx] = p
    diff = coef[:, 0] - prev
    cat = np.where(diff == 0, 0, np.floor(np.log2(np.maximum(np.abs(diff), 1))).astype(np.int64) + 1)
    for b in range(nb):
        t = 0 if comp[b] == 0 else 2
        hist[t, cat[b]] += 1
        run = 0
        for i in range(1, 64):
            v = int(coef[b, i])
            if v == 0:
                run += 1
                continue
            while run > 15:
                hist[t + 1, 0xF0] += 1
                run -= 16
            hist[t + 1, (run << 4) | abs(v).bit_length()] += 1
            run = 0
        if run:
            hist[t + 1, 0] += 1
    return hist


@pytest.mark.parametrize("kind,q", [("synth", 75), ("synth", 95), ("noise", 90), ("smooth", 50), ("gray", 85)])
def test_builder_equals_libjpeg_turbo(kind, q):
    """PIL's optimize=True files (PIL 12.2 is built on libjpeg-turbo 3.1; the same tie rule, so BITS and HUFFVAL match
    exactly): rebuild each table's histogram from the coefficients the oracle reads, run our builder, compare."""
    Image = pytest.importorskip("PIL.Image")
    rng = np.random.default_rng(q)
    if kind == "synth":
        px = EC.synth_content(232, 168, 3, seed=q)
    elif kind == "noise":
        px = rng.integers(0, 256, (96, 128, 3), dtype=np.uint8)
    elif kind == "smooth":
        y, x = np.mgrid[0:160, 0:200]
        px = np.stack([(x + y) % 256, (2 * x) % 256, (3 * y) % 256], -1).astype(np.uint8)
    else:
        px = EC.synth_content(200, 136, 1, seed=q)
    buf = io.BytesIO()
    Image.fromarray(px).save(buf, "JPEG", quality=q, optimize=True, subsampling=0)
    jpg = buf.getvalue()
    plan, _, _ = K.parse_jfif(jpg)
    ref = H.oracle_decode(jpg, parity=False, want_pixels=False)
    hist = symbol_histograms(ref["coef"], plan.ncomp)
    for t in range(4 if plan.ncomp == 3 else 2):
        comp = 0 if t < 2 else 1
        tid = (plan.comp_ta if t & 1 else plan.comp_td)[comp]
        spec = plan.ht[t & 1][tid]
        want_bits = list(spec.counts)
        want_vals = list(spec.symbols[:sum(want_bits)])
        bits, vals = c_optimal_table(hist[t])
        assert (bits, vals) == (want_bits, want_vals), (kind, q, t)


def _grid():
    for (w, h), nc in itertools.product(EC.SIZES, [1, 3]):
        yield w, h, nc


@pytest.mark.parametrize("w,h,nc", list(_grid()))
def test_cpu_replay_matches_the_reference(w, h, nc):
    px = EC.synth_content(w, h, nc, seed=w * 5 + h, noise_amp=0 if w < 100 else 30)
    for q, ri, parity in itertools.product(EC.QUALITIES, EC.restart_intervals(w), [True, False]):
        if w * h > 10000 and q not in (50, 100):
            continue
        got, info = EO.emu_encode(px, q, ri, parity)
        assert info[0] == 0, "a block overwrote a word another block owns"
        want = EO.reference(px, q, ri, parity)
        assert got == want, (q, ri, parity)
        assert len(got) <= K.encode_bound(w, h, nc, q, ri, flags=api.KPEG_FLAG_OPTIMIZE_HUFFMAN)


@pytest.mark.parametrize("name", sorted(EC.adversarial()))
@pytest.mark.parametrize("ri", [0, 5])
def test_cpu_replay_adversarial(name, ri):
    px, q = EC.adversarial()[name]
    for parity in (True, False):
        got, info = EO.emu_encode(px, q, ri, parity)
        assert info[0] == 0
        assert got == EO.reference(px, q, ri, parity)
        assert len(got) <= K.encode_bound(px.shape[1], px.shape[0], 3, q, ri, flags=api.KPEG_FLAG_OPTIMIZE_HUFFMAN)


@pytest.mark.parametrize("w,h,nc,q,ri", [(61, 37, 3, 50, 7), (200, 120, 1, 90, 0), (256, 192, 3, 95, 0), (64, 64, 3, 100, 1)])
def test_coefficient_twins(w, h, nc, q, ri):
    """The optimised and the Annex K reference files carry the same coefficients and decode to the same pixels."""
    px = EC.synth_content(w, h, nc, seed=q + ri)
    for parity in (True, False):
        opt = EO.reference(px, q, ri, parity)
        ak = EC.reference(px, q, ri, parity)
        assert opt != ak
        for mode in (True, False):
            a, b = H.oracle_decode(opt, parity=mode), H.oracle_decode(ak, parity=mode)
            assert np.array_equal(a["coef"], b["coef"]) and np.array_equal(a["pixels"], b["pixels"])


def test_optimised_tables_are_those_of_the_file():
    """Each DHT the reference writes is the builder's table for the symbol counts of the coefficients it codes, the
    DHT order and the rest of the header are the Annex K file's."""
    px = EC.synth_content(120, 80, 3, seed=8)
    opt = EO.reference(px, 80, 4, True)
    ak = EC.reference(px, 80, 4, True)
    p_opt, off_opt, _ = K.parse_jfif(opt)
    p_ak, off_ak, _ = K.parse_jfif(ak)
    assert bytes(p_opt.qt) == bytes(p_ak.qt) and p_opt.restart_interval == p_ak.restart_interval == 4
    hist = symbol_histograms(H.oracle_decode(opt, parity=True, want_pixels=False)["coef"], 3, 4)
    for t in range(4):
        spec = p_opt.ht[t & 1][t >> 1]
        bits, vals = c_optimal_table(hist[t])
        assert list(spec.counts) == bits and list(spec.symbols[:sum(bits)]) == vals
        check_invariants(hist[t], bits, vals, False, annex_t=t)
    # the same segments before the first DHT
    first_dht = ak.index(b"\xff\xc4")
    assert opt[:first_dht] == ak[:first_dht]


def test_argument_checks_for_the_new_flag():
    lib = K.load_cuda_library()
    n = C.c_size_t(0)
    buf = np.zeros(16, np.uint8)
    for flags in (2, 3):
        p = api.EncodeParams(16, 16, 3, 90, 0, flags)
        assert lib.kpeg_encode_bound(C.byref(p)) > 0
    for flags in (4, 8, 2 | 8, 16):
        bad = api.EncodeParams(16, 16, 3, 90, 0, flags)
        assert lib.kpeg_encode_bound(C.byref(bad)) == 0
        assert lib.kpeg_cuda_encode(None, C.byref(bad), buf.ctypes.data, buf.ctypes.data, 16, C.byref(n), None) == api.KPEG_ERR_ARG
    assert K.KPEG_FLAG_OPTIMIZE_HUFFMAN == 2 and OPTIMIZE_HUFFMAN == 16


@pytest.mark.parametrize("w,h,nc,ri", [(1, 1, 1, 0), (61, 37, 3, 7), (1920, 1080, 3, 0), (1920, 1080, 3, 1), (65535, 65535, 3, 0)])
def test_bound_with_the_flag(w, h, nc, ri):
    for q in (1, 90, 100):
        plain = K.encode_bound(w, h, nc, q, ri)
        opt = K.encode_bound(w, h, nc, q, ri, flags=api.KPEG_FLAG_OPTIMIZE_HUFFMAN | api.KPEG_FLAG_REF_PARITY)
        assert opt >= plain
        assert opt == EO.emu().emu_encode_bound_flags(w, h, nc, q, ri, 3)
        blocks = ((w + 7) // 8) * ((h + 7) // 8) * nc
        assert opt - plain == 2 * (-(-blocks * 1665 // 8) - -(-blocks * 1660 // 8))


def test_worst_streams_fit_the_flagged_bound():
    """q100 noise (1920 x 1080 included) and full-swing checkerboards, with a restart marker after every MCU: the
    files with optimised tables, whose blocks are the nearest to 1665 bits, fit the bound."""
    rng = np.random.default_rng(5)
    frames = [rng.integers(0, 256, (64, 64, 3), dtype=np.uint8), EC.adversarial(64, 64)["pixel_checkerboard"][0],
              rng.integers(0, 256, (33, 17), dtype=np.uint8), rng.integers(0, 256, (1080, 1920, 3), dtype=np.uint8)]
    for px in frames:
        h, w = px.shape[:2]
        nc = 1 if px.ndim == 2 else 3
        for ri in (0, 1) if w < 1000 else (0,):
            got = EO.reference(px, 100, ri, True)
            assert len(got) <= K.encode_bound(w, h, nc, 100, ri, flags=3)


# sha256 of kpeg_synth_encode's output before optimised tables were added: without the new flag it must not change
_PINS = [
    (dict(width=61, height=37, file_components=3, quality=75, restart_interval=0, flags=4, seed=3),
     "a509786fd2f7ca7424bf4b4d186cf52d4902bb684303a78826c882b50ab7355c"),
    (dict(width=200, height=120, file_components=1, quality=90, restart_interval=5, flags=5, seed=11),
     "737bbd99f9a132d53e35c4b4b514ee30d1168adcaf03772d2f6fb1a8c43c55a1"),
    (dict(width=333, height=221, file_components=3, quality=100, restart_interval=7, flags=1 | 4 | 8, seed=9, noise_amp=60),
     "70434849d04ce61a5bc97952260daa4ee76e182fbc2c588b46ec97796f295e13"),
    (dict(width=128, height=64, file_components=3, quality=30, restart_interval=16, flags=2 | 1, seed=2),
     "fd04fdf472a0db1a676d023f41dd939c65b6780850558fbfee5a18debab3f219"),
]


@pytest.mark.parametrize("params,digest", _PINS)
def test_synth_without_the_flag_is_unchanged(params, digest):
    assert hashlib.sha256(synth_encode(SynthParams(**params)).tobytes()).hexdigest() == digest
