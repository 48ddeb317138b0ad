"""TEST INFRASTRUCTURE: crafted coefficient fields that drive each reconstruction branch of K3
(libkpeg_b200/csrc/k3_fused.cu), and a float64 reference of the reconstruction that shares no code with the oracle
or with idct_core.h.

A field is [blocks][64] quantised coefficients -- MCU-interleaved, zig-zag order, DC values integrated, what the
oracle returns -- together with one quantiser table per component.  `encode` writes it as a baseline JPEG with the
Annex K Huffman tables (DC categories 0..11, all 162 AC symbols) through tests/jpeg_writer.py.

Families, each named after the branch it targets (A = sum of |dequantised coefficient| of a block):
  dc_only         DC-only blocks over the whole DC range at q = 1 and q = 255: the one-term shortcut, exact x.5 values
                  (F = 8 k + 4) and values next to them, and DC-only blocks with A above SAMPLE_SAFE_A (huge).
  exact_ties      terms only at natural positions (0,0), (0,4), (4,0), (4,4): every sample is
                  (+-F00 +- F04 +- F40 +- F44) / 8, an exact x.5 tie where the signed sum is 4 mod 8.  Whole-block
                  and quarter-block tie patterns, in one, two and three components of an MCU, arranged so that some
                  strips hold at most IDCT_TIE_LIST_CAP tied samples (tie records) and others more (resolved in K3).
  near_band       blocks found by a seeded hill-climb (+-1 steps on coefficients, per-coefficient quantisers): the
                  largest |fast - reference| / band, the reference value just outside the band, and a sample on which
                  the fast value rounds the other way than the reference (what the band exists to catch).
  wide_and_huge   A one quantum below and above COLOUR_SAFE_A and SAMPLE_SAFE_A in every component; a huge Y block
                  beside tied chroma blocks; the maximum-amplitude block (DC +-2047, every AC +-1023, q = 255).
  colour_lattice  constant (y, cb, cr) where G is an exact integer or 1.402 d / 1.772 d is, in COLOUR_PLAIN MCUs (the
                  per-row redo) and in COLOUR_GENERAL ones (a Y block with A > COLOUR_SAFE_A), plus MCUs with one or both
                  chroma blocks zero (COLOUR_FLAT).

Constraints every field meets:
  * SURVEY F1: in parity mode a block whose DC difference is 0 loses its AC terms.  No block with AC terms repeats the
    DC value of the previous block of its component (`avoid_f1` moves the DC of a DC-only predecessor); the tests
    check that the oracle's parity-mode coefficients are the field itself, so no family is silently emptied.
  * The thresholds (COLOUR_SAFE_A, SAMPLE_SAFE_A, IDCT_TIE_LIST_CAP, TIE_REL, TIE_ABS, COLOUR_FAST_RANGE) are read from
    the source text (`thresholds`), and the tests assert that their inputs straddle each of them: change a constant
    and the tests fail instead of testing nothing.

What valid 8-bit baseline streams cannot reach: the largest |sample| is about 1.9e6 (DC +-2047 and every AC +-1023 at
q = 255, all in phase at one sample), below 2^22, where RINT_MAGIC rounding stops being exact; `max_sample_bound`
computes it and a test keeps it below 2^22.

Known open question: an integrated DC value outside int16 (a run of +2047 differences) is truncated to int16 by the
oracle (oracle/kpeg_oracle.c, DC prediction).  Whether the original decoder does the same cannot be checked without
its sources, so no field integrates a DC value beyond +-2047.
"""
from __future__ import annotations

import ctypes as C
import functools
import math
import re
from dataclasses import dataclass, field
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
CSRC = ROOT / "libkpeg_b200" / "csrc"
STRIP_MCUS = 32  # IDCT_MCUS_PER_CTA: a strip is 32 consecutive MCUs of the job

# T.81 Figure A.6: zig-zag index -> natural index (row * 8 + column); written out, not derived, so that a wrong map
# shared by the oracle and idct_core.h would show up
ZZ_TO_NAT = np.array([0, 1, 8, 16, 9, 2, 3, 10, 17, 24, 32, 25, 18, 11, 4, 5, 12, 19, 26, 33, 40, 48, 41, 34, 27, 20,
                      13, 6, 7, 14, 21, 28, 35, 42, 49, 56, 57, 50, 43, 36, 29, 22, 15, 23, 30, 37, 44, 51, 58, 59, 52,
                      45, 38, 31, 39, 46, 53, 60, 61, 54, 47, 55, 62, 63])
NAT_TO_ZZ = np.argsort(ZZ_TO_NAT)


# ---- thresholds, from the source text ------------------------------------------------------------
def _constexpr(text: str, name: str) -> str:
    m = re.search(rf"constexpr\s+\w+\s+{name}\s*=\s*([^;]+);", text)
    assert m, f"{name} not found"
    return m.group(1)


def _eval_c(expr: str, env: dict) -> float:
    expr = re.sub(r"(\d(?:[\d.]*)(?:e[-+]?\d+)?)f\b", r"\1", expr)  # 1.5e-6f -> 1.5e-6
    return float(eval(expr, {"__builtins__": {}}, env))  # noqa: S307 -- constant expressions of our own sources


@functools.lru_cache(maxsize=None)
def thresholds() -> dict:
    core = (CSRC / "idct_core.h").read_text()
    k3 = (CSRC / "k3_fused.cu").read_text()
    kc = (CSRC / "kernels.cuh").read_text()
    t = {}
    for name in ("TIE_REL", "TIE_ABS", "COLOUR_FAST_RANGE", "COLOUR_G_BAND"):
        t[name] = _eval_c(_constexpr(core, name), t)
    for name in ("COLOUR_SAFE_A", "SAMPLE_SAFE_A"):
        t[name] = _eval_c(_constexpr(k3, name), t)
    t["IDCT_TIE_LIST_CAP"] = int(_eval_c(_constexpr(kc, "IDCT_TIE_LIST_CAP"), t))
    assert int(_eval_c(_constexpr(kc, "IDCT_MCUS_PER_CTA"), t)) == STRIP_MCUS
    return t


# ---- float64 reference --------------------------------------------------------------------------
def _basis() -> np.ndarray:
    """B[x, u] = C_u cos((2x + 1) u pi / 16) / 2 (orthonormal 8-point DCT-III)."""
    x = np.arange(8)[:, None]
    u = np.arange(8)[None, :]
    c = np.where(u == 0, 1.0 / math.sqrt(2.0), 1.0)
    return c * np.cos((2 * x + 1) * u * math.pi / 16.0) / 2.0


BASIS = _basis()


def dequantised(zz: np.ndarray, q: np.ndarray) -> np.ndarray:
    """[n][64] zig-zag coefficients, [64] zig-zag quantisers -> [n][8][8] dequantised, natural order (int64)."""
    zz = np.asarray(zz, dtype=np.int64).reshape(-1, 64)
    F = np.zeros_like(zz)
    F[:, ZZ_TO_NAT] = zz * np.asarray(q, dtype=np.int64)[None, :]
    return F.reshape(-1, 8, 8)


def exact_samples(zz, q) -> tuple[np.ndarray, np.ndarray]:
    """-> (samples [n][8][8] float64 before rounding and level shift, A [n] = sum |F| as an exact integer)."""
    F = dequantised(zz, q)
    s = np.einsum("xu,nuv,yv->nxy", BASIS, F.astype(np.float64), BASIS)
    return s, np.abs(F).reshape(F.shape[0], -1).sum(axis=1)


def round_half_away(v: np.ndarray) -> np.ndarray:
    return np.sign(v) * np.floor(np.abs(v) + 0.5)


def tie_distance(v: np.ndarray) -> np.ndarray:
    """distance from the nearest x.5"""
    return np.abs(v - (np.floor(v) + 0.5))


def ycc_to_rgb(y, cb, cr) -> np.ndarray:
    """The JFIF expression in double on unshifted integer samples, floor, clamp (operation order of the reference)."""
    Y = np.asarray(y, dtype=np.float64) + 128.0
    db = np.asarray(cb, dtype=np.float64)
    dr = np.asarray(cr, dtype=np.float64)
    r = np.floor(Y + 1.402 * dr)
    g = np.floor((Y - 0.344136 * db) - 0.714136 * dr)
    b = np.floor(Y + 1.772 * db)
    return np.clip(np.stack([r, g, b], axis=-1), 0, 255).astype(np.uint8)


def reference_pixels(f: "Field") -> tuple[np.ndarray, np.ndarray]:
    """-> (pixels [H][W] or [H][W][3], decided [H][W] bool).  A pixel is decided when every component sample lies
    further than 1e-6 A + 1e-5 from x.5: float64 and the reference's own evaluation then round it the same way."""
    nc, mx, my = f.ncomp, f.mcus_x, f.mcus_y
    comps, ok = [], np.ones((my * 8, mx * 8), dtype=bool)
    for c in range(nc):
        s, A = exact_samples(f.coef[c::nc], f.qt[c])
        far = tie_distance(s) > (1e-6 * A + 1e-5)[:, None, None]
        v = round_half_away(s)
        img = v.reshape(my, mx, 8, 8).transpose(0, 2, 1, 3).reshape(my * 8, mx * 8)
        ok &= far.reshape(my, mx, 8, 8).transpose(0, 2, 1, 3).reshape(my * 8, mx * 8)
        comps.append(img)
    if nc == 1:
        px = np.clip(comps[0] + 128.0, 0, 255).astype(np.uint8)
    else:
        px = ycc_to_rgb(*comps)
    return px[:f.height, :f.width], ok[:f.height, :f.width]


# ---- fields ---------------------------------------------------------------------------------------
@dataclass
class Field:
    name: str
    width: int
    height: int
    ncomp: int
    coef: np.ndarray  # [blocks][64] int16
    qt: list          # per component: 64 quantisers, zig-zag order
    notes: dict = field(default_factory=dict)

    @property
    def mcus_x(self):
        return (self.width + 7) // 8

    @property
    def mcus_y(self):
        return (self.height + 7) // 8


def block(terms: dict | None = None, dc: int = 0) -> np.ndarray:
    """terms {(row, col): value} in natural positions -> zig-zag block"""
    b = np.zeros(64, dtype=np.int64)
    b[0] = dc
    for (r, c), v in (terms or {}).items():
        b[NAT_TO_ZZ[r * 8 + c]] = v
    return b


def avoid_f1(coef: np.ndarray, ncomp: int) -> np.ndarray:
    """Make the DC differences of every component encodable and keep the F1 rule from dropping AC terms:
      * a difference beyond category 11 (|d| > 2047): a DC-only block moves toward its predecessor, or else the
        DC-only predecessor moves half way;
      * a block with AC terms whose DC equals the previous block's (SURVEY F1: its AC terms would be dropped in parity
        mode): the DC-only predecessor moves by 1 or 2.
    Blocks with AC terms are never changed; an arrangement that needs that is an error of the family."""
    coef = coef.copy()
    for c in range(ncomp):
        idx = list(range(c, coef.shape[0], ncomp))
        for k, b in enumerate(idx):
            prev = coef[idx[k - 1], 0] if k else 0
            pp = coef[idx[k - 2], 0] if k > 1 else 0
            cur = coef[b, 0]
            bad_cat = abs(int(cur) - int(prev)) > 2047
            bad_f1 = coef[b, 1:].any() and cur == prev
            if not (bad_cat or bad_f1):
                continue
            if bad_cat and not coef[b, 1:].any():  # a DC-only block moves itself toward its predecessor
                coef[b, 0] = int(prev) + int(np.clip(int(cur) - int(prev), -2047, 2047))
                continue
            assert k > 0 and not coef[idx[k - 1], 1:].any(), f"block {b}: needs a DC-only predecessor to move"
            if bad_cat:
                coef[idx[k - 1], 0] = (int(pp) + int(cur)) // 2
            else:
                for d in (1, -1, 2, -2):
                    v = prev + d
                    if abs(v) <= 2047 and v != pp and abs(int(v) - int(pp)) <= 2047:
                        coef[idx[k - 1], 0] = v
                        break
            prev = coef[idx[k - 1], 0]
            assert abs(int(cur) - int(prev)) <= 2047 and abs(int(prev) - int(pp)) <= 2047, f"block {b}"
            assert not (coef[b, 1:].any() and cur == prev), f"block {b}"
    return coef


def layout(name, mcus: list, width: int, height: int, ncomp: int, qt: list, seed: int, notes=None) -> Field:
    """MCUs (each a list of ncomp zig-zag blocks) in job order, the rest of the image filled with DC-only MCUs of
    random DC (no AC, so no tie and no F1 effect)."""
    mx, my = (width + 7) // 8, (height + 7) // 8
    n = mx * my
    assert len(mcus) <= n, (name, len(mcus), n)
    rng = np.random.default_rng(seed)
    coef = np.zeros((n * ncomp, 64), dtype=np.int64)
    for m in range(n):
        for c in range(ncomp):
            if m < len(mcus):
                coef[m * ncomp + c] = mcus[m][c]
            else:
                coef[m * ncomp + c, 0] = rng.integers(-60, 61)
    coef = avoid_f1(coef, ncomp)
    assert np.abs(coef[:, 0]).max() <= 2047 and np.abs(coef[:, 1:]).max() <= 1023
    return Field(name, width, height, ncomp, coef.astype(np.int16), [np.asarray(q, dtype=np.int64) for q in qt],
                 notes or {})


def _qtable(rng, lo, hi, dc=None):
    q = rng.integers(lo, hi + 1, size=64)
    if dc is not None:
        q[0] = dc
    return q


def dc_only(width, height, ncomp, seed=1) -> list[Field]:
    T = thresholds()
    out = []
    n = ((width + 7) // 8) * ((height + 7) // 8)
    for q00 in (1, 255):
        rng = np.random.default_rng(seed + q00)
        vals = [2047, -2047, 2046, -2046, 1, -1, 0, 4, -4, 12, -12, 3, 5, -3, -5, 2044, -2044, 2043, 2045]
        vals += [8 * k + 4 for k in rng.integers(-255, 255, size=24)]  # exact x.5 at q = 1
        vals += [8 * k + r for k in rng.integers(-255, 255, size=12) for r in (3, 5)]  # next to one
        huge_dc = int(T["SAMPLE_SAFE_A"] // q00)  # A = |DC| q straddles SAMPLE_SAFE_A (reachable at q = 255 only)
        if huge_dc < 2047:
            vals += [huge_dc, huge_dc + 1, -huge_dc, -huge_dc - 1, huge_dc + 2, -huge_dc + 1]
        vals = [v for v in vals if abs(v) <= 2047]
        need = n * ncomp
        rest = rng.permutation(np.arange(-2047, 2048))[:max(0, need - len(vals))]
        vals = np.array(vals + list(rest))[:need]
        # each component's values in ascending order: every DC difference within category 11
        vals = np.stack([np.sort(vals[c::ncomp]) for c in range(ncomp)], axis=1).reshape(-1)
        mcus = [[block(dc=int(vals[m * ncomp + c])) for c in range(ncomp)] for m in range(n)]
        qt = [np.full(64, 1 + (c * 7) % 5) for c in range(ncomp)]
        for q in qt:
            q[0] = q00
        out.append(layout(f"dc_only_q{q00}", mcus, width, height, ncomp, qt, seed))
    return out


# tie patterns at q = 1: samples (F00 + sc F04 + sr F40 + sr sc F44) / 8 with sc / sr the signs of the column / row
WHOLE_TIE = {(0, 4): 8, (4, 0): -16, (4, 4): 24}  # with F00 = 8 k + 4: all 64 samples are x.5
QUARTER_TIE = {(0, 4): 1, (4, 0): 1, (4, 4): 1}    # with F00 = 8 k + 1: 8 k + 4 where sc = sr = +1, else 8 k: 16 ties


def tie_block(kind: str, k: int) -> np.ndarray:
    terms = WHOLE_TIE if kind == "whole" else QUARTER_TIE
    return block(terms, dc=8 * k + (4 if kind == "whole" else 1))


ODD_ROWS = (1, 2, 3, 5, 6, 7)  # frequencies whose cosines are irrational at every sample: no exact ties


def exact_ties(width, height, ncomp, seed=2) -> list[Field]:
    """Strips (32 MCUs) of four kinds: one whole-tie block (64 ties: records); one MCU with the quarter pattern in
    every component (16 pixels tied in all components: records carrying 3 flags, or 1 in gray); quarter patterns in
    two components (Cb and Cr: the record sits on Cb and carries Cr); whole-tie blocks in every MCU (thousands of ties:
    resolved in K3).  Non-tie filler: blocks with a few odd AC terms."""
    rng = np.random.default_rng(seed)
    cap = thresholds()["IDCT_TIE_LIST_CAP"]
    n = ((width + 7) // 8) * ((height + 7) // 8)

    count = [0]

    def filler():  # odd DC stepping through 600 values: never the DC of the previous block of its component
        count[0] += 1
        return block({(int(rng.choice(ODD_ROWS)), int(rng.choice(ODD_ROWS))): int(rng.integers(1, 9)) * 2 + 1},
                     dc=2 * ((37 * count[0]) % 600 - 300) + 1)

    mcus = []
    kinds = ["one_whole", "three_quarter", "two_quarter", "flood"]
    s = 0
    while len(mcus) + STRIP_MCUS <= n:
        kind = kinds[s % len(kinds)]
        strip = [[filler() for _ in range(ncomp)] for _ in range(STRIP_MCUS)]
        at = int(rng.integers(0, STRIP_MCUS))
        k = int(rng.integers(-30, 30))
        if kind == "one_whole":
            strip[at][int(rng.integers(0, ncomp))] = tie_block("whole", k)
        elif kind == "three_quarter":
            strip[at] = [tie_block("quarter", k + c) for c in range(ncomp)]
        elif kind == "two_quarter" and ncomp == 3:
            strip[at][1] = tie_block("quarter", k)
            strip[at][2] = tie_block("quarter", k - 3)
        elif kind == "flood":
            for m in range(0, STRIP_MCUS, 2):
                strip[m][m % ncomp] = tie_block("whole", int(rng.integers(-30, 30)))
        mcus += strip
        s += 1
    qt = [np.array([1] + [int(x) for x in rng.integers(1, 4, size=63)]) for _ in range(ncomp)]
    for q in qt:  # the tie positions at q = 1
        for r, c in ((0, 4), (4, 0), (4, 4)):
            q[NAT_TO_ZZ[r * 8 + c]] = 1
    return [layout("exact_ties", mcus, width, height, ncomp, qt, seed, notes=dict(tie_list_cap=cap))]


# ---- near_band: hill-climbed blocks ----------------------------------------------------------------
def _emu():
    import helpers as H
    lib = H.emu()
    lib.emu_idct_fast_k3.restype = C.c_float
    lib.emu_idct_fast_k3.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(C.c_float)]
    return lib


def fast_and_reference(zz: np.ndarray, q: np.ndarray):
    """-> (fast fp32 samples [64], reference-order float samples [64] before rounding, band, kernel A)"""
    import helpers as H
    lib, orc = _emu(), H.oracle()
    zz16 = np.ascontiguousarray(zz, dtype=np.int16)
    q16 = np.ascontiguousarray(q, dtype=np.uint16)
    fast = np.zeros(64, dtype=np.float32)
    a = C.c_float()
    band = lib.emu_idct_fast_k3(zz16.ctypes.data, q16.ctypes.data, fast.ctypes.data, C.byref(a))
    F = np.zeros(64, dtype=np.int32)
    F[ZZ_TO_NAT] = zz16.astype(np.int32) * q16.astype(np.int32)
    ref = np.zeros(64, dtype=np.float32)
    orc.kpo_idct8x8(F.ctypes.data, ref.ctypes.data)
    return fast.astype(np.float64), ref.astype(np.float64), float(band), float(a.value)


def objective(kind: str, zz, q) -> float:
    fast, ref, band, _ = fast_and_reference(zz, q)
    err = np.abs(fast - ref)
    d = tie_distance(ref)
    if kind == "err":     # the largest |fast - reference| in band units
        return float(err.max() / band)
    if kind == "outside":  # a reference value just outside the band: 1 <= d / band <= 2, as close to 1 as possible
        r = d / band
        r = r[(r >= 1.0) & (r <= 2.0)]
        return float(-(r.min() - 1.0)) if r.size else -10.0
    # "flip": fast and reference on the two sides of the same x.5, as far from it as possible -- the margin the band
    # must have (|fast - h| = err - d when they straddle h)
    return float(((err - d) / band).max())


@functools.lru_cache(maxsize=None)
def hill_climb(kind: str, seed: int, qseed: int, steps: int = 600) -> tuple:
    """Seeded stochastic hill-climb with +-1 steps on single coefficients under a per-coefficient quantiser table.
    -> (zig-zag block, quantiser table, score) as tuples."""
    rng = np.random.default_rng(seed)
    q = _qtable(np.random.default_rng(qseed), 1, 40, dc=int(np.random.default_rng(qseed).integers(1, 20)))
    zz = np.zeros(64, dtype=np.int64)
    dens = int(rng.choice([6, 16, 63]))
    idx = rng.choice(63, size=dens, replace=False) + 1
    zz[idx] = rng.integers(-60, 61, size=dens)
    zz[0] = int(rng.integers(20, 200)) * (1 if rng.random() < 0.5 else -1)
    best = objective(kind, zz, q)
    for _ in range(steps):
        i = int(rng.integers(0, 64)) if rng.random() < 0.8 else int(rng.choice(np.nonzero(zz)[0]))
        d = 1 if rng.random() < 0.5 else -1
        zz[i] += d
        if zz[0] == 0 or abs(zz[i]) > (2047 if i == 0 else 1023):
            zz[i] -= d
            continue
        s = objective(kind, zz, q)
        if s >= best:
            best = s
        else:
            zz[i] -= d
    return tuple(int(v) for v in zz), tuple(int(v) for v in q), best


def near_band_blocks(qseed: int, n_each: int = 3):
    """-> [(kind, zz, score)] for one quantiser table (qseed)"""
    out = []
    for kind in ("err", "outside", "flip"):
        for s in range(n_each):
            zz, q, score = hill_climb(kind, 1000 * qseed + 17 * s + len(kind), qseed)
            out.append((kind, np.array(zz), score))
    return out, np.array(q)


def near_band(width, height, ncomp, seed=3) -> list[Field]:
    """The hill-climbed blocks of each component's table, in that component, every block twice (once negated), the
    rest of the MCU DC-only."""
    rng = np.random.default_rng(seed)
    per_comp, qt = [], []
    for c in range(ncomp):
        blocks, q = near_band_blocks(qseed=seed * 10 + c)
        per_comp.append([b for _, b, _ in blocks] + [-b for _, b, _ in blocks])
        qt.append(q)
    mcus = []
    for k in range(len(per_comp[0])):
        for c in range(ncomp):
            m = [block(dc=int(rng.integers(-500, 500)) | 1) for _ in range(ncomp)]
            m[c] = per_comp[c][k]
            mcus.append(m)
    return [layout("near_band", mcus, width, height, ncomp, qt, seed)]


# ---- wide_and_huge ----------------------------------------------------------------------------------
def straddle_pair(rng, q: np.ndarray, target: float):
    """Two blocks one coefficient step apart whose A = sum |c| q lies below and above `target`."""
    for _ in range(2000):
        zz = np.zeros(64, dtype=np.int64)
        idx = rng.choice(63, size=12, replace=False) + 1
        zz[idx] = rng.integers(-40, 41, size=12)
        zz[0] = int(rng.integers(50, 400)) * (1 if rng.random() < 0.5 else -1)
        A = int((np.abs(zz) * q).sum())
        # scale to just below the target, then one coefficient at a time up to it
        f = target / max(A, 1) * 0.97
        zz = np.round(zz * f).astype(np.int64)
        zz[0] = zz[0] or 1
        if np.abs(zz[0]) > 2047 or np.abs(zz[1:]).max() > 1023:
            continue
        j = int(idx[0])
        while (np.abs(zz) * q).sum() + q[j] <= target:
            zz[j] += 1 if zz[j] >= 0 else -1
        lo = zz.copy()
        hi = zz.copy()
        hi[j] += 1 if hi[j] >= 0 else -1
        A_lo, A_hi = int((np.abs(lo) * q).sum()), int((np.abs(hi) * q).sum())
        if A_lo < target < A_hi and abs(hi[j]) <= 1023:
            return lo, hi
    raise AssertionError(f"no block of 8-bit coefficients reaches A = {target} under this quantiser table")


def wide_and_huge(width, height, ncomp, seed=4) -> list[Field]:
    T = thresholds()
    rng = np.random.default_rng(seed)
    # Y: 255 everywhere (255 = -1 mod 8 keeps the tie patterns); chroma: 1 at the tie positions, random elsewhere
    qt = [np.full(64, 255)] + [_qtable(rng, 1, 60) for _ in range(1, ncomp)]
    for q in qt[1:]:
        q[NAT_TO_ZZ[[0, 4, 32, 36]]] = 1
    mcus = []

    def dc_mcu():
        return [block(dc=int(rng.integers(-300, 300)) * 2 + 1) for _ in range(ncomp)]

    for target in (T["COLOUR_SAFE_A"], T["SAMPLE_SAFE_A"]):
        for c in range(ncomp):
            for b in straddle_pair(rng, qt[c], target):  # same DC: a DC-only MCU between (F1)
                m = dc_mcu()
                m[c] = b
                mcus += [m, dc_mcu()]
    # a huge DC-only Y block (sample ~ 65000, beyond the 16 bits of a tie record) beside tied chroma, in a strip with
    # few ties (records, not the in-kernel path); in a strip of its own, a huge dense Y block beside tied chroma
    while len(mcus) % STRIP_MCUS:
        mcus.append(dc_mcu())
    strip = [dc_mcu() for _ in range(STRIP_MCUS)]
    strip2 = [dc_mcu() for _ in range(STRIP_MCUS)]
    if ncomp == 3:
        strip[3] = [block(dc=2047), tie_block("quarter", 2), tie_block("quarter", -5)]
        strip[9] = [block(dc=-2047), tie_block("quarter", 7), dc_mcu()[2]]
        hz, _ = straddle_pair(rng, qt[0], 4 * T["SAMPLE_SAFE_A"])
        strip2[20] = [hz, dc_mcu()[1], tie_block("quarter", 1)]
    else:
        strip[3] = [block(dc=2047)]
        strip[9] = [block(dc=-2047)]
    strip[27][0] = tie_block("quarter", 3)  # tied, not huge: its record must survive
    mcus += strip + strip2
    # maximum amplitude (Y is quantised by 255 throughout): DC +-2047, every AC +-1023, signs in phase at sample (0, 0) or seeded
    sgn = np.sign(np.concatenate([[1.0], BASIS[0, ZZ_TO_NAT[1:] // 8] * BASIS[0, ZZ_TO_NAT[1:] % 8]]))
    big = np.concatenate([[2047], np.full(63, 1023)]) * sgn
    rnd = np.concatenate([[-2047], rng.choice([-1023, 1023], size=63)])
    for b in (big, -big, rnd):
        m = dc_mcu()
        m[0] = b.astype(np.int64)
        mcus += [m, dc_mcu()]  # a DC-only block between: DC differences stay within category 11
    return [layout("wide_and_huge", mcus, width, height, ncomp, qt, seed)]


def max_sample_bound() -> float:
    """Largest |sample| any valid 8-bit baseline block can have: every coefficient at its category limit (DC 2047, AC
    1023) times q = 255, in phase at one sample."""
    w = np.abs(np.einsum("u,v->uv", BASIS[0], BASIS[0]))  # sample (0, 0) is as large as any
    lim = np.full((8, 8), 1023.0)
    lim[0, 0] = 2047.0
    return float((w * lim * 255.0).sum())


# ---- colour_lattice ----------------------------------------------------------------------------------
def lattice_points(limit: int = 1023):
    """(cb, cr) with G = Y - 0.344136 cb - 0.714136 cr an exact integer, |cb|, |cr| <= limit; and the integer points
    of 1.402 d (d = 500 k) and 1.772 d (d = 250 k)."""
    g = [(cb, cr) for cb in range(-limit, limit + 1) for cr in range(-limit, limit + 1)
         if (43017 * cb + 89267 * cr) % 125000 == 0 and (cb, cr) != (0, 0)]
    rb = [(250 * k, 500 * j) for k in (-4, -3, -2, -1, 1, 2, 3, 4) for j in (-2, -1, 1, 2)]
    return g, rb


def colour_lattice(width, height, ncomp, seed=5) -> list[Field]:
    """DC-only MCUs with constant samples (y, cb, cr): quantiser DC entries 4 (Y) and 2 (chroma) make F00 = 8 s exact.
    COLOUR_GENERAL twins: the Y block gets an (0,4) term so that columns 0, 3, 4, 7 keep y and the others y - 600, and
    A > COLOUR_SAFE_A.  Then MCUs with Cb or Cr or both all-zero, and a Cb block (F00 = F04) whose samples are 0 on
    half the pixels beside a zero Cr block: flat pixels in a non-flat MCU."""
    assert ncomp == 3
    rng = np.random.default_rng(seed)
    qt = [np.ones(64, dtype=np.int64) for _ in range(3)]
    qt[0][0] = 4
    qt[1][0] = qt[2][0] = 4
    qt[0][NAT_TO_ZZ[4]] = 4
    g, rb = lattice_points()
    small = [p for p in g if max(abs(p[0]), abs(p[1])) <= 500]
    large = [p for p in g if max(abs(p[0]), abs(p[1])) > 500]
    pts = small + [p for p in rb if max(abs(p[0]), abs(p[1])) <= 500]
    pts += [large[i] for i in rng.choice(len(large), size=min(12, len(large)), replace=False)]
    pts += [p for p in rb if max(abs(p[0]), abs(p[1])) > 500][:8]
    ys = (-140, -3, 0, 5, 131, -128, 127)
    mcus = []

    def y_plain(y):  # F00 = 4 DC = 8 y
        return block(dc=2 * y)

    def y_general(y):  # F00 = 4 (y + y'), F04 = 4 (y - y'), y' = y - 600
        return block({(0, 4): 600}, dc=2 * y - 600)

    def ch(s):
        return block(dc=2 * s)

    for i, (cb, cr) in enumerate(pts):
        y = ys[i % len(ys)]
        mcus.append([y_plain(y), ch(cb), ch(cr)])
        if y < 92:
            mcus.append([y_general(y), ch(cb), ch(cr)])
    for y in ys:
        mcus.append([y_plain(y), ch(0), ch(37)])        # Cb zero
        mcus.append([y_plain(y), ch(-41), ch(0)])       # Cr zero
        mcus.append([y_plain(y), ch(0), ch(0)])         # both: COLOUR_FLAT
        mcus.append([y_general(min(y, 91)), ch(0), ch(0)])
        mcus.append([y_plain(y), block({(0, 4): 40}, dc=10), ch(0)])  # Cb 10 / 0 by column, Cr zero
        mcus.append([y_general(min(y, 91)), block({(0, 4): 60}, dc=15), ch(0)])
    n = ((width + 7) // 8) * ((height + 7) // 8)
    return [layout("colour_lattice", mcus[:n], width, height, ncomp, qt, seed, notes=dict(points=len(mcus)))]


FAMILIES = {
    "dc_only": dc_only,
    "exact_ties": exact_ties,
    "near_band": near_band,
    "wide_and_huge": wide_and_huge,
    "colour_lattice": colour_lattice,
}


def build(family: str, width: int, height: int, ncomp: int) -> list[Field]:
    return FAMILIES[family](width, height, ncomp)


# ---- encoding ----------------------------------------------------------------------------------------
@functools.lru_cache(maxsize=None)
def annex_k_tables():
    import jpeg_writer as JW
    import libkpeg_b200 as K
    from libkpeg_b200.synth import SynthParams, synth_encode
    plan, _, _ = K.parse_jfif(synth_encode(SynthParams(16, 16, quality=90)).tobytes())
    t = JW.tables_of(plan)
    return t[(0, 0)], t[(1, 0)]


def encode(f: Field) -> bytes:
    import jpeg_writer as JW
    dc, ac = annex_k_tables()
    qts = {c: [int(x) for x in f.qt[c]] for c in range(f.ncomp)}
    z = (0,) * f.ncomp
    return JW.write_jpeg(f.coef, f.width, f.height, f.ncomp, qts, tq=tuple(range(f.ncomp)), dc_tables={0: dc},
                         ac_tables={0: ac}, td=z, ta=z)


# ---- what a field contains, against the thresholds ------------------------------------------------------
def block_facts(f: Field) -> dict:
    """Per block: integer A, the kernel's fp32 A, DC-only, number of samples in the tie band (fast path) -- and per
    strip the tie count, per MCU the colour mode K3 picks."""
    T = thresholds()
    nb = f.coef.shape[0]
    A_int = np.zeros(nb)
    A_k = np.zeros(nb)
    ties = np.zeros(nb, dtype=np.int64)
    dc_only_ = ~f.coef[:, 1:].any(axis=1)
    for b in range(nb):
        c = b % f.ncomp
        fast, _, band, a = fast_and_reference(f.coef[b], f.qt[c])
        A_k[b] = a
        A_int[b] = float((np.abs(f.coef[b].astype(np.int64)) * f.qt[c]).sum())
        if not dc_only_[b] and a <= T["SAMPLE_SAFE_A"]:
            ties[b] = int((tie_distance(fast) < band).sum())
    huge = A_k > T["SAMPLE_SAFE_A"]
    wide = A_k > T["COLOUR_SAFE_A"]
    nz = A_k != 0
    nm = nb // f.ncomp
    mode = np.zeros(nm, dtype=np.int64)  # 0 plain, 1 flat, 2 general
    if f.ncomp == 3:
        w3, nz3 = wide.reshape(nm, 3), nz.reshape(nm, 3)
        mode = np.where(w3.any(axis=1), 2, np.where(nz3[:, 1:].any(axis=1), 0, 1))
    strip_ties = np.add.reduceat(ties.reshape(nm, f.ncomp).sum(axis=1), np.arange(0, nm, STRIP_MCUS))
    return dict(A_int=A_int, A_kernel=A_k, dc_only=dc_only_, huge=huge, wide=wide, ties=ties, mode=mode,
                strip_ties=strip_ties)


def describe(f: Field, facts: dict) -> str:
    T = thresholds()
    A = facts["A_kernel"]
    nt = facts["strip_ties"]
    cap = T["IDCT_TIE_LIST_CAP"]
    parts = [f"{f.name} {f.width}x{f.height}x{f.ncomp}:",
             f"blocks A<=COLOUR_SAFE_A {int((A <= T['COLOUR_SAFE_A']).sum())} / above {int((A > T['COLOUR_SAFE_A']).sum())}",
             f"A<=SAMPLE_SAFE_A {int((A <= T['SAMPLE_SAFE_A']).sum())} / above {int((A > T['SAMPLE_SAFE_A']).sum())}",
             f"dc-only {int(facts['dc_only'].sum())}",
             f"strips ties 1..{cap} {int(((nt > 0) & (nt <= cap)).sum())} / above {int((nt > cap).sum())} / none {int((nt == 0).sum())}"]
    if f.ncomp == 3:
        m = facts["mode"]
        parts.append(f"MCUs plain {int((m == 0).sum())} flat {int((m == 1).sum())} general {int((m == 2).sum())}")
    return "  ".join(parts)


# ---- the cases the tests run ----------------------------------------------------------------------------
SIZES = ((250, 44), (124, 60))  # W % 8 != 0 (byte stores); 32 and 16 MCUs per row (a strip is one row / two rows)


def cases():
    return [(fam, w, h, nc) for fam in FAMILIES for (w, h) in SIZES for nc in (3, 1)
            if not (fam == "colour_lattice" and nc == 1)]  # colour modes need colour


@functools.lru_cache(maxsize=None)
def fields_and_files(family: str, width: int, height: int, ncomp: int) -> tuple:
    """-> ((Field, jpeg bytes), ...), encoded once per session"""
    return tuple((f, encode(f)) for f in build(family, width, height, ncomp))


@functools.lru_cache(maxsize=None)
def facts_of(family: str, width: int, height: int, ncomp: int) -> tuple:
    return tuple(block_facts(f) for f, _ in fields_and_files(family, width, height, ncomp))


def reference_bound(zz: np.ndarray, q: np.ndarray) -> float:
    """Bound on |reference evaluation - exact value| (DESIGN.md "K3 rounding"): each of the nnz non-zero terms is
    rounded into a float partial sum bounded by A, plus the product and the final scaling: 0.25 (nnz + 2) A 2^-24."""
    zz = np.asarray(zz, dtype=np.int64)
    A = float((np.abs(zz) * np.asarray(q, dtype=np.int64)).sum())
    return 0.25 * (int(np.count_nonzero(zz)) + 2) * A * 2.0 ** -24


def narrow_batch(n_images: int = 5, width: int = 44, height: int = 20, seed: int = 6) -> list:
    """Images narrower than a strip (6 MCUs per row, 18 per image): a strip of 32 MCUs spans two or three images.
    Every image has a huge DC-only Y block beside tied chroma in its first MCU and a huge dense Y block beside tied
    chroma in its last, so tied and huge blocks sit on both sides of every image boundary inside a strip.  Image 2
    adds whole-tie blocks: the strips around it hold more ties than the list (resolved in K3), the others fewer
    (tie records)."""
    rng = np.random.default_rng(seed)
    qt = [np.full(64, 255), np.ones(64, dtype=np.int64), np.ones(64, dtype=np.int64)]
    n = ((width + 7) // 8) * ((height + 7) // 8)
    out = []
    for i in range(n_images):
        mcus = [[block(dc=int(rng.integers(-7, 8)) * 2 + 1) for _ in range(3)] for _ in range(n)]
        mcus[0] = [block(dc=2047 - i), tie_block("quarter", i), tie_block("quarter", -i - 2)]
        mcus[n - 1] = [block({(1, 1): 300 + i, (2, 3): -200}, dc=-900), tie_block("quarter", 5), block(dc=9)]
        if i in (0, 4):
            mcus[n - 2][2] = tie_block("quarter", -7)  # tied, in an MCU without a huge block: a tie record
        if i == 2:
            mcus[1][1] = tie_block("whole", 3)
            mcus[n // 2][2] = tie_block("whole", -4)
        f = layout(f"narrow_batch_{i}", mcus, width, height, 3, qt, seed + i)
        out.append((f, encode(f)))
    return out
