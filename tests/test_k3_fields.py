"""The crafted coefficient fields of tests/coef_fields.py on the CPU: they encode what they claim (no family emptied by
the F1 rule), they straddle every threshold K3 branches on (read from the source text), the oracle agrees with an
independent float64 reconstruction wherever that decides a pixel, and the emulator of the kernel logic (tests/emu)
agrees with the oracle.  A failure here without a GPU points at idct_core.h or the host tables; one seen only by
tests/test_gpu_k3_branches.py points at device-only code in k3_fused.cu."""
import numpy as np
import pytest

import coef_fields as CF
import helpers as H

CASE_IDS = lambda c: f"{c[0]}-{c[1]}x{c[2]}x{c[3]}"  # noqa: E731


@pytest.mark.parametrize("case", CF.cases(), ids=CASE_IDS)
def test_oracle_reads_the_intended_field(case):
    """The parity-mode and T.81-mode coefficients are the field itself: no block lost its AC terms to F1."""
    for f, jpg in CF.fields_and_files(*case):
        for parity in (True, False):
            o = H.oracle_decode(jpg, parity=parity, want_pixels=False)
            assert np.array_equal(o["coef"], f.coef), f"{f.name} parity={parity}"


@pytest.mark.parametrize("case", CF.cases(), ids=CASE_IDS)
def test_oracle_against_float64_reconstruction(case):
    """Wherever no component sample lies within 1e-6 A + 1e-5 of x.5, the oracle's pixel is the float64 one."""
    for f, jpg in CF.fields_and_files(*case):
        o = H.oracle_decode(jpg, parity=True)
        px, decided = CF.reference_pixels(f)
        bad = o["pixels"] != px
        if f.ncomp == 3:
            bad = bad.any(axis=-1)
        assert decided.mean() > 0.2, f"{f.name}: too few pixels decided by float64"
        assert not (bad & decided).any(), f"{f.name}: {int((bad & decided).sum())} decided pixels differ"


@pytest.mark.parametrize("parity", [True, False], ids=["parity", "t81"])
@pytest.mark.parametrize("case", CF.cases(), ids=CASE_IDS)
def test_emulator_against_oracle(case, parity):
    for f, jpg in CF.fields_and_files(*case):
        o = H.oracle_decode(jpg, parity=parity)
        e = H.emu_decode(jpg, flags=1 if parity else 0)
        assert e["status"] == 0
        assert np.array_equal(o["coef"], e["coef"]), f.name
        assert np.array_equal(o["pixels"], e["pixels"]), f"{f.name}: {int((o['pixels'] != e['pixels']).sum())} bytes differ"


def test_narrow_batch_emulated_as_one_stream():
    fields = CF.narrow_batch()
    import libkpeg_b200 as K
    parsed = [K.parse_jfif(np.frombuffer(j, dtype=np.uint8)) for _, j in fields]
    scans = [np.frombuffer(j, dtype=np.uint8)[o:o + n] for (_, j), (_, o, n) in zip(fields, parsed)]
    e = H.emu_decode(None, scans=scans, plan=parsed[0][0])
    assert e["status"] == 0
    for i, (f, j) in enumerate(fields):
        assert np.array_equal(H.oracle_decode(j)["coef"], f.coef)
        assert np.array_equal(H.oracle_decode(j)["pixels"], e["pixels"][i]), f.name


def test_fields_straddle_every_threshold(capsys):
    """Each threshold K3 branches on has inputs on both sides of it; the counts are printed per field."""
    T = CF.thresholds()
    cap = T["IDCT_TIE_LIST_CAP"]
    lines = []
    seen = dict(ties_le_cap=0, ties_gt_cap=0, plain=0, flat=0, general=0, huge_dc_only=0, multi_comp_tie_mcus=0)
    for case in CF.cases():
        for (f, _), facts in zip(CF.fields_and_files(*case), CF.facts_of(*case)):
            lines.append(CF.describe(f, facts))
            nt = facts["strip_ties"]
            seen["ties_le_cap"] += int(((nt > 0) & (nt <= cap)).sum())
            seen["ties_gt_cap"] += int((nt > cap).sum())
            seen["huge_dc_only"] += int((facts["huge"] & facts["dc_only"]).sum())
            if f.ncomp == 3:
                for k, name in enumerate(("plain", "flat", "general")):
                    seen[name] += int((facts["mode"] == k).sum())
                tied = (facts["ties"].reshape(-1, 3) > 0).sum(axis=1)
                seen["multi_comp_tie_mcus"] += int((tied >= 2).sum())
            if f.name == "wide_and_huge":
                # per component: two blocks one coefficient step apart on either side of each A threshold
                A = facts["A_kernel"].reshape(-1, f.ncomp)
                for c in range(f.ncomp):
                    q = int(f.qt[c].max())
                    for t in (T["COLOUR_SAFE_A"], T["SAMPLE_SAFE_A"]):
                        assert ((A[:, c] > t - q) & (A[:, c] < t)).any(), (case, c, t, "below")
                        assert ((A[:, c] > t) & (A[:, c] < t + q)).any(), (case, c, t, "above")
                assert facts["A_int"].max() > 64 * 1023 * 255, "the maximum-amplitude block"
    with capsys.disabled():
        print("\n" + "\n".join(lines) + "\n" + repr(seen))
    for k, v in seen.items():
        assert v > 0, k


def test_largest_sample_stays_in_the_rounding_range():
    """RINT_MAGIC rounding ((x + M) - M) is exact for |x| < 2^22; no valid 8-bit baseline block comes near it, and the
    wide_and_huge field holds the block that comes nearest."""
    bound = CF.max_sample_bound()
    assert bound < 2 ** 22
    f = CF.build("wide_and_huge", 250, 44, 1)[0]
    s, _ = CF.exact_samples(f.coef, f.qt[0])
    assert np.abs(s).max() > 0.99 * bound


def _bound_blocks():
    """Dense blocks at full amplitude, sparse and dense random blocks, all with per-coefficient quantisers, and the
    hill-climbed worst cases."""
    rng = np.random.default_rng(12)
    out = []
    for trial in range(1500):
        q = rng.integers(1, 256, size=64) if trial % 3 else rng.integers(1, 9, size=64) * rng.integers(1, 32)
        dens = int(rng.choice([1, 3, 8, 20, 63]))
        amp = int(rng.choice([4, 40, 400, 1023]))
        zz = np.zeros(64, dtype=np.int64)
        idx = rng.choice(63, size=dens, replace=False) + 1
        zz[idx] = rng.integers(-amp, amp + 1, size=dens)
        zz[0] = rng.integers(-2047, 2048)
        out.append((zz, q))
    for _ in range(40):  # every coefficient at its limit
        zz = rng.choice([-1, 1], size=64) * np.concatenate([[2047], np.full(63, 1023)])
        out.append((zz, rng.integers(200, 256, size=64)))
    for qseed in range(30, 33):
        blocks, q = CF.near_band_blocks(qseed)
        out += [(b, q) for _, b, _ in blocks]
    return out


def test_tie_band_covers_fast_and_reference_errors():
    """The band K3 derives from A (fp32, accumulated as dequant_dezigzag does) covers:
      * the measured |fast - reference evaluation| with margin (worst ratio below 0.9), and
      * |fast - exact| plus the proven bound on the reference's own error, 0.25 (nnz + 2) A 2^-24: the band must hold
        for whatever rounding the reference's float accumulator does, not only for the blocks tried."""
    worst_measured = worst_proven = 0.0
    for zz, q in _bound_blocks():
        fast, ref, band, a = CF.fast_and_reference(zz, q)
        exact, A = CF.exact_samples(zz, q)
        assert abs(a - float(A[0])) <= 1e-5 * float(A[0]) + 1e-3, "the kernel's fp32 A"
        measured = float(np.abs(fast - ref).max())
        proven = float(np.abs(fast - exact.reshape(64)).max()) + CF.reference_bound(zz, q)
        assert measured <= band, (zz.tolist(), q.tolist(), measured, band)
        assert proven <= band, (zz.tolist(), q.tolist(), proven, band)
        worst_measured = max(worst_measured, measured / band)
        worst_proven = max(worst_proven, proven / band)
    assert worst_measured < 0.9
    assert worst_proven < 1.0


def test_hill_climb_reaches_the_targets():
    """The near_band blocks do what they are for: a reference value within 1..2 bands of x.5, and a sample on which the
    fast value and the reference lie on the two sides of one x.5."""
    blocks, q = CF.near_band_blocks(30)
    T = CF.thresholds()
    assert T["TIE_REL"] > 0 and T["TIE_ABS"] > 0
    outside = flip = 0
    for kind, zz, score in blocks:
        fast, ref, band, _ = CF.fast_and_reference(zz, q)
        d = CF.tie_distance(ref) / band
        outside += int(((d >= 1.0) & (d <= 2.0)).any())
        flip += int(((np.floor(fast + 0.5) != np.floor(ref + 0.5)) & (np.abs(fast - ref) > 0)).any())
    assert outside > 0 and flip > 0
