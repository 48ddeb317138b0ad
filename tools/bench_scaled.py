"""Reduced-size decode benchmark (KPEG_FLAG_SCALE_*): BASELINE.json configs[2] -- 8 synthetic 3840x2160 RGB 4:4:4 q95
JPEGs per step, no restart markers -- decoded at 1/1, 1/2, 1/4 and 1/8, the scales alternated step by step in one
process so that they share the clocks and the neighbours' load.

Two modes:
  device  scans resident in device memory, pixels to device memory (kpeg_cuda_decode_batch_packed_device_split)
  e2e     pinned host scans in, pinned host pixels out (kpeg_cuda_decode_batch: copies in, kernels, copies out)
Reported per scale and mode: median step time, Gpixel/s of INPUT pixels, MB of output per step.  A separate profiled run
(CUDA events after every stage, one lane) gives the per-stage split; the reconstruction kernel -- K3 at 1/1, the
reduced-size kernel otherwise -- is in ms["idct"].  For the reduced-size kernel, its algorithmic bytes (coefficient
tiles and quantisers read, pixels written) over that time.  The card's name and power limit come from an nvidia-smi
query in the same run.  Every scale's output is checked once against the C reference of tests/scaled_cases.py.

    python tools/bench_scaled.py [--steps 20] [--warmup 3] [--out result.json]
"""
from __future__ import annotations

import argparse
import json
import re
import subprocess
import sys
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
sys.path[:0] = [str(ROOT), str(ROOT / "tests")]

import libkpeg_b200 as K  # noqa: E402
from libkpeg_b200 import api  # noqa: E402
from libkpeg_b200.synth import QUIRK_FREE, SynthParams, synth_encode  # noqa: E402

SEED0 = 0x6B706567  # bench.py's image 0
W, H, Q, N = 3840, 2160, 95, 8
SCALES = (1, 2, 4, 8)
# MCUs per strip of the reconstruction kernels, read from the source they are built from
MCUS_PER_STRIP = int(re.search(r"constexpr\s+int\s+IDCT_MCUS_PER_CTA\s*=\s*(\d+);",
                               (ROOT / "libkpeg_b200" / "csrc" / "kernels.cuh").read_text()).group(1))


def card() -> dict:
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                             text=True, timeout=30).stdout.splitlines()[0]
        name, power = [s.strip() for s in out.split(",")]
        return {"name": name, "power_limit": power}
    except Exception as e:  # noqa: BLE001
        return {"name": "unknown", "power_limit": "unknown", "error": str(e)}


def kernel_bytes(scale: int, nc: int = 3) -> int:
    """What the reduced-size kernel has to move for one step: every strip's coefficient tile and the quantisers read,
    the output pixels written."""
    mcus = N * ((W + 7) // 8) * ((H + 7) // 8)
    strips = -(-mcus // MCUS_PER_STRIP)
    out = N * -(-W // scale) * -(-H // scale) * nc
    return strips * MCUS_PER_STRIP * nc * 128 + strips * nc * 256 + out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", type=str, default="")
    args = ap.parse_args()

    jpgs = [synth_encode(SynthParams(W, H, quality=Q, seed=SEED0 + i, flags=QUIRK_FREE)).tobytes() for i in range(N)]
    plan, _, _ = api.parse_jfif(jpgs[0])
    plan.flags = api.KPEG_FLAG_REF_PARITY
    scans = []
    for j in jpgs:
        _, off, ln = api.parse_jfif(j)
        scans.append(np.frombuffer(j, np.uint8)[off:off + ln].copy())
    plans = {s: api._scaled_plan(plan, s) for s in SCALES}
    nbytes = {s: int(np.prod(api.output_shape(plans[s]))) for s in SCALES}

    dec = K.Decoder(0)
    packed = api.pack_batch(scans)
    offs = api.packed_offsets(scans)
    d_in = dec.device_alloc(packed.size + 64)
    dec.h2d(d_in, packed)
    d_out = dec.device_alloc(nbytes[1] * N + 64)
    pin_in = [api.PinnedArray(s.size) for s in scans]
    for p, s in zip(pin_in, scans):
        p.array[:] = s
    pin_out = api.PinnedArray(nbytes[1] * N)

    def device_step(s):
        dec.decode_batch_packed_device_split(plans[s], N, d_in, offs, d_out)

    def e2e_step(s):
        one = nbytes[s]
        dec.decode_batch(plans[s], [p.array for p in pin_in], [pin_out.array[k * one:(k + 1) * one] for k in range(N)])

    # correctness, once per scale: images 0 and 7 against the C reference (1/1: against the plain full-size decode)
    import scaled_cases as SC
    checked = {}
    for s in SCALES:
        e2e_step(s)
        one = nbytes[s]
        for k in (0, N - 1):
            got = pin_out.array[k * one:(k + 1) * one]
            want = dec.decode_file(jpgs[k]) if s == 1 else SC.reference(jpgs[k], s, True)
            assert np.array_equal(got, want.reshape(-1)), f"1/{s} image {k} differs"
        checked[s] = True

    times = {m: {s: [] for s in SCALES} for m in ("device", "e2e")}
    for mode, step in (("device", device_step), ("e2e", e2e_step)):
        for _ in range(args.warmup):
            for s in SCALES:
                step(s)
        for _ in range(args.steps):
            for s in SCALES:
                t0 = time.perf_counter()
                step(s)  # synchronous: returns after the device work (and the copies out) are complete
                times[mode][s].append(time.perf_counter() - t0)

    prof = K.Decoder(0, profiling=True)
    stages = {}
    for s in SCALES:
        acc = None
        for i in range(args.warmup + args.steps):
            prof.decode_batch_packed_device(plans[s], N, d_in, packed.size, d_out)
            if i >= args.warmup:
                ms = prof.last_stats.stage_ms()
                acc = ms if acc is None else {k: acc[k] + ms[k] for k in ms}
        stages[s] = {k: round(v / args.steps, 4) for k, v in acc.items()}
        stages[s]["kernel_launches"] = int(prof.last_stats.kernel_launches)
    prof.close()

    res = {"tool": "tools/bench_scaled.py", "card": card(),
           "workload": f"{N} x synthetic {W}x{H} RGB 4:4:4 baseline q={Q}, no restart markers (BASELINE.json configs[2]) per step",
           "steps": args.steps, "warmup": args.warmup, "checked_against_reference": checked, "scales": {}}
    in_px = N * W * H
    for s in SCALES:
        r = {"output_mb_per_step": round(nbytes[s] * N / 1e6, 3), "stages_ms": stages[s]}
        for mode in ("device", "e2e"):
            med = float(np.median(times[mode][s]))
            r[mode] = {"median_step_ms": round(med * 1e3, 4), "min_step_ms": round(min(times[mode][s]) * 1e3, 4),
                       "gpixel_per_s_input": round(in_px / med / 1e9, 2)}
        if s > 1:
            kb = kernel_bytes(s)
            r["reduced_kernel"] = {"algorithmic_bytes": kb, "ms": stages[s]["idct"],
                                   "gb_per_s": round(kb / (stages[s]["idct"] * 1e-3) / 1e9, 1) if stages[s]["idct"] > 0 else None}
        res["scales"][f"1/{s}"] = r
    line = json.dumps(res)
    print(line)
    if args.out:
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        Path(args.out).write_text(json.dumps(res, indent=1) + "\n")
    for p in pin_in:
        p.free()
    pin_out.free()
    dec.device_free(d_in)
    dec.device_free(d_out)
    dec.close()


if __name__ == "__main__":
    main()
