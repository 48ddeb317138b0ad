"""Crop decode benchmark (kpeg_cuda_decode_crop*): what decoding only a rectangle saves against the full decode.

Workloads, the legs of each alternated step by step in one process so that they share the clocks and the neighbours' load:
  (a) 8 synthetic 3840x2160 RGB 4:4:4 q95 JPEGs per step, no restart markers (BASELINE.json configs[2]): the full image,
      a 224x224 centre crop, a 1920x1080 centre crop and one MCU row (3840x8 at y = 1080).
        device  scans resident in device memory, pixels to device memory: 8 x kpeg_cuda_decode_device against
                8 x kpeg_cuda_decode_crop_device (one job each, lane 0)
        e2e     pinned host scans in, pinned host pixels out: kpeg_cuda_decode_batch against kpeg_cuda_decode_batch_crop
  (b) 4096 synthetic 512x512 gray q90 JPEGs per step, pinned host buffers: kpeg_cuda_decode_batch against
      kpeg_cuda_decode_batch_crop with a seeded random 224x224 rectangle per image.
  (c) a separately profiled pass (CUDA events after every stage, one image of (a) per call): K2 (ms["entropy_write"]) and
      K3 + patch (ms["idct"]) per leg, and the strips the crop lists against all strips.
Every leg's output is checked once against the full decode sliced.  The card's name and power limit come from an
nvidia-smi query in the same run.

    python tools/bench_crop.py [--steps 20] [--warmup 3] [--out result.json]
"""
from __future__ import annotations

import argparse
import json
import os
import re
import subprocess
import sys
import time
from concurrent.futures import ThreadPoolExecutor
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
sys.path[:0] = [str(ROOT)]

import libkpeg_b200 as K  # noqa: E402
from libkpeg_b200 import api  # noqa: E402
from libkpeg_b200.synth import GRAY_CONTENT, QUIRK_FREE, SynthParams, synth_encode  # noqa: E402

SEED0 = 0x6B706567  # bench.py's image 0
W, H, Q, N = 3840, 2160, 95, 8
GW, GN, GQ, GC = 512, 4096, 90, 224
MCUS_PER_STRIP = int(re.search(r"constexpr\s+int\s+IDCT_MCUS_PER_CTA\s*=\s*(\d+);",
                               (ROOT / "libkpeg_b200" / "csrc" / "kernels.cuh").read_text()).group(1))
LEGS = {"full": None, "centre_224": ((W - 224) // 2, (H - 224) // 2, 224, 224),
        "centre_1920x1080": ((W - 1920) // 2, (H - 1080) // 2, 1920, 1080), "one_mcu_row": (0, 1080, W, 8)}


def card() -> dict:
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                             text=True, timeout=30).stdout.splitlines()[0]
        name, power = [s.strip() for s in out.split(",")]
        return {"name": name, "power_limit": power}
    except Exception as e:  # noqa: BLE001
        return {"name": "unknown", "power_limit": "unknown", "error": str(e)}


def listed_strips(w, h, rect) -> int:
    """strips of MCUS_PER_STRIP MCUs that hold an MCU meeting the rectangle (full size, one image)"""
    mx = -(-w // 8)
    x, y, cw, ch = rect
    strips = set()
    for by in range(y // 8, (y + ch - 1) // 8 + 1):
        strips.update(range((by * mx + x // 8) // MCUS_PER_STRIP, (by * mx + (x + cw - 1) // 8) // MCUS_PER_STRIP + 1))
    return len(strips)


def split(jpg):
    plan, off, ln = api.parse_jfif(jpg)
    plan.flags = api.KPEG_FLAG_REF_PARITY
    return plan, np.frombuffer(jpg, np.uint8)[off:off + ln].copy()


def timed(legs: dict, warmup: int, steps: int) -> dict:
    for _ in range(warmup):
        for f in legs.values():
            f()
    t = {k: [] for k in legs}
    for _ in range(steps):
        for k, f in legs.items():
            t0 = time.perf_counter()
            f()  # synchronous: returns after the device work (and the copies out) are complete
            t[k].append(time.perf_counter() - t0)
    return {k: {"median_step_ms": round(float(np.median(v)) * 1e3, 4), "min_step_ms": round(min(v) * 1e3, 4)} for k, v in t.items()}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", type=str, default="")
    args = ap.parse_args()
    dec = K.Decoder(0)

    # ---- (a) 8 x 4K q95 -------------------------------------------------------------------------------------------
    jpgs = [synth_encode(SynthParams(W, H, quality=Q, seed=SEED0 + i, flags=QUIRK_FREE)).tobytes() for i in range(N)]
    plan, _ = split(jpgs[0])
    scans = [split(j)[1] for j in jpgs]
    full_bytes = W * H * 3
    d_scans = []
    for s in scans:
        d = dec.device_alloc(s.size + 64)
        dec.h2d(d, s)
        d_scans.append(d)
    d_out = dec.device_alloc(full_bytes * N + 64)
    pin_in = [api.PinnedArray(s.size) for s in scans]
    for p, s in zip(pin_in, scans):
        p.array[:] = s
    pin_out = api.PinnedArray(full_bytes * N)
    nbytes = {k: full_bytes if r is None else r[2] * r[3] * 3 for k, r in LEGS.items()}

    def device_leg(rect):
        def f():
            for k in range(N):
                dec.decode_device(plan, d_scans[k], scans[k].size, d_out + k * nbytes_of(rect), crop=rect)
        return f

    def nbytes_of(rect):
        return full_bytes if rect is None else rect[2] * rect[3] * 3

    def e2e_leg(rect):
        one = nbytes_of(rect)
        outs = [pin_out.array[k * one:(k + 1) * one] for k in range(N)]

        def f():
            dec.decode_batch(plan, [p.array for p in pin_in], outs, crops=None if rect is None else [rect] * N)
        return f

    checked = {}
    for k, r in LEGS.items():  # each leg once against the full decode sliced: images 0 and N - 1
        e2e_leg(r)()
        e2e = pin_out.array[:nbytes[k] * N].copy()
        device_leg(r)()
        dev = np.empty(nbytes[k] * N, np.uint8)
        dec.d2h(dev, d_out)
        for i in (0, N - 1):
            full = dec.decode_file(jpgs[i])
            want = full if r is None else full[r[1]:r[1] + r[3], r[0]:r[0] + r[2]]
            for got in (e2e, dev):
                assert np.array_equal(got[i * nbytes[k]:(i + 1) * nbytes[k]], want.reshape(-1)), f"{k} image {i} differs"
        checked[k] = True
    device = timed({k: device_leg(r) for k, r in LEGS.items()}, args.warmup, args.steps)
    e2e = timed({k: e2e_leg(r) for k, r in LEGS.items()}, args.warmup, args.steps)
    for p in pin_in:
        p.free()
    pin_out.free()
    dec.device_free(d_out)

    # ---- (c) stage times, profiled pass: one image per call, device-resident --------------------------------------
    prof = K.Decoder(0, profiling=True)
    d_one = prof.device_alloc(full_bytes + 64)
    stages = {}
    for k, r in LEGS.items():
        acc = None
        for i in range(args.warmup + args.steps):
            prof.decode_device(plan, d_scans[0], scans[0].size, d_one, crop=r)
            if i >= args.warmup:
                ms = prof.last_stats.stage_ms()
                acc = ms if acc is None else {s: acc[s] + ms[s] for s in ms}
        stages[k] = {s: round(v / args.steps, 4) for s, v in acc.items()}
        stages[k]["kernel_launches"] = int(prof.last_stats.kernel_launches)
    prof.device_free(d_one)
    prof.close()
    for d in d_scans:
        dec.device_free(d)
    all_strips = -(-((W + 7) // 8) * ((H + 7) // 8) // MCUS_PER_STRIP)

    # ---- (b) 4096 x 512x512 gray q90, a random 224x224 rectangle per image ----------------------------------------
    with ThreadPoolExecutor(max_workers=os.cpu_count() or 1) as ex:  # bench.py's gray images
        gj = list(ex.map(lambda i: synth_encode(SynthParams(GW, GW, file_components=1, quality=GQ, flags=QUIRK_FREE | GRAY_CONTENT,
                                                            seed=0xC30000 + i)).tobytes(), range(GN)))
    gplan, _ = split(gj[0])
    gscans = [split(j)[1] for j in gj]
    rng = np.random.default_rng(7)
    crops = [(int(rng.integers(0, GW - GC + 1)), int(rng.integers(0, GW - GC + 1)), GC, GC) for _ in range(GN)]
    gin = [api.PinnedArray(s.size) for s in gscans]
    for p, s in zip(gin, gscans):
        p.array[:] = s
    gout = api.PinnedArray(GW * GW * GN)
    full_outs = [gout.array[k * GW * GW:(k + 1) * GW * GW] for k in range(GN)]
    crop_outs = [gout.array[k * GC * GC:(k + 1) * GC * GC] for k in range(GN)]

    def gfull():
        dec.decode_batch(gplan, [p.array for p in gin], full_outs)

    def gcrop():
        dec.decode_batch(gplan, [p.array for p in gin], crop_outs, crops=crops)

    gfull()
    ref = [full_outs[k].reshape(GW, GW)[crops[k][1]:crops[k][1] + GC, crops[k][0]:crops[k][0] + GC].copy() for k in (0, GN - 1)]
    gcrop()
    for k, want in zip((0, GN - 1), ref):
        assert np.array_equal(crop_outs[k].reshape(GC, GC), want), f"gray batch image {k} differs"
    gray = timed({"full": gfull, "crop_224": gcrop}, args.warmup, args.steps)
    gray["checked_against_full"] = True
    for p in gin:
        p.free()
    gout.free()

    res = {"tool": "tools/bench_crop.py", "card": card(), "steps": args.steps, "warmup": args.warmup,
           "a_4k": {"workload": f"{N} x synthetic {W}x{H} RGB 4:4:4 baseline q={Q}, no restart markers, per step",
                    "legs": {k: {"rect_xywh": r, "output_mb_per_step": round(nbytes[k] * N / 1e6, 3),
                                 "device": device[k], "e2e_pinned": e2e[k]} for k, r in LEGS.items()},
                    "checked_against_full": checked},
           "c_stages_one_image": {"note": "profiled pass, separate from the timed steps; K2 = entropy_write, K3 + patch = idct",
                                  "all_strips": all_strips,
                                  "legs": {k: {"listed_strips": all_strips if r is None else listed_strips(W, H, r),
                                               "stages_ms": stages[k]} for k, r in LEGS.items()}},
           "b_gray_batch": {"workload": f"{GN} x synthetic {GW}x{GW} gray baseline q={GQ}, random {GC}x{GC} rectangle per image",
                            "legs": gray}}
    print(json.dumps(res))
    if args.out:
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        Path(args.out).write_text(json.dumps(res, indent=1) + "\n")
    dec.close()


if __name__ == "__main__":
    main()
