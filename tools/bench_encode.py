"""Throughput of the GPU baseline-JPEG encoder (kpeg_cuda_encode_device), device-resident: pixels already on the
device, the file assembled in device memory.  Prints one JSON document.

    python tools/bench_encode.py [--optimize] [--steps K] [--warmup W] [--out FILE]

Workloads (synth_pixels content):
  4k_rgb_q95   3840x2160 RGB, q95, no restart interval, 8 images per step
  1080p_q90    1920x1080 RGB, q90, restart interval 16
  512_gray_q90 512x512 gray, q90
For each: encode Gpixel/s and MB/s of output (host clock around synchronous calls), then -- in a separate pass with
profiling on -- the per-stage CUDA-event times the library reports (FDCT, DC nudge, bit lengths + emission, stuffing),
and the multi-threaded host reference encoder (kpeg_synth_encode_pixels) on the same pixels.  Also the card's name
and power limit (nvidia-smi query), which belong with the numbers.

--optimize: every workload twice, with the Annex K tables and with KPEG_FLAG_OPTIMIZE_HUFFMAN (the legs alternate
step by step, so they see the same machine state); the optimised leg adds the histogram + table-build stage
(`huffman_opt`), and each workload reports the file-size ratio optimised / Annex K."""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))

import numpy as np  # noqa: E402

import libkpeg_b200 as K  # noqa: E402
from libkpeg_b200.synth import EMIT_RESTART, OPTIMIZE_HUFFMAN, QUIRK_FREE, SynthParams, synth_encode_pixels, synth_pixels  # noqa: E402

WORKLOADS = [
    ("4k_rgb_q95", 3840, 2160, 3, 95, 0, 8),
    ("1080p_q90", 1920, 1080, 3, 90, 16, 1),
    ("512_gray_q90", 512, 512, 1, 90, 0, 1),
]
STAGES = {"fdct": 8, "dc_nudge": 7, "bits_and_emit": 6, "stuffing": 2}  # KPEG_T_IDCT, _DC_SCAN, _ENTROPY_WRITE, _UNSTUFF
OPT_STAGES = {**STAGES, "huffman_opt": 5}  # + KPEG_T_ENTROPY_SCAN


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                             text=True, timeout=60).stdout.strip().splitlines()[0]
        name, power = [s.strip() for s in out.split(",")]
        return {"name": name, "power_limit": power}
    except Exception as e:  # the numbers are still reported; the card is then unknown
        return {"name": "unknown", "power_limit": "unknown", "error": str(e)}


def leg(dec, a, w, h, nc, q, ri, per_step, px, d_px, d_out, cap, optimize, timed):
    """Times `timed` encodes (added to timed["s"]); then, once called with timed=None, the profiled stage times, the
    bytes and the host reference check."""
    flags = K.KPEG_FLAG_REF_PARITY | (K.KPEG_FLAG_OPTIMIZE_HUFFMAN if optimize else 0)
    args = dict(quality=q, restart_interval=ri, flags=flags)
    if timed is not None:
        t0 = time.perf_counter()
        for _ in range(per_step):
            timed["n"] = dec.encode_device(d_px, w, h, nc, d_out, cap, **args)
        timed["s"] += time.perf_counter() - t0
        timed["launches"] = dec.last_stats.kernel_launches
        return None
    stages = OPT_STAGES if optimize else STAGES
    dec.set_profiling(True)
    stage_ms = {k: 0.0 for k in stages}
    total_ms = 0.0
    reps = max(3, a.steps // 2)
    for _ in range(reps):
        n = dec.encode_device(d_px, w, h, nc, d_out, cap, **args)
        for k, i in stages.items():
            stage_ms[k] += dec.last_stats.ms[i] / reps
        total_ms += dec.last_stats.ms_total / reps
    dec.set_profiling(False)
    got = np.empty(n, np.uint8)
    dec.d2h(got, d_out)
    sp = SynthParams(w, h, file_components=nc, quality=q, restart_interval=ri,
                     flags=QUIRK_FREE | (EMIT_RESTART if ri else 0) | (OPTIMIZE_HUFFMAN if optimize else 0))
    t0 = time.perf_counter()
    ref = synth_encode_pixels(sp, px)
    host_s = time.perf_counter() - t0
    assert got.tobytes() == ref.tobytes(), f"{w}x{h} q{q} optimize={optimize}: GPU bytes differ from the host reference"
    return {"stage_ms_profiled": {k: round(v, 4) for k, v in stage_ms.items()}, "kernels_ms_profiled": round(total_ms, 4),
            "host_reference_ms": round(host_s * 1e3, 1), "host_reference_threads": os.cpu_count(),
            "bytes_equal_host_reference": True}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--optimize", action="store_true", help="also the KPEG_FLAG_OPTIMIZE_HUFFMAN leg, and the size ratio")
    ap.add_argument("--out", type=str, default=None)
    a = ap.parse_args()
    dec = K.Decoder(device=0)
    results = {"card": card(), "steps": a.steps, "warmup": a.warmup, "workloads": {}}
    modes = (False, True) if a.optimize else (False,)
    for name, w, h, nc, q, ri, per_step in WORKLOADS:
        sp = SynthParams(w, h, file_components=nc, quality=q, restart_interval=ri,
                         flags=QUIRK_FREE | (EMIT_RESTART if ri else 0), seed=0x6B706567)
        px = np.ascontiguousarray(synth_pixels(sp))
        cap = K.encode_bound(w, h, nc, q, ri, flags=K.KPEG_FLAG_REF_PARITY | (K.KPEG_FLAG_OPTIMIZE_HUFFMAN if a.optimize else 0))
        d_px, d_out = dec.device_alloc(px.nbytes), dec.device_alloc(cap)
        dec.h2d(d_px, px)
        common = (dec, a, w, h, nc, q, ri, per_step, px, d_px, d_out, cap)
        timed = {m: {"s": 0.0} for m in modes}
        for _ in range(a.warmup):
            for m in modes:
                leg(*common, m, {"s": 0.0})
        for _ in range(a.steps):
            for m in modes:
                leg(*common, m, timed[m])
        out = {}
        for m in modes:
            n, dt = timed[m]["n"], timed[m]["s"] / (a.steps * per_step)
            out[m] = {
                "width": w, "height": h, "ncomp": nc, "quality": q, "restart_interval": ri, "images_per_step": per_step,
                "bytes_out": int(n), "bits_per_pixel": round(n * 8 / (w * h), 3),
                "ms_per_image": round(dt * 1e3, 4), "gpixel_per_s": round(w * h / dt / 1e9, 3),
                "mb_per_s_out": round(n / dt / 1e6, 1), "mb_out": round(n / 1e6, 3),
                "bytes_in_plus_out_per_image": int(w * h * nc + n), "kernel_launches": int(timed[m]["launches"]),
                **leg(*common, m, None),
            }
        dec.device_free(d_px)
        dec.device_free(d_out)
        if a.optimize:
            results["workloads"][name] = {
                "annex_k": out[False], "optimized": out[True],
                "size_ratio_optimized_to_annex_k": round(out[True]["bytes_out"] / out[False]["bytes_out"], 4),
                "time_ratio_optimized_to_annex_k": round(out[True]["ms_per_image"] / out[False]["ms_per_image"], 3),
            }
        else:
            results["workloads"][name] = out[False]
    dec.close()
    text = json.dumps(results, indent=1)
    print(text)
    if a.out:
        Path(a.out).parent.mkdir(parents=True, exist_ok=True)
        Path(a.out).write_text(text + "\n")


if __name__ == "__main__":
    main()
