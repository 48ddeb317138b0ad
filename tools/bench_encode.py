"""Throughput of the GPU baseline-JPEG encoder (kpeg_cuda_encode_device), device-resident: pixels already on the
device, the file assembled in device memory.  Prints one JSON document.

    python tools/bench_encode.py [--steps K] [--warmup W] [--out FILE]

Workloads (synth_pixels content):
  4k_rgb_q95   3840x2160 RGB, q95, no restart interval, 8 images per step
  1080p_q90    1920x1080 RGB, q90, restart interval 16
  512_gray_q90 512x512 gray, q90
For each: encode Gpixel/s and MB/s of output (host clock around synchronous calls), then -- in a separate pass with
profiling on -- the per-stage CUDA-event times the library reports (FDCT, DC nudge, bit lengths + emission, stuffing),
and the multi-threaded host reference encoder (kpeg_synth_encode_pixels) on the same pixels.  Also the card's name
and power limit (nvidia-smi query), which belong with the numbers."""
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
from libkpeg_b200.synth import EMIT_RESTART, QUIRK_FREE, SynthParams, synth_encode_pixels, synth_pixels  # noqa: E402

WORKLOADS = [
    ("4k_rgb_q95", 3840, 2160, 3, 95, 0, 8),
    ("1080p_q90", 1920, 1080, 3, 90, 16, 1),
    ("512_gray_q90", 512, 512, 1, 90, 0, 1),
]
STAGES = {"fdct": 8, "dc_nudge": 7, "bits_and_emit": 6, "stuffing": 2}  # KPEG_T_IDCT, _DC_SCAN, _ENTROPY_WRITE, _UNSTUFF


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                             text=True, timeout=60).stdout.strip().splitlines()[0]
        name, power = [s.strip() for s in out.split(",")]
        return {"name": name, "power_limit": power}
    except Exception as e:  # the numbers are still reported; the card is then unknown
        return {"name": "unknown", "power_limit": "unknown", "error": str(e)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", type=str, default=None)
    a = ap.parse_args()
    dec = K.Decoder(device=0)
    results = {"card": card(), "steps": a.steps, "warmup": a.warmup, "workloads": {}}
    for name, w, h, nc, q, ri, per_step in WORKLOADS:
        sp = SynthParams(w, h, file_components=nc, quality=q, restart_interval=ri,
                         flags=QUIRK_FREE | (EMIT_RESTART if ri else 0), seed=0x6B706567)
        px = np.ascontiguousarray(synth_pixels(sp))
        cap = K.encode_bound(w, h, nc, q, ri)
        d_px, d_out = dec.device_alloc(px.nbytes), dec.device_alloc(cap)
        dec.h2d(d_px, px)
        args = dict(quality=q, restart_interval=ri)
        for _ in range(a.warmup):
            n = dec.encode_device(d_px, w, h, nc, d_out, cap, **args)
        t0 = time.perf_counter()
        for _ in range(a.steps * per_step):
            n = dec.encode_device(d_px, w, h, nc, d_out, cap, **args)
        dt = (time.perf_counter() - t0) / (a.steps * per_step)
        launches = dec.last_stats.kernel_launches
        # per-stage CUDA-event times (profiling adds events between stages: a separate pass)
        dec.set_profiling(True)
        stage_ms = {k: 0.0 for k in STAGES}
        total_ms = 0.0
        reps = max(3, a.steps // 2)
        for _ in range(reps):
            dec.encode_device(d_px, w, h, nc, d_out, cap, **args)
            for k, i in STAGES.items():
                stage_ms[k] += dec.last_stats.ms[i] / reps
            total_ms += dec.last_stats.ms_total / reps
        dec.set_profiling(False)
        got = np.empty(n, np.uint8)
        dec.d2h(got, d_out)
        t0 = time.perf_counter()
        ref = synth_encode_pixels(sp, px)
        host_s = time.perf_counter() - t0
        assert got.tobytes() == ref.tobytes(), f"{name}: GPU bytes differ from the host reference"
        dec.device_free(d_px)
        dec.device_free(d_out)
        results["workloads"][name] = {
            "width": w, "height": h, "ncomp": nc, "quality": q, "restart_interval": ri, "images_per_step": per_step,
            "bytes_out": int(n), "bits_per_pixel": round(n * 8 / (w * h), 3),
            "ms_per_image": round(dt * 1e3, 4), "gpixel_per_s": round(w * h / dt / 1e9, 3),
            "mb_per_s_out": round(n / dt / 1e6, 1), "bytes_in_plus_out_per_image": int(w * h * nc + n),
            "kernel_launches": int(launches),
            "stage_ms_profiled": {k: round(v, 4) for k, v in stage_ms.items()}, "kernels_ms_profiled": round(total_ms, 4),
            "host_reference_ms": round(host_s * 1e3, 1), "host_reference_threads": os.cpu_count(),
            "bytes_equal_host_reference": True,
        }
    dec.close()
    text = json.dumps(results, indent=1)
    print(text)
    if a.out:
        Path(a.out).parent.mkdir(parents=True, exist_ok=True)
        Path(a.out).write_text(text + "\n")


if __name__ == "__main__":
    main()
