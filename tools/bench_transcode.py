"""Lossless transcode on the GPU (kpeg_cuda_transcode): host buffers in and out (pinned), a host clock around the
synchronous calls.  Prints one JSON document.

    python tools/bench_transcode.py [--steps K] [--warmup W] [--out FILE]

Workloads (synthetic files, the bench's content):
  a  3840x2160 RGB q95, no restart markers (bench.py's image 0), --optimize
  b  the same, restart interval of one MCU row (480 MCUs): the markers banded and multi-GPU decodes need
  c  the same, rot90
  d  1920x1080 RGB q90 with DRI 16, --optimize, interval kept
  e  512x512 gray q90
For each: ms per file and input MB/s (end to end, host clock), output size / input size, and from a separate pass with
profiling on the stage split the library reports (the decode's K0..K2 slots; the gather TG plus the coded stages in the
`idct` slot), with TG's kernel time from torch.profiler against the bytes it moves (128 B read + 2 B, 130 B written
per block).  Two comparisons: the decode-side stages of (a) against a plain T.81 decode of the same file, and the coded
stages (the `idct` slot minus TG) against the encoder's bit lengths + emission + stuffing (+ histogram and table build)
for the same geometry and tables.  Where several GPUs are visible, (b) also times decode_file_tiled of its output on
all of them against the single-GPU decode of its input.  The card's name and power limit come from an nvidia-smi query.
Inputs and outputs stay in host memory, so the end-to-end figures include both PCIe copies."""
from __future__ import annotations

import argparse
import json
import subprocess
import sys
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))

import numpy as np  # noqa: E402

import libkpeg_b200 as K  # noqa: E402
from libkpeg_b200 import api  # noqa: E402
from libkpeg_b200.synth import EMIT_RESTART, QUIRK_FREE, GRAY_CONTENT, SynthParams, synth_encode, synth_pixels  # noqa: E402

SEED0 = 0x6B706567  # bench.py's image 0
DECODE_STAGES = ("memset", "unstuff", "entropy_cold", "entropy_relay", "entropy_scan", "entropy_write", "relay_sparse")
ENCODE_CODED = ("entropy_scan", "entropy_write", "unstuff")  # the encoder's EH/EB, E3 + E4, E5 slots


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                             text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power = [s.strip() for s in out.split(",")]
        return {"name": name, "power_limit": power}
    except Exception as e:  # noqa: BLE001
        return {"name": "unknown", "power_limit": "unknown", "error": str(e)}


def workloads():
    sp4k = SynthParams(3840, 2160, quality=95, seed=SEED0, flags=QUIRK_FREE)
    a = synth_encode(sp4k).tobytes()
    d = synth_encode(SynthParams(1920, 1080, quality=90, restart_interval=16, flags=QUIRK_FREE | EMIT_RESTART, seed=5)).tobytes()
    e = synth_encode(SynthParams(512, 512, file_components=1, quality=90, flags=QUIRK_FREE | GRAY_CONTENT, seed=6)).tobytes()
    return [
        ("a_4k_q95_optimize", a, dict(optimize=True)),
        ("b_4k_q95_restart_row", a, dict(restart_interval=480)),
        ("c_4k_q95_rot90", a, dict(transform=K.KPEG_XFORM_ROT90)),
        ("d_1080p_q90_dri16_optimize", d, dict(optimize=True)),
        ("e_512_gray_q90", e, dict()),
    ], sp4k


def pinned_copy(data: bytes):
    p = api.PinnedArray(len(data))
    p.array[:] = np.frombuffer(data, np.uint8)
    return p


def tg_kernel_ms(dec, src, out, kw, reps=5):
    """Mean tc_gather_kernel time in ms (torch.profiler, CUDA activities)."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            dec.transcode_into(src, out, **kw)
        torch.cuda.synchronize()
    tg = [e for e in prof.events() if "tc_gather_kernel" in e.name]
    return sum(e.device_time for e in tg) / 1000.0 / max(len(tg), 1) if tg else None


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", type=str, default="")
    args = ap.parse_args()
    info = {"gpu": gpu_info(), "steps": args.steps, "warmup": args.warmup, "workloads": {}}
    wl, sp4k = workloads()
    dec = K.Decoder(0)
    for name, jpg, kw in wl:
        src = pinned_copy(jpg)
        cap = K.transcode_bound(jpg, **kw)
        out = api.PinnedArray(cap)
        for _ in range(args.warmup):
            n = dec.transcode_into(src.array, out.array, **kw)
        times = []
        for _ in range(args.steps):
            t0 = time.perf_counter()
            n = dec.transcode_into(src.array, out.array, **kw)
            times.append((time.perf_counter() - t0) * 1e3)
        result = bytes(out.array[:n])
        dec.set_profiling(True)
        stage = {k: 0.0 for k in api.Stats.STAGES}
        for _ in range(args.steps):
            dec.transcode_into(src.array, out.array, **kw)
            for k, v in dec.last_stats.stage_ms().items():
                stage[k] += v / args.steps
        launches = int(dec.last_stats.kernel_launches)
        dec.set_profiling(False)
        tg_ms = tg_kernel_ms(dec, src.array, out.array, kw)
        nblk = int(dec.last_stats.width + 7) // 8 * ((int(dec.last_stats.height) + 7) // 8) * int(dec.last_stats.ncomp)
        med = float(np.median(times))
        r = {
            "params": {k: int(v) if not isinstance(v, bool) else v for k, v in kw.items()},
            "input_bytes": len(jpg), "output_bytes": n, "output_over_input": n / len(jpg),
            "ms_per_file_median": med, "ms_per_file_min": float(np.min(times)), "input_MB_per_s": len(jpg) / med / 1e3,
            "stage_ms_profiled": stage, "kernel_launches": launches,
            "tg": {"blocks": nblk, "ms": tg_ms, "bytes": nblk * 260,
                   "GB_per_s": (nblk * 260 / (tg_ms * 1e-3) / 1e9) if tg_ms else None},
        }
        r["coded_stages_ms"] = stage["idct"] - (tg_ms or 0.0)
        if name.startswith("a_"):
            # the same file decoded plainly (T.81), its decode-side stages
            dec.set_profiling(True)
            dstage = {k: 0.0 for k in DECODE_STAGES}
            for _ in range(args.steps):
                dec.decode_file(jpg, flags=0)
                for k in DECODE_STAGES:
                    dstage[k] += dec.last_stats.stage_ms()[k] / args.steps
            r["plain_decode_stage_ms"] = dstage
            r["decode_side_transcode_ms"] = sum(stage[k] for k in DECODE_STAGES)
            r["decode_side_plain_ms"] = sum(dstage.values())
            # the encoder's coded stages for the same geometry and table mode
            px = synth_pixels(sp4k)
            estage = {k: 0.0 for k in ENCODE_CODED}
            for _ in range(args.steps):
                dec.encode(px, quality=95, flags=K.KPEG_FLAG_OPTIMIZE_HUFFMAN)
                for k in ENCODE_CODED:
                    estage[k] += dec.last_stats.stage_ms()[k] / args.steps
            dec.set_profiling(False)
            r["encoder_coded_stage_ms"] = estage
            r["encoder_coded_ms"] = sum(estage.values())
        if name.startswith("b_") and K.api.load_cuda_library().kpeg_cuda_device_count() > 1:
            ndev = K.api.load_cuda_library().kpeg_cuda_device_count()
            frame = np.empty((2160, 3840, 3), np.uint8)
            for _ in range(2):
                api.decode_file_tiled(list(range(ndev)), result, flags=0, out=frame)
                dec.decode_file(jpg, flags=0, out=frame)
            tt, ts = [], []
            for _ in range(args.steps):
                t0 = time.perf_counter()
                api.decode_file_tiled(list(range(ndev)), result, flags=0, out=frame)
                tt.append((time.perf_counter() - t0) * 1e3)
                t0 = time.perf_counter()
                dec.decode_file(jpg, flags=0, out=frame)
                ts.append((time.perf_counter() - t0) * 1e3)
            r["tiled_decode_of_output"] = {"devices": ndev, "ms_median": float(np.median(tt)),
                                           "single_gpu_decode_of_input_ms_median": float(np.median(ts))}
        info["workloads"][name] = r
        out.free()
        src.free()
    dec.close()
    text = json.dumps(info, indent=1)
    print(text)
    if args.out:
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        Path(args.out).write_text(text + "\n")


if __name__ == "__main__":
    main()
