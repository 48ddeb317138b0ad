#!/usr/bin/env python
"""bench.py -- decode throughput of the B200 baseline-JPEG hot path (BASELINE.json metric).

  python bench.py --gpus N --steps K --warmup W            # the CUDA path (this repo)
  python bench.py --impl reference --gpus N --steps K ...  # the reference's own CPU decoder

Workload (config.workload): BASELINE.json configs[2], the configuration the metric is quoted on --
synthetic 3840x2160 RGB 4:4:4 baseline JPEGs, q=95, NO restart markers (one entropy segment per
image, which forces the self-synchronising speculative Huffman decode).  One "step" decodes one
batch of `--batch` such images per GPU (distinct seeds; 8 by default: 51 MB of bit stream, 398 MB of
coefficients, 199 MB of pixels per step -- all far larger than the 126 MB L2, so no flush is needed
between iterations).  Images come from the committed deterministic encoder (libkpeg_b200/host/
synth_encoder.cpp); the reference's own encoder is non-functional.

  value  : whole-job Mpixel/s with the packed bit streams already resident in HBM and the pixels left
           in HBM (CUDA events on the decode stream, max over ranks).
  e2e    : the same metric through the host-pointer C-ABI call (kpeg_cuda_decode_batch) with pinned
           HOST buffers: packing, H2D of the bit streams and D2H of the pixels inside the timed region.
  roofline / kernels : per-kernel CUDA-event times from the timed region, algorithmic bytes per launch
           (DESIGN.md "Algorithmic bytes") and the fraction of the measured HBM peak.
  cpu_baseline : the compiled, unmodified reference (oracle/_ref/kpeg_ref_quiet) on the box's host
           cores, one process per core, on a bounded sample (512x512 images of the same generator).

  sustained : the device-resident leg repeated until at least 2 s have passed (the 20-step burst is 17 ms).
  gray_batch_4096 : BASELINE.json configs[3] -- 4096 synthetic 512x512 one-component JPEGs sharded over the ranks
           (contiguous index ranges), device-resident and end to end (pinned host scans in, ONE pinned frame of
           consecutive images out).
  tiles_16k : BASELINE.json configs[4] -- one 16384x16384 RGB image with a restart interval per MCU row, cut at its
           RSTn markers into one band of whole MCU rows per rank; end to end every rank's rows land in ITS slice of
           one host frame shared by the ranks (a host gather: no device-to-device traffic, no collective).
  parity : every image of every rank against the CPU oracle before timing (coefficients bit-exact, pixel
           max-abs-error and PSNR against the reference-exact oracle).

With torchrun (N > 1) every rank drives its own GPU on its own images (weak scaling, no collective in
the data path; torch.distributed is used only for the barrier, the max-over-ranks of the times and -- untimed
set-up of the tiles leg -- handing the encoded 16k image from rank 0 to the others).

  --dump-outputs DIR : after the timed steps, the RGB pixels the last timed step wrote, as float32: DIR/pixels.npy
           [rows, width, 3] holds a fixed, seeded sample of whole image rows (all of them when they fit in 56 MB) and
           DIR/pixels_rows.npy [rows, 2] float64 the (image, row) of each; with N > 1 every rank writes its own pair
           (pixels_rank<r>.npy, pixels_rank<r>_rows.npy).  The inputs depend on the arguments only, so two builds run
           with the same arguments can be compared file for file.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import threading
import time
from concurrent.futures import ThreadPoolExecutor
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tests"))

METRIC = "decode_mpixel_per_s"
UNIT = "Mpixel/s"
W4K, H4K, Q4K = 3840, 2160, 95
WORKLOAD = "synthetic 3840x2160 RGB 4:4:4 baseline q=95, no restart markers (BASELINE.json configs[2])"
SEED0 = 0x6B706567
REF_SAMPLE_WH = 512
DUMP_PIXEL_BYTES = 56 << 20  # the pixel sample of --dump-outputs; with its row index and headers it stays under 64 MB


def env_int(name, default):
    try:
        return int(os.environ.get(name, default))
    except ValueError:
        return default


def ncu_traffic(kernel, pixels):
    """DRAM bytes per launch of `kernel` (read + write) scaled from the committed ncu capture; None if absent."""
    try:
        with open(os.path.join(ROOT, "profiles", "ncu_traffic.json")) as f:
            t = json.load(f)
        k = t["kernels"][kernel]
        return (k["read_mb"] + k["write_mb"]) * 1e6 / t["pixels_per_captured_launch"] * pixels
    except (OSError, KeyError, ValueError):
        return None


def measured_peaks():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        try:
            d = json.loads(p.read_text())
            return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


# ---- clocks sampling -------------------------------------------------------------------------------
class ClockSampler:
    FIELDS = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu = gpu_index
        self.samples = []
        self._stop = threading.Event()
        self._t = None

    def _nvml_sample(self):
        pynvml, h, mx = self._nvml
        sm = pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM)
        rs = pynvml.nvmlDeviceGetCurrentClocksEventReasons(h) if hasattr(pynvml, "nvmlDeviceGetCurrentClocksEventReasons") \
            else pynvml.nvmlDeviceGetCurrentClocksThrottleReasons(h)
        pw = pynvml.nvmlDeviceGetPowerUsage(h) / 1000.0
        flags = ["Active" if rs & getattr(pynvml, n, 0) else "Not Active" for n in (
            "nvmlClocksThrottleReasonHwSlowdown", "nvmlClocksThrottleReasonHwThermalSlowdown",
            "nvmlClocksThrottleReasonSwThermalSlowdown", "nvmlClocksThrottleReasonSwPowerCap")]
        self.samples.append([str(sm), str(mx), str(pw), *flags])

    def _run(self):
        # NVML in-process (2 ms period; the handle is opened by start(), BEFORE the timed region: the headline region is
        # only ~17 ms long); falls back to polling nvidia-smi if pynvml is unavailable
        if self._nvml is not None:
            while not self._stop.is_set():
                try:
                    self._nvml_sample()
                except Exception:
                    break
                self._stop.wait(0.002)
            return
        while not self._stop.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--id={self.gpu}", f"--query-gpu={self.FIELDS}",
                                      "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5).stdout
                parts = [x.strip() for x in out.strip().split(",")]
                if len(parts) >= 7:
                    self.samples.append(parts)
            except Exception:
                pass
            self._stop.wait(0.2)

    def start(self):
        self._nvml = None
        try:
            import pynvml
            pynvml.nvmlInit()
            h = pynvml.nvmlDeviceGetHandleByIndex(self.gpu)
            self._nvml = (pynvml, h, pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM))
        except Exception:
            self._nvml = None
        self._t = threading.Thread(target=self._run, daemon=True)
        self._t.start()

    def stop(self):
        if self._nvml is not None:
            try:
                self._nvml_sample()  # one sample at the end of the region (the GPU is still under load: stop() is called before the final wait returns control for long)
            except Exception:
                pass
        self._stop.set()
        if self._t:
            self._t.join(timeout=6)
        sm, mx, reasons = [], 0.0, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for s in self.samples:
            try:
                sm.append(float(s[0]))
                mx = max(mx, float(s[1]))
            except ValueError:
                continue
            for nm, v in zip(names, s[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": mx or None, "reasons": sorted(reasons),
                "samples": len(sm)}


# ---- reference arm / cpu baseline ---------------------------------------------------------------------
def _ref_binary():
    p = ROOT / "oracle" / "_ref" / "kpeg_ref_quiet"
    return p if p.exists() and os.access(p, os.X_OK) else None


def _ref_decode_one(binary, jpg_bytes, workdir):
    d = tempfile.mkdtemp(dir=workdir)
    p = Path(d) / "img.jpg"
    p.write_bytes(jpg_bytes)
    subprocess.run([str(binary), str(p)], cwd=d, stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL, check=True)
    ok = (Path(d) / "img.ppm").exists()
    return ok


def _oracle_decode_one(jpg_bytes):
    import helpers as H
    H.oracle_decode(jpg_bytes, parity=True, want_pixels=True, threads=1)
    return True


def reference_step_runner(cores: int, build: str = "quiet"):
    """Returns (kind, run_step, pixels_per_step, sample_description).  One step = `cores` images of
    REF_SAMPLE_WH^2, one reference process per core (the reference is single-threaded and keeps
    decoder state in statics, so one process per image: SURVEY F5).  build = "quiet" (stock sources,
    log level ERROR in main()) or "debug" (the stock build as shipped: DEBUG logging to kpeg.log and stdout)."""
    from libkpeg_b200.synth import QUIRK_FREE, SynthParams, synth_encode
    jpgs = [synth_encode(SynthParams(REF_SAMPLE_WH, REF_SAMPLE_WH, quality=Q4K, seed=SEED0 + 1000 + i,
                                     flags=QUIRK_FREE)).tobytes() for i in range(cores)]
    binary = _ref_binary() if build == "quiet" else _ref_binary_debug()
    workdir = tempfile.mkdtemp(prefix="kpeg_ref_")
    pool = ThreadPoolExecutor(max_workers=cores)
    if binary is not None:
        kind = "reference"

        def run_step():
            assert all(pool.map(lambda j: _ref_decode_one(binary, j, workdir), jpgs))
    else:
        kind = "port"

        def run_step():
            assert all(pool.map(_oracle_decode_one, jpgs))
    what = {"quiet": "oracle/_ref/kpeg_ref_quiet: stock sources, log level ERROR",
            "debug": "oracle/_ref/kpeg_ref: the stock build, DEBUG logging, stdout to /dev/null"}[build]
    sample = (f"NOT the 4K workload: {cores} images {REF_SAMPLE_WH}x{REF_SAMPLE_WH} RGB 4:4:4 q={Q4K} no-RST from the same generator per step "
              f"(a 4K image costs the reference ~160 s: its unstuffing is O(n^2)), "
              f"one {'unmodified reference process (' + what + ')' if kind == 'reference' else 'oracle-port thread'} per core")
    return kind, run_step, cores * REF_SAMPLE_WH * REF_SAMPLE_WH, sample


def _ref_binary_debug():
    p = ROOT / "oracle" / "_ref" / "kpeg_ref"
    return p if p.exists() and os.access(p, os.X_OK) else None


class Reference4K:
    """ONE same-configuration figure for the reference: a single 3840x2160 q95 decode by the quiet build, started in the
    background when the bench starts (it takes ~160 s on one core) and collected at the end."""

    def __init__(self):
        self.proc = None
        self.t0 = None
        self.dir = None
        binary = _ref_binary()
        if binary is None:
            return
        from libkpeg_b200.synth import QUIRK_FREE, SynthParams, synth_encode
        self.dir = tempfile.mkdtemp(prefix="kpeg_ref4k_")
        (Path(self.dir) / "img.jpg").write_bytes(synth_encode(SynthParams(W4K, H4K, quality=Q4K, seed=SEED0, flags=QUIRK_FREE)).tobytes())
        self.t0 = time.perf_counter()
        self.proc = subprocess.Popen([str(binary), "img.jpg"], cwd=self.dir, stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)

    def collect(self, timeout_s=420):
        if self.proc is None:
            return None
        try:
            self.proc.wait(timeout=timeout_s)
        except subprocess.TimeoutExpired:
            self.proc.kill()
            return {"unavailable": f"not finished after {timeout_s} s"}
        dt = time.perf_counter() - self.t0
        ok = (Path(self.dir) / "img.ppm").exists()
        return {"value": W4K * H4K / dt / 1e6 if ok else None, "unit": UNIT, "cores": 1, "seconds": dt, "same_config": True,
                "sample": "ONE 3840x2160 q95 image of the bench workload (seed of image 0), quiet build, one process on one core, "
                          "run in the background while the GPU legs ran"}


def run_reference_arm(args):
    rank = env_int("RANK", 0)
    if rank != 0:
        return 0
    cores = os.cpu_count() or 1
    kind, run_step, px, sample = reference_step_runner(cores)
    for _ in range(max(args.warmup, 0)):
        run_step()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        run_step()
    dt = time.perf_counter() - t0
    value = px * args.steps / dt / 1e6
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32/f64 (CPU)", "data": "synthetic",
        "config": {"workload": WORKLOAD, "sample": sample},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": kind, "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)
    return 0



# ---- the other BASELINE configurations, at the same N ---------------------------------------------------------
def _max_over_ranks(torch, dist, device, seconds):
    t = torch.tensor([seconds], dtype=torch.float64, device=torch.device("cuda", device))
    if dist is not None:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t[0])


def leg_gray_batch(dec, K, rank, world, dist, device, torch, quick):
    """BASELINE.json configs[3]: 4096 synthetic 512x512 one-component baseline JPEGs, sharded over the ranks by contiguous
    index ranges (libkpeg_b200.shard.shard_range), no collective.  Device-resident: the rank's packed scans already in
    HBM, 1024 images per submission.  End to end: kpeg_cuda_submit_batch with pinned host scans in and ONE pinned
    frame of consecutive images out (copies inside the timed region)."""
    import helpers as H
    from libkpeg_b200.api import PinnedArray, pack_batch, packed_offsets
    from libkpeg_b200.shard import shard_range
    from libkpeg_b200.synth import GRAY_CONTENT, QUIRK_FREE, SynthParams, synth_encode
    total, side = (4096 if not quick else 256), 512
    total = int(os.environ.get("KPEG_BENCH_GRAY_TOTAL", total))  # development: a rank's share at N > 1, on one GPU
    idx = list(shard_range(total, rank, world))
    n = len(idx)
    threads = max(1, (os.cpu_count() or 1) // max(world, 1))

    def enc(i):
        return synth_encode(SynthParams(side, side, file_components=1, quality=90, flags=QUIRK_FREE | GRAY_CONTENT, seed=0xC30000 + i))

    with ThreadPoolExecutor(max_workers=threads) as ex:
        jpgs = list(ex.map(enc, idx))
    parsed = [K.parse_jfif(j) for j in jpgs]
    plan = parsed[0][0]
    plan.flags = K.KPEG_FLAG_REF_PARITY
    scans = [j[o:o + m] for j, (_, o, m) in zip(jpgs, parsed)]
    px = side * side
    # pinned host buffers: one arena of scans, one frame of images
    arena = PinnedArray(int(sum(s.size for s in scans)))
    in_views, o = [], 0
    for sc in scans:
        arena.array[o:o + sc.size] = sc
        in_views.append(arena.array[o:o + sc.size])
        o += sc.size
    frame = PinnedArray(n * px)
    out_views = [frame.array[i * px:(i + 1) * px].reshape(side, side) for i in range(n)]
    packed, offs = pack_batch(scans), packed_offsets(scans)
    d_in = dec.device_alloc(packed.size + 64)
    d_out = [dec.device_alloc(n * px + 64) for _ in range(2)]
    dec.h2d(d_in, packed)
    per_sub = 1024

    def run_device(reps):
        for r in range(reps):
            for a in range(0, n, per_sub):
                b = min(n, a + per_sub)
                dec.submit_batch_packed_device(plan, b - a, d_in + int(offs[a]), offs[a:b + 1] - offs[a], d_out[r & 1] + a * px)
        dec.wait()

    def sync():
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()

    reps = 5 if not quick else 2
    # the device-resident pass is short (a few ms per rep at N = 8): the same number of images per rank at every N, so that
    # neither filling the lanes nor a moment of host jitter on one rank (the time is the max over ranks) dominates
    dev_reps = 4 * reps * max(1, total // max(n, 1))
    # warm-up: every one of the context's eight lanes must have sized its scratch (a lane allocates at its first job)
    subs_per_rep = max(1, -(-n // per_sub))
    run_device(max(3, -(-16 // subs_per_rep)))
    sync()
    t0 = time.perf_counter()
    run_device(dev_reps)
    torch.cuda.synchronize()
    dev_s = _max_over_ranks(torch, dist, device, time.perf_counter() - t0)

    prepared = dec.prepare_batch(in_views, out_views)  # pointer arrays built once: the buffers are the same every rep

    def run_e2e(reps):
        for _ in range(reps):
            dec.submit_prepared(plan, prepared)
        dec.wait()

    run_e2e(max(2, -(-16 // max(1, min(8, n // max(1, per_sub // 8))))))  # the chunks of a submission rotate through the lanes
    sync()
    e2e_reps = reps * max(1, min(4, total // max(n, 1)))  # more repetitions where a rank's share is small (see dev_reps)
    t0 = time.perf_counter()
    run_e2e(e2e_reps)
    torch.cuda.synchronize()
    e2e_s = _max_over_ranks(torch, dist, device, time.perf_counter() - t0)
    # parity: a sample of this rank's images against the oracle, bit for bit (out_views hold the last end-to-end run)
    ok = True
    for i in sorted({0, n // 3, n - 1}):
        ok = ok and bool(np.array_equal(out_views[i], H.oracle_decode(jpgs[i].tobytes(), threads=threads)["pixels"]))
    okt = torch.tensor([1 if ok else 0], device=torch.device("cuda", device))
    if dist is not None:
        dist.all_reduce(okt, op=dist.ReduceOp.MIN)
    res = {"workload": f"{total} synthetic {side}x{side} one-component baseline JPEGs q=90 (BASELINE.json configs[3]), {n} per GPU (contiguous index ranges)",
           "device_resident_mpixel_per_s": total * px * dev_reps / dev_s / 1e6, "e2e_mpixel_per_s": total * px * e2e_reps / e2e_s / 1e6,
           "images_per_submission": min(per_sub, n), "reps": e2e_reps, "device_resident_reps": dev_reps, "scan_bytes_per_gpu": int(packed.size),
           "e2e_h2d_bytes_per_rep": int(arena.nbytes), "e2e_d2h_bytes_per_rep": int(n * px),
           "e2e_d2h_gbs_per_gpu": n * px * reps / e2e_s / 1e9,
           "pixels_match_oracle": bool(int(okt[0])), "checked": "3 images per rank, bit for bit, from the end-to-end run's host frame",
           "timer": "host clock around submit .. wait after a device sync and barrier, max over ranks"}
    for b in d_out + [d_in]:
        dec.device_free(b)
    arena.free()
    frame.free()
    return res


def leg_tiles(dec, K, rank, world, dist, device, torch, quick):
    """BASELINE.json configs[4]: one 16384x16384 RGB 4:4:4 image with a restart interval per MCU row, cut at its RSTn
    markers into one band of whole MCU rows per rank (kpeg_split_restart_bands); every GPU decodes its band.  End to
    end each rank's rows land in its slice of ONE host frame shared by the rank processes (/dev/shm mapping, the
    rank's slice pinned with kpeg_cuda_host_register): a host gather, no device-to-device traffic, no collective."""
    import helpers as H
    from libkpeg_b200.api import PinnedArray, load_cuda_library, pack_batch, packed_offsets
    from libkpeg_b200.shard import split_restart_bands
    from libkpeg_b200.synth import EMIT_RESTART, QUIRK_FREE, SynthParams, synth_encode
    side = 16384 if not quick else 2048
    lib = load_cuda_library()
    dev = torch.device("cuda", device)
    if rank == 0:
        jpg = synth_encode(SynthParams(width=side, height=side, quality=90, restart_interval=side // 8,
                                       flags=QUIRK_FREE | EMIT_RESTART, seed=5))
    if dist is not None:  # set-up, untimed: the encoded image from rank 0 to everybody
        nbytes = torch.tensor([jpg.size if rank == 0 else 0], dtype=torch.int64, device=dev)
        dist.broadcast(nbytes, 0)
        buf = torch.from_numpy(jpg).to(dev) if rank == 0 else torch.empty(int(nbytes[0]), dtype=torch.uint8, device=dev)
        dist.broadcast(buf, 0)
        jpg = buf.cpu().numpy()
        del buf
    plan, off, m = K.parse_jfif(jpg)
    plan.flags = K.KPEG_FLAG_REF_PARITY
    scan = jpg[off:off + m]
    band = split_restart_bands(plan, scan, world)[rank]
    nbytes_band = plan.width * band.rows * plan.ncomp
    packed, offs = pack_batch([band.scan]), packed_offsets([band.scan])
    d_in = dec.device_alloc(packed.size + 64)
    d_out = [dec.device_alloc(nbytes_band + 64) for _ in range(2)]
    dec.h2d(d_in, packed)

    def sync():
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()

    def run_device(k):
        for i in range(k):
            dec.submit_batch_packed_device(band.plan, 1, d_in, offs, d_out[i & 1])
        dec.wait()

    steps = 10 if not quick else 3
    run_device(10)
    sync()
    t0 = time.perf_counter()
    run_device(steps)
    torch.cuda.synchronize()
    dev_s = _max_over_ranks(torch, dist, device, time.perf_counter() - t0)

    # ONE host frame for all ranks
    path = f"/dev/shm/kpeg_bench_frame_{os.environ.get('MASTER_PORT', '0')}_{side}"
    frame_bytes = side * side * 3
    if rank == 0:
        with open(path, "wb") as f:
            f.truncate(frame_bytes)
    sync()
    frame = np.memmap(path, dtype=np.uint8, mode="r+", shape=(frame_bytes,))
    lo = band.row0 * plan.width * 3
    mine = frame[lo:lo + nbytes_band]
    pinned = nbytes_band > 0 and lib.kpeg_cuda_host_register(mine.ctypes.data, nbytes_band) == 0
    h_in = PinnedArray(band.scan.size)
    h_in.array[:] = band.scan
    # kpeg_cuda_decode on the rank's band: a large restart-marked image from host memory goes through the context's
    # lanes as sub-bands, so its copies in, kernels and copies out overlap (kpeg_cuda.cu decode_banded)
    dec.decode_scan(band.plan, h_in.array, out=mine)
    sync()
    t0 = time.perf_counter()
    for _ in range(steps):
        dec.decode_scan(band.plan, h_in.array, out=mine)
    e2e_s = _max_over_ranks(torch, dist, device, time.perf_counter() - t0)
    sync()
    # parity, on rank 0, from the SHARED frame: narrow bands out of the regions different ranks wrote against the oracle's
    # decode of the same band as an image of its own
    ok = True
    if rank == 0:
        narrow = split_restart_bands(plan, scan, side // 64)
        head = bytearray(jpg[:off].tobytes())
        i = head.find(b"\xff\xc0")
        for b in (narrow[0], narrow[len(narrow) // 2 + 1], narrow[-1]):
            head[i + 5:i + 7] = int(b.rows).to_bytes(2, "big")
            ref = H.oracle_decode(bytes(head) + b.scan.tobytes() + b"\xff\xd9")["pixels"]
            got = np.asarray(frame[b.row0 * side * 3:(b.row0 + b.rows) * side * 3]).reshape(b.rows, side, 3)
            ok = ok and bool(np.array_equal(ref, got))
    sync()
    if pinned:
        lib.kpeg_cuda_host_unregister(mine.ctypes.data)
    del mine, frame
    sync()
    if rank == 0:
        os.unlink(path)
    res = {"workload": f"{side}x{side} RGB 4:4:4 q=90, restart interval = one MCU row (BASELINE.json configs[4]), {world} band(s) of whole MCU rows, one per GPU",
           "device_resident_mpixel_per_s": side * side * steps / dev_s / 1e6, "e2e_mpixel_per_s": side * side * steps / e2e_s / 1e6,
           "band_rows_rank0": int(band.rows), "band_scan_bytes_rank0": int(band.scan.size), "steps": steps,
           "e2e_call": "kpeg_cuda_decode per rank on its band (host buffers; the band goes through the context's lanes as four sub-bands whose copies and kernels overlap)",
           "e2e_frame": "one host frame shared by the rank processes (/dev/shm), each rank's rows pinned with kpeg_cuda_host_register" if pinned
                        else "one host frame shared by the rank processes (/dev/shm), NOT pinned (registration refused)",
           "pixels_match_oracle": ok, "checked": "three 64-row bands of the shared frame (first, middle, last) against the oracle, on rank 0",
           "timer": "host clock around the calls after a device sync and barrier, max over ranks"}
    h_in.free()
    for b in d_out + [d_in]:
        dec.device_free(b)
    return res


# ---- CUDA arm -----------------------------------------------------------------------------------------
def dump_pixels(out_dir, name, pixels):
    """pixels [N, H, W, C] uint8 -> out_dir/<name>.npy [R, W, C] float32, R whole rows drawn with a fixed seed (every row
    when all fit in DUMP_PIXEL_BYTES, in order), and out_dir/<name>_rows.npy [R, 2] float64: (image, row) of each."""
    n, h, w, c = pixels.shape
    # a JPEG is at most 65535 samples wide, so one float32 RGB row stays under 1 MB and at least one row fits
    assert w * c * 4 <= DUMP_PIXEL_BYTES, f"a {w}-pixel row does not fit the dump budget"
    rows_all = pixels.reshape(n * h, w, c)
    r = min(n * h, DUMP_PIXEL_BYTES // (w * c * 4))
    pick = np.arange(n * h) if r == n * h else np.sort(np.random.default_rng(SEED0).choice(n * h, size=r, replace=False))
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, f"{name}.npy"), rows_all[pick].astype(np.float32))
    np.save(os.path.join(out_dir, f"{name}_rows.npy"), np.stack([pick // h, pick % h], axis=1).astype(np.float64))


def run_cuda_arm(args):
    import torch

    import libkpeg_b200 as K
    from libkpeg_b200.api import PinnedArray, pack_batch, packed_offsets
    from libkpeg_b200.synth import QUIRK_FREE, SynthParams, synth_encode

    rank, world, local = env_int("RANK", 0), env_int("WORLD_SIZE", 1), env_int("LOCAL_RANK", 0)
    ref4k = Reference4K() if (world == 1 and not args.no_cpu_baseline and not args.quick) else None
    dist = None
    if world > 1:
        import torch.distributed as dist_mod
        dist = dist_mod
        torch.cuda.set_device(local)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    device = local if world > 1 else 0
    torch.cuda.set_device(device)

    NB = args.batch
    W, Hh = args.width, args.height
    # ---- inputs: NB distinct images per rank -----------------------------------------------------
    jpgs = [synth_encode(SynthParams(W, Hh, quality=args.quality, seed=SEED0 + rank * 4096 + i, flags=QUIRK_FREE))
            for i in range(NB)]
    parsed = [K.parse_jfif(j) for j in jpgs]
    plan = parsed[0][0]
    plan.flags = K.KPEG_FLAG_REF_PARITY
    scans = [j[o:o + n] for j, (_, o, n) in zip(jpgs, parsed)]
    scan_bytes = int(sum(s.size for s in scans))
    npix_img = W * Hh
    pix_bytes_img = npix_img * 3

    dec = K.Decoder(device=device)  # raises without the CUDA library / a GPU: no fallback
    if args.sub_bits or args.relay_rounds:
        dec.set_tuning(args.sub_bits, args.relay_rounds)
    packed = pack_batch(scans)
    d_packed = dec.device_alloc(packed.size + 64)
    d_out = dec.device_alloc(NB * pix_bytes_img + 64)
    d_outs = [d_out, dec.device_alloc(NB * pix_bytes_img + 64)]
    dec.h2d(d_packed, packed)

    stream = torch.cuda.ExternalStream(dec.stream, device=torch.device("cuda", device))

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- correctness gate (untimed): EVERY image of this rank against the CPU oracle ---------------------
    import helpers as H
    dec.decode_batch_packed_device(plan, NB, d_packed, packed.size, d_out)
    got_all = np.empty((NB, Hh, W, 3), dtype=np.uint8)
    dec.d2h(got_all, d_out)
    got0 = got_all[0]
    nblk = (W // 8) * (Hh // 8) * 3
    coef_all = dec.read_coefficients(nblk * NB).reshape(NB, nblk, 64)
    cores_here = max(1, (os.cpu_count() or 1) // max(world, 1))
    coef_ok, max_abs_err, sq_err, n_checked = True, 0, 0.0, 0
    check_pixels = not args.skip_pixel_check
    for i in range(NB if not args.quick else 1):
        ref = H.oracle_decode(jpgs[i], parity=True, want_pixels=check_pixels, threads=cores_here)
        coef_ok = coef_ok and bool(np.array_equal(coef_all[i], ref["coef"]))
        if ref["pixels"] is not None:
            d = got_all[i].astype(np.int16) - ref["pixels"].astype(np.int16)
            max_abs_err = max(max_abs_err, int(np.abs(d).max()))
            sq_err += float((d.astype(np.float64) ** 2).sum())
            n_checked += d.size
    if (not coef_ok or max_abs_err > 1) and os.environ.get("KPEG_BENCH_WHATIF") == "1":
        # timing experiments with deliberately broken kernels (tools/whatif.sh): exit at once, without a bench line
        print("bench: WHATIF run, parity gate failed as expected; no measurement", file=sys.stderr)
        raise SystemExit(0)
    if not coef_ok or max_abs_err > 1:
        raise SystemExit(f"bench: parity gate failed on rank {rank} (coefficients equal: {coef_ok}, pixel max-abs-err: {max_abs_err})")
    images_checked = NB if not args.quick else 1
    del coef_all

    # ---- device-resident timing ------------------------------------------------------------------------
    # (1) throughput: the batch as two concurrent half-batches (one per lane of the context), no
    #     per-kernel events;  (2) the same steps again with an event after every kernel, one lane, for the
    #     per-kernel / roofline figures (kernel times are only meaningful without a concurrent lane).
    offsets = packed_offsets(scans)
    # every step is SUBMITTED (kpeg_cuda_submit_batch_packed_device: enqueue only), one wait at the end of the
    # timed region completes and checks all of them: consecutive steps overlap on the device, as they do for
    # any caller that keeps a decoder fed.  --sync-steps completes every step before the next is submitted.
    def run_steps(k):
        n_launch = 0
        for _ in range(k):
            if args.sync_steps:
                dec.decode_batch_packed_device_split(plan, NB, d_packed, offsets, d_out)
                n_launch += dec.last_stats.kernel_launches
            else:
                dec.submit_batch_packed_device(plan, NB, d_packed, offsets, d_outs[_ & 1])  # steps in flight never share an output
        if not args.sync_steps:
            dec.wait()
            n_launch += dec.last_stats.kernel_launches
        return n_launch

    run_steps(max(args.warmup, 3) + 16)  # + enough steps for every lane of the context to have sized its scratch
    sampler = ClockSampler(device)
    barrier()
    sampler.start()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record(stream)
    t_wall0 = time.perf_counter()
    launches = run_steps(args.steps)
    t_wall = time.perf_counter() - t_wall0
    ev1.record(stream)
    barrier()
    # all lanes are drained when wait() returns, so the event pair on lane 0 brackets all the work;
    # take the larger of the event time and the host wall clock around the same region
    dev_ms = max(ev0.elapsed_time(ev1), t_wall * 1e3)
    clocks = sampler.stop()
    if args.dump_outputs:
        # read back now: the legs below write into the same output buffers
        last = np.empty((NB, Hh, W, 3), dtype=np.uint8)
        dec.d2h(last, d_out if args.sync_steps else d_outs[(args.steps - 1) & 1])
        dump_pixels(args.dump_outputs, "pixels" if world == 1 else f"pixels_rank{rank}", last)
        del last

    # ---- sustained: the same steps until at least 2 s have passed (chunks of 256 steps, one wait per chunk) ----
    sustained = None
    if not args.quick:
        sampler2 = ClockSampler(device)
        barrier()
        sampler2.start()
        ev2, ev3 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev2.record(stream)
        t0 = time.perf_counter()
        sus_steps = 0
        while time.perf_counter() - t0 < args.sustain_s:
            run_steps(256)
            sus_steps += 256
        ev3.record(stream)
        torch.cuda.synchronize()
        sus_ms = max(ev2.elapsed_time(ev3), (time.perf_counter() - t0) * 1e3)
        sus_clocks = sampler2.stop()
        # every rank runs until ITS clock says 2 s: ranks differ in step count; per-rank rates are summed
        sus_rate = torch.tensor([NB * npix_img * sus_steps / (sus_ms / 1e3) / 1e6], dtype=torch.float64, device=torch.device("cuda", device))
        if dist is not None:
            dist.all_reduce(sus_rate, op=dist.ReduceOp.SUM)
        sustained = {"value": float(sus_rate[0]), "unit": UNIT, "seconds": sus_ms / 1e3, "steps_rank0": sus_steps,
                     "clocks": sus_clocks, "how": "device-resident steps submitted in chunks of 256 with one wait per chunk until 2 s have passed; sum of the ranks' rates"}
        barrier()

    if not clocks.get("samples") and sustained is not None:
        clocks = dict(sustained["clocks"], source="sustained leg (no sample fell into the short headline region)")
    dec.set_profiling(True)
    stage_ms = {k: 0.0 for k in K.Stats.STAGES}
    for _ in range(2):
        dec.decode_batch_packed_device(plan, NB, d_packed, packed.size, d_out)
    barrier()
    for _ in range(args.steps):
        dec.decode_batch_packed_device(plan, NB, d_packed, packed.size, d_out)
        for k, v in dec.last_stats.stage_ms().items():
            stage_ms[k] += v
    barrier()
    st = dec.last_stats
    stats_snapshot = dict(subsequences=st.subsequences, sync_rounds=st.sync_rounds, exact_pixels=st.exact_samples,
                          unstuffed_bytes=int(st.unstuffed_bytes), launches_per_step=st.kernel_launches)
    single_lane_ms = sum(stage_ms.values()) / args.steps
    dec.set_profiling(False)

    # ---- end to end: host pinned buffers in, host pinned buffers out -----------------------------------
    pin_in = [PinnedArray(s.size) for s in scans]
    for p, s in zip(pin_in, scans):
        p.array[:] = s
    pin_out = [PinnedArray(pix_bytes_img) for _ in range(2 * NB)]  # two sets: steps in flight never share an output
    in_views = [p.array for p in pin_in]
    out_sets = [[p.array.reshape(Hh, W, 3) for p in pin_out[k * NB:(k + 1) * NB]] for k in range(2)]
    out_views = out_sets[0]

    def run_e2e(k):
        for i in range(k):
            if args.sync_steps:
                dec.decode_batch(plan, in_views, out_sets[i & 1])
            else:
                dec.submit_batch(plan, in_views, out_sets[i & 1])  # kpeg_cuda_submit_batch: copies + kernels enqueued
        if not args.sync_steps:
            dec.wait()                                              # kpeg_cuda_wait: pixels are in host memory

    run_e2e(max(min(args.warmup, 3), 1) + 2)
    # what the link alone allows: the step's pixel bytes, device -> pinned host, nothing else running
    flat_out = [p.array for p in pin_out[:NB]]
    dec.d2h(flat_out[0], d_out)
    t0 = time.perf_counter()
    for rep in range(3):
        for i, o in enumerate(flat_out):
            dec.d2h(o, d_out + i * pix_bytes_img)
    pcie_d2h_gbs = 3 * NB * pix_bytes_img / (time.perf_counter() - t0) / 1e9
    barrier()
    t0 = time.perf_counter()
    run_e2e(args.steps)
    torch.cuda.synchronize()
    e2e_s = time.perf_counter() - t0
    e2e_ok = all(bool(np.array_equal(out_sets[k][i], got_all[i])) for k in range(2) for i in range(NB))
    barrier()

    # ---- the other configurations at this N ------------------------------------------------------------------
    gray = tiles = None
    if not args.no_extras:
        for p_ in pin_in + pin_out:
            p_.free()
        pin_in, pin_out = [], []
        gray = leg_gray_batch(dec, K, rank, world, dist, device, torch, args.quick)
        tiles = leg_tiles(dec, K, rank, world, dist, device, torch, args.quick)
        barrier()

    # ---- max over ranks -----------------------------------------------------------------------------------
    times = torch.tensor([dev_ms, e2e_s * 1e3], dtype=torch.float64, device=torch.device("cuda", device))
    if dist is not None:
        dist.all_reduce(times, op=dist.ReduceOp.MAX)
    dev_ms_max, e2e_ms_max = float(times[0]), float(times[1])
    par = torch.tensor([float(max_abs_err), sq_err, float(n_checked), 1.0 if (coef_ok and e2e_ok) else 0.0], dtype=torch.float64,
                       device=torch.device("cuda", device))
    if dist is not None:
        pmax = par.clone()
        dist.all_reduce(pmax, op=dist.ReduceOp.MAX)
        psum = par.clone()
        dist.all_reduce(psum, op=dist.ReduceOp.SUM)
        pmin = par.clone()
        dist.all_reduce(pmin, op=dist.ReduceOp.MIN)
        max_abs_err, sq_err, n_checked, all_ok = int(pmax[0]), float(psum[1]), float(psum[2]), bool(pmin[3] > 0.5)
    else:
        all_ok = bool(coef_ok and e2e_ok)
    mse = sq_err / n_checked if n_checked else None
    psnr = None if mse is None else ("inf" if mse == 0.0 else 10.0 * float(np.log10(255.0 ** 2 / mse)))
    total_px = world * NB * npix_img * args.steps
    value = total_px / (dev_ms_max / 1e3) / 1e6
    e2e_value = total_px / (e2e_ms_max / 1e3) / 1e6

    if rank == 0:
        peak, peak_src = measured_peaks()
        per_step = {k: v / args.steps for k, v in stage_ms.items()}
        unstuffed = stats_snapshot["unstuffed_bytes"]
        coef_bytes = NB * npix_img * 6
        alg = {  # algorithmic bytes per launch (group) -- DESIGN.md "Algorithmic bytes"
            "unstuff": packed.size + unstuffed,       # stuffed bytes in, unstuffed bytes out
            "entropy_cold": unstuffed,                # one read of the bit stream
            "entropy_relay": unstuffed,               # one read of the bit stream (records are not algorithmic)
            "entropy_write": coef_bytes,              # K2 (record expansion + DC prediction): the coefficient tiles, written once
            "idct": NB * npix_img * 9,                # 6 B/px of int16 coefficients in, 3 B/px of RGB out
            "dc_scan": NB * (npix_img // 64) * 3 * 4,
        }
        kernels = {}
        for k, ms in per_step.items():
            if k in ("h2d", "d2h") or ms <= 0:
                continue
            e = {"ms_per_step": ms}
            if k in alg:
                e["algorithmic_bytes"] = alg[k]
                e["achieved_gbs"] = alg[k] / (ms * 1e-3) / 1e9
                e["frac_of_hbm_peak"] = e["achieved_gbs"] / peak
            kernels[k] = e
        dom = max((k for k in kernels if k not in ("memset", "relay_sparse")), key=lambda k: kernels[k]["ms_per_step"])
        px_per_launch = NB * npix_img  # the per-kernel pass runs the whole batch as one job: one launch per kernel
        ncu_names = {"idct": "idct_kernel<3>", "entropy_write": "expand_kernel<3>", "entropy_relay": "entropy_relay_full_kernel",
                     "entropy_cold": "entropy_cold_kernel", "unstuff": "unstuff_count/scan/write_kernel"}
        roof = lambda k: {"kernel": k, "cuda_kernel": ncu_names.get(k, k), "bound": "hbm", "achieved": kernels[k].get("achieved_gbs"), "peak": peak,
                          "unit": "GB/s", "frac": kernels[k].get("frac_of_hbm_peak"),
                          "algorithmic_bytes_per_launch": kernels[k].get("algorithmic_bytes"),
                          "traffic": ncu_traffic(k, px_per_launch) if (W, Hh, args.quality) == (W4K, H4K, Q4K) else None,
                          "traffic_source": "profiles/ncu_traffic.json (ncu --set full dram bytes per pixel x pixels per launch)",
                          "peak_source": peak_src, "ms_per_launch_group": kernels[k]["ms_per_step"],
                          "share_of_step": kernels[k]["ms_per_step"] / sum(x["ms_per_step"] for x in kernels.values())}
        entropy_ms = sum(per_step[k] for k in ("memset", "unstuff", "entropy_cold", "entropy_relay", "relay_sparse",
                                               "entropy_scan", "entropy_write", "dc_scan"))
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
            "ms_per_step": dev_ms_max / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "u8/int16 entropy decode, f32 IDCT (f64 on the exact path)", "data": "synthetic",
            "config": {"workload": WORKLOAD if (W, Hh, args.quality) == (W4K, H4K, Q4K) else f"synthetic {W}x{Hh} q={args.quality}",
                       "images_per_step_per_gpu": NB, "width": W, "height": Hh, "quality": args.quality,
                       "restart_interval": 0, "parallelism": f"{world} GPU(s), images sharded, no collective",
                       "l2_policy": "inputs larger than L2 (no flush): per step %.0f MB bit stream + %.0f MB coefficients + %.0f MB pixels"
                                    % (packed.size / 1e6, coef_bytes / 1e6, NB * pix_bytes_img / 1e6),
                       "sub_bits": args.sub_bits or "default", "parity_mode": "reference (F1 quirk on)",
                       "concurrency": ("steps completed one at a time; " if args.sync_steps else "steps submitted back to back, one wait at the end of the timed region; ") + ("each step = up to 4 concurrent jobs on the lanes (streams) of one context" if args.sync_steps else "each step = one job, consecutive steps on different lanes (streams) of one context")},
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": int(packed.size),
                    "d2h_bytes_per_step": int(NB * pix_bytes_img), "ms_per_step": e2e_ms_max / args.steps,
                    "pcie_d2h_gbs_measured": pcie_d2h_gbs,
                    "frac_of_pcie_d2h": (NB * pix_bytes_img / (e2e_ms_max / args.steps * 1e-3) / 1e9) / pcie_d2h_gbs,
                    "timer": "host wall clock around the C-ABI calls, pinned host buffers in and out: " + ("kpeg_cuda_decode_batch per step" if args.sync_steps else "kpeg_cuda_submit_batch per step + one kpeg_cuda_wait"),
                    "matches_device_path": e2e_ok},
            "gpu_launches": int(launches),
            "clocks": clocks,
            "roofline": roof(dom),
            "roofline_idct": roof("idct"),
            "kernels": kernels,
            "entropy_bitstream_gbs": scan_bytes / (entropy_ms * 1e-3) / 1e9 if entropy_ms > 0 else None,
            "parity": {"coefficients_bit_exact": all_ok, "pixel_max_abs_err_vs_oracle": max_abs_err if check_pixels else None,
                       "pixel_psnr_db_vs_oracle": psnr if check_pixels else None,
                       "e2e_pixels_equal_device_path": all_ok,
                       "checked": f"all {images_checked} image(s) of every rank ({world} rank(s)) against the CPU oracle before timing: quantised "
                                  "coefficients bit for bit, pixels by max-abs-error and PSNR ('inf' = every byte identical); every image "
                                  "of both end-to-end output sets byte-compared with the device-resident decode"},
            "sustained": sustained,
            "gray_batch_4096": gray,
            "tiles_16k": tiles,
            "decode_stats": stats_snapshot,
            "kernel_timing": {"how": "same steps repeated on ONE lane with a CUDA event after every kernel",
                              "ms_per_step_sum_of_kernels": single_lane_ms},
        }
        if world == 1 and not args.no_cpu_baseline:
            cores = os.cpu_count() or 1
            kind, run_step, px, sample = reference_step_runner(cores)
            run_step()
            t0 = time.perf_counter()
            reps = 0
            while reps < 2 or (time.perf_counter() - t0 < 10 and reps < 8):
                run_step()
                reps += 1
            dt = time.perf_counter() - t0
            line["cpu_baseline"] = {"value": px * reps / dt / 1e6, "unit": UNIT, "cores": cores, "kind": kind,
                                    "sample": sample + f"; {reps} timed steps"}
            if not args.quick and _ref_binary_debug() is not None:
                kind_d, run_d, px_d, sample_d = reference_step_runner(cores, build="debug")
                run_d()
                t0 = time.perf_counter()
                reps_d = 0
                while reps_d < 2 or (time.perf_counter() - t0 < 8 and reps_d < 6):
                    run_d()
                    reps_d += 1
                line["cpu_baseline"]["stock_debug_build"] = {"value": px_d * reps_d / (time.perf_counter() - t0) / 1e6, "unit": UNIT, "cores": cores,
                                                             "kind": kind_d, "sample": sample_d + f"; {reps_d} timed steps"}
            if ref4k is not None:
                line["cpu_baseline"]["same_config_4k"] = ref4k.collect()
        print(json.dumps(line), flush=True)

    for p in pin_in + pin_out:
        p.free()
    dec.device_free(d_packed)
    for p in d_outs:
        dec.device_free(p)
    dec.close()
    if dist is not None:
        dist.destroy_process_group()
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="cuda", choices=["cuda", "reference"])
    ap.add_argument("--batch", type=int, default=8, help="images per step per GPU")
    ap.add_argument("--width", type=int, default=W4K)
    ap.add_argument("--height", type=int, default=H4K)
    ap.add_argument("--quality", type=int, default=Q4K)
    ap.add_argument("--sub-bits", type=int, default=0)
    ap.add_argument("--relay-rounds", type=int, default=0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--skip-pixel-check", action="store_true")
    ap.add_argument("--sync-steps", action="store_true", help="complete every step before submitting the next")
    ap.add_argument("--quick", action="store_true", help="development runs: parity gate on one image, no sustained leg, small extra legs")
    ap.add_argument("--no-extras", action="store_true", help="skip the gray-batch and 16k-tiles legs")
    ap.add_argument("--sustain-s", type=float, default=2.0)
    ap.add_argument("--dump-outputs", metavar="DIR", help="write a seeded sample of the pixels of the last timed step to "
                                                          "DIR/*.npy (float32, under 64 MB; CUDA arm only)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "cuda":
        ap.error("--dump-outputs applies to the CUDA arm")
    # stdout carries exactly ONE JSON line: whatever libraries write to file descriptor 1 (NCCL's version
    # banner, for one) is sent to stderr, and Python's own stdout keeps the original descriptor
    sys.stdout.flush()
    real_stdout = os.dup(1)
    os.dup2(2, 1)
    sys.stdout = os.fdopen(real_stdout, "w")
    if args.impl == "reference":
        return run_reference_arm(args)
    return run_cuda_arm(args)


if __name__ == "__main__":
    sys.exit(main())
