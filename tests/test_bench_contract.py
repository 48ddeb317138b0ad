"""bench.py's output contract, the part that can be checked without a GPU: the reference arm (`--impl reference`) runs
the compiled reference (or, where it did not travel, the oracle port) on the host cores and prints ONE JSON line with
the keys the driver reads; the CUDA arm must refuse to run without a device instead of falling back to anything."""
import json
import os
import subprocess
import sys
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent


def _run(args, timeout=600):
    return subprocess.run([sys.executable, str(ROOT / "bench.py"), *args], cwd=ROOT, capture_output=True, text=True, timeout=timeout)


def test_reference_arm_prints_one_contract_line():
    r = _run(["--impl", "reference", "--steps", "1", "--warmup", "0"])
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.strip().startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "decode_mpixel_per_s" and d["unit"] == "Mpixel/s"
    assert d["higher_is_better"] is True and d["n_gpus"] == 1 and d["value"] > 0
    assert d["cpu_baseline"]["kind"] in ("reference", "port") and d["cpu_baseline"]["cores"] >= 1
    assert d["cpu_baseline"]["value"] == d["value"] and "sample" in d["cpu_baseline"]
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["gpu_launches"] == 0 and "workload" in d["config"]


def test_dump_pixels_rows_and_budget(tmp_path, monkeypatch):
    """--dump-outputs: whole rows as float32 with their (image, row); all rows when they fit, else the same seeded sample
    on every call, within the byte budget."""
    import numpy as np
    import bench
    px = np.random.default_rng(1).integers(0, 256, size=(3, 10, 7, 3), dtype=np.uint8)
    bench.dump_pixels(str(tmp_path / "all"), "pixels", px)
    got, idx = np.load(tmp_path / "all" / "pixels.npy"), np.load(tmp_path / "all" / "pixels_rows.npy")
    assert got.dtype == np.float32 and idx.dtype == np.float64
    assert np.array_equal(got, px.reshape(30, 7, 3)) and np.array_equal(idx[:, 0] * 10 + idx[:, 1], np.arange(30))
    monkeypatch.setattr(bench, "DUMP_PIXEL_BYTES", 8 * 7 * 3 * 4)
    for d in ("a", "b"):
        bench.dump_pixels(str(tmp_path / d), "pixels", px)
    got, idx = np.load(tmp_path / "a" / "pixels.npy"), np.load(tmp_path / "a" / "pixels_rows.npy").astype(int)
    assert got.shape == (8, 7, 3) and got.nbytes <= bench.DUMP_PIXEL_BYTES
    assert np.array_equal(got, px[idx[:, 0], idx[:, 1]]) and (np.diff(idx[:, 0] * 10 + idx[:, 1]) > 0).all()
    assert np.array_equal(got, np.load(tmp_path / "b" / "pixels.npy"))


def test_dump_outputs_and_steps_are_checked():
    r = _run(["--impl", "reference", "--steps", "1", "--dump-outputs", "x"], timeout=120)
    assert r.returncode != 0 and "--dump-outputs" in r.stderr
    r = _run(["--steps", "0"], timeout=120)
    assert r.returncode != 0 and "--steps" in r.stderr


def test_cuda_arm_fails_loudly_without_a_device():
    import torch
    if torch.cuda.is_available():
        import pytest
        pytest.skip("a GPU is present: the CUDA arm would run")
    r = _run(["--steps", "1", "--warmup", "3", "--quick", "--no-extras", "--no-cpu-baseline"], timeout=300)
    assert r.returncode != 0
    assert not [l for l in r.stdout.splitlines() if l.strip().startswith("{")], "no bench line may be printed without the GPU path"
