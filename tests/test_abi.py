"""The C-ABI library: loads, exports every symbol include/kpeg_cuda.h declares, the host-side
entry points work without a GPU, and the compute entry points fail loudly (no CPU fallback)."""
import ctypes as C
import re
import subprocess
from pathlib import Path

import numpy as np
import pytest

import libkpeg_b200 as K
from libkpeg_b200 import api

ROOT = Path(__file__).resolve().parent.parent


def declared_functions(header: Path):
    text = re.sub(r"/\*.*?\*/", "", header.read_text(), flags=re.S)
    return sorted(set(re.findall(r"\b(kpeg_[a-z0-9_]+)\s*\(", text)))


def test_library_exports_every_declared_symbol():
    lib = K.load_cuda_library()
    names = declared_functions(ROOT / "include" / "kpeg_cuda.h")
    assert len(names) >= 20
    for n in names:
        assert hasattr(lib, n), f"libkpeg_cuda.so does not export {n}"
    assert set(names) == set(api.SYMBOLS), "python binding and header disagree"


def test_synth_library_exports():
    lib = C.CDLL(str(ROOT / "libkpeg_b200" / "lib" / "libkpeg_synth.so"))
    for n in declared_functions(ROOT / "include" / "kpeg_synth.h"):
        assert hasattr(lib, n)


def test_struct_layouts_match_the_header(tmp_path):
    """sizeof(kpeg_plan) / sizeof(kpeg_stats) as the C compiler sees them == the ctypes mirrors."""
    src = '#include <stdio.h>\n#include "kpeg_cuda.h"\nint main(){printf("%zu %zu %d\\n", sizeof(kpeg_plan), sizeof(kpeg_stats), KPEG_T_COUNT);return 0;}\n'
    exe = tmp_path / "kpeg_sizeof"
    subprocess.run(["gcc", "-x", "c", "-", f"-I{ROOT / 'include'}", "-o", str(exe)], input=src.encode(), check=True)
    a, b, c = map(int, subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.split())
    assert a == C.sizeof(api.Plan) and b == C.sizeof(api.Stats) and c == len(api.Stats.STAGES)


def test_parse_jfif_lena(lena_jpg):
    plan, off, n = K.parse_jfif(lena_jpg)
    assert (plan.width, plan.height, plan.ncomp, plan.restart_interval) == (512, 512, 3, 0)
    assert n == 104113  # SURVEY §4: scan bytes of lena.jpg
    assert lena_jpg[off + n:off + n + 2] == b"\xff\xd9"
    assert list(plan.comp_tq) == [0, 1, 1] and list(plan.comp_td) == [0, 1, 1] and list(plan.comp_ta) == [0, 1, 1]
    assert list(plan.ht[0][0].counts) == [0, 1, 5, 1, 1, 1, 1, 1, 1, 0, 0, 0, 0, 0, 0, 0]  # Annex K luminance DC


def test_error_codes():
    lib = K.load_cuda_library()
    with pytest.raises(K.KpegError) as e:
        K.parse_jfif(b"not a jpeg at all")
    assert e.value.code == api.KPEG_ERR_FORMAT
    assert lib.kpeg_cuda_decode(None, None, None, 0, None, None) == api.KPEG_ERR_ARG
    assert lib.kpeg_cuda_read_coefficients(None, None, 0) == api.KPEG_ERR_ARG
    assert lib.kpeg_cuda_last_error(None) == b"no context"


def test_no_gpu_means_error_not_fallback():
    lib = K.load_cuda_library()
    if lib.kpeg_cuda_device_count() > 0:
        pytest.skip("a GPU is present")
    with pytest.raises(K.KpegError) as e:
        K.Decoder(device=0)
    assert e.value.code == api.KPEG_ERR_CUDA


def test_cli_without_gpu_reports_and_exits_like_the_reference(tmp_path, lena_jpg):
    lib = K.load_cuda_library()
    exe = ROOT / "libkpeg_b200" / "lib" / "kpeg"
    r = subprocess.run([str(exe), "-h"], cwd=tmp_path, capture_output=True, text=True)
    assert r.returncode == 0 and "K-PEG - Simple JPEG Encoder & Decoder" in r.stdout
    r = subprocess.run([str(exe)], cwd=tmp_path, capture_output=True, text=True)
    assert r.returncode != 0 and "No arguments provided." in r.stdout  # main.cpp:56-60
    r = subprocess.run([str(exe), "a.jpg", "b.jpg", "c.jpg"], cwd=tmp_path, capture_output=True, text=True)
    assert r.returncode != 0
    if lib.kpeg_cuda_device_count() == 0:
        p = tmp_path / "lena.jpg"
        p.write_bytes(lena_jpg)
        r = subprocess.run([str(exe), str(p)], cwd=tmp_path, capture_output=True, text=True)
        assert r.returncode == 0  # main.cpp:66-70: EXIT_SUCCESS for any one-file run
        assert "no CPU decode path" in r.stdout and not (tmp_path / "lena.ppm").exists()
        assert (tmp_path / "kpeg.log").exists()


def test_batch_pack_format():
    scans = [np.arange(5, dtype=np.uint8), np.arange(3, dtype=np.uint8) + 100]
    packed = api.pack_batch(scans)
    assert packed.tolist() == [0, 1, 2, 3, 4, 0xFF, 0xD0, 100, 101, 102, 0xFF, 0xD1]
