"""In-tree build of the native artefacts (nvcc / g++ via make).  Used by __graft_entry__.build()
and, lazily, by the ctypes loader when a library is missing or older than its sources."""
from __future__ import annotations

import os
import subprocess
from pathlib import Path

PKG = Path(__file__).resolve().parent
ROOT = PKG.parent
LIB = PKG / "lib"


def _run(cmd, cwd):
    proc = subprocess.run(cmd, cwd=cwd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    if proc.returncode != 0:
        raise RuntimeError(f"build failed: {' '.join(map(str, cmd))}\n{proc.stdout[-4000:]}")
    return proc.stdout


def build_product(targets=("all",)) -> None:
    """libkpeg_cuda.so (sm_100a kernels + C ABI), libkpeg_synth.so, kpeg CLI."""
    _run(["make", "-j8", *targets], cwd=PKG)


def build_oracle() -> None:
    """oracle/_ref: the CPU restatement, and the unmodified reference when /root/reference exists."""
    _run(["make", "all"], cwd=ROOT / "oracle")
    # the reference's own executable with its hot path replaced by the C ABI (INTEGRATION.md section 2), when
    # /root/reference is present; needs libkpeg_cuda.so, so build_product() first
    import sys
    _run([sys.executable, str(ROOT / "oracle" / "hybrid" / "build.py")], cwd=ROOT)


def build_emu() -> None:
    """tests/emu: CPU single-stepper of the kernel logic (test infrastructure)."""
    emu = ROOT / "tests" / "emu"
    out = emu / "libkpeg_emu.so"
    src = emu / "emu.cpp"
    deps = [src, *sorted((PKG / "csrc").glob("*.h"))]
    if out.exists() and all(out.stat().st_mtime >= d.stat().st_mtime for d in deps):
        return
    _run(["g++", "-std=c++17", "-O2", "-fPIC", "-shared", "-ffp-contract=off", "-fno-fast-math",
          "-Wno-unknown-pragmas", f"-I{ROOT / 'include'}", f"-I{PKG / 'csrc'}", "-o", str(out), str(src)], cwd=emu)


def build_emu_encode() -> None:
    """tests/emu/emu_encode.cpp: CPU single-stepper of the encoder's kernel logic (test infrastructure)."""
    emu = ROOT / "tests" / "emu"
    out = emu / "libkpeg_emu_encode.so"
    src = emu / "emu_encode.cpp"
    deps = [src, *sorted((PKG / "csrc").glob("*.h")), ROOT / "include" / "kpeg_cuda.h"]
    if out.exists() and all(out.stat().st_mtime >= d.stat().st_mtime for d in deps):
        return
    _run(["g++", "-std=c++17", "-O2", "-fPIC", "-shared", "-ffp-contract=off", "-fno-fast-math",
          "-Wno-unknown-pragmas", f"-I{ROOT / 'include'}", f"-I{PKG / 'csrc'}", "-o", str(out), str(src)], cwd=emu)


def build_emu_encode_opt() -> None:
    """tests/emu/emu_encode_opt.cpp: CPU replay of the encoder with optimised Huffman tables (test infrastructure)."""
    emu = ROOT / "tests" / "emu"
    out = emu / "libkpeg_emu_encode_opt.so"
    src = emu / "emu_encode_opt.cpp"
    deps = [src, *sorted((PKG / "csrc").glob("*.h")), ROOT / "include" / "kpeg_cuda.h"]
    if out.exists() and all(out.stat().st_mtime >= d.stat().st_mtime for d in deps):
        return
    _run(["g++", "-std=c++17", "-O2", "-fPIC", "-shared", "-ffp-contract=off", "-fno-fast-math",
          "-Wno-unknown-pragmas", f"-I{ROOT / 'include'}", f"-I{PKG / 'csrc'}", "-o", str(out), str(src)], cwd=emu)


def build_emu_transcode() -> None:
    """tests/emu/emu_transcode.cpp: CPU replay of the lossless transcoder's gather and coded stages (test infrastructure)."""
    emu = ROOT / "tests" / "emu"
    out = emu / "libkpeg_emu_transcode.so"
    src = emu / "emu_transcode.cpp"
    deps = [src, *sorted((PKG / "csrc").glob("*.h")), ROOT / "include" / "kpeg_cuda.h"]
    if out.exists() and all(out.stat().st_mtime >= d.stat().st_mtime for d in deps):
        return
    _run(["g++", "-std=c++17", "-O2", "-fPIC", "-shared", "-ffp-contract=off", "-fno-fast-math",
          "-Wno-unknown-pragmas", f"-I{ROOT / 'include'}", f"-I{PKG / 'csrc'}", "-o", str(out), str(src)], cwd=emu)


def build_emu_scaled() -> None:
    """tests/emu: CPU replay of the reduced-size reconstruction (emu_scaled.cpp, over csrc/idct_reduced.h) and its C
    reference restated from libjpeg (ref_scaled.c) -- test infrastructure."""
    emu = ROOT / "tests" / "emu"
    hdrs = [*sorted((PKG / "csrc").glob("*.h")), ROOT / "include" / "kpeg_cuda.h"]
    for out, src, cmd in (
        (emu / "libkpeg_emu_scaled.so", emu / "emu_scaled.cpp",
         ["g++", "-std=c++17", "-O2", "-fPIC", "-shared", "-Wall", "-Wno-unknown-pragmas", f"-I{ROOT / 'include'}",
          f"-I{PKG / 'csrc'}"]),
        (emu / "libkpeg_ref_scaled.so", emu / "ref_scaled.c", ["gcc", "-std=c11", "-O2", "-fPIC", "-shared", "-Wall"]),
    ):
        deps = [src, *hdrs]
        if out.exists() and all(out.stat().st_mtime >= d.stat().st_mtime for d in deps):
            continue
        _run([*cmd, "-o", str(out), str(src)], cwd=emu)


def build_emu_crop() -> None:
    """tests/emu/emu_crop.cpp: the crop decode's geometry (csrc/crop_geom.h) compiled for the host (test infrastructure)."""
    emu = ROOT / "tests" / "emu"
    out = emu / "libkpeg_emu_crop.so"
    src = emu / "emu_crop.cpp"
    deps = [src, *sorted((PKG / "csrc").glob("*.h"))]
    if out.exists() and all(out.stat().st_mtime >= d.stat().st_mtime for d in deps):
        return
    _run(["g++", "-std=c++17", "-O2", "-fPIC", "-shared", "-Wall", "-Wno-unknown-pragmas", f"-I{ROOT / 'include'}",
          f"-I{PKG / 'csrc'}", "-o", str(out), str(src)], cwd=emu)


def have_nvcc() -> bool:
    from shutil import which
    return which(os.environ.get("NVCC", "nvcc")) is not None
