"""libkpeg_b200 -- B200-native (sm_100a) baseline-JPEG decode hot path of libKPEG.

The product is native: ``lib/libkpeg_cuda.so`` (hand-written CUDA kernels behind the C ABI of
``include/kpeg_cuda.h``) and the C++ drop-in ``kpeg::JPEGDecoder`` / ``kpeg`` CLI in ``host/``.
This Python package is only the thin ctypes binding the tests and ``bench.py`` drive it with; it
contains no decode logic and no CPU fallback -- every decode call goes to the CUDA library and
raises when that library or a GPU is missing.
"""
from .api import (  # noqa: F401
    KPEG_FLAG_OPTIMIZE_HUFFMAN,
    KPEG_FLAG_REF_PARITY,
    Decoder,
    EncodeParams,
    KpegError,
    Plan,
    Stats,
    load_cuda_library,
    encode_bound,
    parse_jfif,
    ppm_header,
)
from .synth import SynthParams, synth_encode, synth_pixels  # noqa: F401
