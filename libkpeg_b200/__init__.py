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
    KPEG_FLAG_SCALE_1_2,
    KPEG_FLAG_SCALE_1_4,
    KPEG_FLAG_SCALE_1_8,
    KPEG_FLAG_SCALE_MASK,
    KPEG_TRANSCODE_KEEP_RESTART,
    KPEG_XFORM_FLIP_H,
    KPEG_XFORM_FLIP_V,
    KPEG_XFORM_NONE,
    KPEG_XFORM_ROT90,
    KPEG_XFORM_ROT180,
    KPEG_XFORM_ROT270,
    KPEG_XFORM_TRANSPOSE,
    KPEG_XFORM_TRANSVERSE,
    Crop,
    Decoder,
    EncodeParams,
    KpegError,
    Plan,
    Stats,
    crop_shape,
    crop_struct,
    load_cuda_library,
    output_shape,
    encode_bound,
    parse_jfif,
    ppm_header,
    TranscodeParams,
    transcode_bound,
)
from .synth import SynthParams, synth_encode, synth_pixels  # noqa: F401
