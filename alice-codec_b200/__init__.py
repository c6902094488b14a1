"""alice-codec_b200 — B200-native (sm_100a) implementation of ALICE-Codec's encode/decode hot path.

The product is `lib/libalice_codec.so` (CUDA kernels + C ABI, built from `csrc/` by
`build.py`); this package is the thin host-side mirror of the reference's operator
interface on top of that C ABI.  The directory name carries a hyphen, so import it through
`__graft_entry__.load_package()` (which registers it as `alice_codec_b200`).
"""
from . import _capi, sharding  # noqa: F401
from .api import (Api, ChunkBatch, CodecError, EncodedChunk, FrameDecoder, FrameEncoder, LosslessSet, ReferenceAbi,  # noqa: F401
                  SUBBANDS, WAVELET_BYTES, WAVELET_NAMES, default_api, quality_for_step, quality_to_step,
                  rgb_to_ycocg_r_numpy, version, ycocg_r_to_rgb_numpy)

__all__ = ["Api", "ChunkBatch", "CodecError", "EncodedChunk", "FrameDecoder", "FrameEncoder", "LosslessSet", "ReferenceAbi",
           "default_api", "WAVELET_NAMES", "WAVELET_BYTES", "SUBBANDS", "rgb_to_ycocg_r_numpy", "ycocg_r_to_rgb_numpy", "version",
           "quality_to_step", "quality_for_step"]
