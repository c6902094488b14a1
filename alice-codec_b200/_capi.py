"""ctypes declarations of every symbol of include/alice_codec.h.

`load(path)` opens a libalice_codec build and attaches argument / result types.  The
default path is the in-tree product library (sm_100a CUDA build); there is no CPU build
of the product and no fallback: if the library is missing this raises.
"""
from __future__ import annotations

import ctypes as C
import os
import re

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
HEADER = os.path.join(ROOT, "include", "alice_codec.h")
PRODUCT_LIB = os.path.join(HERE, "lib", "libalice_codec.so")

u8p = C.POINTER(C.c_uint8)
u16p = C.POINTER(C.c_uint16)
i16p = C.POINTER(C.c_int16)
i32p = C.POINTER(C.c_int32)
u32p = C.POINTER(C.c_uint32)
u64p = C.POINTER(C.c_uint64)
vp = C.c_void_p
u8, u32, u64, i32, cint, dbl = C.c_uint8, C.c_uint32, C.c_uint64, C.c_int32, C.c_int, C.c_double

# name -> (restype, argtypes); opaque handles are void*
SIGNATURES = {
    # ---- Part 1: reference ABI (src/ffi.rs:16-315)
    "alice_codec_wavelet1d_haar": (vp, []),
    "alice_codec_wavelet1d_cdf53": (vp, []),
    "alice_codec_wavelet1d_cdf97": (vp, []),
    "alice_codec_wavelet1d_destroy": (None, [vp]),
    "alice_codec_wavelet1d_forward": (None, [vp, i32p, u32]),
    "alice_codec_wavelet1d_inverse": (None, [vp, i32p, u32]),
    "alice_codec_encoder_create": (vp, [u8]),
    "alice_codec_encoder_destroy": (None, [vp]),
    "alice_codec_encode": (vp, [vp, u8p, u32, u32, u32, u32]),
    "alice_codec_decode": (vp, [vp, u32p]),
    "alice_codec_chunk_destroy": (None, [vp]),
    "alice_codec_chunk_to_bytes": (vp, [vp, u32p]),
    "alice_codec_chunk_from_bytes": (vp, [u8p, u32]),
    "alice_codec_chunk_width": (u32, [vp]),
    "alice_codec_chunk_height": (u32, [vp]),
    "alice_codec_chunk_frames": (u32, [vp]),
    "alice_codec_psnr": (dbl, [u8p, u8p, u32]),
    "alice_codec_data_free": (None, [vp, u32]),
    "alice_codec_string_free": (None, [vp]),
    "alice_codec_version": (vp, []),
    # ---- Part 2: extensions
    "alice_codec_last_error": (i32, []),
    "alice_codec_last_error_message": (C.c_char_p, []),
    "alice_codec_encoder_create_with_wavelet": (vp, [u8, u8]),
    "alice_codec_encoder_create_ex": (vp, [u8, u8, u32]),
    "alice_codec_chunk_wavelet": (u8, [vp]),
    "alice_codec_chunk_compressed_size": (u64, [vp]),
    "alice_codec_chunk_channel_header": (cint, [vp, u32, u32p, i32p, i32p, u32p, u32p]),
    "alice_codec_chunk_to_bytes64": (vp, [vp, u64p]),
    "alice_codec_chunk_from_bytes64": (vp, [u8p, u64]),
    "alice_codec_data_free64": (None, [vp, u64]),
    "alice_codec_rgb_to_ycocg_r": (cint, [u8p, u64, i16p, i16p, i16p, u64]),
    "alice_codec_ycocg_r_to_rgb": (cint, [i16p, i16p, i16p, u64, u8p, u64]),
    "alice_codec_wavelet2d_forward": (cint, [u8, i32p, u32, u32]),
    "alice_codec_wavelet2d_inverse": (cint, [u8, i32p, u32, u32]),
    "alice_codec_wavelet3d_forward": (cint, [u8, i32p, u32, u32, u32]),
    "alice_codec_wavelet3d_inverse": (cint, [u8, i32p, u32, u32, u32]),
    "alice_codec_wavelet2d_device": (cint, [u8, cint, C.c_void_p, C.c_void_p, u32, u32, u32, C.c_void_p]),
    "alice_codec_wavelet3d_device": (cint, [u8, cint, C.c_void_p, C.c_void_p, u32, u32, u32, C.c_void_p]),
    "alice_codec_lossless_create": (vp, [u32, u32, u32, vp]),
    "alice_codec_lossless_destroy": (None, [vp]),
    "alice_codec_lossless_encode_device": (cint, [vp, C.c_void_p]),
    "alice_codec_lossless_decode_device": (cint, [vp]),
    "alice_codec_lossless_fetch": (cint, [vp, cint, cint, C.c_void_p, u64, u64p]),
    "alice_codec_lossless_timings": (cint, [vp, C.POINTER(C.c_float)]),
    "alice_codec_quantize_buffer": (cint, [i32, i32, i32p, u64, i32p, u64]),
    "alice_codec_dequantize_buffer": (cint, [i32, i32p, u64, i32p, u64]),
    "alice_codec_fast_quantize_buffer": (cint, [i32, i32, i32p, u64, i32p, u64]),
    "alice_codec_to_symbols": (cint, [i32p, u64, u8p, u64]),
    "alice_codec_from_symbols": (cint, [u8p, u64, i32p, u64]),
    "alice_codec_build_histogram": (cint, [u8p, u64, u32p]),
    "alice_codec_rdo_bpp_from_quality": (dbl, [u8]),
    "alice_codec_rdo_compute_quantizer": (cint, [dbl, i32p, u64, u8, i32p, i32p]),
    "alice_codec_rdo_estimate_variance": (cint, [i32p, u64, C.POINTER(C.c_double)]),
    "alice_codec_rdo_compute_all_quantizers": (cint, [dbl, i32p, u32, u32, u32, i32p, i32p]),
    "alice_codec_rdo_compute_all_quantizers_device": (cint, [dbl, C.c_void_p, u32, u32, u32, i32p, i32p]),
    "alice_codec_rdo_quantize_volume": (cint, [dbl, i32p, u32, u32, u32, i32p, u64, i32p, i32p]),
    "alice_codec_psnr_device": (cint, [C.c_void_p, C.c_void_p, u64, C.c_void_p, C.POINTER(C.c_double)]),
    "alice_codec_freq_table_from_histogram": (cint, [u32p, u32, u16p, u16p, u8p]),
    "alice_codec_rans_encode": (cint, [u8p, u64, u32p, u32, C.POINTER(vp), u64p]),
    "alice_codec_rans_encode_interleaved": (cint, [u8p, u64, u32p, u32, C.POINTER(vp), u64p]),
    "alice_codec_rans_decode": (cint, [u8p, u64, u32p, u32, u8p, u64]),
    "alice_codec_rans_decode_interleaved": (cint, [u8p, u64, u32p, u32, u8p, u64]),
    "alice_codec_encode_stages": (vp, [vp, u8p, u64, u32, u32, u32, i32p, u8p]),
    "alice_codec_decode_stages": (vp, [vp, u64p, u8p]),
    "alice_codec_batch_create": (vp, [u8, u8, u32, u32, u32, u32, vp]),
    "alice_codec_batch_create_ex": (vp, [u8, u8, u32, u32, u32, u32, vp, u32]),
    "alice_codec_batch_create_ex2": (vp, [u8, u8, u32, u32, u32, u32, vp, u32, u64]),
    "alice_codec_batch_workspace_bytes": (u64, [vp]),
    "alice_codec_batch_encode_device_ws": (cint, [vp, C.POINTER(vp), C.POINTER(vp), u32]),
    "alice_codec_batch_destroy": (None, [vp]),
    "alice_codec_batch_encode_device": (cint, [vp, C.POINTER(vp), u32]),
    "alice_codec_batch_decode_device": (cint, [vp, C.POINTER(vp), u32]),
    "alice_codec_batch_encode_host": (cint, [vp, C.POINTER(vp), u32, C.POINTER(vp)]),
    "alice_codec_batch_decode_host": (cint, [vp, C.POINTER(vp), u32, C.POINTER(vp)]),
    "alice_codec_batch_submit_host": (cint, [vp, u32, vp]),
    "alice_codec_batch_collect": (cint, [vp, u32, C.POINTER(vp)]),
    "alice_codec_batch_sync": (cint, [vp]),
    "alice_codec_batch_submit_device": (cint, [vp, u32, vp, vp]),
    "alice_codec_batch_encode_finish": (cint, [vp, u32]),
    "alice_codec_batch_decode_begin": (cint, [vp, u32]),
    "alice_codec_batch_decode_next_device": (cint, [vp, u32, vp]),
    "alice_codec_batch_decode_end": (cint, [vp]),
    "alice_codec_batch_get_chunk": (vp, [vp, u32]),
    "alice_codec_batch_timings": (cint, [vp, C.POINTER(C.c_float)]),
    "alice_codec_batch_device_bytes": (u64, [vp]),
    "alice_codec_rate_curve": (cint, [u8, u8p, u64, u32, u32, u32, u64p, u32p]),
    "alice_codec_rate_curve_device": (cint, [u8, vp, u32, u32, u32, u64p, u32p, vp]),
    "alice_codec_encode_to_size": (vp, [u8, u8p, u64, u32, u32, u32, u64, u8p]),
    "alice_codec_rate_curve_ex": (cint, [u8, u8p, u64, u32, u32, u32, u64p, u32p, u32]),
    "alice_codec_rate_curve_device_ex": (cint, [u8, vp, u32, u32, u32, u64p, u32p, vp, u32]),
    "alice_codec_encode_to_size_ex": (vp, [u8, u8p, u64, u32, u32, u32, u64, u8p, u32]),
    "alice_codec_batch_encode_host_to_size": (cint, [vp, C.POINTER(vp), u32, u64, C.POINTER(vp), u8p]),
    "alice_codec_synth_rgb_device": (cint, [cint, u32, u32, u32, u32, vp, vp]),
    "alice_codec_pinned_alloc": (vp, [u64]),
    "alice_codec_pinned_free": (None, [vp]),
    "alice_codec_trim_host_pool": (None, []),
    "alice_codec_device_count": (cint, []),
    "alice_codec_set_device": (cint, [cint]),
}


def declared_symbols(header: str = HEADER):
    """Every function name the C header declares (comments stripped)."""
    text = open(header).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(alice_codec_[a-z0-9_]+)\s*\(", text)))


def load(path: str | None = None) -> C.CDLL:
    path = path or PRODUCT_LIB
    if not os.path.exists(path):
        raise RuntimeError(
            f"{path} not found: build it with `python alice-codec_b200/build.py` (nvcc, sm_100a). "
            "libalice_codec has no CPU build and no fallback.")
    lib = C.CDLL(path)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError if the build does not export a declared symbol
        fn.restype = res
        fn.argtypes = args
    return lib
