"""Host-side mirror of the reference's operator interface, on top of the C ABI.

Names, argument meaning and error behaviour follow the reference's Python module
(/root/reference/src/python.rs: FrameEncoder :365-435, FrameDecoder :443-482, EncodedChunk
:287-357, rgb_to_ycocg_r_numpy :497, ycocg_r_to_rgb_numpy :541) and, for the stage
functions the reference only exposes in Rust, the Rust names (Wavelet1D/2D/3D, Quantizer,
FastQuantizer, AnalyticalRDO, to_symbols, from_symbols, build_histogram, FrequencyTable,
RansEncoder, RansDecoder).  Every call goes through libalice_codec's C ABI
(include/alice_codec.h) and computes on the CUDA device; errors become CodecError
(a ValueError, like python.rs:61-63).
"""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import _capi

WAVELET_NAMES = {"cdf53": 0, "cdf97": 1, "haar": 2}  # pipeline.rs:34-41, python.rs:380-384
WAVELET_BYTES = {v: k for k, v in WAVELET_NAMES.items()}
ERR_NAMES = {1: "InvalidBufferSize", 2: "InvalidDimensions", 3: "DimensionOverflow", 4: "InvalidBitstream",
             5: "InvalidQuantStep", 6: "ReferencePanic", 7: "NullArgument", 100: "CudaError"}
SUBBANDS = ("LLL", "LLH", "LHL", "LHH", "HLL", "HLH", "HHL", "HHH")  # lib.rs:115-132


class CodecError(ValueError):
    """CodecError of the reference (error.rs:12-23) + the CUDA failure class of this build."""

    def __init__(self, code: int, message: str = ""):
        self.code = code
        self.kind = ERR_NAMES.get(code, f"Error{code}")
        super().__init__(f"{self.kind}: {message}" if message else self.kind)


RATE_STEPS = 64
UINT64_MAX = (1 << 64) - 1


def quality_to_step(quality: int) -> int:
    """pipeline.rs:456-457: the quantiser step (1..64) of a quality byte"""
    q = min(int(quality), 100)
    return max(1, 64 - q * 63 // 100)


def quality_for_step(step: int) -> int:
    """the largest quality in 0..=100 whose quantiser step is `step` (1..64)"""
    return max(q for q in range(101) if quality_to_step(q) == step)


def _by_quality(curve):
    """{quality: curve[step - 1]} over the 64 steps (highest quality first): a rate curve's predicted .alc bytes (None
    where the reference aborts) or a PSNR curve's dB"""
    return {quality_for_step(s): None if curve.dtype == np.uint64 and int(v) == UINT64_MAX else v.item()
            for s, v in enumerate(curve, 1)}


def _wavelet_byte(wavelet) -> int:
    if isinstance(wavelet, str):
        if wavelet not in WAVELET_NAMES:
            raise ValueError(f"unknown wavelet type '{wavelet}'; expected 'cdf53', 'cdf97', or 'haar'")
        return WAVELET_NAMES[wavelet]
    w = int(wavelet)
    if w not in WAVELET_BYTES:
        raise ValueError(f"unknown wavelet byte {w}")
    return w


def _u8(a):
    a = np.ascontiguousarray(a, dtype=np.uint8).reshape(-1)
    return a, a.ctypes.data_as(_capi.u8p)


def _i32(a, copy=False):
    a = np.array(a, dtype=np.int32, copy=True).reshape(-1) if copy else np.ascontiguousarray(a, dtype=np.int32).reshape(-1)
    return a, a.ctypes.data_as(_capi.i32p)


def _i16(a):
    a = np.ascontiguousarray(a, dtype=np.int16).reshape(-1)
    return a, a.ctypes.data_as(_capi.i16p)


class Api:
    """One loaded libalice_codec build.  `Api()` = the in-tree product library."""

    def __init__(self, lib_path: str | None = None):
        self.lib = _capi.load(lib_path)
        self.path = lib_path or _capi.PRODUCT_LIB

    # ---- error plumbing
    def _raise(self, default_code=100):
        code = self.lib.alice_codec_last_error() or default_code
        msg = self.lib.alice_codec_last_error_message()
        raise CodecError(code, msg.decode() if msg else "")

    def _chk(self, rc):
        if rc != 0:
            self._raise(rc)

    def _take(self, ptr, n) -> bytes:
        try:
            return C.string_at(ptr, n)
        finally:
            self.lib.alice_codec_data_free64(ptr, n)

    def _take_np(self, ptr, n) -> np.ndarray:
        try:
            out = np.empty(n, np.uint8)
            if n:
                C.memmove(out.ctypes.data, ptr, n)
            return out
        finally:
            self.lib.alice_codec_data_free64(ptr, n)

    def version(self) -> str:
        p = self.lib.alice_codec_version()
        try:
            return C.string_at(p).decode()
        finally:
            self.lib.alice_codec_string_free(p)

    def device_count(self) -> int:
        return self.lib.alice_codec_device_count()

    def set_device(self, device: int):
        self._chk(self.lib.alice_codec_set_device(device))

    # ---- colour (color.rs:199, :245)
    def rgb_to_ycocg_r(self, rgb_bytes):
        a, pa = _u8(rgb_bytes)
        if a.size % 3:
            raise ValueError("rgb_bytes length must be a multiple of 3")
        n = a.size // 3
        y, co, cg = (np.empty(n, np.int16) for _ in range(3))
        self._chk(self.lib.alice_codec_rgb_to_ycocg_r(pa, a.size, y.ctypes.data_as(_capi.i16p),
                                                      co.ctypes.data_as(_capi.i16p), cg.ctypes.data_as(_capi.i16p), n))
        return y, co, cg

    def ycocg_r_to_rgb(self, y, co, cg):
        (y, py), (co, pco), (cg, pcg) = _i16(y), _i16(co), _i16(cg)
        if not (y.size == co.size == cg.size):
            raise ValueError("y, co, cg arrays must have the same length")
        out = np.empty(y.size * 3, np.uint8)
        self._chk(self.lib.alice_codec_ycocg_r_to_rgb(py, pco, pcg, y.size, out.ctypes.data_as(_capi.u8p), out.size))
        return out

    # ---- wavelets (wavelet.rs)
    def wavelet1d(self, wavelet, data, inverse=False):
        wb = _wavelet_byte(wavelet)
        ctor = (self.lib.alice_codec_wavelet1d_cdf53, self.lib.alice_codec_wavelet1d_cdf97,
                self.lib.alice_codec_wavelet1d_haar)[wb]
        h = ctor()
        try:
            a, pa = _i32(data, copy=True)
            (self.lib.alice_codec_wavelet1d_inverse if inverse else self.lib.alice_codec_wavelet1d_forward)(h, pa, a.size)
            if a.size >= 2 and self.lib.alice_codec_last_error() == 100:
                self._raise()
            return a
        finally:
            self.lib.alice_codec_wavelet1d_destroy(h)

    def wavelet2d(self, wavelet, data, width, height, inverse=False):
        a, pa = _i32(data, copy=True)
        if a.size != width * height:
            raise ValueError("buffer size != width*height")
        fn = self.lib.alice_codec_wavelet2d_inverse if inverse else self.lib.alice_codec_wavelet2d_forward
        self._chk(fn(_wavelet_byte(wavelet), pa, width, height))
        return a

    def wavelet3d(self, wavelet, data, width, height, depth, inverse=False):
        a, pa = _i32(data, copy=True)
        if a.size != width * height * depth:
            raise ValueError("buffer size != width*height*depth")
        fn = self.lib.alice_codec_wavelet3d_inverse if inverse else self.lib.alice_codec_wavelet3d_forward
        self._chk(fn(_wavelet_byte(wavelet), pa, width, height, depth))
        return a

    # ---- quantisation / symbols / histogram (quant.rs)
    def quantize_buffer(self, step, dead_zone, data):
        a, pa = _i32(data)
        out = np.empty_like(a)
        self._chk(self.lib.alice_codec_quantize_buffer(step, dead_zone, pa, a.size, out.ctypes.data_as(_capi.i32p), out.size))
        return out

    def fast_quantize_buffer(self, step, dead_zone, data):
        a, pa = _i32(data)
        out = np.empty_like(a)
        self._chk(self.lib.alice_codec_fast_quantize_buffer(step, dead_zone, pa, a.size, out.ctypes.data_as(_capi.i32p), out.size))
        return out

    def dequantize_buffer(self, step, data):
        a, pa = _i32(data)
        out = np.empty_like(a)
        self._chk(self.lib.alice_codec_dequantize_buffer(step, pa, a.size, out.ctypes.data_as(_capi.i32p), out.size))
        return out

    def to_symbols(self, coeffs):
        a, pa = _i32(coeffs)
        out = np.empty(a.size, np.uint8)
        self._chk(self.lib.alice_codec_to_symbols(pa, a.size, out.ctypes.data_as(_capi.u8p), out.size))
        return out

    def from_symbols(self, symbols):
        a, pa = _u8(symbols)
        out = np.empty(a.size, np.int32)
        self._chk(self.lib.alice_codec_from_symbols(pa, a.size, out.ctypes.data_as(_capi.i32p), out.size))
        return out

    def build_histogram(self, symbols):
        a, pa = _u8(symbols)
        h = np.zeros(256, np.uint32)
        self._chk(self.lib.alice_codec_build_histogram(pa, a.size, h.ctypes.data_as(_capi.u32p)))
        return h

    def rdo_bpp_from_quality(self, quality):
        return self.lib.alice_codec_rdo_bpp_from_quality(quality)

    def rdo_compute_quantizer(self, target_bpp, coeffs, subband):
        sb = SUBBANDS.index(subband) if isinstance(subband, str) else int(subband)
        a, pa = _i32(coeffs)
        s, d = C.c_int32(), C.c_int32()
        self._chk(self.lib.alice_codec_rdo_compute_quantizer(target_bpp, pa, a.size, sb, C.byref(s), C.byref(d)))
        return s.value, d.value

    def rdo_estimate_variance(self, coeffs) -> float:
        a, pa = _i32(coeffs)
        v = C.c_double()
        self._chk(self.lib.alice_codec_rdo_estimate_variance(pa, a.size, C.byref(v)))
        return v.value

    def rdo_compute_all_quantizers(self, target_bpp, volume, width, height, depth):
        """AnalyticalRDO::compute_all_quantizers on the 8 octants of a forward-transformed volume:
        returns [(step, dead_zone)] * 8 indexed by the SubBand3D byte."""
        a, pa = _i32(volume)
        assert a.size == width * height * depth
        s, d = np.zeros(8, np.int32), np.zeros(8, np.int32)
        self._chk(self.lib.alice_codec_rdo_compute_all_quantizers(target_bpp, pa, width, height, depth,
                                                                  s.ctypes.data_as(_capi.i32p), d.ctypes.data_as(_capi.i32p)))
        return list(zip(s.tolist(), d.tolist()))

    def rdo_compute_all_quantizers_device(self, target_bpp, d_volume: int, width, height, depth):
        """as rdo_compute_all_quantizers for an i32 volume in device memory (raw device pointer)."""
        s, d = np.zeros(8, np.int32), np.zeros(8, np.int32)
        self._chk(self.lib.alice_codec_rdo_compute_all_quantizers_device(target_bpp, C.c_void_p(d_volume), width, height,
                                                                         depth, s.ctypes.data_as(_capi.i32p),
                                                                         d.ctypes.data_as(_capi.i32p)))
        return list(zip(s.tolist(), d.tolist()))

    def rdo_quantize_volume(self, target_bpp, volume, width, height, depth):
        """statistics -> quantisers -> FastQuantizer per octant; returns (quantised i32 volume, [(step, dz)] * 8)."""
        a, pa = _i32(volume)
        assert a.size == width * height * depth
        out = np.empty(a.size, np.int32)
        s, d = np.zeros(8, np.int32), np.zeros(8, np.int32)
        self._chk(self.lib.alice_codec_rdo_quantize_volume(target_bpp, pa, width, height, depth,
                                                           out.ctypes.data_as(_capi.i32p), out.size,
                                                           s.ctypes.data_as(_capi.i32p), d.ctypes.data_as(_capi.i32p)))
        return out, list(zip(s.tolist(), d.tolist()))

    def psnr_device(self, d_a: int, d_b: int, n: int, stream: int = 0) -> float:
        """alice_codec_psnr for two device buffers (raw device pointers)."""
        v = C.c_double()
        self._chk(self.lib.alice_codec_psnr_device(C.c_void_p(d_a), C.c_void_p(d_b), n, C.c_void_p(stream), C.byref(v)))
        return v.value

    # ---- rANS (rans.rs)
    def freq_table_from_histogram(self, hist):
        h = np.ascontiguousarray(hist, dtype=np.uint32).reshape(-1)
        cum, freq, lut = np.zeros(256, np.uint16), np.zeros(256, np.uint16), np.zeros(4096, np.uint8)
        self._chk(self.lib.alice_codec_freq_table_from_histogram(
            h.ctypes.data_as(_capi.u32p), h.size, cum.ctypes.data_as(_capi.u16p), freq.ctypes.data_as(_capi.u16p),
            lut.ctypes.data_as(_capi.u8p)))
        return cum[:h.size].copy(), freq[:h.size].copy(), lut

    def rans_encode(self, symbols, hist) -> bytes:
        a, pa = _u8(symbols)
        h = np.ascontiguousarray(hist, dtype=np.uint32).reshape(-1)
        out, n = C.c_void_p(), C.c_uint64()
        self._chk(self.lib.alice_codec_rans_encode(pa, a.size, h.ctypes.data_as(_capi.u32p), h.size, C.byref(out), C.byref(n)))
        return self._take(out, n.value)

    def rans_decode(self, stream: bytes, n: int, hist) -> np.ndarray:
        buf = np.frombuffer(bytes(stream), dtype=np.uint8)
        h = np.ascontiguousarray(hist, dtype=np.uint32).reshape(-1)
        out = np.empty(n, np.uint8)
        self._chk(self.lib.alice_codec_rans_decode(buf.ctypes.data_as(_capi.u8p) if buf.size else None, buf.size,
                                                   h.ctypes.data_as(_capi.u32p), h.size,
                                                   out.ctypes.data_as(_capi.u8p), n))
        return out

    def rans_encode_interleaved(self, symbols, hist) -> bytes:
        """InterleavedRansEncoder::encode + finish (rans.rs:393-459); not the .alc stream format."""
        a, pa = _u8(symbols)
        h = np.ascontiguousarray(hist, dtype=np.uint32).reshape(-1)
        out, n = C.c_void_p(), C.c_uint64()
        self._chk(self.lib.alice_codec_rans_encode_interleaved(pa, a.size, h.ctypes.data_as(_capi.u32p), h.size,
                                                               C.byref(out), C.byref(n)))
        return self._take(out, n.value)

    def rans_decode_interleaved(self, stream: bytes, n: int, hist) -> np.ndarray:
        """InterleavedRansDecoder::new + decode_n (rans.rs:465-524)."""
        buf = np.frombuffer(bytes(stream), dtype=np.uint8)
        h = np.ascontiguousarray(hist, dtype=np.uint32).reshape(-1)
        out = np.empty(n, np.uint8)
        self._chk(self.lib.alice_codec_rans_decode_interleaved(
            buf.ctypes.data_as(_capi.u8p) if buf.size else None, buf.size, h.ctypes.data_as(_capi.u32p), h.size,
            out.ctypes.data_as(_capi.u8p), n))
        return out

    def psnr(self, a, b) -> float:
        (a, pa), (b, pb) = _u8(a), _u8(b)
        assert a.size == b.size
        return self.lib.alice_codec_psnr(pa, pb, a.size)


_default_api: Api | None = None


def default_api() -> Api:
    global _default_api
    if _default_api is None:
        _default_api = Api()
    return _default_api


# ---- module-level functions of the reference's Python module (python.rs:274-277, 496-583, 598-609)
def version() -> str:
    """python.rs:274: the crate version the library is ABI-compatible with."""
    return default_api().version()


def rgb_to_ycocg_r_numpy(rgb_bytes):
    """python.rs:496-527: 1-D uint8 [R0,G0,B0, R1,...] -> (y, co, cg) 1-D int16 arrays."""
    a = np.asarray(rgb_bytes)
    if a.dtype != np.uint8 or a.ndim != 1:
        raise TypeError("rgb_bytes must be a 1-D uint8 NumPy array")
    if not a.flags.c_contiguous:
        raise ValueError("rgb_bytes must be C-contiguous")
    return default_api().rgb_to_ycocg_r(a)


def ycocg_r_to_rgb_numpy(y, co, cg):
    """python.rs:540-583: three 1-D int16 arrays of equal length -> 1-D uint8 interleaved RGB."""
    arrs = []
    for name, v in (("y", y), ("co", co), ("cg", cg)):
        a = np.asarray(v)
        if a.dtype != np.int16 or a.ndim != 1:
            raise TypeError(f"{name} must be a 1-D int16 NumPy array")
        arrs.append(a)
    if not (arrs[0].size == arrs[1].size == arrs[2].size):
        raise ValueError("y, co, cg arrays must have the same length")
    for name, a in zip(("y", "co", "cg"), arrs):
        if not a.flags.c_contiguous:
            raise ValueError(f"{name} must be C-contiguous")
    return default_api().ycocg_r_to_rgb(*arrs)


class EncodedChunk:
    """python.rs:287-357 / pipeline.rs:172-313."""

    def __init__(self, handle, api: Api):
        self._h = handle.value if isinstance(handle, C.c_void_p) else handle
        self._api = api

    def __del__(self):
        if getattr(self, "_h", None):
            self._api.lib.alice_codec_chunk_destroy(self._h)
            self._h = None

    @property
    def width(self):
        return self._api.lib.alice_codec_chunk_width(self._h)

    @property
    def height(self):
        return self._api.lib.alice_codec_chunk_height(self._h)

    @property
    def frames(self):
        return self._api.lib.alice_codec_chunk_frames(self._h)

    @property
    def wavelet(self):
        return WAVELET_BYTES[self._api.lib.alice_codec_chunk_wavelet(self._h)]

    @property
    def compressed_size(self):
        return self._api.lib.alice_codec_chunk_compressed_size(self._h)

    def channel_header(self, channel: int):
        clen, step, dz, ns = C.c_uint32(), C.c_int32(), C.c_int32(), C.c_uint32()
        hist = np.zeros(256, np.uint32)
        self._api._chk(self._api.lib.alice_codec_chunk_channel_header(
            self._h, channel, C.byref(clen), C.byref(step), C.byref(dz), C.byref(ns), hist.ctypes.data_as(_capi.u32p)))
        return {"compressed_len": clen.value, "quant_step": step.value, "quant_dead_zone": dz.value,
                "num_symbols": ns.value, "histogram": hist}

    def to_bytes(self) -> bytes:
        n = C.c_uint64()
        p = self._api.lib.alice_codec_chunk_to_bytes64(self._h, C.byref(n))
        if not p:
            self._api._raise()
        return self._api._take(p, n.value)

    @staticmethod
    def from_bytes(data, api: Api | None = None) -> "EncodedChunk":
        api = api or default_api()
        buf = np.frombuffer(bytes(data), dtype=np.uint8)
        h = api.lib.alice_codec_chunk_from_bytes64(buf.ctypes.data_as(_capi.u8p) if buf.size else None, buf.size)
        if not h:
            api._raise(4)
        return EncodedChunk(h, api)

    def __repr__(self):
        # python.rs:343-355
        return f"EncodedChunk({self.width}x{self.height}x{self.frames}, {self.compressed_size} bytes, {self.wavelet})"


ENCODE_WELL_FORMED_TABLES = 1   # ALICE_ENCODE_WELL_FORMED_TABLES
BATCH_WELL_FORMED_TABLES = 4    # ALICE_BATCH_WELL_FORMED_TABLES


class FrameEncoder:
    """python.rs:365-435: FrameEncoder(quality=90, wavelet="cdf53").encode(rgb_frames, width, height, frames).

    well_formed_tables=True: every encode (and rate_curve / encode_to_size) stores, per channel, a histogram whose
    rANS table keeps every used symbol inside [0, 4096), so that the chunk decodes to exactly what was encoded on any
    decoder of the format (DESIGN.md 4.8).  The header histogram is then a table specification, not symbol counts."""

    def __init__(self, quality: int = 90, wavelet="cdf53", api: Api | None = None, well_formed_tables: bool = False):
        if not 0 <= int(quality) <= 255:
            raise OverflowError("quality must fit in u8")
        self._api = api or default_api()
        self.quality, self.wavelet = int(quality), _wavelet_byte(wavelet)
        self.well_formed_tables = bool(well_formed_tables)
        self._flags = ENCODE_WELL_FORMED_TABLES if self.well_formed_tables else 0
        self._h = self._api.lib.alice_codec_encoder_create_ex(self.quality, self.wavelet, self._flags)
        if not self._h:
            self._api._raise()

    def __del__(self):
        if getattr(self, "_h", None):
            self._api.lib.alice_codec_encoder_destroy(self._h)
            self._h = None

    def encode(self, rgb_frames, width: int, height: int, frames: int) -> EncodedChunk:
        a, pa = _u8(rgb_frames)
        h = self._api.lib.alice_codec_encode_stages(self._h, pa if a.size else a.ctypes.data_as(_capi.u8p), a.size,
                                                    width, height, frames, None, None)
        if not h:
            self._api._raise()
        return EncodedChunk(h, self._api)

    def encode_stages(self, rgb_frames, width, height, frames, want_coeffs=True):
        """encode + stage dumps for parity tests: (chunk, coeffs i32 [3][N] or None, symbols u8 [3][N])."""
        a, pa = _u8(rgb_frames)
        pw, ph = width + (width & 1), height + (height & 1)
        pf = 2 if frames == 1 else frames + (frames & 1)
        n = pw * ph * pf if width * height * frames else 0
        coeffs = np.zeros((3, n), np.int32) if want_coeffs else None
        syms = np.zeros((3, n), np.uint8)
        h = self._api.lib.alice_codec_encode_stages(
            self._h, pa, a.size, width, height, frames,
            coeffs.ctypes.data_as(_capi.i32p) if want_coeffs and n else None,
            syms.ctypes.data_as(_capi.u8p) if n else None)
        if not h:
            self._api._raise()
        return EncodedChunk(h, self._api), coeffs, syms

    def rate_curve(self, rgb_frames, width: int, height: int, frames: int, with_hist: bool = False):
        """Predicted .alc size of the chunk at every quantiser step, before any rANS work: {quality: bytes}, one entry per
        step (the largest quality with that step), each an upper bound on len(encode at that quality).to_bytes(); None
        where the reference aborts.  The encoder's wavelet and table mode are used, its quality is not.  with_hist=True
        also returns the symbol histograms, uint32 [64][3][256] (row step - 1): what the headers of default encodes hold.
        With well_formed_tables the sizes bound the well-formed encodes, and no step is None."""
        return self._curve(False, rgb_frames, width, height, frames, with_hist)

    def rate_curve_device(self, d_rgb: int, width: int, height: int, frames: int, stream: int = 0, with_hist: bool = False):
        """rate_curve for RGB in device memory (raw device pointer); waits for the work enqueued on `stream` first"""
        return self._curve(False, d_rgb, width, height, frames, with_hist, device=True, stream=stream)

    def encode_to_size(self, rgb_frames, width: int, height: int, frames: int, max_bytes: int):
        """The chunk at the highest quality whose .alc (to_bytes) is at most max_bytes: (EncodedChunk, quality), the
        chunk byte-identical to FrameEncoder(quality, wavelet, well_formed_tables=...).encode.  The encoder's quality is
        not used.  Raises CodecError InvalidBufferSize if no quality fits."""
        return self._encode_to(self._api.lib.alice_codec_encode_to_size_ex, rgb_frames, width, height, frames,
                               int(max_bytes), self._flags)

    def _need_well_formed(self):
        if not self.well_formed_tables:
            raise ValueError("the PSNR curve describes the well-formed-tables encode only: "
                             "make the encoder with well_formed_tables=True")

    def psnr_curve(self, rgb_frames, width: int, height: int, frames: int, with_sse: bool = False):
        """Exact PSNR of the decode of this encoder's encode at every quantiser step, without any rANS work:
        {quality: dB}, one entry per step (the largest quality with that step), each equal to
        psnr(rgb, FrameDecoder().decode(FrameEncoder(quality, wavelet, well_formed_tables=True).encode(rgb, ...))) bit
        for bit; inf where the decode is exact.  Not monotone in the quality.  with_sse=True also returns the sums of
        squared differences, uint64 [64] (index step - 1).  Well-formed-tables encoders only (DESIGN.md 4.9)."""
        return self._curve(True, rgb_frames, width, height, frames, with_sse)

    def psnr_curve_device(self, d_rgb: int, width: int, height: int, frames: int, stream: int = 0,
                          with_sse: bool = False):
        """psnr_curve for RGB in device memory (raw device pointer); waits for the work enqueued on `stream` first"""
        return self._curve(True, d_rgb, width, height, frames, with_sse, device=True, stream=stream)

    def encode_to_psnr(self, rgb_frames, width: int, height: int, frames: int, min_psnr: float):
        """The chunk at the lowest quality whose decode reaches min_psnr dB: (EncodedChunk, quality), the chunk
        byte-identical to FrameEncoder(quality, wavelet, well_formed_tables=True).encode.  The encoder's quality is not
        used.  Raises CodecError InvalidQuantStep if no quality reaches the target, or if it is NaN."""
        self._need_well_formed()
        return self._encode_to(self._api.lib.alice_codec_encode_to_psnr, rgb_frames, width, height, frames,
                               float(min_psnr))

    def _curve(self, psnr, rgb, width, height, frames, with_extra, device=False, stream=0):
        """The rate curve, or (psnr=True) the PSNR curve, of host RGB or (device=True) of the RGB at device pointer rgb:
        {quality: value}, and with_extra the histograms or the sums of squared differences."""
        L = self._api.lib
        if psnr:
            self._need_well_formed()
            curve, extra = np.zeros(RATE_STEPS, np.float64), np.zeros(RATE_STEPS, np.uint64)
            fn = L.alice_codec_psnr_curve_device if device else L.alice_codec_psnr_curve
            outs, flags = (curve.ctypes.data_as(C.POINTER(C.c_double)), extra.ctypes.data_as(_capi.u64p)), ()
        else:
            curve = np.zeros(RATE_STEPS, np.uint64)
            extra = np.zeros((RATE_STEPS, 3, 256), np.uint32) if with_extra else None
            fn = L.alice_codec_rate_curve_device_ex if device else L.alice_codec_rate_curve_ex
            outs = (curve.ctypes.data_as(_capi.u64p), extra.ctypes.data_as(_capi.u32p) if with_extra else None)
            flags = (self._flags,)
        if device:
            self._api._chk(fn(self.wavelet, C.c_void_p(int(rgb)), width, height, frames, *outs, C.c_void_p(stream), *flags))
        else:
            a, pa = _u8(rgb)
            self._api._chk(fn(self.wavelet, pa, a.size, width, height, frames, *outs, *flags))
        return (_by_quality(curve), extra) if with_extra else _by_quality(curve)

    def _encode_to(self, fn, rgb_frames, width, height, frames, target, *flags):
        """the chunk and quality that alice_codec_encode_to_size_ex or _to_psnr (fn) choose for target"""
        a, pa = _u8(rgb_frames)
        q = C.c_uint8()
        h = fn(self.wavelet, pa, a.size, width, height, frames, target, C.byref(q), *flags)
        if not h:
            self._api._raise()
        return EncodedChunk(h, self._api), q.value


class FrameDecoder:
    """python.rs:443-482: FrameDecoder().decode(chunk) -> 1-D uint8 RGB array."""

    def __init__(self, api: Api | None = None):
        self._api = api or default_api()

    def decode(self, chunk: EncodedChunk) -> np.ndarray:
        n = C.c_uint64()
        p = self._api.lib.alice_codec_decode_stages(chunk._h, C.byref(n), None)
        if not p:
            self._api._raise()
        return self._api._take_np(p, n.value)

    def decode_stages(self, chunk: EncodedChunk):
        hdr = chunk.channel_header(0)
        ns = hdr["num_symbols"]
        syms = np.zeros((3, ns), np.uint8)
        n = C.c_uint64()
        p = self._api.lib.alice_codec_decode_stages(chunk._h, C.byref(n), syms.ctypes.data_as(_capi.u8p) if ns else None)
        if not p:
            self._api._raise()
        return self._api._take_np(p, n.value), syms


class ReferenceAbi:
    """The 20 reference symbols exactly as a Unity/UE5/ctypes consumer of the reference's cdylib would call them
    (ffi.rs:16-315; u32 lengths, null on error)."""

    def __init__(self, api: Api | None = None):
        self._api = api or default_api()
        self.lib = self._api.lib

    def encode_to_bytes(self, rgb, width, height, frames, quality=90):
        L = self.lib
        a, pa = _u8(rgb)
        enc = L.alice_codec_encoder_create(quality)
        try:
            ck = L.alice_codec_encode(enc, pa, a.size, width, height, frames)
            if not ck:
                return None
            try:
                n = C.c_uint32()
                p = L.alice_codec_chunk_to_bytes(ck, C.byref(n))
                try:
                    return C.string_at(p, n.value)
                finally:
                    L.alice_codec_data_free(p, n.value)
            finally:
                L.alice_codec_chunk_destroy(ck)
        finally:
            L.alice_codec_encoder_destroy(enc)

    def decode_from_bytes(self, alc: bytes):
        L = self.lib
        buf = np.frombuffer(bytes(alc), dtype=np.uint8)
        ck = L.alice_codec_chunk_from_bytes(buf.ctypes.data_as(_capi.u8p), buf.size)
        if not ck:
            return None
        try:
            n = C.c_uint32()
            p = L.alice_codec_decode(ck, C.byref(n))
            if not p:
                return None
            try:
                out = np.empty(n.value, np.uint8)
                if n.value:
                    C.memmove(out.ctypes.data, p, n.value)
                return out
            finally:
                L.alice_codec_data_free(p, n.value)
        finally:
            L.alice_codec_chunk_destroy(ck)


class ChunkBatch:
    """Many independent chunks of one shape in flight on one GPU (the throughput path):
    wraps the alice_codec_batch_* entry points.  Device pointers are plain integers
    (e.g. torch.Tensor.data_ptr()); `stream` is a cudaStream_t value (0 = default stream).
    well_formed_tables=True: every encode of the batch stores well-formed table specifications, as
    FrameEncoder(..., well_formed_tables=True) does."""

    def __init__(self, quality, wavelet, width, height, frames, n_chunks, stream: int = 0, api: Api | None = None,
                 shared_workspace: bool = False, payload_bytes_per_chunk: int = 0, small_smem_kernels: bool = False,
                 well_formed_tables: bool = False):
        self._api = api or default_api()
        self.n_chunks = n_chunks
        self.shape = (width, height, frames)
        self.shared_workspace = shared_workspace
        self.well_formed_tables = bool(well_formed_tables)
        flags = ((1 if shared_workspace else 0) | (2 if small_smem_kernels else 0) |
                 (BATCH_WELL_FORMED_TABLES if well_formed_tables else 0))
        self._h = self._api.lib.alice_codec_batch_create_ex2(int(quality), _wavelet_byte(wavelet), width, height, frames,
                                                             n_chunks, C.c_void_p(stream), flags,
                                                             int(payload_bytes_per_chunk))
        if not self._h:
            self._api._raise()

    def close(self):
        if getattr(self, "_h", None):
            self._api.lib.alice_codec_batch_destroy(self._h)
            self._h = None

    __del__ = close

    @staticmethod
    def _ptr_array(ptrs):
        arr = (C.c_void_p * len(ptrs))(*[C.c_void_p(int(p)) for p in ptrs])
        return arr

    def workspace_bytes(self):
        return self._api.lib.alice_codec_batch_workspace_bytes(self._h)

    def encode_device(self, d_rgb_ptrs, d_workspace_ptrs=None):
        """d_workspace_ptrs: per-chunk buffers of workspace_bytes() (shared-workspace batches only); a workspace may
        be the chunk's RGB input or the buffer it is decoded into later."""
        arr = self._ptr_array(d_rgb_ptrs)
        if d_workspace_ptrs is not None:
            ws = self._ptr_array(d_workspace_ptrs)
            self._api._chk(self._api.lib.alice_codec_batch_encode_device_ws(self._h, arr, ws, len(d_rgb_ptrs)))
            return
        self._api._chk(self._api.lib.alice_codec_batch_encode_device(self._h, arr, len(d_rgb_ptrs)))

    def decode_device(self, d_rgb_out_ptrs):
        arr = self._ptr_array(d_rgb_out_ptrs)
        self._api._chk(self._api.lib.alice_codec_batch_decode_device(self._h, arr, len(d_rgb_out_ptrs)))

    def encode_host(self, h_rgb_ptrs):
        n = len(h_rgb_ptrs)
        arr = self._ptr_array(h_rgb_ptrs)
        out = (C.c_void_p * n)()
        self._api._chk(self._api.lib.alice_codec_batch_encode_host(self._h, arr, n, out))
        return [EncodedChunk(C.c_void_p(out[i]), self._api) for i in range(n)]

    def encode_host_to_size(self, h_rgb_ptrs, max_bytes: int):
        """encode_host with every chunk at the highest quality whose .alc fits max_bytes: (chunks, qualities).  The
        batch's quality is not used."""
        return self._encode_host_to(self._api.lib.alice_codec_batch_encode_host_to_size, h_rgb_ptrs, int(max_bytes))

    def encode_host_to_psnr(self, h_rgb_ptrs, min_psnr: float):
        """encode_host with every chunk at the lowest quality whose decode reaches min_psnr dB: (chunks, qualities).
        Batches made with well_formed_tables=True only; the batch's quality is not used."""
        if not self.well_formed_tables:
            raise ValueError("the PSNR curve describes the well-formed-tables encode only: "
                             "make the batch with well_formed_tables=True")
        return self._encode_host_to(self._api.lib.alice_codec_batch_encode_host_to_psnr, h_rgb_ptrs, float(min_psnr))

    def _encode_host_to(self, fn, h_rgb_ptrs, target):
        """the chunks and qualities that alice_codec_batch_encode_host_to_size or _to_psnr (fn) choose for target"""
        n = len(h_rgb_ptrs)
        arr = self._ptr_array(h_rgb_ptrs)
        out = (C.c_void_p * n)()
        q = np.zeros(max(n, 1), np.uint8)
        self._api._chk(fn(self._h, arr, n, target, out, q.ctypes.data_as(_capi.u8p)))
        return [EncodedChunk(C.c_void_p(out[i]), self._api) for i in range(n)], [int(x) for x in q[:n]]

    def submit_host(self, i, h_rgb_ptr):
        """chunk-at-a-time encode: enqueue the copy and the front-end of chunk i (submit 0, 1, ... in order)"""
        self._api._chk(self._api.lib.alice_codec_batch_submit_host(self._h, i, C.c_void_p(int(h_rgb_ptr))))

    def sync(self):
        self._api._chk(self._api.lib.alice_codec_batch_sync(self._h))

    def collect(self, n):
        out = (C.c_void_p * n)()
        self._api._chk(self._api.lib.alice_codec_batch_collect(self._h, n, out))
        return [EncodedChunk(C.c_void_p(out[i]), self._api) for i in range(n)]

    def submit_device(self, i, d_rgb_ptr, d_workspace_ptr=None):
        """streaming encode with device pointers: enqueue the front-end of chunk i (submit 0, 1, ... in order); the RGB
        buffer may be rewritten by work enqueued on the batch's stream afterwards"""
        self._api._chk(self._api.lib.alice_codec_batch_submit_device(
            self._h, i, C.c_void_p(int(d_rgb_ptr)), C.c_void_p(int(d_workspace_ptr)) if d_workspace_ptr else None))

    def encode_finish(self, n):
        """tables + all 3n rANS streams of the submitted chunks, one synchronisation (results stay on the device)"""
        self._api._chk(self._api.lib.alice_codec_batch_encode_finish(self._h, n))

    def decode_begin(self, n):
        self._api._chk(self._api.lib.alice_codec_batch_decode_begin(self._h, n))

    def decode_next_device(self, i, d_rgb_out_ptr):
        self._api._chk(self._api.lib.alice_codec_batch_decode_next_device(self._h, i, C.c_void_p(int(d_rgb_out_ptr))))

    def decode_end(self):
        self._api._chk(self._api.lib.alice_codec_batch_decode_end(self._h))

    def decode_host(self, chunks, h_rgb_out_ptrs):
        n = len(chunks)
        cks = (C.c_void_p * n)(*[c._h for c in chunks])
        arr = self._ptr_array(h_rgb_out_ptrs)
        self._api._chk(self._api.lib.alice_codec_batch_decode_host(self._h, cks, n, arr))

    def get_chunk(self, i) -> EncodedChunk:
        h = self._api.lib.alice_codec_batch_get_chunk(self._h, i)
        if not h:
            self._api._raise()
        return EncodedChunk(C.c_void_p(h), self._api)

    def timings(self):
        ms = (C.c_float * 8)()
        self._api._chk(self._api.lib.alice_codec_batch_timings(self._h, ms))
        return list(ms)

    def device_bytes(self):
        return self._api.lib.alice_codec_batch_device_bytes(self._h)


class LosslessSet:
    """BASELINE config 4 on the device (alice_codec_lossless_*): the reference's lossless module (src/lossless.rs:
    transform_2d / inverse_2d = Wavelet2D::cdf53) over a frame set, with the reference's symbol, histogram, table and rANS
    stages per colour channel.  `d_rgb` is a device pointer (integer)."""

    STAGES = {"coeffs": (0, np.int32), "symbols": (1, np.uint8), "hist": (2, np.uint32), "decoded": (3, np.uint8),
              "inverse": (4, np.int32)}

    def __init__(self, width, height, frames, stream: int = 0, api: Api | None = None):
        self._api = api or default_api()
        self.shape = (width, height, frames)
        self.n = width * height * frames
        self._h = self._api.lib.alice_codec_lossless_create(width, height, frames, C.c_void_p(stream))
        if not self._h:
            self._api._raise()

    def close(self):
        if getattr(self, "_h", None):
            self._api.lib.alice_codec_lossless_destroy(self._h)
            self._h = None

    __del__ = close

    def encode_device(self, d_rgb):
        self._api._chk(self._api.lib.alice_codec_lossless_encode_device(self._h, C.c_void_p(int(d_rgb))))

    def decode_device(self):
        self._api._chk(self._api.lib.alice_codec_lossless_decode_device(self._h))

    def fetch(self, what):
        which, dt = self.STAGES[what]
        count = 3 * 256 if what == "hist" else 3 * self.n
        out = np.empty(count, dtype=dt)
        n = C.c_uint64(0)
        self._api._chk(self._api.lib.alice_codec_lossless_fetch(self._h, which, 0, out.ctypes.data_as(C.c_void_p), out.nbytes, C.byref(n)))
        return out.reshape(3, -1)

    def stream(self, channel) -> bytes:
        buf = np.empty(2 * self.n + 2048, dtype=np.uint8)
        n = C.c_uint64(0)
        self._api._chk(self._api.lib.alice_codec_lossless_fetch(self._h, 5, channel, buf.ctypes.data_as(C.c_void_p), buf.nbytes, C.byref(n)))
        return buf[:n.value].tobytes()

    def timings(self):
        ms = (C.c_float * 8)()
        self._api._chk(self._api.lib.alice_codec_lossless_timings(self._h, ms))
        return list(ms)
