// capi.cu — the C ABI of libalice_codec (declared in include/alice_codec.h).
// Part 1 mirrors src/ffi.rs of the reference symbol for symbol; Part 2 are the extensions.
// Every compute entry point runs on the CUDA device; there is no CPU fallback.
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <new>

#include "../../include/alice_codec.h"
#include "engine.h"
#include "lifting.cuh"

using namespace alice;

struct Wavelet1D { int kind; };                       // wavelet.rs:47-50 (step list chosen by kind)
struct FrameEncoder { uint8_t quality; uint8_t wavelet; bool well_formed = false; };   // pipeline.rs:335-340
struct EncodedChunk { Chunk c; };
struct AliceBatch {
    Engine *eng = nullptr;
    uint8_t quality = 0, wavelet = 0;
    std::vector<uint8_t *> stage_ptrs, work_ptrs;
};

#define CU_CHECK_RC(expr)                                                                   \
    do {                                                                                    \
        cudaError_t _e = (expr);                                                            \
        if (_e != cudaSuccess) {                                                            \
            set_error(kErrCuda, std::string(#expr) + ": " + cudaGetErrorString(_e));        \
            return kErrCuda;                                                                \
        }                                                                                   \
    } while (0)

namespace {
// scoped device buffer
struct DevBuf {
    void *p = nullptr;
    bool alloc(size_t bytes) {
        if (cudaMalloc(&p, bytes ? bytes : 16) != cudaSuccess) {
            cudaGetLastError();
            p = nullptr;
            set_error(kErrCuda, "device memory allocation failed");
            return false;
        }
        return true;
    }
    ~DevBuf() { if (p) cudaFree(p); }
    template <class T> T *as() { return reinterpret_cast<T *>(p); }
};

// Rust's Box<[u8]> of length 0 is a dangling non-null pointer that data_free(ptr, 0) ignores (ffi.rs:288-296).  Empty
// results get the address of this static byte: non-null, never malloc'ed, never freed.
uint8_t g_empty_box;
uint8_t *boxed_copy(const uint8_t *src, size_t len) {
    if (len == 0) return &g_empty_box;
    uint8_t *p = (uint8_t *)malloc(len);
    if (p) memcpy(p, src, len);
    return p;
}

// wavelet.rs:392-438 / 441-484 (3-D), :292-340 (2-D), :133-176 (1-D) on device buffers A (data) and B (scratch of the same
// size).  *result = the buffer that holds the transform afterwards: A, except for the fast 2-D path (one out-of-place pass).
int wavelet_nd_device(uint8_t wavelet, bool inverse, int32_t *A, int32_t *B, uint64_t w, uint64_t h, uint64_t d, int ndim,
                      cudaStream_t st, int32_t **result) {
    *result = A;
    if (wavelet_fast_eligible(A, B, (long long)w, (long long)h, (long long)d, ndim)) {
        const size_t fs = (size_t)w * h;
        if (ndim == 2) {               // d images, each transformed on its own
            wavelet_xy_i32(wavelet, inverse, A, B, (int)w, (int)h, (long long)d, st);
            *result = B;
        } else if (!inverse) {
            wavelet_xy_i32(wavelet, false, A, B, (int)w, (int)h, (long long)d, st);
            wavelet_t_i32(wavelet, false, B, A, fs, (int)d, st);
        } else {
            wavelet_t_i32(wavelet, true, A, B, fs, (int)d, st);
            wavelet_xy_i32(wavelet, true, B, A, (int)w, (int)h, (long long)d, st);
        }
        return kOk;
    }
    if (ndim == 2 && d != 1) {         // the step-by-step path transforms one image at a time
        for (uint64_t t = 0; t < d; t++) {
            lift_axis(A + t * w * h, B + t * w * h, wavelet, inverse, inverse ? 1 : 0, (long long)w, (long long)h, 1, st);
            lift_axis(A + t * w * h, B + t * w * h, wavelet, inverse, inverse ? 0 : 1, (long long)w, (long long)h, 1, st);
        }
        return kOk;
    }
    if (!inverse) {
        lift_axis(A, B, wavelet, false, 0, (long long)w, (long long)h, (long long)d, st);
        if (ndim >= 2) lift_axis(A, B, wavelet, false, 1, (long long)w, (long long)h, (long long)d, st);
        if (ndim >= 3) lift_axis(A, B, wavelet, false, 2, (long long)w, (long long)h, (long long)d, st);
    } else {
        if (ndim >= 3) lift_axis(A, B, wavelet, true, 2, (long long)w, (long long)h, (long long)d, st);
        if (ndim >= 2) lift_axis(A, B, wavelet, true, 1, (long long)w, (long long)h, (long long)d, st);
        lift_axis(A, B, wavelet, true, 0, (long long)w, (long long)h, (long long)d, st);
    }
    return kOk;
}

int wavelet_nd(uint8_t wavelet, bool inverse, int32_t *data, uint64_t w, uint64_t h, uint64_t d, int ndim) {
    if (!data) { set_error(kErrNull, "null data"); return kErrNull; }
    if (wavelet > 2) { set_error(kErrBitstream, "unknown wavelet type byte"); return kErrBitstream; }
    unsigned __int128 tot = (unsigned __int128)w * h * d;
    if (tot > ((unsigned __int128)1 << 40)) { set_error(kErrOverflow, "volume too large"); return kErrOverflow; }
    const size_t n = (size_t)tot;
    if (n == 0) return kOk;
    if (!cuda_ready()) return kErrCuda;
    DevBuf a, b;
    if (!a.alloc(n * 4) || !b.alloc(n * 4)) return kErrCuda;
    CU_CHECK_RC(cudaMemcpy(a.p, data, n * 4, cudaMemcpyHostToDevice));
    int32_t *A = a.as<int32_t>(), *B = b.as<int32_t>();
    int32_t *res = A;
    int rc = wavelet_nd_device(wavelet, inverse, A, B, w, h, d, ndim, nullptr, &res);
    if (rc) return rc;
    CU_CHECK_RC(cudaGetLastError());
    CU_CHECK_RC(cudaMemcpy(data, res, n * 4, cudaMemcpyDeviceToHost));
    return kOk;
}

// FrameEncoder::encode validation (pipeline.rs:384-427); returns kOk with empty=true for zero-area input
int validate_encode(uint64_t rgb_len, uint32_t w, uint32_t h, uint32_t f, Dims &d, bool &empty) {
    empty = false;
    int rc = make_dims(w, h, f, d);
    if (rc) return rc;
    if (d.n_pixels == 0) {
        if (rgb_len != 0) { set_error(kErrBufferSize, "buffer size mismatch: expected 0"); return kErrBufferSize; }
        empty = true;
        return kOk;
    }
    if (w == 0 || h == 0) { set_error(kErrDimensions, "invalid dimensions"); return kErrDimensions; }
    unsigned __int128 e = (unsigned __int128)d.n_pixels * 3;
    if (e > (unsigned __int128)UINT64_MAX) { set_error(kErrOverflow, "dimensions overflow usize"); return kErrOverflow; }
    if (rgb_len != (uint64_t)e) { set_error(kErrBufferSize, "buffer size mismatch"); return kErrBufferSize; }
    if (d.padded > 0xffffffffull) {
        // num_symbols and the histogram counts are u32 in the .alc format (pipeline.rs:131-133)
        set_error(kErrOverflow, "padded volume exceeds the u32 symbol count of the .alc format");
        return kErrOverflow;
    }
    return kOk;
}

// Stage 0 of a pooled single-chunk engine, with the copy of the host chunk `rgb` enqueued on the engine's stream; null
// (error set) on failure.
const uint8_t *stage_host_chunk(Engine *e, const uint8_t *rgb, uint64_t rgb_len) {
    uint8_t *stage = e->rgb_stage(0);
    if (stage && cudaMemcpyAsync(stage, rgb, (size_t)rgb_len, cudaMemcpyHostToDevice, e->stream()) != cudaSuccess) {
        set_error(kErrCuda, "H2D copy failed");
        return nullptr;
    }
    return stage;
}

EncodedChunk *encode_impl(const FrameEncoder *enc, const uint8_t *rgb, uint64_t rgb_len, uint32_t w, uint32_t h,
                          uint32_t f, int32_t *coeffs_out, uint8_t *symbols_out) {
    set_error(0, "");
    if (!enc || !rgb) { set_error(kErrNull, "null argument"); return nullptr; }
    Dims d;
    bool empty;
    if (validate_encode(rgb_len, w, h, f, d, empty)) return nullptr;
    EncodedChunk *out = new (std::nothrow) EncodedChunk();
    if (!out) return nullptr;
    out->c.width = w; out->c.height = h; out->c.frames = f;
    out->c.wavelet = enc->wavelet;
    if (empty) return out;  // three default headers, empty payload (pipeline.rs:391-412)
    if (!cuda_ready()) { delete out; return nullptr; }
    Engine *e = acquire_engine(d, enc->well_formed);
    if (!e) { delete out; return nullptr; }
    int rc = kOk;
    DevBuf coef;
    do {
        const uint8_t *stage = stage_host_chunk(e, rgb, rgb_len);
        if (!stage) { rc = kErrCuda; break; }
        if (coeffs_out && !coef.alloc((size_t)d.padded * 3 * 4)) { rc = kErrCuda; break; }
        const uint8_t *ptrs[1] = {stage};
        rc = e->encode_device(enc->quality, enc->wavelet, ptrs, 1, coef.as<int32_t>());
        if (rc) break;
        rc = e->fetch_chunk(0, out->c);
        if (rc) break;
        if (coeffs_out && cudaMemcpy(coeffs_out, coef.p, (size_t)d.padded * 3 * 4, cudaMemcpyDeviceToHost) != cudaSuccess) {
            set_error(kErrCuda, "D2H copy failed"); rc = kErrCuda; break;
        }
        if (symbols_out && cudaMemcpy(symbols_out, e->symbols_dev(0), (size_t)d.padded * 3, cudaMemcpyDeviceToHost) != cudaSuccess) {
            set_error(kErrCuda, "D2H copy failed"); rc = kErrCuda; break;
        }
    } while (0);
    release_engine(e);
    if (rc) { delete out; return nullptr; }
    return out;
}

// ------------------------------------------------------------------------------ rate control
constexpr uint64_t kAlcHeaderBytes = kFixedHeaderBytes + 3 * kChannelHeaderBytes;   // 3138

// the largest quality in 0..=100 whose step is s (every step has one: 63q/100 takes every integer 0..63)
uint8_t quality_for_step(int s) {
    for (int q = 100; q >= 0; q--)
        if (quality_to_step((uint8_t)q) == s) return (uint8_t)q;
    return 100;
}

// the smallest step >= first whose prediction fits max_bytes (the highest quality; sizes are not assumed monotone in the
// step), 0 if there is none
int pick_step(const uint64_t pred[kRateSteps], uint64_t max_bytes, int first) {
    for (int s = first; s <= kRateSteps; s++)
        if (pred[s - 1] != UINT64_MAX && pred[s - 1] <= max_bytes) return s;
    return 0;
}

void set_no_fit_error(const uint64_t pred[kRateSteps], uint64_t max_bytes) {
    uint64_t best = UINT64_MAX;
    for (int i = 0; i < kRateSteps; i++) best = std::min(best, pred[i]);
    set_error(kErrBufferSize, "no quality fits " + std::to_string(max_bytes) + " bytes: the smallest predicted size is " +
                                  (best == UINT64_MAX ? std::string("unbounded (the reference aborts at every step)")
                                                      : std::to_string(best) + " bytes"));
}

bool encode_flags_ok(uint32_t flags) {
    if (flags & ~(uint32_t)ALICE_ENCODE_WELL_FORMED_TABLES) { set_error(kErrDimensions, "unknown encode flag"); return false; }
    return true;
}

// Predicted .alc size of every step for one chunk whose RGB is on the host (device == false) or the device.
int rate_curve_impl(uint8_t wavelet, const uint8_t *rgb, bool device, uint64_t rgb_len, uint32_t w, uint32_t h,
                    uint32_t f, uint64_t *bytes64, uint32_t *hist_out, cudaStream_t user_st, uint32_t flags) {
    set_error(0, "");
    if (!bytes64) { set_error(kErrNull, "null output"); return kErrNull; }
    if (wavelet > 2) { set_error(kErrBitstream, "unknown wavelet type byte"); return kErrBitstream; }
    if (!encode_flags_ok(flags)) return kErrDimensions;
    Dims d;
    bool empty;
    int rc = validate_encode(rgb_len, w, h, f, d, empty);
    if (rc) return rc;
    if (empty) {   // the empty chunk (three default headers) at every step
        for (int i = 0; i < kRateSteps; i++) bytes64[i] = kAlcHeaderBytes;
        if (hist_out) memset(hist_out, 0, (size_t)kRateSteps * 3 * 256 * sizeof(uint32_t));
        return kOk;
    }
    if (!rgb) { set_error(kErrNull, "null argument"); return kErrNull; }
    if (!cuda_ready()) return kErrCuda;
    Engine *e = acquire_engine(d, (flags & ALICE_ENCODE_WELL_FORMED_TABLES) != 0);
    if (!e) return kErrCuda;
    do {
        const uint8_t *src = rgb;
        if (device) {   // the engine's stream waits for the caller's work on the input
            cudaEvent_t ev = nullptr;
            if (cudaEventCreateWithFlags(&ev, cudaEventDisableTiming) != cudaSuccess) { cudaGetLastError(); set_error(kErrCuda, "event creation failed"); rc = kErrCuda; break; }
            cudaError_t ce = cudaEventRecord(ev, user_st);
            if (ce == cudaSuccess) ce = cudaStreamWaitEvent(e->stream(), ev, 0);
            cudaEventDestroy(ev);
            if (ce != cudaSuccess) { cudaGetLastError(); set_error(kErrCuda, "stream ordering failed"); rc = kErrCuda; break; }
        } else {
            src = stage_host_chunk(e, rgb, rgb_len);
            if (!src) { rc = kErrCuda; break; }
        }
        rc = e->rate_curve(wavelet, src, bytes64, hist_out);
    } while (0);
    release_engine(e);
    return rc;
}

// The highest quality whose chunk fits max_bytes, trying steps from first_step on: the rate curve picks the step, one
// real encode checks it (an encode larger than its prediction, which the bound rules out, moves on to the next step).
EncodedChunk *encode_to_size_impl(uint8_t wavelet, const uint8_t *rgb, uint64_t rgb_len, uint32_t w, uint32_t h,
                                  uint32_t f, uint64_t max_bytes, int first_step, uint8_t *quality_out, uint32_t flags) {
    set_error(0, "");
    if (!rgb || !quality_out) { set_error(kErrNull, "null argument"); return nullptr; }
    if (wavelet > 2) { set_error(kErrBitstream, "unknown wavelet type byte"); return nullptr; }
    if (!encode_flags_ok(flags)) return nullptr;
    Dims d;
    bool empty;
    if (validate_encode(rgb_len, w, h, f, d, empty)) return nullptr;
    if (empty) {
        uint64_t pred[kRateSteps];
        for (int i = 0; i < kRateSteps; i++) pred[i] = kAlcHeaderBytes;
        if (max_bytes < kAlcHeaderBytes) { set_no_fit_error(pred, max_bytes); return nullptr; }
        EncodedChunk *out = new (std::nothrow) EncodedChunk();
        if (!out) return nullptr;
        out->c.width = w; out->c.height = h; out->c.frames = f;
        out->c.wavelet = wavelet;
        *quality_out = 100;
        return out;
    }
    if (!cuda_ready()) return nullptr;
    Engine *e = acquire_engine(d, (flags & ALICE_ENCODE_WELL_FORMED_TABLES) != 0);
    if (!e) return nullptr;
    EncodedChunk *out = nullptr;
    do {
        const uint8_t *stage = stage_host_chunk(e, rgb, rgb_len);
        if (!stage) break;
        uint64_t pred[kRateSteps];
        if (e->rate_curve(wavelet, stage, pred, nullptr)) break;
        const uint8_t *ptrs[1] = {stage};
        int step = pick_step(pred, max_bytes, first_step);
        if (!step) { set_no_fit_error(pred, max_bytes); break; }
        for (; step; step = pick_step(pred, max_bytes, step + 1)) {
            out = new (std::nothrow) EncodedChunk();
            if (!out) break;
            if (e->encode_device(quality_for_step(step), wavelet, ptrs, 1, nullptr) || e->fetch_chunk(0, out->c)) {
                delete out; out = nullptr;
                break;
            }
            if (kAlcHeaderBytes + out->c.data.size() <= max_bytes) {
                *quality_out = quality_for_step(step);
                break;
            }
            delete out; out = nullptr;
            set_error(kErrBufferSize, "no quality fits " + std::to_string(max_bytes) + " bytes");
        }
    } while (0);
    release_engine(e);
    return out;
}

uint8_t *decode_impl(const EncodedChunk *chunk, uint64_t *out_len, uint8_t *symbols_out) {
    set_error(0, "");
    if (!chunk || !out_len) { set_error(kErrNull, "null argument"); return nullptr; }
    const Chunk &c = chunk->c;
    Dims d;
    if (make_dims(c.width, c.height, c.frames, d)) return nullptr;
    if (d.n_pixels == 0) { *out_len = 0; return boxed_copy(nullptr, 0); }  // pipeline.rs:543-545
    if (d.padded > 0xffffffffull) { set_error(kErrBitstream, "num_symbols != padded_pixels"); return nullptr; }
    if (!cuda_ready()) return nullptr;
    // cheap header validation first, so that malformed chunks fail without touching the device
    {
        size_t off = 0;
        for (int k = 0; k < 3; k++) {
            if ((uint64_t)c.ch[k].num_symbols != d.padded) { set_error(kErrBitstream, "num_symbols != padded_pixels"); return nullptr; }
            if (off + c.ch[k].compressed_len > c.data.size()) { set_error(kErrBitstream, "compressed data overrun"); return nullptr; }
            off += c.ch[k].compressed_len;
        }
    }
    Engine *e = acquire_engine(d);
    if (!e) return nullptr;
    uint8_t *res = nullptr;
    do {
        uint8_t *stage = e->rgb_stage(0);
        if (!stage) break;
        const Chunk *cks[1] = {&c};
        uint8_t *outs[1] = {stage};
        if (e->decode_chunks(cks, 1, outs)) break;
        const size_t len = (size_t)d.n_pixels * 3;
        res = (uint8_t *)malloc(len);
        if (!res) break;
        if (cudaMemcpy(res, stage, len, cudaMemcpyDeviceToHost) != cudaSuccess) {
            set_error(kErrCuda, "D2H copy failed"); free(res); res = nullptr; break;
        }
        if (symbols_out && cudaMemcpy(symbols_out, e->symbols_dev(0), (size_t)d.padded * 3, cudaMemcpyDeviceToHost) != cudaSuccess) {
            set_error(kErrCuda, "D2H copy failed"); free(res); res = nullptr; break;
        }
        *out_len = len;
    } while (0);
    release_engine(e);
    return res;
}
}  // namespace

#pragma GCC visibility push(default)
extern "C" {

// =============================================================== Part 1: reference ABI
Wavelet1D *alice_codec_wavelet1d_haar(void) { return new (std::nothrow) Wavelet1D{WT_HAAR}; }
Wavelet1D *alice_codec_wavelet1d_cdf53(void) { return new (std::nothrow) Wavelet1D{WT_CDF53}; }
Wavelet1D *alice_codec_wavelet1d_cdf97(void) { return new (std::nothrow) Wavelet1D{WT_CDF97}; }
void alice_codec_wavelet1d_destroy(Wavelet1D *p) { delete p; }

void alice_codec_wavelet1d_forward(const Wavelet1D *wv, int32_t *data, uint32_t len) {
    set_error(0, "");                     // void entry point: callers read alice_codec_last_error() afterwards
    if (!wv || !data || len < 2) return;  // ffi.rs:57
    wavelet_nd((uint8_t)wv->kind, false, data, len, 1, 1, 1);
}
void alice_codec_wavelet1d_inverse(const Wavelet1D *wv, int32_t *data, uint32_t len) {
    set_error(0, "");
    if (!wv || !data || len < 2) return;  // ffi.rs:78
    wavelet_nd((uint8_t)wv->kind, true, data, len, 1, 1, 1);
}

FrameEncoder *alice_codec_encoder_create(uint8_t quality) { return new (std::nothrow) FrameEncoder{quality, WT_CDF53}; }
void alice_codec_encoder_destroy(FrameEncoder *p) { delete p; }

EncodedChunk *alice_codec_encode(const FrameEncoder *enc, const uint8_t *rgb, uint32_t rgb_len, uint32_t width,
                                 uint32_t height, uint32_t frames) {
    return encode_impl(enc, rgb, rgb_len, width, height, frames, nullptr, nullptr);
}

uint8_t *alice_codec_decode(const EncodedChunk *chunk, uint32_t *out_len) {
    if (!chunk || !out_len) return nullptr;
    uint64_t n = 0;
    uint8_t *p = decode_impl(chunk, &n, nullptr);
    if (p) *out_len = (uint32_t)n;  // `rgb.len() as u32`, ffi.rs:157
    return p;
}

void alice_codec_chunk_destroy(EncodedChunk *p) { delete p; }

uint8_t *alice_codec_chunk_to_bytes(const EncodedChunk *chunk, uint32_t *out_len) {
    if (!chunk || !out_len) return nullptr;
    std::vector<uint8_t> b = chunk->c.to_bytes();
    *out_len = (uint32_t)b.size();
    return boxed_copy(b.data(), b.size());
}
EncodedChunk *alice_codec_chunk_from_bytes(const uint8_t *data, uint32_t len) {
    return alice_codec_chunk_from_bytes64(data, len);
}
uint32_t alice_codec_chunk_width(const EncodedChunk *c) { return c ? c->c.width : 0; }
uint32_t alice_codec_chunk_height(const EncodedChunk *c) { return c ? c->c.height : 0; }
uint32_t alice_codec_chunk_frames(const EncodedChunk *c) { return c ? c->c.frames : 0; }

// metrics.rs:16-63 — a 10-line host-side f64 reduction used by callers for reporting; not on the codec path.
double alice_codec_psnr(const uint8_t *a, const uint8_t *b, uint32_t len) {
    if (!a || !b) return -1.0;
    if (len == 0) return INFINITY;
    double sum = 0.0;
    for (uint32_t i = 0; i < len; i++) {
        double diff = (double)a[i] - (double)b[i];
        sum += diff * diff;
    }
    double mse = sum / (double)len;
    if (mse == 0.0) return INFINITY;
    return 10.0 * log10(255.0 * 255.0 / mse);
}

void alice_codec_data_free(uint8_t *ptr, uint32_t len) { if (ptr && len > 0 && ptr != &g_empty_box) free(ptr); }
void alice_codec_string_free(char *s) { free(s); }
char *alice_codec_version(void) {
    const char v[] = "0.1.2";  // CARGO_PKG_VERSION of the reference this library is ABI-compatible with
    char *p = (char *)malloc(sizeof(v));
    if (p) memcpy(p, v, sizeof(v));
    return p;
}

// =============================================================== Part 2: extensions
int32_t alice_codec_last_error(void) { return last_error_code(); }
const char *alice_codec_last_error_message(void) { return last_error_msg(); }

FrameEncoder *alice_codec_encoder_create_with_wavelet(uint8_t quality, uint8_t wavelet) {
    if (wavelet > 2) { set_error(kErrBitstream, "unknown wavelet type byte"); return nullptr; }
    return new (std::nothrow) FrameEncoder{quality, wavelet};
}
FrameEncoder *alice_codec_encoder_create_ex(uint8_t quality, uint8_t wavelet, uint32_t flags) {
    set_error(0, "");
    if (wavelet > 2) { set_error(kErrBitstream, "unknown wavelet type byte"); return nullptr; }
    if (!encode_flags_ok(flags)) return nullptr;
    return new (std::nothrow) FrameEncoder{quality, wavelet, (flags & ALICE_ENCODE_WELL_FORMED_TABLES) != 0};
}
uint8_t alice_codec_chunk_wavelet(const EncodedChunk *c) { return c ? c->c.wavelet : 0; }
uint64_t alice_codec_chunk_compressed_size(const EncodedChunk *c) { return c ? c->c.data.size() : 0; }
int alice_codec_chunk_channel_header(const EncodedChunk *c, uint32_t channel, uint32_t *compressed_len,
                                     int32_t *quant_step, int32_t *quant_dead_zone, uint32_t *num_symbols,
                                     uint32_t *hist256) {
    if (!c || channel > 2) { set_error(kErrNull, "null chunk or channel > 2"); return kErrNull; }
    const ChannelHeader &h = c->c.ch[channel];
    if (compressed_len) *compressed_len = h.compressed_len;
    if (quant_step) *quant_step = h.quant_step;
    if (quant_dead_zone) *quant_dead_zone = h.quant_dead_zone;
    if (num_symbols) *num_symbols = h.num_symbols;
    if (hist256) memcpy(hist256, h.histogram, sizeof(h.histogram));
    return kOk;
}
uint8_t *alice_codec_chunk_to_bytes64(const EncodedChunk *chunk, uint64_t *out_len) {
    if (!chunk || !out_len) return nullptr;
    std::vector<uint8_t> b = chunk->c.to_bytes();
    *out_len = b.size();
    return boxed_copy(b.data(), b.size());
}
EncodedChunk *alice_codec_chunk_from_bytes64(const uint8_t *data, uint64_t len) {
    set_error(0, "");
    if (!data) { set_error(kErrNull, "null data"); return nullptr; }
    EncodedChunk *c = new (std::nothrow) EncodedChunk();
    if (!c) return nullptr;
    if (Chunk::from_bytes(data, (size_t)len, c->c)) { delete c; return nullptr; }
    return c;
}
void alice_codec_data_free64(uint8_t *ptr, uint64_t) { if (ptr != &g_empty_box) free(ptr); }

int alice_codec_rgb_to_ycocg_r(const uint8_t *rgb, uint64_t rgb_len, int16_t *y, int16_t *co, int16_t *cg,
                               uint64_t out_len) {
    set_error(0, "");
    if (rgb_len % 3 != 0) { set_error(kErrBufferSize, "rgb length not a multiple of 3"); return kErrBufferSize; }
    const size_t n = (size_t)(rgb_len / 3);
    if (out_len < n) { set_error(kErrBufferSize, "output smaller than pixel count"); return kErrBufferSize; }
    if (n == 0) return kOk;
    if (!rgb || !y || !co || !cg) { set_error(kErrNull, "null argument"); return kErrNull; }
    if (!cuda_ready()) return kErrCuda;
    DevBuf in, o;
    if (!in.alloc(n * 3) || !o.alloc(n * 6)) return kErrCuda;
    CU_CHECK_RC(cudaMemcpy(in.p, rgb, n * 3, cudaMemcpyHostToDevice));
    int16_t *dy = o.as<int16_t>();
    rgb_to_ycocg(in.as<uint8_t>(), dy, dy + n, dy + 2 * n, n, nullptr);
    CU_CHECK_RC(cudaGetLastError());
    CU_CHECK_RC(cudaMemcpy(y, dy, n * 2, cudaMemcpyDeviceToHost));
    CU_CHECK_RC(cudaMemcpy(co, dy + n, n * 2, cudaMemcpyDeviceToHost));
    CU_CHECK_RC(cudaMemcpy(cg, dy + 2 * n, n * 2, cudaMemcpyDeviceToHost));
    return kOk;
}
int alice_codec_ycocg_r_to_rgb(const int16_t *y, const int16_t *co, const int16_t *cg, uint64_t n64, uint8_t *rgb,
                               uint64_t rgb_len) {
    set_error(0, "");
    const size_t n = (size_t)n64;
    if (rgb_len < (uint64_t)n * 3) { set_error(kErrBufferSize, "rgb_out smaller than 3*n"); return kErrBufferSize; }
    if (n == 0) return kOk;
    if (!rgb || !y || !co || !cg) { set_error(kErrNull, "null argument"); return kErrNull; }
    if (!cuda_ready()) return kErrCuda;
    DevBuf in, o;
    if (!in.alloc(n * 6) || !o.alloc(n * 3)) return kErrCuda;
    int16_t *dy = in.as<int16_t>();
    CU_CHECK_RC(cudaMemcpy(dy, y, n * 2, cudaMemcpyHostToDevice));
    CU_CHECK_RC(cudaMemcpy(dy + n, co, n * 2, cudaMemcpyHostToDevice));
    CU_CHECK_RC(cudaMemcpy(dy + 2 * n, cg, n * 2, cudaMemcpyHostToDevice));
    ycocg_to_rgb(dy, dy + n, dy + 2 * n, o.as<uint8_t>(), n, nullptr);
    CU_CHECK_RC(cudaGetLastError());
    CU_CHECK_RC(cudaMemcpy(rgb, o.p, n * 3, cudaMemcpyDeviceToHost));
    return kOk;
}

int alice_codec_wavelet2d_forward(uint8_t wv, int32_t *data, uint32_t w, uint32_t h) {
    set_error(0, "");
    return wavelet_nd(wv, false, data, w, h, 1, 2);
}
int alice_codec_wavelet2d_inverse(uint8_t wv, int32_t *data, uint32_t w, uint32_t h) {
    set_error(0, "");
    return wavelet_nd(wv, true, data, w, h, 1, 2);
}
int alice_codec_wavelet3d_forward(uint8_t wv, int32_t *data, uint32_t w, uint32_t h, uint32_t d) {
    set_error(0, "");
    return wavelet_nd(wv, false, data, w, h, d, 3);
}
int alice_codec_wavelet3d_inverse(uint8_t wv, int32_t *data, uint32_t w, uint32_t h, uint32_t d) {
    set_error(0, "");
    return wavelet_nd(wv, true, data, w, h, d, 3);
}

// Device-pointer forms of Wavelet2D / Wavelet3D (no host copies; asynchronous on `cuda_stream`).
//   2-D: n_images images of w x h, out of place (d_src -> d_dst, the buffers must not overlap);
//   3-D: one w x h x d volume, in place in d_data with a scratch volume d_tmp of the same size.
int alice_codec_wavelet2d_device(uint8_t wv, int inverse, const int32_t *d_src, int32_t *d_dst, uint32_t w, uint32_t h,
                                 uint32_t n_images, void *cuda_stream) {
    set_error(0, "");
    if (!d_src || !d_dst) { set_error(kErrNull, "null argument"); return kErrNull; }
    if (wv > 2) { set_error(kErrBitstream, "unknown wavelet type byte"); return kErrBitstream; }
    if (!cuda_ready()) return kErrCuda;
    cudaStream_t st = (cudaStream_t)cuda_stream;
    const size_t n = (size_t)w * h * n_images;
    if (n == 0) return kOk;
    if (wavelet_fast_eligible(d_src, d_dst, w, h, n_images, 2)) {
        wavelet_xy_i32(wv, inverse != 0, d_src, d_dst, (int)w, (int)h, (long long)n_images, st);
    } else {
        int32_t *tmp = (int32_t *)scratch_device(n * 4);
        if (!tmp) { set_error(kErrCuda, "scratch allocation failed"); return kErrCuda; }
        CU_CHECK_RC(cudaMemcpyAsync(d_dst, d_src, n * 4, cudaMemcpyDeviceToDevice, st));
        int32_t *res = nullptr;
        int rc = wavelet_nd_device(wv, inverse != 0, d_dst, tmp, w, h, n_images, 2, st, &res);
        if (rc) return rc;
        if (res != d_dst) CU_CHECK_RC(cudaMemcpyAsync(d_dst, res, n * 4, cudaMemcpyDeviceToDevice, st));
    }
    CU_CHECK_RC(cudaGetLastError());
    return kOk;
}
int alice_codec_wavelet3d_device(uint8_t wv, int inverse, int32_t *d_data, int32_t *d_tmp, uint32_t w, uint32_t h, uint32_t d,
                                 void *cuda_stream) {
    set_error(0, "");
    if (!d_data || !d_tmp) { set_error(kErrNull, "null argument"); return kErrNull; }
    if (wv > 2) { set_error(kErrBitstream, "unknown wavelet type byte"); return kErrBitstream; }
    if (!cuda_ready()) return kErrCuda;
    if ((size_t)w * h * d == 0) return kOk;
    int32_t *res = nullptr;
    int rc = wavelet_nd_device(wv, inverse != 0, d_data, d_tmp, w, h, d, 3, (cudaStream_t)cuda_stream, &res);
    if (rc) return rc;
    CU_CHECK_RC(cudaGetLastError());
    return kOk;
}

namespace {
enum ElemOp { OP_QUANT, OP_FASTQ, OP_DEQUANT };
int elementwise_i32(ElemOp op, int32_t step, int32_t dz, const int32_t *in, uint64_t n64, int32_t *out,
                    uint64_t out_len) {
    set_error(0, "");
    unsigned long long recip = 0;
    unsigned shift = 0;
    if (op == OP_FASTQ) {
        // FastQuantizer::new (quant.rs:190-217)
        if (step <= 0) { set_error(kErrQuantStep, "quantization step must be positive"); return kErrQuantStep; }
        const uint32_t su = (uint32_t)step;
        const uint32_t extra = 32 - (uint32_t)__builtin_clz(su);
        shift = 32 + extra;
        const unsigned __int128 power = (unsigned __int128)1 << shift;
        recip = (unsigned long long)((power + su - 1) / su);
    }
    if (out_len < n64) { set_error(kErrBufferSize, "output smaller than input"); return kErrBufferSize; }
    const size_t n = (size_t)n64;
    if (n == 0) return kOk;
    if (!in || !out) { set_error(kErrNull, "null argument"); return kErrNull; }
    if (!cuda_ready()) return kErrCuda;
    DevBuf a, b, flag;
    if (!a.alloc(n * 4) || !b.alloc(n * 4) || !flag.alloc(4)) return kErrCuda;
    CU_CHECK_RC(cudaMemcpy(a.p, in, n * 4, cudaMemcpyHostToDevice));
    CU_CHECK_RC(cudaMemset(flag.p, 0, 4));
    if (op == OP_QUANT) quantize_i32(a.as<int32_t>(), b.as<int32_t>(), n, step, dz, flag.as<int>(), nullptr);
    else if (op == OP_FASTQ) fast_quantize_i32(a.as<int32_t>(), b.as<int32_t>(), n, dz, recip, shift, nullptr);
    else dequantize_i32(a.as<int32_t>(), b.as<int32_t>(), n, step, nullptr);
    CU_CHECK_RC(cudaGetLastError());
    int panic = 0;
    CU_CHECK_RC(cudaMemcpy(&panic, flag.p, 4, cudaMemcpyDeviceToHost));
    CU_CHECK_RC(cudaMemcpy(out, b.p, n * 4, cudaMemcpyDeviceToHost));
    if (panic) { set_error(kErrPanic, "division by zero / overflow: the reference panics"); return kErrPanic; }
    return kOk;
}
}  // namespace

int alice_codec_quantize_buffer(int32_t step, int32_t dz, const int32_t *in, uint64_t n, int32_t *out, uint64_t out_len) {
    return elementwise_i32(OP_QUANT, step, dz, in, n, out, out_len);
}
int alice_codec_dequantize_buffer(int32_t step, const int32_t *in, uint64_t n, int32_t *out, uint64_t out_len) {
    return elementwise_i32(OP_DEQUANT, step, 0, in, n, out, out_len);
}
int alice_codec_fast_quantize_buffer(int32_t step, int32_t dz, const int32_t *in, uint64_t n, int32_t *out, uint64_t out_len) {
    return elementwise_i32(OP_FASTQ, step, dz, in, n, out, out_len);
}

int alice_codec_to_symbols(const int32_t *coeffs, uint64_t n64, uint8_t *symbols, uint64_t symbols_len) {
    set_error(0, "");
    if (symbols_len < n64) { set_error(kErrBufferSize, "symbols smaller than coeffs"); return kErrBufferSize; }
    const size_t n = (size_t)n64;
    if (n == 0) return kOk;
    if (!coeffs || !symbols) { set_error(kErrNull, "null argument"); return kErrNull; }
    if (!cuda_ready()) return kErrCuda;
    DevBuf a, b;
    if (!a.alloc(n * 4) || !b.alloc(n)) return kErrCuda;
    CU_CHECK_RC(cudaMemcpy(a.p, coeffs, n * 4, cudaMemcpyHostToDevice));
    to_symbols_u8(a.as<int32_t>(), b.as<uint8_t>(), n, nullptr);
    CU_CHECK_RC(cudaGetLastError());
    CU_CHECK_RC(cudaMemcpy(symbols, b.p, n, cudaMemcpyDeviceToHost));
    return kOk;
}
int alice_codec_from_symbols(const uint8_t *symbols, uint64_t n64, int32_t *coeffs, uint64_t coeffs_len) {
    set_error(0, "");
    if (coeffs_len < n64) { set_error(kErrBufferSize, "coeffs smaller than symbols"); return kErrBufferSize; }
    const size_t n = (size_t)n64;
    if (n == 0) return kOk;
    if (!coeffs || !symbols) { set_error(kErrNull, "null argument"); return kErrNull; }
    if (!cuda_ready()) return kErrCuda;
    DevBuf a, b;
    if (!a.alloc(n) || !b.alloc(n * 4)) return kErrCuda;
    CU_CHECK_RC(cudaMemcpy(a.p, symbols, n, cudaMemcpyHostToDevice));
    from_symbols_i32(a.as<uint8_t>(), b.as<int32_t>(), n, nullptr);
    CU_CHECK_RC(cudaGetLastError());
    CU_CHECK_RC(cudaMemcpy(coeffs, b.p, n * 4, cudaMemcpyDeviceToHost));
    return kOk;
}
int alice_codec_build_histogram(const uint8_t *symbols, uint64_t n64, uint32_t *hist256) {
    set_error(0, "");
    if (!hist256) { set_error(kErrNull, "null argument"); return kErrNull; }
    const size_t n = (size_t)n64;
    if (n == 0) { memset(hist256, 0, 1024); return kOk; }
    if (!symbols) { set_error(kErrNull, "null argument"); return kErrNull; }
    if (!cuda_ready()) return kErrCuda;
    DevBuf a, h;
    if (!a.alloc(n) || !h.alloc(1024)) return kErrCuda;
    CU_CHECK_RC(cudaMemcpy(a.p, symbols, n, cudaMemcpyHostToDevice));
    CU_CHECK_RC(cudaMemset(h.p, 0, 1024));
    histogram_u8(a.as<uint8_t>(), n, h.as<unsigned>(), nullptr);
    CU_CHECK_RC(cudaGetLastError());
    CU_CHECK_RC(cudaMemcpy(hist256, h.p, 1024, cudaMemcpyDeviceToHost));
    return kOk;
}

double alice_codec_rdo_bpp_from_quality(uint8_t quality) {
    // quant.rs:398-412 — scalar host arithmetic on the configuration byte
    const double RCP_100 = 1.0 / 100.0;
    if (quality > 100) quality = 100;
    double q = (double)quality * RCP_100;
    return fma(q * q, 23.9, 0.1);
}
namespace {
// quant.rs:440-468 — closed form on two scalars: lambda, base step, sub-band strength, dead zone
void rdo_step_from_variance(double target_bpp, double variance, int subband, int32_t *step, int32_t *dead_zone) {
    const double ln2 = 0.693147180559945309417232121458176568;
    const double lambda = (6.0 * ln2 * variance) / target_bpp;
    const double r = round(sqrt(12.0 * lambda));
    int32_t base;
    if (r != r) base = 0;                               // `as i32` saturates, NaN -> 0
    else if (r >= 2147483647.0) base = INT32_MAX;
    else if (r <= -2147483648.0) base = INT32_MIN;
    else base = (int32_t)r;
    if (base < 1) base = 1;
    static const int strength[8] = {1, 2, 2, 4, 2, 4, 4, 8};  // lib.rs:152-159
    int32_t st = (int32_t)((uint32_t)base * (uint32_t)strength[subband]);
    if (st < 1) st = 1;
    *step = st;
    *dead_zone = (int32_t)((uint32_t)st + (uint32_t)(st / 2));
}
// quant.rs:415-435 for up to 8 device-resident views; variance[i] = max(acc / n, 1.0), 1.0 for an empty view
int rdo_variances(const RdoViewHost *views, int n_views, double *variance) {
    double acc[8], mean[8];
    cudaError_t e = rdo_seq_sums(views, n_views, acc, mean, nullptr);
    if (e != cudaSuccess) { set_error(kErrCuda, cudaGetErrorString(e)); return kErrCuda; }
    for (int i = 0; i < n_views; i++) {
        double v = 1.0;
        if (views[i].n > 0) {
            const double inv_n = 1.0 / (double)views[i].n;
            v = acc[i] * inv_n;
            if (!(v > 1.0)) v = 1.0;                    // f64::max(1.0)
        }
        variance[i] = v;
    }
    return kOk;
}
// the 8 octants of a w x h x d volume (lib.rs:115-132: letters are x, y, t; index 4*[x high] + 2*[y high] + [t high]);
// along each axis low = [0, dim/2), high = [dim/2, 2*(dim/2)) (an odd last sample belongs to no sub-band, wavelet.rs:220-233)
void octant_views(const int32_t *d_vol, uint32_t w, uint32_t h, uint32_t d, RdoViewHost v[8]) {
    const uint32_t hx = w / 2, hy = h / 2, ht = d / 2;
    for (int sb = 0; sb < 8; sb++) {
        const uint32_t x0 = (sb & 4) ? hx : 0, y0 = (sb & 2) ? hy : 0, t0 = (sb & 1) ? ht : 0;
        v[sb].base = d_vol + ((size_t)t0 * h + y0) * w + x0;
        v[sb].n = (unsigned long long)hx * hy * ht;
        v[sb].sw = hx ? hx : 1;
        v[sb].sh = hy ? hy : 1;
        v[sb].row = w;
        v[sb].plane = (unsigned long long)w * h;
    }
}
bool fastq_constants(int32_t step, unsigned long long *recip, unsigned *shift) {
    if (step <= 0) return false;                        // FastQuantizer::new (quant.rs:190-217)
    const uint32_t su = (uint32_t)step;
    const uint32_t extra = 32 - (uint32_t)__builtin_clz(su);
    *shift = 32 + extra;
    const unsigned __int128 power = (unsigned __int128)1 << *shift;
    *recip = (unsigned long long)((power + su - 1) / su);
    return true;
}
}  // namespace

int alice_codec_rdo_compute_quantizer(double target_bpp, const int32_t *coeffs, uint64_t n64, uint8_t subband,
                                      int32_t *step, int32_t *dead_zone) {
    set_error(0, "");
    if (subband > 7 || !step || !dead_zone) { set_error(kErrNull, "bad subband or null output"); return kErrNull; }
    const size_t n = (size_t)n64;
    double variance = 1.0;  // quant.rs:416-418
    if (n > 0) {
        if (!coeffs) { set_error(kErrNull, "null argument"); return kErrNull; }
        if (!cuda_ready()) return kErrCuda;
        DevBuf a;
        if (!a.alloc(n * 4)) return kErrCuda;
        CU_CHECK_RC(cudaMemcpy(a.p, coeffs, n * 4, cudaMemcpyHostToDevice));
        RdoViewHost v;
        v.base = a.as<int32_t>(); v.n = n; v.sw = 1u << 20; v.sh = 1u << 20;   // a flat slice: rows of 2^20 elements
        v.row = v.sw; v.plane = (unsigned long long)v.sw * v.sh;
        int rc = rdo_variances(&v, 1, &variance);
        if (rc != kOk) return rc;
    }
    rdo_step_from_variance(target_bpp, variance, subband, step, dead_zone);
    return kOk;
}

// AnalyticalRDO::estimate_variance (quant.rs:415-435; private in the reference, exported for the parity tests)
int alice_codec_rdo_estimate_variance(const int32_t *coeffs, uint64_t n64, double *variance_out) {
    set_error(0, "");
    if (!variance_out) { set_error(kErrNull, "null output"); return kErrNull; }
    const size_t n = (size_t)n64;
    *variance_out = 1.0;
    if (n == 0) return kOk;
    if (!coeffs) { set_error(kErrNull, "null argument"); return kErrNull; }
    if (!cuda_ready()) return kErrCuda;
    DevBuf a;
    if (!a.alloc(n * 4)) return kErrCuda;
    CU_CHECK_RC(cudaMemcpy(a.p, coeffs, n * 4, cudaMemcpyHostToDevice));
    RdoViewHost v;
    v.base = a.as<int32_t>(); v.n = n; v.sw = 1u << 20; v.sh = 1u << 20;
    v.row = v.sw; v.plane = (unsigned long long)v.sw * v.sh;
    return rdo_variances(&v, 1, variance_out);
}

// AnalyticalRDO::compute_all_quantizers (quant.rs:472-490) on the octants of a forward-transformed volume, each
// octant gathered in row-major (t, y, x) order; steps8 / dead_zones8 are indexed by the SubBand3D byte.
int alice_codec_rdo_compute_all_quantizers(double target_bpp, const int32_t *volume, uint32_t w, uint32_t h, uint32_t d,
                                           int32_t *steps8, int32_t *dead_zones8) {
    set_error(0, "");
    if (!steps8 || !dead_zones8) { set_error(kErrNull, "null output"); return kErrNull; }
    const unsigned __int128 tot = (unsigned __int128)w * h * d;
    if (tot > ((unsigned __int128)1 << 40)) { set_error(kErrOverflow, "dimension overflow"); return kErrOverflow; }
    const size_t n = (size_t)tot;
    double variance[8];
    for (int i = 0; i < 8; i++) variance[i] = 1.0;
    if (n > 0) {
        if (!volume) { set_error(kErrNull, "null argument"); return kErrNull; }
        if (!cuda_ready()) return kErrCuda;
        DevBuf a;
        if (!a.alloc(n * 4)) return kErrCuda;
        CU_CHECK_RC(cudaMemcpy(a.p, volume, n * 4, cudaMemcpyHostToDevice));
        RdoViewHost v[8];
        octant_views(a.as<int32_t>(), w, h, d, v);
        int rc = rdo_variances(v, 8, variance);
        if (rc != kOk) return rc;
    }
    for (int sb = 0; sb < 8; sb++) rdo_step_from_variance(target_bpp, variance[sb], sb, &steps8[sb], &dead_zones8[sb]);
    return kOk;
}

// the same for a volume that is already on the device (synchronises the default stream)
int alice_codec_rdo_compute_all_quantizers_device(double target_bpp, const int32_t *d_volume, uint32_t w, uint32_t h,
                                                  uint32_t d, int32_t *steps8, int32_t *dead_zones8) {
    set_error(0, "");
    if (!steps8 || !dead_zones8) { set_error(kErrNull, "null output"); return kErrNull; }
    const unsigned __int128 tot = (unsigned __int128)w * h * d;
    if (tot > ((unsigned __int128)1 << 40)) { set_error(kErrOverflow, "dimension overflow"); return kErrOverflow; }
    double variance[8];
    for (int i = 0; i < 8; i++) variance[i] = 1.0;
    if (tot > 0) {
        if (!d_volume) { set_error(kErrNull, "null argument"); return kErrNull; }
        if (!cuda_ready()) return kErrCuda;
        RdoViewHost v[8];
        octant_views(d_volume, w, h, d, v);
        int rc = rdo_variances(v, 8, variance);
        if (rc != kOk) return rc;
    }
    for (int sb = 0; sb < 8; sb++) rdo_step_from_variance(target_bpp, variance[sb], sb, &steps8[sb], &dead_zones8[sb]);
    return kOk;
}

// statistics -> quantisers -> FastQuantizer::quantize_buffer per octant (README.md:143-147 "manual pipeline", applied
// per sub-band): out[i] = FastQuantizer::from(quantizers[octant(i)]).quantize(volume[i]).  The volume stays on the device
// between the statistics and the quantiser pass.
int alice_codec_rdo_quantize_volume(double target_bpp, const int32_t *volume, uint32_t w, uint32_t h, uint32_t d,
                                    int32_t *out, uint64_t out_len, int32_t *steps8, int32_t *dead_zones8) {
    set_error(0, "");
    if (!steps8 || !dead_zones8) { set_error(kErrNull, "null output"); return kErrNull; }
    const unsigned __int128 tot = (unsigned __int128)w * h * d;
    if (tot > ((unsigned __int128)1 << 40)) { set_error(kErrOverflow, "dimension overflow"); return kErrOverflow; }
    const size_t n = (size_t)tot;
    if (out_len < n) { set_error(kErrBufferSize, "output smaller than input"); return kErrBufferSize; }
    double variance[8];
    for (int i = 0; i < 8; i++) variance[i] = 1.0;
    DevBuf a, b;
    if (n > 0) {
        if (!volume || !out) { set_error(kErrNull, "null argument"); return kErrNull; }
        if (!cuda_ready()) return kErrCuda;
        if (!a.alloc(n * 4) || !b.alloc(n * 4)) return kErrCuda;
        CU_CHECK_RC(cudaMemcpy(a.p, volume, n * 4, cudaMemcpyHostToDevice));
        RdoViewHost v[8];
        octant_views(a.as<int32_t>(), w, h, d, v);
        int rc = rdo_variances(v, 8, variance);
        if (rc != kOk) return rc;
    }
    int dz[8];
    unsigned long long recip[8];
    unsigned shift[8];
    for (int sb = 0; sb < 8; sb++) {
        rdo_step_from_variance(target_bpp, variance[sb], sb, &steps8[sb], &dead_zones8[sb]);
        dz[sb] = dead_zones8[sb];
        fastq_constants(steps8[sb], &recip[sb], &shift[sb]);    // steps are >= 1 by construction
    }
    if (n > 0) {
        rdo_quantize_volume(a.as<int32_t>(), b.as<int32_t>(), w, h, d, dz, recip, shift, nullptr);
        CU_CHECK_RC(cudaGetLastError());
        CU_CHECK_RC(cudaMemcpy(out, b.p, n * 4, cudaMemcpyDeviceToHost));
    }
    return kOk;
}

int alice_codec_freq_table_from_histogram(const uint32_t *hist, uint32_t n_symbols, uint16_t *cum256,
                                          uint16_t *freq256, uint8_t *lut4096) {
    set_error(0, "");
    if (!hist) { set_error(kErrNull, "null argument"); return kErrNull; }
    if (n_symbols == 0) { set_error(kErrPanic, "empty histogram: the reference divides by zero"); return kErrPanic; }
    if (n_symbols > 256) { set_error(kErrDimensions, "n_symbols > 256"); return kErrDimensions; }
    if (!cuda_ready()) return kErrCuda;
    DevBuf h, enc, dec, aux, fr, cu, l8;
    if (!h.alloc(1024) || !enc.alloc(kEncTableBytes) || !dec.alloc(kDecLutEntries * 4) || !aux.alloc(sizeof(DecAux)) ||
        !fr.alloc(512) || !cu.alloc(512) || !l8.alloc(4096))
        return kErrCuda;
    CU_CHECK_RC(cudaMemset(h.p, 0, 1024));
    CU_CHECK_RC(cudaMemcpy(h.p, hist, n_symbols * 4, cudaMemcpyHostToDevice));
    build_tables(h.as<unsigned>(), 1, (int)n_symbols, enc.as<EncSym>(), dec.as<uint32_t>(), aux.as<DecAux>(),
                 fr.as<uint16_t>(), cu.as<uint16_t>(), l8.as<uint8_t>(), nullptr);
    CU_CHECK_RC(cudaGetLastError());
    if (freq256) CU_CHECK_RC(cudaMemcpy(freq256, fr.p, 512, cudaMemcpyDeviceToHost));
    if (cum256) CU_CHECK_RC(cudaMemcpy(cum256, cu.p, 512, cudaMemcpyDeviceToHost));
    if (lut4096) CU_CHECK_RC(cudaMemcpy(lut4096, l8.p, 4096, cudaMemcpyDeviceToHost));
    return kOk;
}

int alice_codec_rans_encode(const uint8_t *symbols, uint64_t n64, const uint32_t *hist, uint32_t n_symbols,
                            uint8_t **out, uint64_t *out_len) {
    set_error(0, "");
    if (!hist || !out || !out_len || (n64 && !symbols)) { set_error(kErrNull, "null argument"); return kErrNull; }
    if (n_symbols == 0) { set_error(kErrPanic, "empty histogram"); return kErrPanic; }
    if (n_symbols > 256) { set_error(kErrDimensions, "n_symbols > 256"); return kErrDimensions; }
    const size_t n = (size_t)n64;
    for (size_t i = 0; i < n; i++)
        if (symbols[i] >= n_symbols) {  // table.get_symbol would index out of bounds (rans.rs:195)
            set_error(kErrPanic, "symbol outside the table");
            return kErrPanic;
        }
    if (!cuda_ready()) return kErrCuda;
    const size_t cap = rans_enc_worst_case(n);
    DevBuf h, enc, dec, aux, sy, pay, job, res;
    if (!h.alloc(1024) || !enc.alloc(kEncTableBytes) || !dec.alloc(kDecLutEntries * 4) || !aux.alloc(sizeof(DecAux)) ||
        !sy.alloc(n) || !pay.alloc(cap) || !job.alloc(sizeof(RansEncJob)) || !res.alloc(16))
        return kErrCuda;
    CU_CHECK_RC(cudaMemset(h.p, 0, 1024));
    CU_CHECK_RC(cudaMemcpy(h.p, hist, n_symbols * 4, cudaMemcpyHostToDevice));
    if (n) CU_CHECK_RC(cudaMemcpy(sy.p, symbols, n, cudaMemcpyHostToDevice));
    build_tables(h.as<unsigned>(), 1, (int)n_symbols, enc.as<EncSym>(), dec.as<uint32_t>(), aux.as<DecAux>(), nullptr,
                 nullptr, nullptr, nullptr);
    RansEncJob j;
    j.symbols = sy.as<uint8_t>(); j.n = n; j.out = pay.as<uint8_t>(); j.cap = cap;
    CU_CHECK_RC(cudaMemcpy(job.p, &j, sizeof(j), cudaMemcpyHostToDevice));
    rans_encode(job.as<RansEncJob>(), enc.as<EncSym>(), nullptr, res.as<unsigned long long>(), 1, nullptr);
    CU_CHECK_RC(cudaGetLastError());
    unsigned long long r[2] = {0, 0};
    CU_CHECK_RC(cudaMemcpy(r, res.p, 16, cudaMemcpyDeviceToHost));
    if (r[1] & 2) { set_error(kErrPanic, "symbol with zero frequency in use: the reference aborts"); return kErrPanic; }
    if (r[1]) { set_error(kErrCuda, "rANS output overflow"); return kErrCuda; }
    uint8_t *p = (uint8_t *)malloc((size_t)r[0] ? (size_t)r[0] : 1);
    if (!p) { set_error(kErrCuda, "host allocation failed"); return kErrCuda; }
    CU_CHECK_RC(cudaMemcpy(p, pay.as<uint8_t>() + cap - r[0], (size_t)r[0], cudaMemcpyDeviceToHost));
    *out = p;
    *out_len = r[0];
    return kOk;
}

int alice_codec_rans_decode(const uint8_t *stream, uint64_t len64, const uint32_t *hist, uint32_t n_symbols,
                            uint8_t *symbols_out, uint64_t n64) {
    set_error(0, "");
    if (!hist || (n64 && !symbols_out) || (len64 && !stream)) { set_error(kErrNull, "null argument"); return kErrNull; }
    if (n_symbols == 0) { set_error(kErrPanic, "empty histogram"); return kErrPanic; }
    if (n_symbols > 256) { set_error(kErrDimensions, "n_symbols > 256"); return kErrDimensions; }
    const size_t n = (size_t)n64, len = (size_t)len64;
    if (n == 0) return kOk;
    if (!cuda_ready()) return kErrCuda;
    DevBuf h, enc, dec, aux, sy, in, job;
    if (!h.alloc(1024) || !enc.alloc(kEncTableBytes) || !dec.alloc(kDecLutEntries * 4) || !aux.alloc(sizeof(DecAux)) ||
        !sy.alloc(n) || !in.alloc(len + 32) || !job.alloc(sizeof(RansDecJob)))
        return kErrCuda;
    CU_CHECK_RC(cudaMemset(h.p, 0, 1024));
    CU_CHECK_RC(cudaMemcpy(h.p, hist, n_symbols * 4, cudaMemcpyHostToDevice));
    if (len) CU_CHECK_RC(cudaMemcpy(in.p, stream, len, cudaMemcpyHostToDevice));
    build_tables(h.as<unsigned>(), 1, (int)n_symbols, enc.as<EncSym>(), dec.as<uint32_t>(), aux.as<DecAux>(), nullptr,
                 nullptr, nullptr, nullptr);
    RansDecJob j;
    j.in = in.as<uint8_t>(); j.len = len; j.symbols = sy.as<uint8_t>(); j.n = n;
    CU_CHECK_RC(cudaMemcpy(job.p, &j, sizeof(j), cudaMemcpyHostToDevice));
    rans_decode(job.as<RansDecJob>(), dec.as<uint32_t>(), aux.as<DecAux>(), 1, nullptr);
    CU_CHECK_RC(cudaGetLastError());
    CU_CHECK_RC(cudaMemcpy(symbols_out, sy.p, n, cudaMemcpyDeviceToHost));
    return kOk;
}

// InterleavedRansEncoder::{encode, finish} (rans.rs:393-459): four independent RansEncoder streams over symbols
// i % 4 == k, run as four lanes of the one-warp-per-stream kernel; container = 4 lengths + 4 counts + the streams.
int alice_codec_rans_encode_interleaved(const uint8_t *symbols, uint64_t n64, const uint32_t *hist, uint32_t n_symbols,
                                        uint8_t **out, uint64_t *out_len) {
    set_error(0, "");
    if (!hist || !out || !out_len || (n64 && !symbols)) { set_error(kErrNull, "null argument"); return kErrNull; }
    if (n_symbols == 0) { set_error(kErrPanic, "empty histogram"); return kErrPanic; }
    if (n_symbols > 256) { set_error(kErrDimensions, "n_symbols > 256"); return kErrDimensions; }
    const size_t n = (size_t)n64;
    for (size_t i = 0; i < n; i++)
        if (symbols[i] >= n_symbols) { set_error(kErrPanic, "symbol outside the table"); return kErrPanic; }
    if (!cuda_ready()) return kErrCuda;
    size_t count[4];
    for (int k = 0; k < 4; k++) count[k] = (n + 3 - (size_t)k) / 4;             // rans.rs:421-423
    const size_t stride = (count[0] + 15) / 16 * 16 + 16;
    const size_t cap = rans_enc_worst_case(count[0]);
    DevBuf h, enc, dec, aux, sy, pl, pay, job, res;
    if (!h.alloc(4 * 1024) || !enc.alloc(4 * kEncTableBytes) || !dec.alloc(4 * kDecLutEntries * 4) ||
        !aux.alloc(4 * sizeof(DecAux)) || !sy.alloc(n) || !pl.alloc(4 * stride) || !pay.alloc(4 * cap) ||
        !job.alloc(4 * sizeof(RansEncJob)) || !res.alloc(4 * 16))
        return kErrCuda;
    CU_CHECK_RC(cudaMemset(h.p, 0, 4 * 1024));
    for (int k = 0; k < 4; k++)
        CU_CHECK_RC(cudaMemcpy(h.as<uint8_t>() + 1024 * k, hist, n_symbols * 4, cudaMemcpyHostToDevice));
    if (n) CU_CHECK_RC(cudaMemcpy(sy.p, symbols, n, cudaMemcpyHostToDevice));
    deinterleave4_u8(sy.as<uint8_t>(), n, pl.as<uint8_t>(), stride, nullptr);
    build_tables(h.as<unsigned>(), 4, (int)n_symbols, enc.as<EncSym>(), dec.as<uint32_t>(), aux.as<DecAux>(), nullptr,
                 nullptr, nullptr, nullptr);
    RansEncJob j[4];
    for (int k = 0; k < 4; k++) {
        j[k].symbols = pl.as<uint8_t>() + k * stride; j[k].n = count[k];
        j[k].out = pay.as<uint8_t>() + k * cap; j[k].cap = cap;
    }
    CU_CHECK_RC(cudaMemcpy(job.p, j, sizeof(j), cudaMemcpyHostToDevice));
    rans_encode(job.as<RansEncJob>(), enc.as<EncSym>(), nullptr, res.as<unsigned long long>(), 4, nullptr);
    CU_CHECK_RC(cudaGetLastError());
    unsigned long long r[8];
    CU_CHECK_RC(cudaMemcpy(r, res.p, sizeof(r), cudaMemcpyDeviceToHost));
    size_t total = 32;
    for (int k = 0; k < 4; k++) {
        if (r[2 * k + 1] & 2) { set_error(kErrPanic, "symbol with zero frequency in use: the reference aborts"); return kErrPanic; }
        if (r[2 * k + 1]) { set_error(kErrCuda, "rANS output overflow"); return kErrCuda; }
        total += (size_t)r[2 * k];
    }
    uint8_t *p = (uint8_t *)malloc(total);
    if (!p) { set_error(kErrCuda, "host allocation failed"); return kErrCuda; }
    size_t o = 32;
    for (int k = 0; k < 4; k++) {
        const uint32_t len = (uint32_t)r[2 * k], cnt = (uint32_t)count[k];     // `as u32` (rans.rs:443, 449)
        memcpy(p + 4 * k, &len, 4);
        memcpy(p + 16 + 4 * k, &cnt, 4);
        if (cudaMemcpy(p + o, pay.as<uint8_t>() + k * cap + cap - r[2 * k], (size_t)r[2 * k], cudaMemcpyDeviceToHost) != cudaSuccess) {
            free(p);
            set_error(kErrCuda, "copy failed");
            return kErrCuda;
        }
        o += (size_t)r[2 * k];
    }
    *out = p;
    *out_len = total;
    return kOk;
}

// InterleavedRansDecoder::{new, decode_n} (rans.rs:465-524).  Slices past the input (the reference panics) and
// n larger than the four symbol counts (the reference spins forever, rans.rs:511-513) return ALICE_ERR_PANIC.
int alice_codec_rans_decode_interleaved(const uint8_t *stream, uint64_t len64, const uint32_t *hist, uint32_t n_symbols,
                                        uint8_t *symbols_out, uint64_t n64) {
    set_error(0, "");
    if (!hist || (n64 && !symbols_out) || (len64 && !stream)) { set_error(kErrNull, "null argument"); return kErrNull; }
    if (n_symbols == 0) { set_error(kErrPanic, "empty histogram"); return kErrPanic; }
    if (n_symbols > 256) { set_error(kErrDimensions, "n_symbols > 256"); return kErrDimensions; }
    const size_t n = (size_t)n64, len = (size_t)len64;
    if (len < 32) { set_error(kErrPanic, "container shorter than its 32-byte header: the reference panics"); return kErrPanic; }
    size_t slen[4], start[4];
    unsigned long long cnt[4], total = 0;
    size_t o = 32;
    for (int k = 0; k < 4; k++) {
        uint32_t l, c;
        memcpy(&l, stream + 4 * k, 4);
        memcpy(&c, stream + 16 + 4 * k, 4);
        slen[k] = l; cnt[k] = c; total += c; start[k] = o;
        o += l;
        if (o > len) { set_error(kErrPanic, "stream lengths exceed the container: the reference panics"); return kErrPanic; }
    }
    if (n > total) { set_error(kErrPanic, "more symbols requested than the streams hold: the reference never returns"); return kErrPanic; }
    if (n == 0) return kOk;
    if (!cuda_ready()) return kErrCuda;
    // symbols each stream contributes to the first n outputs: rounds are complete up to r, then a partial round
    unsigned long long need[4] = {0, 0, 0, 0};
    {
        unsigned long long left = n, r = 0;
        while (left) {
            unsigned m = 0;
            unsigned long long r_next = ~0ull;
            for (int k = 0; k < 4; k++) if (cnt[k] > r) { m++; if (cnt[k] < r_next) r_next = cnt[k]; }
            const unsigned long long full = (r_next - r) * m;
            if (left >= full) { for (int k = 0; k < 4; k++) if (cnt[k] > r) need[k] = r_next; left -= full; r = r_next; continue; }
            const unsigned long long q = left / m, rem = left % m;
            unsigned seen = 0;
            for (int k = 0; k < 4; k++) if (cnt[k] > r) { need[k] = r + q + (seen < rem ? 1 : 0); seen++; }
            left = 0;
        }
    }
    unsigned long long max_need = 0;
    for (int k = 0; k < 4; k++) if (need[k] > max_need) max_need = need[k];
    const size_t stride = ((size_t)max_need + 15) / 16 * 16 + 16;
    DevBuf h, enc, dec, aux, pl, in, job, outb;
    if (!h.alloc(4 * 1024) || !enc.alloc(4 * kEncTableBytes) || !dec.alloc(4 * kDecLutEntries * 4) ||
        !aux.alloc(4 * sizeof(DecAux)) || !pl.alloc(4 * stride) || !in.alloc(len + 32) ||
        !job.alloc(4 * sizeof(RansDecJob)) || !outb.alloc(n))
        return kErrCuda;
    CU_CHECK_RC(cudaMemset(h.p, 0, 4 * 1024));
    for (int k = 0; k < 4; k++)
        CU_CHECK_RC(cudaMemcpy(h.as<uint8_t>() + 1024 * k, hist, n_symbols * 4, cudaMemcpyHostToDevice));
    CU_CHECK_RC(cudaMemcpy(in.p, stream, len, cudaMemcpyHostToDevice));
    build_tables(h.as<unsigned>(), 4, (int)n_symbols, enc.as<EncSym>(), dec.as<uint32_t>(), aux.as<DecAux>(), nullptr,
                 nullptr, nullptr, nullptr);
    RansDecJob j[4];
    for (int k = 0; k < 4; k++) {
        j[k].in = in.as<uint8_t>() + start[k]; j[k].len = slen[k];
        j[k].symbols = pl.as<uint8_t>() + k * stride; j[k].n = need[k];
    }
    CU_CHECK_RC(cudaMemcpy(job.p, j, sizeof(j), cudaMemcpyHostToDevice));
    rans_decode(job.as<RansDecJob>(), dec.as<uint32_t>(), aux.as<DecAux>(), 4, nullptr);
    interleave_rr_u8(pl.as<uint8_t>(), stride, outb.as<uint8_t>(), n, cnt, nullptr);
    CU_CHECK_RC(cudaGetLastError());
    CU_CHECK_RC(cudaMemcpy(symbols_out, outb.p, n, cudaMemcpyDeviceToHost));
    return kOk;
}

EncodedChunk *alice_codec_encode_stages(const FrameEncoder *enc, const uint8_t *rgb, uint64_t rgb_len, uint32_t w,
                                        uint32_t h, uint32_t f, int32_t *coeffs_out, uint8_t *symbols_out) {
    return encode_impl(enc, rgb, rgb_len, w, h, f, coeffs_out, symbols_out);
}
uint8_t *alice_codec_decode_stages(const EncodedChunk *chunk, uint64_t *out_len, uint8_t *symbols_out) {
    return decode_impl(chunk, out_len, symbols_out);
}

// ------------------------------------------------------------------------------ batch API
namespace {
// Host staging of chunk i of a batch: `rgb` receives its RGB, `work` its symbol planes (null: the engine's own).
// Shared-workspace batches keep the symbol planes of chunk i in the RGB staging buffer of chunk i - 1 (chunk 0: one spare
// buffer): the front-end of chunk i runs after that of chunk i - 1 has consumed its RGB, and a workspace that is not the
// chunk's own RGB lets the fused kernels run.  A decode writes chunk i's RGB over the planes of chunk i + 1, which the
// back-end's descending order has consumed by then (Engine::run_backend).
// Batches that own their symbol planes need ONE staging buffer: copy, front-end, next chunk, all in stream order, so a
// chunk in flight costs 3 B/px (its symbol planes) + its payload, not 3 B/px more for its RGB.
bool host_stage(Engine *e, uint32_t i, uint8_t *&rgb, uint8_t *&work) {
    const bool shared = e->shared_workspace();
    rgb = e->rgb_stage(shared ? i + 1 : 0);
    work = shared ? e->rgb_stage(i) : nullptr;
    return rgb && (work || !shared);
}

// n new chunks filled from the engine's last encode (every payload copy enqueued, one synchronisation); on failure none
// is left allocated
int fetch_new_chunks(Engine *e, uint32_t n, EncodedChunk **out_chunks) {
    int rc = kOk;
    std::vector<Chunk *> cks(n);
    for (uint32_t i = 0; i < n; i++) {
        out_chunks[i] = new (std::nothrow) EncodedChunk();
        if (!out_chunks[i]) { rc = kErrCuda; set_error(kErrCuda, "host allocation failed"); }
        else cks[i] = &out_chunks[i]->c;
    }
    if (!rc) rc = e->fetch_chunks(n, cks.data());
    if (rc)
        for (uint32_t k = 0; k < n; k++) { delete out_chunks[k]; out_chunks[k] = nullptr; }
    return rc;
}
}  // namespace

AliceBatch *alice_codec_batch_create(uint8_t quality, uint8_t wavelet, uint32_t w, uint32_t h, uint32_t f,
                                     uint32_t n_chunks, void *cuda_stream) {
    return alice_codec_batch_create_ex(quality, wavelet, w, h, f, n_chunks, cuda_stream, 0);
}
AliceBatch *alice_codec_batch_create_ex(uint8_t quality, uint8_t wavelet, uint32_t w, uint32_t h, uint32_t f,
                                        uint32_t n_chunks, void *cuda_stream, uint32_t flags) {
    return alice_codec_batch_create_ex2(quality, wavelet, w, h, f, n_chunks, cuda_stream, flags, 0);
}
AliceBatch *alice_codec_batch_create_ex2(uint8_t quality, uint8_t wavelet, uint32_t w, uint32_t h, uint32_t f,
                                         uint32_t n_chunks, void *cuda_stream, uint32_t flags,
                                         uint64_t payload_bytes_per_chunk) {
    set_error(0, "");
    if (wavelet > 2 || n_chunks == 0) { set_error(kErrDimensions, "bad wavelet byte or n_chunks == 0"); return nullptr; }
    Dims d;
    if (make_dims(w, h, f, d)) return nullptr;
    if (d.n_pixels == 0 || d.padded > 0xffffffffull) { set_error(kErrDimensions, "empty or oversized shape"); return nullptr; }
    if (!cuda_ready()) return nullptr;
    AliceBatch *b = new (std::nothrow) AliceBatch();
    if (!b) return nullptr;
    // Payload arena.  Single chunks keep the worst case (two bytes per symbol); batches budget N + 192 KiB per chunk, or
    // what the caller says its chunks need on average (the streams are placed back to back, so the arena only has to
    // hold the batch's real payload); a stream that finds no room falls back to a worst-case buffer of its own
    // (Engine::run_rans_encode).
    uint64_t cap = n_chunks == 1 ? 0 : d.padded / 3 + 65536;
    if (payload_bytes_per_chunk) cap = payload_bytes_per_chunk / 3 + 16;
    b->eng = new (std::nothrow) Engine(d, n_chunks, cap, (cudaStream_t)cuda_stream, false,
                                       (flags & ALICE_BATCH_SHARED_WORKSPACE) != 0,
                                       (flags & ALICE_BATCH_WELL_FORMED_TABLES) != 0);
    if (!b->eng || !b->eng->ok()) { delete b->eng; delete b; return nullptr; }
    b->eng->set_prefer_small_smem((flags & ALICE_BATCH_SMALL_SMEM_KERNELS) != 0);
    b->quality = quality;
    b->wavelet = wavelet;
    return b;
}
void alice_codec_batch_destroy(AliceBatch *b) {
    if (!b) return;
    delete b->eng;
    delete b;
}
int alice_codec_batch_encode_device(AliceBatch *b, const uint8_t *const *d_rgb, uint32_t n) {
    set_error(0, "");
    if (!b || !d_rgb) { set_error(kErrNull, "null argument"); return kErrNull; }
    return b->eng->encode_device(b->quality, b->wavelet, d_rgb, n, nullptr);
}
int alice_codec_batch_encode_device_ws(AliceBatch *b, const uint8_t *const *d_rgb, uint8_t *const *d_workspace,
                                       uint32_t n) {
    set_error(0, "");
    if (!b || !d_rgb || !d_workspace) { set_error(kErrNull, "null argument"); return kErrNull; }
    if (!b->eng->shared_workspace()) { set_error(kErrDimensions, "batch was not created with ALICE_BATCH_SHARED_WORKSPACE"); return kErrDimensions; }
    return b->eng->encode_device(b->quality, b->wavelet, d_rgb, n, nullptr, d_workspace);
}
uint64_t alice_codec_batch_workspace_bytes(const AliceBatch *b) { return b ? b->eng->workspace_bytes() : 0; }
int alice_codec_batch_decode_device(AliceBatch *b, uint8_t *const *d_rgb_out, uint32_t n) {
    set_error(0, "");
    if (!b || !d_rgb_out) { set_error(kErrNull, "null argument"); return kErrNull; }
    return b->eng->decode_device_resident(d_rgb_out, n);
}
EncodedChunk *alice_codec_batch_get_chunk(AliceBatch *b, uint32_t i) {
    set_error(0, "");
    if (!b) { set_error(kErrNull, "null argument"); return nullptr; }
    EncodedChunk *c = new (std::nothrow) EncodedChunk();
    if (!c) return nullptr;
    if (b->eng->fetch_chunk(i, c->c)) { delete c; return nullptr; }
    return c;
}
int alice_codec_batch_encode_host(AliceBatch *b, const uint8_t *const *h_rgb, uint32_t n, EncodedChunk **out_chunks) {
    set_error(0, "");
    if (!b || !h_rgb || !out_chunks) { set_error(kErrNull, "null argument"); return kErrNull; }
    if (n > b->eng->cap_chunks()) { set_error(kErrBufferSize, "batch larger than capacity"); return kErrBufferSize; }
    // submit_host begins the encode at chunk 0; an empty batch begins it here, so that collect finds 0 chunks submitted
    int rc = n ? kOk : b->eng->encode_begin(b->quality, b->wavelet);
    for (uint32_t i = 0; i < n && !rc; i++) rc = alice_codec_batch_submit_host(b, i, h_rgb[i]);
    return rc ? rc : alice_codec_batch_collect(b, n, out_chunks);
}
// Chunk-at-a-time form of alice_codec_batch_encode_host: submit chunk 0, 1, ... as they arrive (the host -> device copy
// and the front-end of that chunk are enqueued and the call returns at once), then collect.  The host does not have to
// hold all chunks at once: a pinned host buffer may be reused as soon as its copy has completed (alice_codec_batch_sync).
int alice_codec_batch_submit_host(AliceBatch *b, uint32_t i, const uint8_t *h_rgb) {
    set_error(0, "");
    if (!b || !h_rgb) { set_error(kErrNull, "null argument"); return kErrNull; }
    Engine *e = b->eng;
    if (i >= e->cap_chunks()) { set_error(kErrBufferSize, "chunk index beyond the batch capacity"); return kErrBufferSize; }
    if (i == 0) {
        int rc = e->encode_begin(b->quality, b->wavelet);
        if (rc) return rc;
    }
    uint8_t *s, *work;
    if (!host_stage(e, i, s, work)) return kErrCuda;
    CU_CHECK_RC(cudaMemcpyAsync(s, h_rgb, (size_t)e->dims().n_pixels * 3, cudaMemcpyHostToDevice, e->stream()));
    return e->encode_submit(i, s, work);
}
// Device-pointer form of submit / collect: chunk i's RGB is already on the device (d_workspace as in
// alice_codec_batch_encode_device_ws, null for batches that own their symbol planes).  Work is enqueued on the batch's stream
// and the call returns; d_rgb may be overwritten by work enqueued on that stream afterwards (e.g. the next chunk's producer).
int alice_codec_batch_submit_device(AliceBatch *b, uint32_t i, const uint8_t *d_rgb, uint8_t *d_workspace) {
    set_error(0, "");
    if (!b || !d_rgb) { set_error(kErrNull, "null argument"); return kErrNull; }
    Engine *e = b->eng;
    if (i >= e->cap_chunks()) { set_error(kErrBufferSize, "chunk index beyond the batch capacity"); return kErrBufferSize; }
    if (i == 0) {
        int rc = e->encode_begin(b->quality, b->wavelet);
        if (rc) return rc;
    }
    return e->encode_submit(i, d_rgb, d_workspace);
}
int alice_codec_batch_encode_finish(AliceBatch *b, uint32_t n) {
    set_error(0, "");
    if (!b) { set_error(kErrNull, "null argument"); return kErrNull; }
    return b->eng->encode_finish(n);
}
int alice_codec_batch_decode_begin(AliceBatch *b, uint32_t n) {
    set_error(0, "");
    if (!b) { set_error(kErrNull, "null argument"); return kErrNull; }
    return b->eng->decode_resident_begin(n);
}
int alice_codec_batch_decode_next_device(AliceBatch *b, uint32_t i, uint8_t *d_rgb_out) {
    set_error(0, "");
    if (!b) { set_error(kErrNull, "null argument"); return kErrNull; }
    return b->eng->decode_resident_next(i, d_rgb_out);
}
int alice_codec_batch_decode_end(AliceBatch *b) {
    set_error(0, "");
    if (!b) { set_error(kErrNull, "null argument"); return kErrNull; }
    return b->eng->decode_resident_end();
}
int alice_codec_batch_collect(AliceBatch *b, uint32_t n, EncodedChunk **out_chunks) {
    set_error(0, "");
    if (!b || !out_chunks) { set_error(kErrNull, "null argument"); return kErrNull; }
    int rc = b->eng->encode_finish(n);
    return rc ? rc : fetch_new_chunks(b->eng, n, out_chunks);
}
int alice_codec_batch_decode_host(AliceBatch *b, const EncodedChunk *const *chunks, uint32_t n,
                                  uint8_t *const *h_rgb_out) {
    set_error(0, "");
    if (!b || !chunks || !h_rgb_out) { set_error(kErrNull, "null argument"); return kErrNull; }
    Engine *e = b->eng;
    if (n > e->cap_chunks()) { set_error(kErrBufferSize, "batch larger than capacity"); return kErrBufferSize; }
    const bool shared = e->shared_workspace();
    std::vector<const Chunk *> cks(n);
    b->stage_ptrs.resize(n);
    b->work_ptrs.resize(n);
    for (uint32_t i = 0; i < n; i++) {
        if (!chunks[i] || !h_rgb_out[i]) { set_error(kErrNull, "null chunk or output pointer"); return kErrNull; }
        cks[i] = &chunks[i]->c;
        if (!host_stage(e, i, b->stage_ptrs[i], b->work_ptrs[i])) return kErrCuda;
    }
    // engine-owned symbol planes: back-end and device -> host copy chunk by chunk (Engine::decode_chunks synchronises)
    int rc = e->decode_chunks(cks.data(), n, b->stage_ptrs.data(), b->work_ptrs.data(), shared ? nullptr : h_rgb_out);
    if (rc || !shared) return rc;
    for (uint32_t i = 0; i < n; i++)
        CU_CHECK_RC(cudaMemcpyAsync(h_rgb_out[i], b->stage_ptrs[i], (size_t)e->dims().n_pixels * 3, cudaMemcpyDeviceToHost,
                                    e->stream()));
    CU_CHECK_RC(cudaStreamSynchronize(e->stream()));
    return kOk;
}
int alice_codec_batch_sync(AliceBatch *b) {
    set_error(0, "");
    if (!b) { set_error(kErrNull, "null argument"); return kErrNull; }
    CU_CHECK_RC(cudaStreamSynchronize(b->eng->stream()));
    return kOk;
}
int alice_codec_batch_timings(AliceBatch *b, float *ms8) {
    if (!b || !ms8) return kErrNull;
    memcpy(ms8, b->eng->timings.ms, sizeof(float) * 8);
    return kOk;
}
uint64_t alice_codec_batch_device_bytes(const AliceBatch *b) { return b ? b->eng->device_bytes() : 0; }

// ------------------------------------------------------------------------------ rate control
int alice_codec_rate_curve(uint8_t wavelet, const uint8_t *rgb, uint64_t rgb_len, uint32_t width, uint32_t height,
                           uint32_t frames, uint64_t *bytes64, uint32_t *hist_out) {
    return alice_codec_rate_curve_ex(wavelet, rgb, rgb_len, width, height, frames, bytes64, hist_out, 0);
}
int alice_codec_rate_curve_ex(uint8_t wavelet, const uint8_t *rgb, uint64_t rgb_len, uint32_t width, uint32_t height,
                              uint32_t frames, uint64_t *bytes64, uint32_t *hist_out, uint32_t flags) {
    return rate_curve_impl(wavelet, rgb, false, rgb_len, width, height, frames, bytes64, hist_out, nullptr, flags);
}
int alice_codec_rate_curve_device(uint8_t wavelet, const uint8_t *d_rgb, uint32_t width, uint32_t height,
                                  uint32_t frames, uint64_t *bytes64, uint32_t *hist_out, void *cuda_stream) {
    return alice_codec_rate_curve_device_ex(wavelet, d_rgb, width, height, frames, bytes64, hist_out, cuda_stream, 0);
}
int alice_codec_rate_curve_device_ex(uint8_t wavelet, const uint8_t *d_rgb, uint32_t width, uint32_t height,
                                     uint32_t frames, uint64_t *bytes64, uint32_t *hist_out, void *cuda_stream,
                                     uint32_t flags) {
    const unsigned __int128 len = (unsigned __int128)width * height * frames * 3;
    if (len > (unsigned __int128)UINT64_MAX) { set_error(kErrOverflow, "dimensions overflow usize"); return kErrOverflow; }
    return rate_curve_impl(wavelet, d_rgb, true, (uint64_t)len, width, height, frames, bytes64, hist_out,
                           (cudaStream_t)cuda_stream, flags);
}
EncodedChunk *alice_codec_encode_to_size(uint8_t wavelet, const uint8_t *rgb, uint64_t rgb_len, uint32_t width,
                                         uint32_t height, uint32_t frames, uint64_t max_bytes, uint8_t *quality_out) {
    return alice_codec_encode_to_size_ex(wavelet, rgb, rgb_len, width, height, frames, max_bytes, quality_out, 0);
}
EncodedChunk *alice_codec_encode_to_size_ex(uint8_t wavelet, const uint8_t *rgb, uint64_t rgb_len, uint32_t width,
                                            uint32_t height, uint32_t frames, uint64_t max_bytes, uint8_t *quality_out,
                                            uint32_t flags) {
    return encode_to_size_impl(wavelet, rgb, rgb_len, width, height, frames, max_bytes, 1, quality_out, flags);
}
// Per chunk, in stream order as alice_codec_batch_encode_host stages it: copy, rate curve, one host read of 64 sizes, the
// front-end at the chosen step; then one table build and one rANS launch for the whole batch.
int alice_codec_batch_encode_host_to_size(AliceBatch *b, const uint8_t *const *h_rgb, uint32_t n, uint64_t max_bytes,
                                          EncodedChunk **out_chunks, uint8_t *qualities_out) {
    set_error(0, "");
    if (!b || !h_rgb || !out_chunks || !qualities_out) { set_error(kErrNull, "null argument"); return kErrNull; }
    Engine *e = b->eng;
    if (n > e->cap_chunks()) { set_error(kErrBufferSize, "batch larger than capacity"); return kErrBufferSize; }
    const Dims &d = e->dims();
    const size_t bytes = (size_t)d.n_pixels * 3;
    std::vector<int> steps(n);
    int rc = e->encode_begin(100, b->wavelet);    // the batch's quality is not used: every chunk names its step
    for (uint32_t i = 0; i < n && !rc; i++) {
        if (!h_rgb[i]) { set_error(kErrNull, "null chunk pointer"); return kErrNull; }
        uint8_t *s, *work;
        if (!host_stage(e, i, s, work)) return kErrCuda;
        CU_CHECK_RC(cudaMemcpyAsync(s, h_rgb[i], bytes, cudaMemcpyHostToDevice, e->stream()));
        uint64_t pred[kRateSteps];
        rc = e->rate_curve(b->wavelet, s, pred, nullptr, i, work);
        if (rc) return rc;
        steps[i] = pick_step(pred, max_bytes, 1);
        if (!steps[i]) {
            set_no_fit_error(pred, max_bytes);
            set_error(kErrBufferSize, "chunk " + std::to_string(i) + ": " + last_error_msg());
            return kErrBufferSize;
        }
        rc = e->encode_submit(i, s, work, steps[i]);
    }
    if (!rc) rc = e->encode_finish(n);
    if (!rc) rc = fetch_new_chunks(e, n, out_chunks);
    if (rc) return rc;
    for (uint32_t i = 0; i < n && !rc; i++) {
        qualities_out[i] = quality_for_step(steps[i]);
        if (kAlcHeaderBytes + out_chunks[i]->c.data.size() <= max_bytes) continue;
        // larger than its prediction (the bound rules this out): this chunk alone, from the next step on
        delete out_chunks[i];
        out_chunks[i] = encode_to_size_impl(b->wavelet, h_rgb[i], bytes, d.w, d.h, d.f, max_bytes, steps[i] + 1,
                                            &qualities_out[i],
                                            e->well_formed_tables() ? (uint32_t)ALICE_ENCODE_WELL_FORMED_TABLES : 0u);
        if (!out_chunks[i]) rc = last_error_code() ? last_error_code() : kErrCuda;
    }
    if (rc) {
        for (uint32_t k = 0; k < n; k++) { delete out_chunks[k]; out_chunks[k] = nullptr; }
        return rc;
    }
    return kOk;
}

int alice_codec_synth_rgb_device(int kind, uint32_t seed, uint32_t w, uint32_t h, uint32_t f, uint8_t *d_rgb,
                                 void *cuda_stream) {
    set_error(0, "");
    if (!d_rgb) { set_error(kErrNull, "null argument"); return kErrNull; }
    if (!cuda_ready()) return kErrCuda;
    synth_rgb(kind, seed, (int)w, (int)h, (int)f, d_rgb, (cudaStream_t)cuda_stream);
    CU_CHECK_RC(cudaGetLastError());
    return kOk;
}
// alice_codec_psnr (ffi.rs:270, metrics.rs:16-63) for two device buffers: the squared differences are summed exactly
// on the device (integers, total < 2^53, so equal to the reference's sequential f64 sum), the closed form runs here.
int alice_codec_psnr_device(const uint8_t *d_a, const uint8_t *d_b, uint64_t len, void *cuda_stream, double *psnr_out) {
    set_error(0, "");
    if (!psnr_out) { set_error(kErrNull, "null output"); return kErrNull; }
    if (len == 0) { *psnr_out = INFINITY; return kOk; }
    if (!d_a || !d_b) { set_error(kErrNull, "null argument"); return kErrNull; }
    if (!cuda_ready()) return kErrCuda;
    cudaStream_t st = (cudaStream_t)cuda_stream;
    unsigned long long *d_acc = (unsigned long long *)scratch_device(8);
    unsigned long long *h_acc = (unsigned long long *)scratch_pinned(8);
    if (!d_acc || !h_acc) { set_error(kErrCuda, "scratch allocation failed"); return kErrCuda; }
    CU_CHECK_RC(cudaMemsetAsync(d_acc, 0, 8, st));
    sq_diff_sum_u8(d_a, d_b, (size_t)len, d_acc, st);
    CU_CHECK_RC(cudaGetLastError());
    CU_CHECK_RC(cudaMemcpyAsync(h_acc, d_acc, 8, cudaMemcpyDeviceToHost, st));
    CU_CHECK_RC(cudaStreamSynchronize(st));
    const unsigned long long sum = *h_acc;
    const double mse = (double)sum / (double)len;
    *psnr_out = mse == 0.0 ? INFINITY : 10.0 * log10(255.0 * 255.0 / mse);
    return kOk;
}
void *alice_codec_pinned_alloc(uint64_t bytes) {
    void *p = nullptr;
    if (cudaMallocHost(&p, (size_t)bytes) != cudaSuccess) { cudaGetLastError(); set_error(kErrCuda, "pinned allocation failed"); return nullptr; }
    return p;
}
void alice_codec_pinned_free(void *p) { if (p) cudaFreeHost(p); }
void alice_codec_trim_host_pool(void) { trim_pinned_pool(); }
int alice_codec_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
    return n;
}
int alice_codec_set_device(int device) {
    CU_CHECK_RC(cudaSetDevice(device));
    return kOk;
}

}  // extern "C"
#pragma GCC visibility pop
