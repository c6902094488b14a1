/*
 * alice_codec.h — C ABI of libalice_codec (B200 / sm_100a implementation).
 *
 * Part 1 is the reference's C ABI verbatim: the 20 `alice_codec_*` symbols of
 * /root/reference/src/ffi.rs (declared for consumers in bindings/ue5/AliceCodec.h:14-68 and
 * bindings/unity/AliceCodec.cs:187-229).  A consumer of the reference's cdylib can load this
 * library instead without changing a line: same names, argument meaning, ownership rules
 * (library-allocated buffers returned with their length, freed by alice_codec_data_free with
 * the same length), and error behaviour (null / 0 / -1.0 returns; no error code crosses).
 * Every call runs its compute on the current CUDA device; there is no CPU fallback — without
 * a usable device the compute entry points fail (null / non-zero) and
 * alice_codec_last_error() reports ALICE_ERR_CUDA.
 *
 * Part 2 are extension entry points with the same conventions for the rest of the hot-path
 * API the north-star names but the reference never exported over FFI (with_wavelet,
 * Wavelet2D/3D, Quantizer, FastQuantizer, AnalyticalRDO, to/from_symbols, build_histogram,
 * FrequencyTable, RansEncoder/RansDecoder, colour transforms), stage dumps for parity tests,
 * and batch / device-pointer entry points for throughput use.
 */
#ifndef ALICE_CODEC_H
#define ALICE_CODEC_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* ---- opaque handles (ffi.rs; bindings/ue5/AliceCodec.h:17-19) ---- */
typedef struct Wavelet1D Wavelet1D;
typedef struct FrameEncoder FrameEncoder;
typedef struct EncodedChunk EncodedChunk;

/* ================= Part 1: the reference ABI (ffi.rs:16-315) ================= */

Wavelet1D *alice_codec_wavelet1d_haar(void);                                   /* ffi.rs:16  */
Wavelet1D *alice_codec_wavelet1d_cdf53(void);                                  /* ffi.rs:22  */
Wavelet1D *alice_codec_wavelet1d_cdf97(void);                                  /* ffi.rs:28  */
void alice_codec_wavelet1d_destroy(Wavelet1D *ptr);                            /* ffi.rs:38  null ok */
/* in place; no-op if wavelet/data is null or len < 2  (ffi.rs:52, :73; wavelet.rs:133,157) */
void alice_codec_wavelet1d_forward(const Wavelet1D *wavelet, int32_t *data, uint32_t len);
void alice_codec_wavelet1d_inverse(const Wavelet1D *wavelet, int32_t *data, uint32_t len);

FrameEncoder *alice_codec_encoder_create(uint8_t quality);                     /* ffi.rs:92  always CDF 5/3 */
void alice_codec_encoder_destroy(FrameEncoder *ptr);                           /* ffi.rs:102 */
/* FrameEncoder::encode (pipeline.rs:377-507); null on any error (ffi.rs:116-133) */
EncodedChunk *alice_codec_encode(const FrameEncoder *encoder, const uint8_t *rgb, uint32_t rgb_len,
                                 uint32_t width, uint32_t height, uint32_t frames);
/* FrameDecoder::decode (pipeline.rs:537-624); null on error; free with alice_codec_data_free (ffi.rs:145) */
uint8_t *alice_codec_decode(const EncodedChunk *chunk, uint32_t *out_len);

void alice_codec_chunk_destroy(EncodedChunk *ptr);                             /* ffi.rs:171 */
uint8_t *alice_codec_chunk_to_bytes(const EncodedChunk *chunk, uint32_t *out_len);   /* ffi.rs:185; pipeline.rs:200 */
EncodedChunk *alice_codec_chunk_from_bytes(const uint8_t *data, uint32_t len);       /* ffi.rs:207; pipeline.rs:235 */
uint32_t alice_codec_chunk_width(const EncodedChunk *chunk);                   /* ffi.rs:226 (0 if null) */
uint32_t alice_codec_chunk_height(const EncodedChunk *chunk);                  /* ffi.rs:240 */
uint32_t alice_codec_chunk_frames(const EncodedChunk *chunk);                  /* ffi.rs:254 */

double alice_codec_psnr(const uint8_t *a, const uint8_t *b, uint32_t len);     /* ffi.rs:270; metrics.rs:57 */

void alice_codec_data_free(uint8_t *ptr, uint32_t len);                        /* ffi.rs:288 (no-op if null or len==0) */
void alice_codec_string_free(char *s);                                         /* ffi.rs:302 */
char *alice_codec_version(void);                                               /* ffi.rs:311 "0.1.2" */

/* ================= Part 2: extensions ================= */

/* error codes of the extension entry points = CodecError variants (error.rs:12-23) */
enum {
    ALICE_OK = 0,
    ALICE_ERR_BUFFER_SIZE = 1,  /* InvalidBufferSize */
    ALICE_ERR_DIMENSIONS = 2,   /* InvalidDimensions */
    ALICE_ERR_OVERFLOW = 3,     /* DimensionOverflow */
    ALICE_ERR_BITSTREAM = 4,    /* InvalidBitstream  */
    ALICE_ERR_QUANT_STEP = 5,   /* InvalidQuantStep  */
    ALICE_ERR_PANIC = 6,        /* the reference would panic / abort here (division by zero, ...) */
    ALICE_ERR_NULL = 7,         /* null argument */
    ALICE_ERR_CUDA = 100        /* no device, CUDA failure or device out of memory */
};
/* thread-local code / text of the last failure of any entry point on this thread (0 / "" if none) */
int32_t alice_codec_last_error(void);
const char *alice_codec_last_error_message(void);

enum { ALICE_WAVELET_CDF53 = 0, ALICE_WAVELET_CDF97 = 1, ALICE_WAVELET_HAAR = 2 }; /* pipeline.rs:34-41 */

/* FrameEncoder::with_wavelet (pipeline.rs:356); null if wavelet > 2 */
FrameEncoder *alice_codec_encoder_create_with_wavelet(uint8_t quality, uint8_t wavelet);
/* ALICE_ENCODE_WELL_FORMED_TABLES — encodes whose chunks decode exactly on every decoder of the format.  The default
 * encode stores each channel's symbol counts, and the table FrequencyTable::from_histogram derives from them gives
 * every empty bin a frequency of 1; where empty bins lie below used symbols, the ranges of the high symbols run past
 * 4096 and the stream does not decode to what was encoded (SURVEY.md 0.7).  In this mode the 256-bin histogram of a
 * channel header is a TABLE SPECIFICATION that sums to 4096, not the symbol counts: the counts themselves where their
 * table is already well formed (the chunk is then byte-identical to the default encode), otherwise the counts scaled
 * to the 4096 - (empty bins among 0..254) slots left by the empty bins, with the rest on symbol 255 (DESIGN.md 4.8).
 * The .alc format and every decoder, including the reference's, are unchanged; where the rule rescales, a chunk costs a
 * few percent more bytes than the default encode.  Unknown flag bits: null, ALICE_ERR_DIMENSIONS. */
enum { ALICE_ENCODE_WELL_FORMED_TABLES = 1 };
/* with_wavelet + flags; alice_codec_encode and alice_codec_encode_stages honour the encoder's flags */
FrameEncoder *alice_codec_encoder_create_ex(uint8_t quality, uint8_t wavelet, uint32_t flags);
uint8_t alice_codec_chunk_wavelet(const EncodedChunk *chunk);                  /* EncodedChunk::wavelet_type */
uint64_t alice_codec_chunk_compressed_size(const EncodedChunk *chunk);         /* pipeline.rs:190 */
/* per-channel header fields (pipeline.rs:123-134); hist256 may be null */
int alice_codec_chunk_channel_header(const EncodedChunk *chunk, uint32_t channel, uint32_t *compressed_len,
                                     int32_t *quant_step, int32_t *quant_dead_zone, uint32_t *num_symbols,
                                     uint32_t *hist256);
/* 64-bit-length variants of to_bytes / from_bytes / decode for buffers beyond u32 */
uint8_t *alice_codec_chunk_to_bytes64(const EncodedChunk *chunk, uint64_t *out_len);
EncodedChunk *alice_codec_chunk_from_bytes64(const uint8_t *data, uint64_t len);
void alice_codec_data_free64(uint8_t *ptr, uint64_t len);

/* colour (color.rs:199, :245) — host pointers */
int alice_codec_rgb_to_ycocg_r(const uint8_t *rgb, uint64_t rgb_len, int16_t *y, int16_t *co, int16_t *cg,
                               uint64_t out_len);
int alice_codec_ycocg_r_to_rgb(const int16_t *y, const int16_t *co, const int16_t *cg, uint64_t n, uint8_t *rgb,
                               uint64_t rgb_len);

/* Wavelet2D / Wavelet3D forward & inverse, in place on host i32 data (wavelet.rs:292,319,392,441);
 * LosslessEncoder::transform_2d / inverse_2d (lossless.rs:45-54) == wavelet2d with CDF 5/3 */
int alice_codec_wavelet2d_forward(uint8_t wavelet, int32_t *data, uint32_t width, uint32_t height);
int alice_codec_wavelet2d_inverse(uint8_t wavelet, int32_t *data, uint32_t width, uint32_t height);
int alice_codec_wavelet3d_forward(uint8_t wavelet, int32_t *data, uint32_t width, uint32_t height, uint32_t depth);
int alice_codec_wavelet3d_inverse(uint8_t wavelet, int32_t *data, uint32_t width, uint32_t height, uint32_t depth);

/* Quantizer::{quantize_buffer, dequantize_buffer} (quant.rs:117,135); FastQuantizer (quant.rs:190-311) */
int alice_codec_quantize_buffer(int32_t step, int32_t dead_zone, const int32_t *in, uint64_t n, int32_t *out,
                                uint64_t out_len);
int alice_codec_dequantize_buffer(int32_t step, const int32_t *in, uint64_t n, int32_t *out, uint64_t out_len);
int alice_codec_fast_quantize_buffer(int32_t step, int32_t dead_zone, const int32_t *in, uint64_t n, int32_t *out,
                                     uint64_t out_len);
/* to_symbols / from_symbols / build_histogram (quant.rs:547,572,594) */
int alice_codec_to_symbols(const int32_t *coeffs, uint64_t n, uint8_t *symbols, uint64_t symbols_len);
int alice_codec_from_symbols(const uint8_t *symbols, uint64_t n, int32_t *coeffs, uint64_t coeffs_len);
int alice_codec_build_histogram(const uint8_t *symbols, uint64_t n, uint32_t *hist256);
/* AnalyticalRDO (quant.rs:377-505): with_quality -> target_bpp; compute_quantizer for one sub-band
 * (SubBand3D byte 0..7, lib.rs:115-132) */
double alice_codec_rdo_bpp_from_quality(uint8_t quality);
int alice_codec_rdo_compute_quantizer(double target_bpp, const int32_t *coeffs, uint64_t n, uint8_t subband,
                                      int32_t *step, int32_t *dead_zone);
/* AnalyticalRDO::estimate_variance (quant.rs:415-435; private in the reference): max(1.0, f64 sum of squared
 * deviations accumulated in slice order / n), 1.0 for an empty slice */
int alice_codec_rdo_estimate_variance(const int32_t *coeffs, uint64_t n, double *variance_out);
/* AnalyticalRDO::compute_all_quantizers (quant.rs:472-490) over the 8 octants of a forward-transformed w x h x d
 * volume (index t*h*w + y*w + x).  Octant = SubBand3D byte = 4*[x >= w/2] + 2*[y >= h/2] + [t >= d/2] (lib.rs:115-132);
 * each octant is the slice a caller would gather in row-major (t, y, x) order.  The f64 variance sum of every
 * octant is bit-identical to the reference's sequential loop (quant.rs:425-432). */
int alice_codec_rdo_compute_all_quantizers(double target_bpp, const int32_t *volume, uint32_t width, uint32_t height,
                                           uint32_t depth, int32_t *steps8, int32_t *dead_zones8);
/* the same for a volume already in device memory */
int alice_codec_rdo_compute_all_quantizers_device(double target_bpp, const int32_t *d_volume, uint32_t width,
                                                  uint32_t height, uint32_t depth, int32_t *steps8, int32_t *dead_zones8);
/* statistics -> quantisers -> FastQuantizer::quantize_buffer (quant.rs:272-299) with the constants of each
 * element's octant, the volume staying on the device in between; also returns the 8 (step, dead_zone) pairs */
int alice_codec_rdo_quantize_volume(double target_bpp, const int32_t *volume, uint32_t width, uint32_t height,
                                    uint32_t depth, int32_t *out, uint64_t out_len, int32_t *steps8,
                                    int32_t *dead_zones8);

/* FrequencyTable::from_histogram / uniform (rans.rs:102,158); n_symbols in 1..=256; outputs sized 256/256/4096 */
int alice_codec_freq_table_from_histogram(const uint32_t *hist, uint32_t n_symbols, uint16_t *cum256,
                                          uint16_t *freq256, uint8_t *lut4096);
/* RansEncoder::encode_symbols + finish with the table of from_histogram(hist) (an all-zero histogram
 * gives the uniform table); *out is library-allocated, free with alice_codec_data_free64 (rans.rs:249-308) */
int alice_codec_rans_encode(const uint8_t *symbols, uint64_t n, const uint32_t *hist, uint32_t n_symbols,
                            uint8_t **out, uint64_t *out_len);
/* RansDecoder::new + decode_n (rans.rs:330-381) */
int alice_codec_rans_decode(const uint8_t *stream, uint64_t len, const uint32_t *hist, uint32_t n_symbols,
                            uint8_t *symbols_out, uint64_t n);

/* InterleavedRansEncoder / InterleavedRansDecoder (rans.rs:393-524): the reference's 4-stream container (4 stream
 * lengths + 4 symbol counts, u32 LE, then the streams; symbol i in stream i % 4).  Opt-in and NOT the .alc format:
 * the only intra-channel entropy-coding parallelism the reference defines (SURVEY.md 8f-4).  Same table rules and
 * ownership as alice_codec_rans_encode / _decode. */
int alice_codec_rans_encode_interleaved(const uint8_t *symbols, uint64_t n, const uint32_t *hist, uint32_t n_symbols,
                                        uint8_t **out, uint64_t *out_len);
int alice_codec_rans_decode_interleaved(const uint8_t *stream, uint64_t len, const uint32_t *hist, uint32_t n_symbols,
                                        uint8_t *symbols_out, uint64_t n);

/* stage dumps for parity tests: as alice_codec_encode / alice_codec_decode, additionally copying out the
 * wavelet coefficients before quantisation (i32 [3][N], only via the generic path when requested) and the
 * symbol planes (u8 [3][N]), N = padded pixels.  Any dump pointer may be null. */
EncodedChunk *alice_codec_encode_stages(const FrameEncoder *encoder, const uint8_t *rgb, uint64_t rgb_len,
                                        uint32_t width, uint32_t height, uint32_t frames, int32_t *coeffs_out,
                                        uint8_t *symbols_out);
uint8_t *alice_codec_decode_stages(const EncodedChunk *chunk, uint64_t *out_len, uint8_t *symbols_out);

/* Wavelet2D / Wavelet3D on DEVICE buffers (same arithmetic as the host-pointer entry points; asynchronous on cuda_stream).
 * 2-D: n_images images of width x height, out of place (d_src and d_dst must not overlap) — LosslessEncoder::transform_2d /
 * inverse_2d (lossless.rs:45-54) over a stack of frames is wavelet 0 (CDF 5/3).  3-D: in place in d_data, d_tmp = scratch of
 * the same size.  Volumes with width % 4 == 0 and even height (and depth) take the one-pass-per-plane / per-line kernels
 * (16 B per sample of memory traffic for a 3-D transform); other shapes the step-by-step path. */
int alice_codec_wavelet2d_device(uint8_t wavelet, int inverse, const int32_t *d_src, int32_t *d_dst, uint32_t width,
                                 uint32_t height, uint32_t n_images, void *cuda_stream);
int alice_codec_wavelet3d_device(uint8_t wavelet, int inverse, int32_t *d_data, int32_t *d_tmp, uint32_t width,
                                 uint32_t height, uint32_t depth, void *cuda_stream);

/* ---- the lossless module over a frame set, on the device (BASELINE config 4; src/lossless.rs + the reference's own
 * entropy stages): per colour channel of a width x height x frames RGB volume, rgb_bytes_to_ycocg_r -> i32 planes ->
 * LosslessEncoder::transform_2d of every frame -> to_symbols (step 1, wrapping) -> build_histogram ->
 * FrequencyTable::from_histogram -> RansEncoder (one stream per channel) ; decode = RansDecoder + inverse_2d of the
 * coefficients.  fetch copies a stage buffer to the host for parity checks: which = 0 coefficients (i32 [3][n]),
 * 1 symbols (u8 [3][n]), 2 histograms (u32 [3][256]), 3 decoded symbols, 4 inverse-transformed planes (i32 [3][n]),
 * 5 the rANS stream of `channel`.  timings: [0] colour, [1] 2-D forward, [2] symbols + histograms + tables,
 * [3] rANS encode, [4] rANS decode, [5] 2-D inverse (ms, CUDA events). */
typedef struct AliceLossless AliceLossless;
AliceLossless *alice_codec_lossless_create(uint32_t width, uint32_t height, uint32_t frames, void *cuda_stream);
void alice_codec_lossless_destroy(AliceLossless *l);
int alice_codec_lossless_encode_device(AliceLossless *l, const uint8_t *d_rgb);
int alice_codec_lossless_decode_device(AliceLossless *l);
int alice_codec_lossless_fetch(AliceLossless *l, int which, int channel, void *host_out, uint64_t cap, uint64_t *out_len);
int alice_codec_lossless_timings(AliceLossless *l, float *ms8);

/* ---- batch / device-pointer API: many independent chunks of one shape in flight ---- */
typedef struct AliceBatch AliceBatch;
/* cuda_stream: a cudaStream_t (may be null = the legacy default stream) on which all work is issued */
AliceBatch *alice_codec_batch_create(uint8_t quality, uint8_t wavelet, uint32_t width, uint32_t height,
                                     uint32_t frames, uint32_t n_chunks, void *cuda_stream);
/* flags: ALICE_BATCH_SHARED_WORKSPACE — the batch owns no symbol planes (3 bytes per padded pixel and chunk): with
 * device pointers the caller passes one workspace of alice_codec_batch_workspace_bytes() per chunk to
 * alice_codec_batch_encode_device_ws.  Chunks are encoded in index order, so workspace i may be the RGB buffer of any
 * chunk j < i (already consumed), or the buffer chunk i is decoded into later (decode finishes reading the planes
 * before it writes RGB).  It may even be chunk i's own RGB input, but that chunk then takes the slower two-kernel
 * front-end (the fused kernel reads RGB and writes symbols in the same launch).  With host pointers the batch's RGB
 * staging buffers double as the workspaces (chunk i's planes live in the staging buffer of chunk i-1).
 * Saves 3 B/px of device memory per chunk in flight. */
/* ALICE_BATCH_SMALL_SMEM_KERNELS — the batch takes the two-kernel front-end / back-end (next to no shared memory) instead
 * of the fused kernels (one 106-210 KB block per SM).  For batches that run NEXT TO other batches' rANS launches (several
 * host threads, one batch each): a fused block cannot start on an SM whose shared memory is held by resident rANS streams
 * and would wait for a whole rANS launch to end; the small kernels slip in beside them.  Same results. */
/* ALICE_BATCH_WELL_FORMED_TABLES — every encode of the batch (encode_host_to_size included) stores well-formed table
 * specifications as ALICE_ENCODE_WELL_FORMED_TABLES does; alice_codec_batch_decode_device builds its tables from them.
 * Costs 3 KiB per chunk of device memory. */
enum { ALICE_BATCH_SHARED_WORKSPACE = 1, ALICE_BATCH_SMALL_SMEM_KERNELS = 2, ALICE_BATCH_WELL_FORMED_TABLES = 4 };
AliceBatch *alice_codec_batch_create_ex(uint8_t quality, uint8_t wavelet, uint32_t width, uint32_t height,
                                        uint32_t frames, uint32_t n_chunks, void *cuda_stream, uint32_t flags);
/* payload_bytes_per_chunk: device memory reserved for the encoded payload, per chunk on average (0 = the default, one
 * byte per padded pixel + 192 KiB).  The batch places its streams back to back, each with the upper bound its histogram
 * gives, so this only has to cover what the chunks really compress to; a stream that finds no room is redone in a
 * worst-case buffer of its own (slow, never wrong). */
AliceBatch *alice_codec_batch_create_ex2(uint8_t quality, uint8_t wavelet, uint32_t width, uint32_t height,
                                         uint32_t frames, uint32_t n_chunks, void *cuda_stream, uint32_t flags,
                                         uint64_t payload_bytes_per_chunk);
uint64_t alice_codec_batch_workspace_bytes(const AliceBatch *b);
int alice_codec_batch_encode_device_ws(AliceBatch *b, const uint8_t *const *d_rgb, uint8_t *const *d_workspace,
                                       uint32_t n);
void alice_codec_batch_destroy(AliceBatch *b);
/* d_rgb[i]: device pointer to chunk i's interleaved RGB (3*w*h*f bytes).  Runs front-end, table build and
 * all 3*n rANS streams; results stay on the device.  Synchronises the stream before returning. */
int alice_codec_batch_encode_device(AliceBatch *b, const uint8_t *const *d_rgb, uint32_t n);
/* decodes what the last encode left on the device into d_rgb_out[i] (tables rebuilt from the histograms) */
int alice_codec_batch_decode_device(AliceBatch *b, uint8_t *const *d_rgb_out, uint32_t n);
/* host-buffer variants: host<->device copies are part of the call.  encode_host returns after ONE stream
 * synchronisation for the whole batch (every payload copy is enqueued first).  A batch that owns its symbol planes (no
 * ALICE_BATCH_SHARED_WORKSPACE) stages the RGB of all chunks through ONE device buffer, in stream order: a chunk in flight
 * costs 3 B per padded pixel + its payload of device memory.
 * Call order: alice_codec_batch_decode_host reuses the histogram / table / payload buffers of the batch, so whatever
 * the last encode left resident on the device is gone afterwards: alice_codec_batch_get_chunk and
 * alice_codec_batch_decode_device then fail with ALICE_ERR_BUFFER_SIZE until the next encode. */
int alice_codec_batch_encode_host(AliceBatch *b, const uint8_t *const *h_rgb, uint32_t n, EncodedChunk **out_chunks);
int alice_codec_batch_decode_host(AliceBatch *b, const EncodedChunk *const *chunks, uint32_t n,
                                  uint8_t *const *h_rgb_out);
/* The same encode, one chunk at a time (the reference encodes one chunk per call, src/bin/main.rs:107-145): submit chunk
 * 0, 1, ... in index order as they become available — each call enqueues the host -> device copy and the front-end of
 * that chunk and returns at once — then collect(n) runs the tables and all 3n rANS streams and returns the chunks after
 * ONE synchronisation.  The host never has to hold the whole batch: a (pinned) host buffer may be reused once its copy has
 * completed, e.g. after alice_codec_batch_sync, which waits for everything enqueued so far. */
int alice_codec_batch_submit_host(AliceBatch *b, uint32_t i, const uint8_t *h_rgb);
int alice_codec_batch_collect(AliceBatch *b, uint32_t n, EncodedChunk **out_chunks);
int alice_codec_batch_sync(AliceBatch *b);
/* Device-pointer streaming: the same pipeline with the RGB already on the device, for batches whose chunks in flight do not
 * fit HBM as RGB (a chunk in flight then costs its symbol planes, 3 B per padded pixel, + its payload).
 *   encode: submit_device(0), (1), ... in index order — each call enqueues that chunk's front-end on the batch's stream and
 *           returns; d_rgb may be rewritten by work enqueued on that stream afterwards (d_workspace: as in
 *           alice_codec_batch_encode_device_ws, null for batches that own their symbol planes) — then encode_finish(n) =
 *           tables + all 3n rANS streams + one synchronisation; alice_codec_batch_get_chunk fetches a result.
 *   decode: decode_begin(n) enqueues the tables and all 3n rANS streams of what the last encode left resident,
 *           decode_next_device(i, d_rgb_out) the back-end of chunk i (any order); d_rgb_out is valid on the batch's stream
 *           after the call, so the caller may hand the same buffer to a later chunk once its own stream-ordered consumer
 *           has been enqueued; decode_end synchronises. */
int alice_codec_batch_submit_device(AliceBatch *b, uint32_t i, const uint8_t *d_rgb, uint8_t *d_workspace);
int alice_codec_batch_encode_finish(AliceBatch *b, uint32_t n);
int alice_codec_batch_decode_begin(AliceBatch *b, uint32_t n);
int alice_codec_batch_decode_next_device(AliceBatch *b, uint32_t i, uint8_t *d_rgb_out);
int alice_codec_batch_decode_end(AliceBatch *b);
/* copy chunk i of the last encode_device to the host as an EncodedChunk */
EncodedChunk *alice_codec_batch_get_chunk(AliceBatch *b, uint32_t i);
/* CUDA-event durations (ms) of the last encode/decode: [0] front-end kernels (all chunks), [1] table build,
 * [2] rANS encode, [3] table build (decode), [4] rANS decode, [5] back-end kernels; [6],[7] reserved */
int alice_codec_batch_timings(AliceBatch *b, float *ms8);
/* bytes of device memory the batch holds */
uint64_t alice_codec_batch_device_bytes(const AliceBatch *b);

/* ---- Byte-budget encoding.  Quality q maps to quantiser step 64 - 63q/100 (1..64); a step's chunk size is bounded
 * before any rANS work from one transform pass and one histogram of the coefficient values (the symbol histogram of
 * every step follows from it, and the table build's size estimate bounds every stream).  The .alc format is unchanged:
 * a rate-controlled chunk is byte-identical to alice_codec_encode at the quality it reports, which is the largest
 * quality with that step.  An empty input (a zero dimension) is the 3138-byte empty chunk at every step. */
/* predicted .alc size of every quantiser step (index i = step i+1), UINT64_MAX where the reference would abort;
 * hist_out (u32 [64][3][256]) may be null */
int alice_codec_rate_curve(uint8_t wavelet, const uint8_t *rgb, uint64_t rgb_len, uint32_t width, uint32_t height,
                           uint32_t frames, uint64_t *bytes64, uint32_t *hist_out);
/* the same for RGB in device memory; the call waits for the work enqueued on cuda_stream before it reads d_rgb */
int alice_codec_rate_curve_device(uint8_t wavelet, const uint8_t *d_rgb, uint32_t width, uint32_t height,
                                  uint32_t frames, uint64_t *bytes64, uint32_t *hist_out, void *cuda_stream);
/* the highest quality whose chunk fits max_bytes; identical to alice_codec_encode at *quality_out.  No quality fits:
 * null, ALICE_ERR_BUFFER_SIZE, and the message names the smallest predicted size */
EncodedChunk *alice_codec_encode_to_size(uint8_t wavelet, const uint8_t *rgb, uint64_t rgb_len, uint32_t width,
                                         uint32_t height, uint32_t frames, uint64_t max_bytes, uint8_t *quality_out);
/* the three calls above for encodes with ALICE_ENCODE_WELL_FORMED_TABLES flags (0 = the calls above): the curve then
 * bounds the well-formed encode at every step and has no UINT64_MAX entry; hist_out still holds the symbol counts */
int alice_codec_rate_curve_ex(uint8_t wavelet, const uint8_t *rgb, uint64_t rgb_len, uint32_t width, uint32_t height,
                              uint32_t frames, uint64_t *bytes64, uint32_t *hist_out, uint32_t flags);
int alice_codec_rate_curve_device_ex(uint8_t wavelet, const uint8_t *d_rgb, uint32_t width, uint32_t height,
                                     uint32_t frames, uint64_t *bytes64, uint32_t *hist_out, void *cuda_stream,
                                     uint32_t flags);
EncodedChunk *alice_codec_encode_to_size_ex(uint8_t wavelet, const uint8_t *rgb, uint64_t rgb_len, uint32_t width,
                                            uint32_t height, uint32_t frames, uint64_t max_bytes, uint8_t *quality_out,
                                            uint32_t flags);
/* host-buffer batch, every chunk with its own quality under the same per-chunk budget; all 3n rANS streams run
 * concurrently as in alice_codec_batch_encode_host.  The batch's own quality is not used.  The first rate call on a
 * batch allocates 12 B per padded pixel of coefficients plus ~4 MB of tables (alice_codec_batch_device_bytes grows). */
int alice_codec_batch_encode_host_to_size(AliceBatch *b, const uint8_t *const *h_rgb, uint32_t n, uint64_t max_bytes,
                                          EncodedChunk **out_chunks, uint8_t *qualities_out);

/* ---- PSNR-target encoding (DESIGN.md 4.9), for ALICE_ENCODE_WELL_FORMED_TABLES encodes only: such a chunk decodes to
 * exactly the symbols it encodes, so the decode at every step follows from one transform pass, without rANS work.  The
 * default encode has no such curve.  sse64[i] = the sum over the chunk's 3*w*h*f bytes of (input - decode)^2 for the
 * well-formed encode at step i+1 (an exact integer), psnr64[i] = 10 log10(255^2 / (sse / len)), +inf where sse == 0:
 * bit for bit what alice_codec_psnr gives for the input and that decode.  PSNR is not monotone in the step (small steps
 * wrap symbols mod 256), so the curve holds every step.  An empty input (a zero dimension) gives +inf and 0 at every
 * step.  These calls take no flags: they always mean the well-formed encode. */
/* sse64 may be null */
int alice_codec_psnr_curve(uint8_t wavelet, const uint8_t *rgb, uint64_t rgb_len, uint32_t width, uint32_t height,
                           uint32_t frames, double *psnr64, uint64_t *sse64);
/* the same for RGB in device memory; the call waits for the work enqueued on cuda_stream before it reads d_rgb */
int alice_codec_psnr_curve_device(uint8_t wavelet, const uint8_t *d_rgb, uint32_t width, uint32_t height,
                                  uint32_t frames, double *psnr64, uint64_t *sse64, void *cuda_stream);
/* the lowest quality that reaches min_psnr_db: the largest step s with psnr64[s-1] >= min_psnr_db, encoded at
 * *quality_out = the largest quality with that step; the chunk is byte-identical to an encode with
 * ALICE_ENCODE_WELL_FORMED_TABLES at that quality.  No step reaches the target, or the target is NaN: null,
 * ALICE_ERR_QUANT_STEP, and the message names the best PSNR of the curve and its quality.  An empty input gives the empty
 * chunk at the quality of step 64. */
EncodedChunk *alice_codec_encode_to_psnr(uint8_t wavelet, const uint8_t *rgb, uint64_t rgb_len, uint32_t width,
                                         uint32_t height, uint32_t frames, double min_psnr_db, uint8_t *quality_out);
/* host-buffer batch form (the batch must have ALICE_BATCH_WELL_FORMED_TABLES, else ALICE_ERR_DIMENSIONS): every chunk at
 * its own lowest quality that reaches min_psnr_db, all 3n rANS streams concurrently.  The batch's own quality is not
 * used.  The first call allocates what the rate curve allocates, and for shapes the fused back-end does not take (or
 * batches with ALICE_BATCH_SMALL_SMEM_KERNELS) an RGB scratch of 3 B per pixel. */
int alice_codec_batch_encode_host_to_psnr(AliceBatch *b, const uint8_t *const *h_rgb, uint32_t n, double min_psnr_db,
                                          EncodedChunk **out_chunks, uint8_t *qualities_out);

/* synthetic RGB volumes generated on the device (SURVEY.md Appendix D): kind 0=G0, 1=G1, 2=G2 */
int alice_codec_synth_rgb_device(int kind, uint32_t seed, uint32_t width, uint32_t height, uint32_t frames,
                                 uint8_t *d_rgb, void *cuda_stream);
/* alice_codec_psnr (ffi.rs:270) for two DEVICE buffers, e.g. a chunk's RGB input and its decode output; the sum of
 * squared differences is an exact integer sum on the device, so the result equals the host function's bit for bit */
int alice_codec_psnr_device(const uint8_t *d_a, const uint8_t *d_b, uint64_t len, void *cuda_stream, double *psnr_out);
/* pinned host memory helpers for the host-buffer batch API */
void *alice_codec_pinned_alloc(uint64_t bytes);
void alice_codec_pinned_free(void *p);
/* Encoded payloads live in page-locked host buffers that the library pools for reuse (idle pool bounded by the
 * environment variable ALICE_CODEC_PINNED_POOL_MB, default 1024); this releases the idle ones. */
void alice_codec_trim_host_pool(void);
/* number of CUDA devices visible (0 if none / no driver); select the device for this thread */
int alice_codec_device_count(void);
int alice_codec_set_device(int device);

#ifdef __cplusplus
}
#endif
#endif /* ALICE_CODEC_H */
