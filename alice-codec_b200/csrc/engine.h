// engine.h — host-side pipeline objects of libalice_codec.
//
//   Chunk         = EncodedChunk (src/pipeline.rs:172-185) with its three ChannelHeaders
//                   (:123-134) and the .alc (de)serialisation (:200-226, :235-313).
//   Engine        = device buffers + CUDA stream for up to `cap_chunks` chunks of one shape
//                   in flight; runs FrameEncoder::encode (:377-507) and FrameDecoder::decode
//                   (:537-624) on the device for each of them.
// Errors are CodecError variants (src/error.rs:12-23) carried as ALICE_ERR_* codes.
#pragma once
#include <cstdint>
#include <string>
#include <vector>

#include "kernels.h"

namespace alice {

constexpr int kOk = 0, kErrBufferSize = 1, kErrDimensions = 2, kErrOverflow = 3, kErrBitstream = 4,
              kErrQuantStep = 5, kErrPanic = 6, kErrNull = 7, kErrCuda = 100;

void set_error(int code, const std::string &msg);
int last_error_code();
const char *last_error_msg();

struct ChannelHeader {              // pipeline.rs:123-134
    uint32_t compressed_len = 0;
    int32_t quant_step = 1;
    int32_t quant_dead_zone = 1;
    uint32_t num_symbols = 0;
    uint32_t histogram[256] = {0};
};
constexpr size_t kChannelHeaderBytes = 1040;  // pipeline.rs:137
constexpr size_t kFixedHeaderBytes = 18;      // pipeline.rs:148

// Payload bytes of a chunk.  Buffers filled by the encoder come from a process-wide pool of page-locked
// (cudaHostRegister) allocations, so the device writes them directly at link speed and a destroyed chunk's buffer is
// reused by the next encode instead of being unmapped and page-faulted in again (ALICE_CODEC_PINNED_POOL_MB bounds
// the idle pool, default 16384).  Buffers filled from user bytes (from_bytes) are plain malloc.
class ByteBuf {
public:
    ByteBuf() = default;
    ~ByteBuf() { release(); }
    ByteBuf(const ByteBuf &) = delete;
    ByteBuf &operator=(const ByteBuf &) = delete;
    ByteBuf(ByteBuf &&o) noexcept { steal(o); }
    ByteBuf &operator=(ByteBuf &&o) noexcept { if (this != &o) { release(); steal(o); } return *this; }
    uint8_t *data() { return p_; }
    const uint8_t *data() const { return p_; }
    size_t size() const { return n_; }
    bool pinned() const { return pinned_; }
    bool assign(const uint8_t *src, size_t n);   // plain heap copy
    bool acquire_pinned(size_t n);               // page-locked storage of n bytes (contents undefined)
    void release();
private:
    void steal(ByteBuf &o) { p_ = o.p_; n_ = o.n_; cap_ = o.cap_; pinned_ = o.pinned_; o.p_ = nullptr; o.n_ = o.cap_ = 0; o.pinned_ = false; }
    uint8_t *p_ = nullptr;
    size_t n_ = 0, cap_ = 0;
    bool pinned_ = false;
};

struct Chunk {                      // pipeline.rs:172-185
    uint32_t width = 0, height = 0, frames = 0;
    uint8_t wavelet = 0;
    ChannelHeader ch[3];
    ByteBuf data;                   // concatenated rANS streams Y | Co | Cg
    std::vector<uint8_t> to_bytes() const;                                   // pipeline.rs:200-226
    static int from_bytes(const uint8_t *data, size_t len, Chunk &out);      // pipeline.rs:235-313
};

struct Dims {
    uint32_t w = 0, h = 0, f = 0;   // as given
    uint32_t pw = 0, ph = 0, pf = 0;  // padded to even (pipeline.rs:437-439)
    uint64_t n_pixels = 0, padded = 0;
};
// pipeline.rs:67-71 checked_pixel_count + padding; returns kErrOverflow like the reference
int make_dims(uint32_t w, uint32_t h, uint32_t f, Dims &d);
int quality_to_step(uint8_t quality);   // pipeline.rs:456-457

struct EngineTimings { float ms[8] = {0, 0, 0, 0, 0, 0, 0, 0}; };

class Engine {
public:
    // payload_cap_per_stream == 0 -> worst case 2N+4 bytes (rANS emits at most 2 bytes per symbol)
    // shared_workspace: the engine owns no symbol planes; every chunk's planes live in a caller-provided buffer of
    // workspace_bytes() (device-pointer calls; it may be the buffer the chunk is later decoded into) or in the
    // chunk's RGB staging buffer (host-pointer calls)
    // well_formed_tables: every encode stores, instead of a channel's symbol counts, the table specification that
    // well_formed_hists derives from them (DESIGN.md 4.8), and builds its rANS tables from that; the rate curve bounds
    // those encodes.  A property of the engine: the decode paths read whatever the headers hold.
    Engine(const Dims &d, uint32_t cap_chunks, uint64_t payload_cap_per_stream, cudaStream_t user_stream,
           bool own_stream, bool shared_workspace = false, bool well_formed_tables = false);
    // prefer_small_smem: take the two-kernel front-end / back-end (k_forward.cu / k_inverse.cu: no shared memory to speak
    // of) instead of the fused kernels (one 106-210 KB block per SM).  For batches that run NEXT TO other batches' rANS
    // launches: a fused block cannot start on an SM whose shared memory is held by eight resident rANS streams and waits
    // for a whole rANS launch to end, the small kernels slip in beside them.
    void set_prefer_small_smem(bool v) { small_smem_ = v; }
    uint64_t workspace_bytes() const { return 3 * d_.padded; }
    bool shared_workspace() const { return shared_ws_; }
    bool well_formed_tables() const { return well_formed_; }
    ~Engine();
    bool ok() const { return ok_; }
    const Dims &dims() const { return d_; }
    uint32_t cap_chunks() const { return cap_; }
    uint64_t device_bytes() const { return dev_bytes_; }
    cudaStream_t stream() const { return st_; }

    // Device-resident encode of n chunks (n <= cap).  d_rgb[i] are device pointers.
    // coef_dump: optional device i32 [3][N] for chunk 0 (parity tests).
    int encode_device(uint8_t quality, uint8_t wavelet, const uint8_t *const *d_rgb, uint32_t n,
                      int32_t *d_coef_dump, uint8_t *const *d_work = nullptr);
    // The same encode, one chunk at a time: begin, submit chunk 0, 1, ... (each call enqueues that chunk's front-end on the
    // stream and returns), finish(n) = tables + all rANS streams + one synchronisation.  d_work as in encode_device.
    // step > 0: chunk c's quantiser step instead of the one encode_begin's quality gives (rate-controlled batches)
    int encode_begin(uint8_t quality, uint8_t wavelet);
    int encode_submit(uint32_t c, const uint8_t *d_rgb, uint8_t *d_work, int step = 0);
    int encode_finish(uint32_t n);
    // Fill a Chunk (headers + payload copied to the host) from the last encode_device.
    int fetch_chunk(uint32_t i, Chunk &out);
    // The first n chunks of the last encode_device at once: all payload copies enqueued, one synchronisation.
    int fetch_chunks(uint32_t n, Chunk *const *out);
    // Decode the payloads the last encode_device left on the device.
    int decode_device_resident(uint8_t *const *d_rgb_out, uint32_t n);
    // The same decode, one chunk at a time: begin(n) enqueues the tables and all 3n rANS streams, next(c, out) the back-end
    // of chunk c (any order; nothing synchronises: `out` is valid on the engine's stream after the call, so it may be a
    // buffer that the caller reuses for a later chunk once its own work on that stream has consumed it).
    int decode_resident_begin(uint32_t n);
    int decode_resident_next(uint32_t c, uint8_t *d_rgb_out);
    int decode_resident_end();        // one synchronisation; fills timings.ms[3..5]
    // Upload n host chunks (headers + payload) and decode them into device buffers d_rgb_out[i].
    // d_work (shared-workspace engines): where chunk i's symbol planes go; default = its output buffer, which keeps the
    // chunk on the two-kernel back-end (see run_backend for the aliasing rules of the fused one)
    // h_rgb_out (engine-owned symbol planes only): copy every chunk to host memory right after its back-end, so that
    // d_rgb_out may name the same device buffer for all chunks
    int decode_chunks(const Chunk *const *chunks, uint32_t n, uint8_t *const *d_rgb_out, uint8_t *const *d_work = nullptr,
                      uint8_t *const *h_rgb_out = nullptr);

    // Rate curve of one chunk (k_rate.cu): bytes[i] = an upper bound on the .alc length an encode at step i + 1 gives
    // (UINT64_MAX where the reference aborts; never for well-formed-tables engines), h_hist_out (host, optional) = the symbol histograms [64][3][256] of every
    // step.  Runs the front-end with the coefficient dump into chunk slot `slot` (its histogram and symbol planes, or
    // d_work for shared-workspace engines, are scratch until that chunk's real front-end), then the value histogram,
    // the step histograms, the table build and the estimate; one synchronisation.  The buffers it needs (12 B per padded
    // pixel of coefficients + the tables of 192 pseudo-streams) are allocated on the first call.
    int rate_curve(uint8_t wavelet, const uint8_t *d_rgb, uint64_t bytes[kRateSteps], unsigned *h_hist_out,
                   uint32_t slot = 0, uint8_t *d_work = nullptr);
    // PSNR curve of one chunk (DESIGN.md 4.9): sse[i] = the sum over the chunk's 3*w*h*f bytes of (input - decode)^2,
    // where the decode is that of a well-formed-tables encode at step i + 1 (such a chunk decodes to exactly the symbols
    // quant_symbol gives, so this is the decode of the quantised coefficient dump; the default encode has no such
    // curve).  Runs the front-end with the coefficient dump as rate_curve does (same slot and d_work rules), then, for
    // the fused back-end's shapes, one launch of its SSE mode over all 64 steps, otherwise per step the symbols, the
    // two-kernel back-end into an RGB scratch and a squared-difference sum; one synchronisation.  Allocates on the first
    // call the rate curve's coefficient buffer, 64 sums, and for the general path an RGB scratch of 3 B per pixel.
    int psnr_curve(uint8_t wavelet, const uint8_t *d_rgb, uint64_t sse[kRateSteps], uint32_t slot = 0,
                   uint8_t *d_work = nullptr);

    // staging buffers for host-pointer entry points
    uint8_t *rgb_stage(uint32_t slot);          // device buffer of 3*n_pixels bytes, allocated on first use
    const uint8_t *symbols_dev(uint32_t chunk) const { return sym_ptr_[chunk]; }
    EngineTimings timings;

private:
    int run_rans_encode(uint32_t n);
    void build_encode_tables(uint32_t n);
    bool overlaps(const uint8_t *sym, const uint8_t *rgb) const;
    bool fused_frontend_ok(const uint8_t *d_rgb, const uint8_t *sym) const;
    int frontend_one(uint32_t c, uint8_t wavelet, const uint8_t *d_rgb, uint8_t *sym, int step, int32_t *coef_dump);
    struct BackendHeader { uint8_t wavelet; int steps[3]; };   // what the back-end needs from a chunk's headers
    bool fused_backend_ok(const uint8_t *sym, const uint8_t *d_rgb, const BackendHeader &hdr) const;
    int run_backend(uint32_t n, const BackendHeader *hdr, uint8_t *const *d_rgb_out);
    int backend_one(uint32_t c, const BackendHeader &hdr, uint8_t *d_rgb_out);
    uint8_t last_wavelet = 0;
    uint32_t last_n = 0;              // chunks of the last successful encode (fetch_chunk, decode_device_resident)
    uint32_t submitted_ = 0;          // chunks whose front-end the current encode has enqueued
    uint32_t resident_decoded_ = 0;   // chunks whose symbol planes decode_resident_begin has queued
    int fetch_enqueue(uint32_t i, Chunk &out, bool &direct);
    Dims d_;
    uint32_t cap_ = 0;
    uint64_t pay_cap_ = 0;
    cudaStream_t st_ = nullptr;
    bool own_stream_ = false, ok_ = false;
    uint64_t dev_bytes_ = 0;
    // device
    void *d_scratch_ = nullptr;       // i16 planes (encode) / i32 coefficients (decode): 4 B * 3 * f*ph*pw
    uint8_t *d_symbols_ = nullptr;    // [cap][3][N] (absent in shared-workspace mode)
    std::vector<uint8_t *> sym_ptr_;  // per chunk: where its symbol planes [3][N] live
    bool shared_ws_ = false;
    bool small_smem_ = false;
    unsigned *d_hist_ = nullptr;      // [cap][3][256] symbol counts
    bool well_formed_ = false;
    unsigned *d_wf_hist_ = nullptr;   // [cap][3][256] table specifications (well-formed engines only)
    unsigned *d_tab_hist_ = nullptr;  // what encode tables are built from and headers store: d_wf_hist_ or d_hist_
    EncSym *d_enc_ = nullptr;         // [cap*3][256]
    uint32_t *d_dec_lut_ = nullptr;   // [cap*3][4096]
    DecAux *d_aux_ = nullptr;         // [cap*3]
    uint8_t *d_payload_ = nullptr;    // [cap*3][pay_cap]
    RansEncJob *d_enc_jobs_ = nullptr;
    RansDecJob *d_dec_jobs_ = nullptr;
    FwdFusedJob *d_fwd_jobs_ = nullptr, *h_fwd_jobs_ = nullptr;   // per chunk: RGB, symbols, histogram (fused front-end)
    InvFusedJob *d_inv_jobs_ = nullptr, *h_inv_jobs_ = nullptr;   // per chunk: symbols, RGB (fused back-end)
    unsigned long long *d_results_ = nullptr;  // [cap*3][2]
    std::vector<uint8_t *> rgb_stage_;
    std::vector<uint8_t *> overflow_bufs_;     // per stream, full-size retry buffers (rare)
    uint8_t *h_pay_ = nullptr;                 // pinned staging for one chunk's payload (host <-> device)
    size_t h_pay_cap_ = 0;
    bool ensure_pinned_payload(size_t bytes);
    std::vector<int> chunk_step_;              // quantiser step of every chunk of the last encode
    int begin_step_ = 1;                       // encode_begin's step, for submits that name none
    // rate curve (allocated by the first rate_curve call)
    bool ensure_rate_buffers();
    int dump_frontend(uint8_t wavelet, const uint8_t *d_rgb, uint32_t slot, uint8_t *d_work, uint8_t *&sym);
    int32_t *d_coef_ = nullptr;                // i32 [3][N] coefficients
    unsigned *d_vhist_ = nullptr;              // [3][2*bound+1] value histogram (largest bound of the three wavelets)
    unsigned *d_rate_hist_ = nullptr;          // [64][3][256]
    unsigned *d_rate_wf_hist_ = nullptr;       // [64][3][256] table specifications (well-formed engines only)
    EncSym *d_rate_enc_ = nullptr;             // [192][256]
    uint32_t *d_rate_lut_ = nullptr;           // [192][4096] (built, not read)
    DecAux *d_rate_aux_ = nullptr;             // [192]
    unsigned long long *d_rate_est_ = nullptr; // [192]
    unsigned long long *d_rate_out_ = nullptr, *h_rate_out_ = nullptr;   // [64] sizes + [1] out-of-range count
    // PSNR curve (allocated by the first psnr_curve call)
    bool ensure_psnr_buffers(bool rgb_scratch);
    unsigned long long *d_sse_ = nullptr, *h_sse_ = nullptr;             // [64]
    InvSseJob *d_sse_jobs_ = nullptr, *h_sse_jobs_ = nullptr;             // [64] (fused path)
    uint8_t *d_sse_rgb_ = nullptr;                                       // decode of one step, 3 B per pixel (general path)
    // pinned host mirrors
    unsigned long long *h_results_ = nullptr;
    unsigned *h_hist_ = nullptr;
    RansEncJob *h_enc_jobs_ = nullptr;
    RansDecJob *h_dec_jobs_ = nullptr;
    std::vector<uint64_t> stream_off_;         // offset of stream s inside d_payload_ (or overflow buf)
    std::vector<uint64_t> stream_len_;
    std::vector<uint8_t *> stream_base_;
    cudaEvent_t ev_[8] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
};

// Pool of single-chunk engines behind the reference-ABI entry points (alice_codec_encode / _decode).
// A well-formed-tables engine only ever serves well_formed_tables calls, and the reverse.
Engine *acquire_engine(const Dims &d, bool well_formed_tables = false);
void release_engine(Engine *e);
bool cuda_ready();   // a device is present and usable; sets the CUDA error otherwise
void trim_pinned_pool();   // release the idle page-locked payload buffers (ByteBuf pool)

}  // namespace alice
