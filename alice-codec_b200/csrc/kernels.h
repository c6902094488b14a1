// kernels.h — host-callable launchers of every CUDA kernel in libalice_codec.
// All pointers are device pointers unless a name says host; every call is asynchronous on `st`.
#pragma once
#include <algorithm>

#include "compat.h"

namespace alice {

// ---- encode front-end / decode back-end (k_forward.cu, k_inverse.cu) -------------------
// planes: i16 [3][f][ph][pw] scratch; symbols: u8 [3][pf*ph*pw]; hist: u32 [3][256] (zeroed by caller)
// coef_dump: optional i32 [3][pf*ph*pw] copy of the 3-D wavelet coefficients (parity tests), else null
void forward_frontend(int wavelet, const uint8_t *d_rgb, int16_t *d_planes, uint8_t *d_symbols, unsigned *d_hist,
                      int w, int h, int f, int pw, int ph, int pf, int step, int32_t *d_coef_dump, cudaStream_t st);
// The fused front-end (k_fwd_fused.cu): one launch for a batch of chunks of one shape, no plane scratch.  Eligible shapes:
// 64 frames, even height, width a multiple of 16 (>= 80), 16-byte aligned RGB.  hist of the batch = [job][3][256], zeroed.
struct FwdFusedJob {
    const uint8_t *rgb;      // [64][h][w][3]
    uint8_t *symbols;        // [3][64][h][w]
    unsigned *hist;          // [3][256] of this chunk
    int32_t *coef_dump;      // optional i32 [3][64][h][w] (parity tests; the launch must say dump = true), else null
};
bool forward_fused_eligible(const uint8_t *d_rgb, int w, int h, int f);
void forward_frontend_fused(int wavelet, const FwdFusedJob *d_jobs, int n_jobs, bool dump, unsigned *d_hist_base, int w, int h,
                            int step, int n_sms, cudaStream_t st);
int device_sm_count();       // multiprocessors of the current device (cached)
// The fused back-end (k_inv_fused.cu): the same shapes as the fused front-end, and quantiser steps within the 32-bit
// lifting bound (128 * |step| <= kInvNarrowMaxCoef, derived in k_inverse.cu).  The kernel reads symbols and writes RGB
// in the same launch: a chunk's RGB output must not overlap the symbol planes of any chunk of the same launch.
constexpr long long kInvNarrowMaxCoef = 15000;
struct InvFusedJob {
    const uint8_t *symbols;  // [3][64][h][w]
    uint8_t *rgb;            // [64][h][w][3]
};
bool inverse_fused_eligible(const uint8_t *d_symbols, const uint8_t *d_rgb, int w, int h, int f, const int steps[3]);
void inverse_backend_fused(int wavelet, const InvFusedJob *d_jobs, int n_jobs, int w, int h, const int steps[3], int n_sms,
                           cudaStream_t st);
// symbols: u8 [3][pf*ph*pw]; coef: i32 [3][f][ph][pw] scratch; steps[3] = per-channel quant_step from the header
void inverse_backend(int wavelet, const uint8_t *d_symbols, int32_t *d_coef, uint8_t *d_rgb, int w, int h, int f,
                     int pw, int ph, int pf, const int steps[3], cudaStream_t st);

// ---- rANS (k_rans.cu) ------------------------------------------------------------------
struct EncSym {          // one per symbol, 16 bytes (read as one uint4 {x_lim, rcp, cmpl, packed})
    uint32_t x_lim;      // renormalise while x > x_lim   (= freq * 2^19 - 1, saturated)
    uint32_t rcp;        // floor(x / freq) == ((x * rcp + rcp) >> 32) >> sh   for x < 2^31 + 2^15
    uint32_t cmpl;       // 4096 - freq  (mod 2^32)
    uint32_t packed;     // sh (low 5 bits: a wrapping shift reads it in place) | cum << 8 (16) | small(freq <= 16) << 24 | wide(freq > 4096) << 25 | zero << 26 | one << 27
};
struct DecAux {          // per stream
    uint32_t wide_sym;   // symbol whose freq is outside [1, 4096] (only the last symbol can be), or 0xffffffff
    uint32_t wide_freq;
    uint32_t wide_reachable;  // 1 if the decoder LUT maps at least one slot to wide_sym
    uint32_t reserved;
};
// the encoder checks for output room once per 512-symbol block, so a stream buffer must hold the worst case
// (2 bytes per symbol + 4 state bytes, rans.rs:269-308) plus one block of slack
constexpr size_t kRansEncSlack = 1104;
ALICE_HD size_t rans_enc_worst_case(size_t n_symbols) { return (2 * n_symbols + 4 + kRansEncSlack + 15) / 16 * 16; }
constexpr int kEncTableBytes = 256 * (int)sizeof(EncSym);
constexpr int kDecLutEntries = 4096;

// hist [n_streams][256] -> enc [n_streams][256], dec_lut [n_streams][4096], aux [n_streams],
// freq/cum u16 [n_streams][256] (optional, may be null).  n_symbols <= 256 (256 in the pipeline).
void build_tables(const unsigned *d_hist, int n_streams, int n_symbols, EncSym *d_enc, uint32_t *d_dec_lut,
                  DecAux *d_aux, uint16_t *d_freq, uint16_t *d_cum, uint8_t *d_lut8, cudaStream_t st);

// out [n_streams][256] = the well-formed table specification of each stream's symbol counts (rule in k_rans.cu,
// DESIGN.md 4.8): a histogram whose from_histogram table keeps every used symbol's range inside [0, 4096)
void well_formed_hists(const unsigned *d_counts, int n_streams, unsigned *d_out, cudaStream_t st);

// est[i] = upper bound on the bytes stream i will take (multiple of 16, includes the encoder's slack), from hist + enc
void estimate_stream_bytes(const unsigned *d_hist, const EncSym *d_enc, int n_streams, unsigned long long n_symbols,
                           unsigned long long *d_est, cudaStream_t st);

struct RansEncJob {      // device-visible description of one stream to encode
    const uint8_t *symbols;
    unsigned long long n;
    uint8_t *out;        // scratch of `cap` bytes; the stream ends at out+cap
    unsigned long long cap;
};
// results[i] = {len, status}: status 0 ok, 1 overflow (cap too small), 2 zero-frequency symbol (reference aborts)
// shared_gpu: other launches run beside this one (several batches in flight): four-warp blocks = one stream per warp
// scheduler and block, so the streams of concurrent launches spread evenly over the schedulers
void rans_encode(const RansEncJob *d_jobs, const EncSym *d_enc, const unsigned *d_hist, unsigned long long *d_results,
                 int n_streams, cudaStream_t st, bool shared_gpu = false);
struct RansDecJob {
    const uint8_t *in;
    unsigned long long len;
    uint8_t *symbols;
    unsigned long long n;
};
void rans_decode(const RansDecJob *d_jobs, const uint32_t *d_dec_lut, const DecAux *d_aux, int n_streams,
                 cudaStream_t st, bool shared_gpu = false);

// ---- rate curve (k_rate.cu): the symbol histograms of every quantiser step from one histogram of coefficient values
constexpr int kRateSteps = 64;   // quantiser steps 1..64 (quality_to_step)
// largest |coefficient| of the pipeline's 3-D transform of u8 RGB for this wavelet (derivation in k_rate.cu)
int rate_value_bound(int wavelet);
// coef: i32 [3][n] (n a multiple of 8); vhist: u32 [3][2*bound+1] (zeroed by caller), bin v + bound = count of v, v != 0;
// *out_of_range (zeroed by caller) += number of coefficients with |v| > bound
void coef_value_hist(const int32_t *d_coef, unsigned long long n, int bound, unsigned *d_vhist,
                     unsigned long long *d_out_of_range, cudaStream_t st);
// hist [kRateSteps][3][256]: row (step-1)*3 + channel = the symbol histogram a front-end at that step would produce
void step_hists(const unsigned *d_vhist, int bound, unsigned long long n, unsigned *d_hist, cudaStream_t st);
// bytes[kRateSteps] = header_bytes + predicted stream bytes of the three channels (from estimate_stream_bytes' est),
// UINT64_MAX where a used symbol has frequency 0
void rate_sizes(const unsigned *d_hist, const EncSym *d_enc, const unsigned long long *d_est, unsigned long long n,
                unsigned long long header_bytes, unsigned long long *d_bytes, cudaStream_t st);

// ---- PSNR curve (DESIGN.md 4.9): the squared error of the decode at every step, from the front-end's coefficient dump
// sym [n] = quant_symbol(coef[i], step): the symbols a front-end at that step writes (k_rate.cu)
void coef_symbols(const int32_t *d_coef, unsigned long long n, int step, uint8_t *d_sym, cudaStream_t st);
// The SSE mode of the fused back-end (k_inv_fused.cu): kRateSteps jobs in one launch, each decodes the coefficient dump
// at its step and adds sum((ref - decode)^2) over the chunk to *sse (zeroed by the caller).  The shapes, alignment and
// bound of inverse_fused_eligible (with ref_rgb in place of the output).
struct InvSseJob {
    const int32_t *coef;       // [3][64][h][w] coefficient dump of the front-end
    const uint8_t *ref_rgb;    // [64][h][w][3] the chunk's input
    unsigned long long *sse;
    int step;
};
void inverse_sse_fused(int wavelet, const InvSseJob *d_jobs, int w, int h, int n_sms, cudaStream_t st);

// ---- generic element-wise / line kernels behind the public stage API (k_generic.cu) -----
void lift_axis(int32_t *d_data, int32_t *d_tmp, int wavelet, bool inverse, int axis, long long w, long long h,
               long long d, cudaStream_t st);  // one 1-D transform along `axis` (0=x,1=y,2=t) of every line
// fast per-pass kernels for volumes with w % 4 == 0 and even transformed dimensions (k_wavelet_i32.cu), out of place:
//   wavelet_xy_i32: the 2-D transform (or its inverse) of each of n_frames images of w x h
//   wavelet_t_i32 : the temporal transform (or its inverse) of a w*h = frame_sz by d volume
bool wavelet_fast_eligible(const int32_t *a, const int32_t *b, long long w, long long h, long long d, int ndim);
void wavelet_xy_i32(int wavelet, bool inverse, const int32_t *d_src, int32_t *d_dst, int w, int h, long long n_frames,
                    cudaStream_t st);
void wavelet_t_i32(int wavelet, bool inverse, const int32_t *d_src, int32_t *d_dst, size_t frame_sz, int d, cudaStream_t st);
void rgb_to_ycocg(const uint8_t *d_rgb, int16_t *d_y, int16_t *d_co, int16_t *d_cg, size_t n, cudaStream_t st);
void ycocg_to_rgb(const int16_t *d_y, const int16_t *d_co, const int16_t *d_cg, uint8_t *d_rgb, size_t n,
                  cudaStream_t st);
void quantize_i32(const int32_t *d_in, int32_t *d_out, size_t n, int step, int dz, int *d_panic, cudaStream_t st);
void fast_quantize_i32(const int32_t *d_in, int32_t *d_out, size_t n, int dz, unsigned long long recip,
                       unsigned shift, cudaStream_t st);
void dequantize_i32(const int32_t *d_in, int32_t *d_out, size_t n, int step, cudaStream_t st);
void to_symbols_u8(const int32_t *d_in, uint8_t *d_out, size_t n, cudaStream_t st);
void from_symbols_i32(const uint8_t *d_in, int32_t *d_out, size_t n, cudaStream_t st);
void histogram_u8(const uint8_t *d_in, size_t n, unsigned *d_hist256, cudaStream_t st);  // adds into d_hist256
void sum_i64(const int32_t *d_in, size_t n, long long *d_sum, cudaStream_t st);          // adds into *d_sum
void sq_diff_sum_u8(const uint8_t *d_a, const uint8_t *d_b, size_t n, unsigned long long *d_sum,
                    cudaStream_t st);                                                      // adds into *d_sum
// InterleavedRansEncoder / Decoder symbol order (rans.rs:420-430, 508-520): planes[k * stride + j] <-> stream k, symbol j
void deinterleave4_u8(const uint8_t *d_in, size_t n, uint8_t *d_planes, size_t stride, cudaStream_t st);
void interleave_rr_u8(const uint8_t *d_planes, size_t stride, uint8_t *d_out, size_t n, const unsigned long long counts[4],
                      cudaStream_t st);
void variance_seq_f64(const int32_t *d_in, size_t n, double mean, double *d_acc, cudaStream_t st);

// ---- AnalyticalRDO statistics and per-octant quantiser (k_rdo.cu; SURVEY.md 8f-2) -------------------------
struct RdoViewHost {     // a sub-box of a w x h x d i32 volume on the device, visited in row-major order
    const int32_t *base; // first element of the sub-box
    unsigned long long n;
    unsigned sw, sh;     // sub-box width and height
    unsigned long long row, plane;   // volume strides W and W*H
};
// h_acc[i] = the f64 sum of squared deviations of view i accumulated in slice order exactly as quant.rs:425-432
// does (bit-identical to the sequential loop), h_mean[i] = its mean.  At most 8 views.  Synchronises `st`.
cudaError_t rdo_seq_sums(const RdoViewHost *h_views, int n_views, double *h_acc, double *h_mean, cudaStream_t st);
// FastQuantizer::quantize of every element with the constants of its octant (index 4*[x>=w/2] + 2*[y>=h/2] + [t>=d/2])
void rdo_quantize_volume(const int32_t *d_in, int32_t *d_out, unsigned w, unsigned h, unsigned d, const int dz[8],
                         const unsigned long long recip[8], const unsigned shift[8], cudaStream_t st);

// ---- small per-thread scratch (k_generic.cu): cudaMalloc / cudaFree cost milliseconds next to other contexts' memory,
// so short reductions keep one growing device block and one pinned host block per calling thread and device.
// Returns nullptr if the allocation fails.  The blocks live until the thread's next request on another device.
void *scratch_device(size_t bytes);
void *scratch_pinned(size_t bytes);

// ---- synthetic inputs (k_synth.cu; SURVEY.md Appendix D) ---------------------------------
void synth_rgb(int kind, uint32_t seed, int w, int h, int f, uint8_t *d_rgb, cudaStream_t st);

}  // namespace alice
