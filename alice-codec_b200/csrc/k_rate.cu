// k_rate.cu — rate curve of one chunk: the exact symbol histograms of all 64 quantiser steps from ONE histogram of the
// wavelet coefficient values, then (engine.cu) the existing build_tables + estimate_stream_bytes on the 64 x 3
// (step, channel) pseudo-streams give a size bound for every step before any rANS work.
//
// A coefficient's symbol depends only on its value and the step (quant_symbol, quant.cuh), so for every step
//     hist_step[c][sym] = sum of count[c][v] over the values v with quant_symbol(v, step) == sym.
//
// Value range (sizes the bins).  The YCoCg-R transform of u8 RGB (color.rs:221-232) gives Y in [0, 255] and Co, Cg in
// [-255, 255], so |x| <= 255 on entry.  One lifting step adds delta = ((a + b) * c + 4096) >> 13 to the samples of one
// parity (lifting.cuh); with |a|, |b| <= B the floor of (2B|c| + 4096) / 8192 is at most 2B|c| / 8192 + 1/2 away from
// zero, so |delta| <= ceil((2B|c| + 4096) / 8192).  A stage (predict cp on the odd samples from the even ones, then
// update cu on the even samples from the new odd ones) with inputs bounded by E (even) and O (odd) gives
//     O' = O + dmax(E, cp),   E' = E + dmax(O', cu).
// The edge mirrors (wavelet.rs:180-217) reuse a neighbour, which keeps the same bound.  One level along one axis runs the
// wavelet's stages in order starting from E = O = M (5/3 and Haar: one stage, 9/7: two), and both output bands are
// bounded by max(E', O').  The pipeline's 3-D transform is one level along x, y and t of the padded volume (padding
// replicates samples), so every coefficient satisfies |v| <= axis(axis(axis(255))):
//     CDF 5/3 (cp = -4096, cu = 1024): 255 -> 511 -> 1023 -> 2047
//     Haar    (cp = -4096, cu = 2048): 255 -> 511 -> 1023 -> 2047
//     CDF 9/7 (cp = -6497, 3616; cu = -217, 1817): 255 -> 918 -> 3299 -> 11846
// (rate_value_bound evaluates this integer recursion; the numbers above are its output.)  k_coef_value_hist still
// counts values outside the bound on the device, and a non-zero count fails the call: the result is never silently
// wrong.
#include "kernels.h"
#include "lifting.cuh"
#include "quant.cuh"

namespace alice {

namespace {
long long dmax(long long b, int c) { return (2 * b * (c < 0 ? -c : c) + 4096 + 8191) / 8192; }
template <int WT> long long axis_bound(long long m) {
    long long e = m, o = m;
    for (int st = 0; st < WaveletTraits<WT>::NST; st++) {
        o += dmax(e, coef_p<WT>(st));
        e += dmax(o, coef_u<WT>(st));
    }
    return e > o ? e : o;
}
template <int WT> int bound3() { return (int)axis_bound<WT>(axis_bound<WT>(axis_bound<WT>(255))); }
}  // namespace

int rate_value_bound(int wavelet) {
    static const int b[3] = {bound3<WT_CDF53>(), bound3<WT_CDF97>(), bound3<WT_HAAR>()};
    return b[wavelet == WT_CDF97 ? 1 : (wavelet == WT_HAAR ? 2 : 0)];
}

// ---------------------------------------------------------------------------------------- value histogram
// vhist: u32 [3][2 * bound + 1], bin v + bound = count of value v (zeroed by the caller).  Most coefficients of a natural
// video are small, so a window [-kWin, kWin) is privatised in shared memory and only the tail goes to global atomics.
// Value 0 is not counted: it is N - the other bins of symbol 0 in k_step_hists, the front-end's bin-0 trick.
constexpr int kWin = 2048;

__global__ void ALICE_LAUNCH_BOUNDS(256, 8)
k_coef_value_hist(const int32_t *__restrict__ coef, unsigned long long n, int bound, unsigned *__restrict__ vhist,
                  unsigned long long *__restrict__ out_of_range) {
    __shared__ unsigned s_win[2 * kWin];
    const int c = blockIdx.y;
    for (int i = threadIdx.x; i < 2 * kWin; i += blockDim.x) s_win[i] = 0;
    __syncthreads();
    unsigned *gh = vhist + (size_t)c * (2 * bound + 1) + bound;   // gh[v] for v in [-bound, bound]
    unsigned oor = 0;
    auto count = [&](int v) {
        if (v == 0) return;
        if ((unsigned)(v + kWin) < 2u * kWin) atomicAdd(&s_win[v + kWin], 1u);
        else if (v >= -bound && v <= bound) atomicAdd(&gh[v], 1u);
        else oor++;
    };
    // n is a multiple of 8 (every padded dimension is even), so a channel is whole int4s and 32-byte aligned
    const int4 *src = reinterpret_cast<const int4 *>(coef + (size_t)c * n);
    const unsigned long long n4 = n / 4;
    for (unsigned long long i = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; i < n4;
         i += (unsigned long long)gridDim.x * blockDim.x) {
        const int4 q = __ldg(src + i);
        count(q.x); count(q.y); count(q.z); count(q.w);
    }
    __syncthreads();
    for (int i = threadIdx.x; i < 2 * kWin; i += blockDim.x) {
        const int v = i - kWin;
        if (!s_win[i]) continue;
        if (v >= -bound && v <= bound) atomicAdd(&gh[v], s_win[i]);
        else oor += s_win[i];
    }
    if (oor) atomicAdd(out_of_range, (unsigned long long)oor);
}

void coef_value_hist(const int32_t *d_coef, unsigned long long n, int bound, unsigned *d_vhist,
                     unsigned long long *d_out_of_range, cudaStream_t st) {
    if (n == 0) return;
    // one wave of 256-thread blocks over the three channels (16 KB of shared memory each, eight per SM)
    const unsigned long long items = n / 4;
    const unsigned gx = (unsigned)std::max<long long>(1, std::min<long long>((long long)((items + 255) / 256),
                                                                          (long long)device_sm_count() * 8 / 3));
    ALICE_LAUNCH(k_coef_value_hist, dim3(gx, 3), dim3(256), 0, st, d_coef, n, bound, d_vhist, d_out_of_range);
}

// ------------------------------------------------------------------------------------ step histograms
// One block per (step, channel): every value bin through the pipeline's own quantiser (quant.cuh) into 256 symbol bins.
// hist: u32 [64][3][256], row (step - 1) * 3 + channel.
__global__ void ALICE_LAUNCH_BOUNDS(256, 4)
k_step_hists(const unsigned *__restrict__ vhist, int bound, unsigned long long n, unsigned *__restrict__ hist) {
    __shared__ unsigned s_h[256];
    const int c = blockIdx.y;
    const QuantDev q = make_quant_dev((int)blockIdx.x + 1);
    s_h[threadIdx.x] = 0;
    __syncthreads();
    const unsigned *gh = vhist + (size_t)c * (2 * bound + 1) + bound;
    for (int a = 1 + (int)threadIdx.x; a <= bound; a += blockDim.x) {
        const unsigned np = gh[a], nn = gh[-a];
        if (np) {
            const uint32_t s = quant_symbol(a, q);
            if (s) atomicAdd(&s_h[s], np);
        }
        if (nn) {
            const uint32_t s = quant_symbol(-a, q);
            if (s) atomicAdd(&s_h[s], nn);
        }
    }
    __syncthreads();
    if (threadIdx.x < 32) {   // bin 0 = N - the other bins (value 0 and the dead zone)
        unsigned s = 0;
        for (int i = 1 + (int)threadIdx.x; i < 256; i += 32) s += s_h[i];
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) s += __shfl_xor_sync(kFullMask, s, d);
        if (threadIdx.x == 0) s_h[0] = (unsigned)n - s;
    }
    __syncthreads();
    hist[((size_t)blockIdx.x * 3 + c) * 256 + threadIdx.x] = s_h[threadIdx.x];
}

void step_hists(const unsigned *d_vhist, int bound, unsigned long long n, unsigned *d_hist, cudaStream_t st) {
    ALICE_LAUNCH(k_step_hists, dim3(kRateSteps, 3), dim3(256), 0, st, d_vhist, bound, n, d_hist);
}

// ------------------------------------------------------------------------------------ PSNR curve, general shapes
// The symbols of one step from the coefficient dump (the front-end's own quantiser), for inverse_backend.
__global__ void k_coef_symbols(const int32_t *__restrict__ coef, unsigned long long n, QuantDev q, uint8_t *__restrict__ sym) {
    const unsigned long long nth = (unsigned long long)gridDim.x * blockDim.x;
    for (unsigned long long i = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += nth)
        sym[i] = (uint8_t)quant_symbol(__ldg(coef + i), q);
}

void coef_symbols(const int32_t *d_coef, unsigned long long n, int step, uint8_t *d_sym, cudaStream_t st) {
    if (n == 0) return;
    const unsigned gx = (unsigned)std::max<long long>(1, std::min<long long>((long long)((n + 255) / 256),
                                                                          (long long)device_sm_count() * 8));
    ALICE_LAUNCH(k_coef_symbols, dim3(gx), dim3(256), 0, st, d_coef, n, make_quant_dev(step), d_sym);
}

// ------------------------------------------------------------------------------------------- chunk sizes
// bytes[i] = header_bytes + the three channels' predicted stream bytes at step i + 1, or UINT64_MAX where a used symbol
// has frequency 0 (EncSym.cmpl == 4096: the reference divides by zero there and the encoder reports ALICE_ERR_PANIC).
// A channel's prediction is the estimate minus the encoder's scratch allowance (kRansEncSlack + 64); a stream the
// estimate sends to the worst case (the out-of-range last symbol of a malformed table is used) is 2n + 4.
__global__ void ALICE_LAUNCH_BOUNDS(96, 1)
k_rate_sizes(const unsigned *__restrict__ hist, const EncSym *__restrict__ enc, const unsigned long long *__restrict__ est,
             unsigned long long n, unsigned long long header_bytes, unsigned long long *__restrict__ bytes) {
    __shared__ unsigned long long s_pred[3];
    __shared__ int s_zero[3];
    const int c = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const size_t s = (size_t)blockIdx.x * 3 + c;
    bool zero = false;
    for (int k = lane; k < 256; k += 32) zero = zero || (hist[s * 256 + k] != 0 && enc[s * 256 + k].cmpl == 4096u);
    zero = __any_sync(kFullMask, zero);
    if (lane == 0) {
        const unsigned long long e = est[s];
        s_pred[c] = e >= (unsigned long long)rans_enc_worst_case(n) ? 2 * n + 4 : e - (kRansEncSlack + 64);
        s_zero[c] = zero ? 1 : 0;
    }
    __syncthreads();
    if (threadIdx.x == 0)
        bytes[blockIdx.x] = (s_zero[0] | s_zero[1] | s_zero[2]) ? ~0ull : header_bytes + s_pred[0] + s_pred[1] + s_pred[2];
}

void rate_sizes(const unsigned *d_hist, const EncSym *d_enc, const unsigned long long *d_est, unsigned long long n,
                unsigned long long header_bytes, unsigned long long *d_bytes, cudaStream_t st) {
    ALICE_LAUNCH(k_rate_sizes, dim3(kRateSteps), dim3(96), 0, st, d_hist, d_enc, d_est, n, header_bytes, d_bytes);
}

}  // namespace alice
