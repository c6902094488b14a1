// k_inv_fused.cu — decode back-end as ONE kernel: three u8 symbol planes -> interleaved RGB u8; the coefficient volume
// between the temporal pass and the y/x pass never leaves the SM (6 B per pixel of HBM traffic instead of ~30).
//
// Replaces, for 64-frame chunks with even height, a width that is a multiple of 16 and headers whose quantiser steps
// keep the coefficients within the 32-bit lifting bound (every step the reference encoder can write; k_inverse.cu keeps
// the general path: any header, any shape) — reference file:line:
//   from_symbols                    src/quant.rs:572-590
//   Quantizer::dequantize_buffer    src/quant.rs:104-110, 135-146
//   Wavelet3D::inverse              src/wavelet.rs:441-484 (t, then per frame y, then x)
//   `as i16`                        src/pipeline.rs:602-611
//   ycocg_r_to_rgb_bytes            src/color.rs:245-276
//
// Mirror image of k_fwd_fused.cu.  Tile = (28-pair column strip + one halo lane per side) x (segment of row pairs) x
// (32 output frames = one half of the temporal axis); a block of 16 warps, one block per SM.
//   t phase   One thread per (row pair, channel, low/high row, column) of the next Q row pairs streams the temporal line of
//             its column: two symbols per pushed t-pair straight from global memory (a warp reads runs of consecutive bytes),
//             dequantise, inverse temporal lifting (lifting.cuh InvLift), the 32 reconstructed frames of the column go to
//             the t buffer in shared memory as i16.  The half that starts in the middle of the temporal axis pushes NST
//             extra pairs as warm-up, the other half NST extra pairs at its end.
//   y/x phase Each half-warp owns one frame, a lane two horizontal pairs: streaming inverse y lifting per owned column out
//             of the t buffer, lane-parallel inverse x lifting (warp shuffles, lanes 0/15 of a half-warp are halo lanes, so
//             the t phase also produces the two halo lanes' columns), i16 truncation, inverse colour transform, clamp,
//             12-byte RGB stores.
//
// SSE mode (SSE = true, PSNR curve of a chunk, DESIGN.md 4.9): the same decode of the coefficient dump at one quantiser
// step per job, compared with the chunk's input instead of stored.  Only two points differ: the t phase reads the i32
// coefficients at the symbols' index and maps each through quant_symbol (quant.cuh) and sym_to_coef_narrow with the
// job's step, and emit_row loads the 12 input bytes it would have stored to and sums the squared differences (a warp
// reduction and one atomicAdd per warp at the end).  A launch runs the kRateSteps jobs of one tile next to each other
// (block = tile * kRateSteps + job), so the 64 decodes of a tile read its coefficients from L2.
#include <stdlib.h>

#include <type_traits>

#include "kernels.h"
#include "lifting.cuh"
#include "quant.cuh"

namespace alice {

constexpr int kIfVP = 28;                  // valid pairs per strip (14 lanes x 2 pairs)
constexpr int kIfCols = 64;                // t-buffer columns per row: 32 low-x + 32 high-x (with the halo lanes' columns)
constexpr int kIfLines = 3 * 2 * kIfCols;  // 384 temporal lines per row pair
constexpr int kIfFrameI16 = 416;           // t-buffer frame stride in i16 (832 bytes = 208 words = 16 banks mod 32)
constexpr int kIfFrames = 32;              // output frames per block
constexpr int kIfNT = 512;
constexpr int kIfQ = 4;                    // row pairs per group: 4 * 384 lines = 3 rounds of 512 threads
constexpr int kIfSmem = kIfQ * kIfFrames * kIfFrameI16 * 2;

ALICE_D int sym_to_coef_narrow(uint32_t s, int step) {
    // quant.rs:580-588 then quant.rs:104-110 (|q| <= 128, |step| small: no wrap)
    const int q = (s & 1) ? (int)((s + 1) >> 1) : -(int)(s >> 1);
    return q * step;
}
ALICE_D uint32_t clamp_u8_i16(int v) {
    const int16_t t = (int16_t)v;
    return t < 0 ? 0u : (t > 255 ? 255u : (uint32_t)t);
}

template <int WT, bool SSE>
__global__ void ALICE_LAUNCH_BOUNDS(kIfNT, 1)
k_inv_fused(const std::conditional_t<SSE, InvSseJob, InvFusedJob> *__restrict__ jobs, int w, int h, int n_strips,
            int seg_pairs, int step0, int step1, int step2) {
    constexpr int NST = WaveletTraits<WT>::NST;
    constexpr int Q = kIfQ;
    ALICE_DYN_SMEM(smem);
    int16_t *tbuf = reinterpret_cast<int16_t *>(smem);

    const auto job = jobs[SSE ? blockIdx.x % (unsigned)kRateSteps : blockIdx.y];
    const unsigned tile = SSE ? blockIdx.x / (unsigned)kRateSteps : blockIdx.x;
    const int tid = threadIdx.x, lane = tid & 31, wv = tid >> 5;
    const int s = (int)(tile % (unsigned)n_strips);
    const int twin = (int)((tile / (unsigned)n_strips) & 1u);
    const int seg = (int)(tile / (2u * (unsigned)n_strips));
    const int halfx = w >> 1, halfy = h >> 1;
    const uint32_t fs32 = (uint32_t)w * (uint32_t)h;
    const int i0 = seg * seg_pairs, i1 = min(halfy, i0 + seg_pairs);
    const int js = max(0, i0 - NST), je = min(halfy, i1 + NST);
    const int fi = 2 * wv + (lane >> 4);          // this half-warp's frame within the block's 32
    const int xl = lane & 15;
    const int p0 = kIfVP * s - 2 + 2 * xl;        // first of this lane's two pairs
    const bool lane_ok = xl >= 1 && xl <= 14 && p0 < halfx;
    // this half-warp's frame of the output (decode) or of the input (SSE mode)
    auto *const out_frame = [&] { if constexpr (SSE) return job.ref_rgb; else return job.rgb; }() +
                            (size_t)(32 * twin + fi) * fs32 * 3;
    unsigned long long sse = 0;   // SSE mode: this thread's sum of squared differences

    // ---- t phase: row pairs [jg, jg + nq) -> t-buffer slots 0 .. nq-1
    auto t_phase = [&](int jg, int nq) {
        const int n_items = nq * kIfLines;
        QuantDev qd;
        if constexpr (SSE) qd = make_quant_dev(job.step);
        for (int item = tid; item < n_items; item += kIfNT) {
            const int qq = item / kIfLines, r = item - qq * kIfLines;
            const int ch = r / (2 * kIfCols), rr = r - ch * (2 * kIfCols);
            const int row = rr / kIfCols, col = rr - row * kIfCols;
            const int xh = col / 32, pair = kIfVP * s - 2 + (col - xh * 32);
            int16_t *dst = tbuf + qq * (kIfFrames * kIfFrameI16) + r;
            if (pair < 0 || pair >= halfx) {      // a halo column outside the image: its lane's results are never stored
#pragma unroll 4
                for (int fr = 0; fr < kIfFrames; fr++) dst[fr * kIfFrameI16] = 0;
                continue;
            }
            const int j = jg + qq;
            int step;
            if constexpr (SSE) step = job.step;
            else step = ch == 0 ? step0 : (ch == 1 ? step1 : step2);
            const uint32_t pos = (uint32_t)(row ? halfy + j : j) * (uint32_t)w + (uint32_t)(xh ? halfx + pair : pair);
            const int tp0 = twin ? 16 - NST : 0;                                   // first t-pair pushed
            const uint32_t hi_delta = 32u * fs32;                                  // its high-t symbol
            // Every symbol of the line first (2 * (16 + NST) one-byte loads in flight per thread: the phase was bound by
            // the latency of these loads when they were issued four pairs at a time), then the lifting.
            constexpr int NP = 16 + NST;
            uint32_t sl[NP], sh[NP];
            if constexpr (SSE) {
                const int32_t *pl = job.coef + ((uint32_t)ch * 64u + (uint32_t)tp0) * fs32 + pos;
#pragma unroll
                for (int jt = 0; jt < NP; jt++) {
                    sl[jt] = quant_symbol(__ldg(pl + (uint32_t)jt * fs32), qd);
                    sh[jt] = quant_symbol(__ldg(pl + hi_delta + (uint32_t)jt * fs32), qd);
                }
            } else {
                const uint8_t *pl = job.symbols + ((uint32_t)ch * 64u + (uint32_t)tp0) * fs32 + pos;   // low-t symbol of the next pair
#pragma unroll
                for (int jt = 0; jt < NP; jt++) {
                    sl[jt] = __ldg(pl + (uint32_t)jt * fs32);
                    sh[jt] = __ldg(pl + hi_delta + (uint32_t)jt * fs32);
                }
            }
            InvLift<WT, false> T;
            int ev, od;
            auto emit = [&](int e, int o) {        // one reconstructed t-pair = two frames of this column
                dst[0] = (int16_t)e;
                dst[kIfFrameI16] = (int16_t)o;
                dst += 2 * kIfFrameI16;
            };
            if (twin == 0) {
                // pairs 0 .. 15+NST are pushed, pairs 0 .. 15 come out (true, mirrored left edge)
#pragma unroll
                for (int jt = 0; jt < NP; jt++) {
                    const int lo = sym_to_coef_narrow(sl[jt], step), hi = sym_to_coef_narrow(sh[jt], step);
                    if (jt <= NST) { if (T.push(lo, hi, jt, jt, ev, od)) emit(ev, od); }
                    else { T.push_steady(lo, hi, ev, od); emit(ev, od); }
                }
            } else {
                // pairs 16-NST .. 31 are pushed; the first NST outputs (pairs 16-NST .. 15) are warm-up and dropped
#pragma unroll
                for (int jt = 0; jt < NP; jt++) {
                    const int lo = sym_to_coef_narrow(sl[jt], step), hi = sym_to_coef_narrow(sh[jt], step);
                    if (jt <= NST) T.push(lo, hi, jt, 16 - NST + jt, ev, od);
                    else T.push_steady(lo, hi, ev, od);
                    if (jt >= 2 * NST) emit(ev, od);
                }
#pragma unroll
                for (int which = 0; which < NST; which++)
                    if (T.flush(16 + NST, which, 32, ev, od)) emit(ev, od);
            }
        }
    };

    // ---- y/x phase
    InvLift<WT, false> L[3][4];   // per channel: columns 0,1 = low-x, 2,3 = high-x
    const bool edge = s == 0 || kIfVP * s + 30 >= halfx;   // some lane owns pair 0 or pair halfx-1 (the mirrored ones)
    // one reconstructed image row from its x-subband values (all lanes take part in the shuffles)
    auto emit_row = [&](int y, bool active, int (&val)[3][4]) {
        int px[3][4];
#pragma unroll
        for (int c = 0; c < 3; c++) {
            int e[2] = {val[c][0], val[c][1]}, o[2] = {val[c][2], val[c][3]};
            if (edge) inv_lanes<WT, false, 2, true>(e, o, p0, halfx);
            else inv_lanes<WT, false, 2, false>(e, o, p0, halfx);
            px[c][0] = e[0]; px[c][1] = o[0]; px[c][2] = e[1]; px[c][3] = o[1];
        }
        if (!active || !lane_ok) return;
        uint32_t bytes[12];
#pragma unroll
        for (int i = 0; i < 4; i++) {
            // pipeline.rs:608 `as i16`, then color.rs:266-273 in wrapping i16
            const int16_t yy = (int16_t)px[0][i], co = (int16_t)px[1][i], cg = (int16_t)px[2][i];
            const int16_t tt = (int16_t)(yy - (cg >> 1));
            const int16_t g = (int16_t)(cg + tt);
            const int16_t b = (int16_t)(tt - (co >> 1));
            const int16_t r = (int16_t)(co + b);
            bytes[3 * i] = clamp_u8_i16(r);
            bytes[3 * i + 1] = clamp_u8_i16(g);
            bytes[3 * i + 2] = clamp_u8_i16(b);
        }
        if constexpr (SSE) {
            const uint32_t *ref = reinterpret_cast<const uint32_t *>(out_frame + ((size_t)y * w + 2 * p0) * 3);
            unsigned part = 0;   // at most 12 * 255^2
#pragma unroll
            for (int q4 = 0; q4 < 3; q4++) {
                const uint32_t r = __ldg(ref + q4);
#pragma unroll
                for (int b = 0; b < 4; b++) {
                    const int d = (int)((r >> (8 * b)) & 0xffu) - (int)bytes[4 * q4 + b];
                    part += (unsigned)(d * d);
                }
            }
            sse += part;
        } else {
            uint32_t *dst = reinterpret_cast<uint32_t *>(out_frame + ((size_t)y * w + 2 * p0) * 3);
#pragma unroll
            for (int q4 = 0; q4 < 3; q4++)
                dst[q4] = bytes[4 * q4] | (bytes[4 * q4 + 1] << 8) | (bytes[4 * q4 + 2] << 16) | (bytes[4 * q4 + 3] << 24);
        }
    };
    auto emit_pair = [&](int jo, int (&ev)[3][4], int (&od)[3][4]) {
        const bool active = jo >= i0 && jo < i1;
        emit_row(2 * jo, active, ev);
        emit_row(2 * jo + 1, active, od);
    };
    auto load_slot = [&](int slot, int (&lo)[3][4], int (&hi)[3][4]) {
        const int16_t *tb = tbuf + slot * (kIfFrames * kIfFrameI16) + fi * kIfFrameI16 + 2 * xl;
#pragma unroll
        for (int c = 0; c < 3; c++) {
            const uint32_t *l0 = reinterpret_cast<const uint32_t *>(tb + (2 * c) * kIfCols);       // low-y row
            const uint32_t *l1 = reinterpret_cast<const uint32_t *>(tb + (2 * c + 1) * kIfCols);   // high-y row
            const uint32_t a = l0[0], b = l0[16], c2 = l1[0], d = l1[16];
            lo[c][0] = (int16_t)(a & 0xffff); lo[c][1] = (int)a >> 16; lo[c][2] = (int16_t)(b & 0xffff); lo[c][3] = (int)b >> 16;
            hi[c][0] = (int16_t)(c2 & 0xffff); hi[c][1] = (int)c2 >> 16; hi[c][2] = (int16_t)(d & 0xffff); hi[c][3] = (int)d >> 16;
        }
    };

    int k = 0;
    const int n_groups = (je - js + Q - 1) / Q;
    // FIRST = the tile's first group: its first NST + 1 steps are the warm-up / top-edge steps (general push)
    auto run_group = [&](int g, auto first_tag) {
        constexpr bool FIRST = decltype(first_tag)::value;
        const int jg = js + g * Q, nq = min(Q, je - jg);
        t_phase(jg, nq);
        __syncthreads();   // the t buffer is complete
        for (int st = 0; st < nq; st++, k++) {
            const int j = jg + st;
            int lo[3][4], hi[3][4], ev[3][4], od[3][4];
            load_slot(st, lo, hi);
            bool has = true;
            if (FIRST && k <= NST) {
#pragma unroll
                for (int c = 0; c < 3; c++)
#pragma unroll
                    for (int i = 0; i < 4; i++) has = L[c][i].push(lo[c][i], hi[c][i], k, j, ev[c][i], od[c][i]);
            } else {
#pragma unroll
                for (int c = 0; c < 3; c++)
#pragma unroll
                    for (int i = 0; i < 4; i++) L[c][i].push_steady(lo[c][i], hi[c][i], ev[c][i], od[c][i]);
            }
            if (has) emit_pair(j - NST, ev, od);   // uniform: k and j are the same for every thread
        }
        __syncthreads();   // the t buffer is free again
    };
    static_assert(kIfQ > 2, "the warm-up steps must fall into the first group");
    if (n_groups > 0) run_group(0, BoolTag<true>());
    for (int g = 1; g < n_groups; g++) run_group(g, BoolTag<false>());
    if (je == halfy && k > 0) {   // bottom of the image: the last NST row pairs come out of the flush
#pragma unroll
        for (int which = 0; which < NST; which++) {
            int ev[3][4], od[3][4];
            bool has = false;
#pragma unroll
            for (int c = 0; c < 3; c++)
#pragma unroll
                for (int i = 0; i < 4; i++) has = L[c][i].flush(k, which, halfy, ev[c][i], od[c][i]);
            if (has) emit_pair(halfy - NST + which, ev, od);
        }
    }
    if constexpr (SSE) {
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) sse += __shfl_xor_sync(kFullMask, sse, d);
        if (lane == 0 && sse) atomicAdd(job.sse, sse);
    }
}

bool inverse_fused_eligible(const uint8_t *d_symbols, const uint8_t *d_rgb, int w, int h, int f, const int steps[3]) {
    if ((unsigned long long)w * (unsigned long long)h * 192ull >= (1ull << 32)) return false;   // 32-bit symbol offsets
    for (int c = 0; c < 3; c++) {
        const long long a = steps[c] < 0 ? -(long long)steps[c] : (long long)steps[c];
        if (128 * a > kInvNarrowMaxCoef) return false;     // coefficients beyond the 32-bit lifting bound (k_inverse.cu)
    }
    (void)d_symbols;
    return f == 64 && (h & 1) == 0 && h >= 2 && (w & 15) == 0 && w >= 80 && (reinterpret_cast<uintptr_t>(d_rgb) & 3) == 0;
}

// SSE = true: n_jobs == kRateSteps, one block per (tile, job), the jobs of a tile adjacent
template <int WT, bool SSE>
static void launch_inv_fused(const std::conditional_t<SSE, InvSseJob, InvFusedJob> *d_jobs, int n_jobs, int w, int h,
                             const int steps[3], int n_sms, cudaStream_t st) {
    constexpr int NST = WaveletTraits<WT>::NST;
    const int halfx = w / 2, halfy = h / 2;
    const int n_strips = (halfx + kIfVP - 1) / kIfVP;
    int best_segs = 1;
    double best_cost = 1e30;
    for (int n_segs = 1; n_segs <= 16 && halfy / n_segs >= 8; n_segs++) {
        const int sp = (halfy + n_segs - 1) / n_segs;
        const long long blocks = (long long)n_jobs * 2 * n_strips * ((halfy + sp - 1) / sp);
        const long long waves = (blocks + n_sms - 1) / n_sms;
        const double cost = (double)waves * (sp + 2 * NST + 2);
        if (cost < best_cost) { best_cost = cost; best_segs = n_segs; }
    }
    const int seg_pairs = (halfy + best_segs - 1) / best_segs;
    const int n_segs = (halfy + seg_pairs - 1) / seg_pairs;
    const unsigned tiles = (unsigned)(2 * n_strips * n_segs);
    const dim3 grid = SSE ? dim3(tiles * (unsigned)n_jobs) : dim3(tiles, (unsigned)n_jobs);
    auto kf = k_inv_fused<WT, SSE>;
#ifndef ALICE_EMUL
    static unsigned long long done = 0;
    int dev = 0;
    cudaGetDevice(&dev);
    if (!(done & (1ull << (dev & 63)))) {
        cudaFuncSetAttribute(kf, cudaFuncAttributeMaxDynamicSharedMemorySize, kIfSmem);
        done |= 1ull << (dev & 63);
    }
#endif
    ALICE_LAUNCH(kf, grid, dim3(kIfNT), kIfSmem, st, d_jobs, w, h, n_strips, seg_pairs, steps[0], steps[1], steps[2]);
}

void inverse_backend_fused(int wavelet, const InvFusedJob *d_jobs, int n_jobs, int w, int h, const int steps[3], int n_sms,
                           cudaStream_t st) {
    if (n_jobs <= 0) return;
    switch (wavelet) {
    case WT_CDF53: launch_inv_fused<WT_CDF53, false>(d_jobs, n_jobs, w, h, steps, n_sms, st); break;
    case WT_CDF97: launch_inv_fused<WT_CDF97, false>(d_jobs, n_jobs, w, h, steps, n_sms, st); break;
    default:       launch_inv_fused<WT_HAAR, false>(d_jobs, n_jobs, w, h, steps, n_sms, st); break;
    }
}

void inverse_sse_fused(int wavelet, const InvSseJob *d_jobs, int w, int h, int n_sms, cudaStream_t st) {
    const int steps[3] = {0, 0, 0};   // each job names its own
    switch (wavelet) {
    case WT_CDF53: launch_inv_fused<WT_CDF53, true>(d_jobs, kRateSteps, w, h, steps, n_sms, st); break;
    case WT_CDF97: launch_inv_fused<WT_CDF97, true>(d_jobs, kRateSteps, w, h, steps, n_sms, st); break;
    default:       launch_inv_fused<WT_HAAR, true>(d_jobs, kRateSteps, w, h, steps, n_sms, st); break;
    }
}

}  // namespace alice
