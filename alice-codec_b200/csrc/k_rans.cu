// k_rans.cu — FrequencyTable construction and the rANS coder, one warp per independent
// (chunk, channel) stream so that every stream is byte-identical to the reference.
//
// Replaces (reference file:line):
//   FrequencyTable::from_histogram / uniform      src/rans.rs:102-189
//   RansEncoder::{new, encode, encode_symbols, finish}   src/rans.rs:249-308
//   RansDecoder::{new, init_state, decode, decode_n}     src/rans.rs:330-381
//
// rANS is a serial recurrence on a 32-bit state and .alc carries no side information, so a
// stream cannot be split bit-exactly: throughput comes from (a) the shortest possible
// dependent chain per symbol and (b) hundreds of streams in flight (grid = streams of all
// in-flight chunks).  Each warp alternates between lane-parallel phases (all 32 lanes move
// symbols, table entries, stream bytes and output through shared memory, 512 symbols at a
// time) and a serial phase in which lane 0 alone runs the state recurrence out of shared
// memory and registers (one active lane keeps every shared access a single wavefront).
// profiles/r01_rans_stalls.md records the measurements behind these choices.
//
// Encoder step (src/rans.rs:269-285), for freq in (16, 4096]:
//     k  = x > freq*2^19 - 1                     (one renormalisation byte at most when freq > 16)
//     q0 = floor(x / freq) = umulhi(x, rcp) >> sh             exact for x < 2^31 + 2^15 (DESIGN.md 4.3)
//     q  = q0 >> 8k        because floor(floor(x / 256) / f) == floor(floor(x / f) / 256)
//     x' = (x >> 8k) + cum + q * (4096 - freq)   == ((x>>8k) / f << 12) + (x>>8k) % f + cum
// so the division does not wait for the renormalisation decision; both outcomes are computed
// and one is selected.  The serial loop only logs the state before each step; all lanes then
// re-derive the emitted bytes from (state, limit) and write them.  Groups of 16 symbols that
// contain a freq in [2, 16] run a two-byte variant; freq == 1, freq > 4096 (the u16-wrapped
// last symbol of a malformed table) or freq == 0 take a literal step with a true division.
//
// Decoder step (src/rans.rs:351-371): {freq, slot - cum} come from two 4096-entry u16 shared tables.  The loop keeps
// the state only as x3 = x << 1: its low bits are the table address, its high bits x >> 12, and the renormalising funnel
// shift produces the next x3 directly.  Stream bytes come from a shared "window" table holding, for every byte
// position, the next eight bytes as two big-endian words (8 bytes per position: the renormalisation shift in bits is
// the address increment), so renormalisation is two selects and two funnel shifts.
#include <math.h>
#include <stdlib.h>

#include "kernels.h"

namespace alice {

constexpr uint32_t kRansL = 1u << 23;   // rans.rs:244
constexpr uint32_t kProbBits = 12;      // rans.rs:50
constexpr uint32_t kProbScale = 1u << 12;

// EncSym.packed flag bits
constexpr uint32_t kEncSmall = 1u << 24;   // freq <= 16: may need two renormalisation bytes
constexpr uint32_t kEncWide = 1u << 25;    // freq > 4096 (u16-wrapped last symbol)
constexpr uint32_t kEncZero = 1u << 26;    // freq == 0: the reference divides by zero
constexpr uint32_t kEncOne = 1u << 27;     // freq == 1: the reciprocal does not fit 32 bits

// ------------------------------------------------------------------------ table building
ALICE_D uint32_t pack_dec(uint32_t sym, uint32_t freq, uint32_t bias) {
    // sym (8) | freq-1 (12) | slot-cum (12); freq outside [1,4096] is resolved through DecAux
    uint32_t fm1 = (freq >= 1 && freq <= kProbScale) ? freq - 1 : 0;
    return sym | (fm1 << 8) | (bias << 20);
}

// FrequencyTable::from_histogram of one stream (rans.rs:102-125; uniform, rans.rs:158-189, for an all-zero histogram):
// freq / cum of symbols [0, n), 0 above.  The normalisation is a serial running sum in the reference; 256 entries are
// cheap enough to do exactly that on one thread.
ALICE_D void normalise_table(const unsigned *h, int n, uint32_t *s_freq, uint32_t *s_cum) {
    unsigned long long total = 0;
    for (int i = 0; i < n; i++) total += h[i];
    if (total == 0) {
        // u16 arithmetic
        uint16_t fps = (uint16_t)(kProbScale / (uint32_t)n);
        uint16_t cum = 0;
        for (int i = 0; i < n; i++) { s_cum[i] = cum; s_freq[i] = fps; cum = (uint16_t)(cum + fps); }
        s_freq[n - 1] = (uint16_t)((uint16_t)kProbScale - (uint16_t)s_cum[n - 1]);
    } else {
        uint32_t cum = 0, norm = 0;
        for (int i = 0; i < n; i++) {
            uint32_t c = h[i];
            uint32_t fr = 1;
            if (c != 0) {
                unsigned long long t = ((unsigned long long)c * kProbScale) / total;
                fr = t < 1 ? 1u : (uint32_t)t;
            }
            norm += fr;
            s_cum[i] = (uint16_t)cum;
            s_freq[i] = (uint16_t)fr;
            cum += fr;
        }
        if (norm != kProbScale) {
            int diff = (int)kProbScale - (int)norm;
            s_freq[n - 1] = (uint16_t)((int)s_freq[n - 1] + diff);
        }
    }
    for (int i = n; i < 256; i++) { s_freq[i] = 0; s_cum[i] = 0; }
}

__global__ void ALICE_LAUNCH_BOUNDS(256, 1)
k_build_tables(const unsigned *__restrict__ hist, int n_symbols, EncSym *__restrict__ enc,
               uint32_t *__restrict__ dec_lut, DecAux *__restrict__ aux, uint16_t *__restrict__ freq_out,
               uint16_t *__restrict__ cum_out, uint8_t *__restrict__ lut8_out) {
    __shared__ uint32_t s_freq[256];
    __shared__ uint32_t s_cum[256];
    const int stream = blockIdx.x;
    const int tid = threadIdx.x;
    const unsigned *h = hist + (size_t)stream * 256;
    const int n = n_symbols;

    if (tid == 0) {
        normalise_table(h, n, s_freq, s_cum);
        const uint32_t fl = s_freq[n - 1];
        const bool last_wide = !(fl >= 1 && fl <= kProbScale);
        DecAux a;
        a.wide_sym = last_wide ? (uint32_t)(n - 1) : 0xffffffffu;
        a.wide_freq = fl;
        // the decoder can meet the out-of-range last symbol only if its slot range starts below 4096
        a.wide_reachable = (last_wide && fl != 0 && s_cum[n - 1] < kProbScale) ? 1u : 0u;
        a.reserved = 0;
        aux[stream] = a;
    }
    __syncthreads();

    {   // encoder entry of symbol `tid`
        const uint32_t f = s_freq[tid], cum = s_cum[tid];
        EncSym e;
        const bool zero = (f == 0), wide = (f > kProbScale), one = (f == 1), small = (f >= 2 && f <= 16);
        e.x_lim = zero ? 0u : (f >= 8192u ? 0xffffffffu : (f << 19) - 1u);
        uint32_t sh = 0, rcp = 0;
        if (f >= 2 && !wide) {
            // floor(x / f) == (umulhi(x, rcp)) >> sh for every x < 2^31 + 2^15 (DESIGN.md "exact division")
            if ((f & (f - 1)) == 0) {
                sh = 30u - (uint32_t)__clz((int)f);            // log2(f) - 1
                rcp = 0x80000000u;
            } else {
                sh = 31u - (uint32_t)__clz((int)f);            // floor(log2 f)
                rcp = (uint32_t)((1ull << (32 + sh)) / f) + 1u;
            }
        }
        e.rcp = rcp;
        e.cmpl = kProbScale - f;
        // sh in the low five bits (a wrapping shift takes it from there), cum in bits 8..23, flags from bit 24
        e.packed = sh | (cum << 8) | (small ? kEncSmall : 0u) | (wide ? kEncWide : 0u) | (zero ? kEncZero : 0u) |
                   (one ? kEncOne : 0u);
        enc[(size_t)stream * 256 + tid] = e;
        if (freq_out) freq_out[(size_t)stream * 256 + tid] = (uint16_t)f;
        if (cum_out) cum_out[(size_t)stream * 256 + tid] = (uint16_t)cum;
    }

    // decoder LUT (rans.rs:134-144): zero-initialised, then each symbol fills [cum, min(cum+f, 4096))
    uint32_t *lut = dec_lut + (size_t)stream * kDecLutEntries;
    uint8_t *l8 = lut8_out ? lut8_out + (size_t)stream * kDecLutEntries : nullptr;
    for (uint32_t slot = tid; slot < kProbScale; slot += blockDim.x) {
        lut[slot] = pack_dec(0, s_freq[0], slot - s_cum[0]) & (n > 0 ? 0xffffffffu : 0u);
        if (l8) l8[slot] = 0;
    }
    __syncthreads();
    if (tid < n) {
        const uint32_t f = s_freq[tid], start = s_cum[tid];
        uint32_t end = start + f;
        if (end > kProbScale) end = kProbScale;
        for (uint32_t slot = start; slot < end; slot++) {
            lut[slot] = pack_dec((uint32_t)tid, f, slot - start);
            if (l8) l8[slot] = (uint8_t)tid;
        }
    }
}

void build_tables(const unsigned *d_hist, int n_streams, int n_symbols, EncSym *d_enc, uint32_t *d_dec_lut,
                  DecAux *d_aux, uint16_t *d_freq, uint16_t *d_cum, uint8_t *d_lut8, cudaStream_t st) {
    if (n_streams <= 0) return;
    ALICE_LAUNCH(k_build_tables, dim3(n_streams), dim3(256), 0, st, d_hist, n_symbols, d_enc, d_dec_lut, d_aux,
                 d_freq, d_cum, d_lut8);
}

// ------------------------------------------------------------------ well-formed table specification
// The histogram a well-formed-tables encode stores in a channel header (DESIGN.md 4.8), from the stream's symbol
// counts c (N = sum c, used = c > 0):
//   1. from_histogram(c) already gives every used symbol 1 <= f <= 4096 and cum + f <= 4096: H' = c.
//   2. otherwise, with Z = empty bins among 0..254 and S = 4096 - Z: F[j] = max(1, c[j] * S / N) for used j, D = S - sum F;
//      D > 0: +1 for the D used symbols with the largest c[j] * S mod N (ties to the lower index); D < 0: -1 from the
//      used symbol with the largest F > 1 (ties to the lower index), -D times.  H'[j] = F[j] for used j < 255, 0 for
//      empty j < 255, H'[255] = 4096 - sum of F[j] over used j < 255.
// H' sums to 4096, so from_histogram(H') gives every used j < 255 exactly F[j], every empty bin 1 and symbol 255 the
// rest: every used range lies inside [0, 4096), and every decoder of the format decodes the stream exactly.
__global__ void ALICE_LAUNCH_BOUNDS(256, 1)
k_well_formed_hists(const unsigned *__restrict__ counts, unsigned *__restrict__ out) {
    __shared__ uint32_t s_freq[256];
    __shared__ uint32_t s_cum[256];
    __shared__ unsigned long long s_rem[256];
    __shared__ unsigned long long s_total;
    __shared__ int s_clean, s_empty, s_d;
    __shared__ uint32_t s_head;          // sum of F over symbols 0..254
    const int stream = blockIdx.x, tid = threadIdx.x;
    const unsigned *c = counts + (size_t)stream * 256;
    unsigned *o = out + (size_t)stream * 256;
    const unsigned cj = c[tid];
    if (tid == 0) {
        normalise_table(c, 256, s_freq, s_cum);
        unsigned long long total = 0;
        int clean = 1, empty = 0;
        for (int i = 0; i < 256; i++) {
            total += c[i];
            if (c[i]) clean &= (s_freq[i] >= 1 && s_freq[i] <= kProbScale && s_cum[i] + s_freq[i] <= kProbScale);
            else if (i < 255) empty++;
        }
        s_total = total;
        s_clean = clean;
        s_empty = empty;
    }
    __syncthreads();
    if (s_clean) { o[tid] = cj; return; }    // block-uniform; also every all-zero histogram (no used symbol)
    const unsigned long long n = s_total, scale = kProbScale - (unsigned long long)s_empty;
    const unsigned long long prod = (unsigned long long)cj * scale;
    const unsigned long long q = prod / n;
    uint32_t f = cj ? (q < 1 ? 1u : (uint32_t)q) : 0u;   // f > 0 marks a used symbol below
    s_freq[tid] = f;
    s_rem[tid] = prod % n;
    __syncthreads();
    if (tid == 0) {
        long long sum = 0;
        for (int i = 0; i < 256; i++) sum += s_freq[i];
        s_d = (int)((long long)scale - sum);
    }
    __syncthreads();
    const int d = s_d;
    if (d > 0 && cj) {   // rank among the used symbols by (remainder descending, index ascending)
        const unsigned long long r = s_rem[tid];
        int rank = 0;
        for (int k = 0; k < 256; k++) {
            const unsigned long long rk = s_rem[k];
            rank += (s_freq[k] != 0 && (rk > r || (rk == r && k < tid))) ? 1 : 0;
        }
        if (rank < d) f++;
    }
    __syncthreads();
    s_freq[tid] = f;
    __syncthreads();
    if (tid == 0) {
        // at most one step per symbol that max(1, .) raised; some used symbol keeps F > 1 since used <= S
        for (int k = d; k < 0; k++) {
            int best = -1;
            for (int i = 0; i < 256; i++)
                if (s_freq[i] > 1 && (best < 0 || s_freq[i] > s_freq[best])) best = i;
            s_freq[best]--;
        }
        uint32_t head = 0;
        for (int i = 0; i < 255; i++) head += s_freq[i];
        s_head = head;
    }
    __syncthreads();
    o[tid] = tid < 255 ? s_freq[tid] : kProbScale - s_head;
}

void well_formed_hists(const unsigned *d_counts, int n_streams, unsigned *d_out, cudaStream_t st) {
    if (n_streams <= 0) return;
    ALICE_LAUNCH(k_well_formed_hists, dim3(n_streams), dim3(256), 0, st, d_counts, d_out);
}

// ------------------------------------------------------------------- stream size estimate
// Upper bound on the bytes a stream will take, from its histogram and table alone, so that a batch can place its
// payloads back to back instead of reserving a fixed slot per stream.  A step multiplies the state by at most
// (4096 / freq) * (1 + 2^-10) -- x' = 4096 * floor(x / f) + (x mod f) + cum < 4096 * (x / f + 2) with x / f >= 2^11 -- so the
// stream holds at most sum(hist * log2(4096 / freq)) / 8 + n * log2(1 + 2^-10) / 8 bytes + the 4 state bytes; the
// estimate adds n / 4096 + the encoder's block slack.  Streams that use the out-of-range last symbol of a malformed
// table (freq > 4096 or 0: SURVEY.md 0.7) get the worst case of two bytes per symbol.
__global__ void ALICE_LAUNCH_BOUNDS(256, 1)
k_estimate_stream_bytes(const unsigned *__restrict__ hist, const EncSym *__restrict__ enc, unsigned long long n_symbols,
                        unsigned long long *__restrict__ est) {
    __shared__ double s_bits[8];
    __shared__ int s_bad;
    const int stream = blockIdx.x, tid = threadIdx.x;
    if (tid == 0) s_bad = 0;
    __syncthreads();
    const unsigned h = hist[(size_t)stream * 256 + tid];
    const EncSym e = enc[(size_t)stream * 256 + tid];
    double bits = 0.0;
    if (h) {
        if (e.packed & (kEncWide | kEncZero)) s_bad = 1;
        else bits = (double)h * log2(4096.0 / (double)(kProbScale - e.cmpl));
    }
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) bits += __shfl_xor_sync(kFullMask, bits, d);
    if ((tid & 31) == 0) s_bits[tid >> 5] = bits;
    __syncthreads();
    if (tid == 0) {
        double t = 0.0;
        for (int i = 0; i < 8; i++) t += s_bits[i];
        unsigned long long b = (unsigned long long)(t / 8.0) + n_symbols / 4096 + 4 + kRansEncSlack + 64;
        const unsigned long long worst = rans_enc_worst_case(n_symbols);
        est[stream] = (s_bad || b > worst) ? worst : (b + 15) / 16 * 16;
    }
}

void estimate_stream_bytes(const unsigned *d_hist, const EncSym *d_enc, int n_streams, unsigned long long n_symbols,
                           unsigned long long *d_est, cudaStream_t st) {
    if (n_streams <= 0) return;
    ALICE_LAUNCH(k_estimate_stream_bytes, dim3(n_streams), dim3(256), 0, st, d_hist, d_enc, n_symbols, d_est);
}

// --------------------------------------------------------------------------------- encode
template <int V> struct IntC { static constexpr int value = V; };
#ifndef ALICE_EMUL
// opt-in to > 48 KB of dynamic shared memory: a per-device function attribute, set once per device and kernel
template <class K> static void ensure_dyn_smem(K kernel, int bytes, unsigned long long &done_mask) {
    int dev = 0;
    cudaGetDevice(&dev);
    const unsigned long long bit = 1ull << (dev & 63);
    if (done_mask & bit) return;   // idempotent; a race only repeats the call
    cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
    done_mask |= bit;
}
#endif
// Block shape per launch (profiles/r02_switches.md).  A launch lasts as long as its slowest stream, and a stream that
// shares its warp scheduler with another runs at ~3/4 of its speed alone (the serial loops are bound by the latency of
// their dependent chains, so the two interleave almost for free: 2 x 0.76 = 1.5x the throughput).
//   * two to eight streams per SM: single-warp blocks; the hardware spreads them evenly over the four schedulers of an
//     SM at four and at eight blocks per SM (measured: 54.9 / 32.4 Msym/s per lane at four, 41.9 / 27.9 at eight);
//   * fewer streams than two per SM: four-warp blocks = one warp per scheduler, so that the blocks of several batches
//     in flight do not pile up on one scheduler (round 1: encode 2.95-3.7 s -> 2.55-2.9 s with three batches in flight);
//   * more than eight per SM do not fit the decoder's shared memory at once; four-warp blocks keep the waves aligned.
// Tried and dropped: two streams per WARP, one per half-warp, lanes 0 and 16 running the two recurrences in the same
// instructions (profiles/r02_rans_two_streams_per_warp.jsonl).  The halves do execute converged (ncu: 2 threads per
// instruction), but a stream then runs at 42 / 28.7 Msym/s whatever the load: the per-half table base costs the decoder
// an address add on its dependent chain (68 instead of 60.6 cycles per symbol), and both kernels lose a fifth of their
// single-stream speed, which is what a one-chunk call through the reference ABI sees.
int device_sm_count() {
#ifdef ALICE_EMUL
    return kNumSMs;
#else
    static int cached[64] = {0};
    int dev = 0;
    cudaGetDevice(&dev);
    int &c = cached[dev & 63];
    if (c == 0) {
        int v = 0;
        if (cudaDeviceGetAttribute(&v, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || v <= 0) { cudaGetLastError(); v = kNumSMs; }
        c = v;
    }
    return c;
#endif
}
template <class F> static void launch_lanes(int n_streams, bool shared_gpu, F f) {
    const int sms = device_sm_count();
    if (!shared_gpu && n_streams >= 2 * sms && n_streams <= 8 * sms) f(IntC<1>());
    else f(IntC<4>());
}

constexpr int kEncBlock = 512;                  // symbols per warp-wide fetch (16 bytes per lane)
constexpr int kEncRing = 2 * kEncBlock + 64;    // bytes one block can emit (2 per symbol) + the 4 state bytes + slack
constexpr uint32_t kGrpSmall = 1u, kGrpGeneric = 2u;

// Streams per block (LPB): with four warps per block = one per SM sub-partition the streams of concurrent launches
// (several batches in flight) spread evenly over the warp schedulers instead of piling up single-warp blocks on a
// few of them (measured: encode 2.95-3.7 s -> 2.55-2.9 s with three batches in flight).  A launch that fills the
// machine on its own uses single-warp blocks, which measured 6-11 % faster there (decode 3.66 s vs 4.06 s).
constexpr int kEncSmemPerWarp = 256 * 16 + kEncBlock * (16 + 4 + 1) + 32 * 4 + kEncRing;   // 16 064 bytes
static_assert(kEncSmemPerWarp % 16 == 0, "per-warp shared memory must keep 16-byte alignment");

template <int LPB>
__global__ void ALICE_LAUNCH_BOUNDS(32 * LPB, 1)
k_rans_encode(const RansEncJob *__restrict__ jobs, const EncSym *__restrict__ enc_all,
              unsigned long long *__restrict__ results, int n_streams) {
    ALICE_DYN_SMEM(smem_all);
    const int stream = blockIdx.x * LPB + (threadIdx.x >> 5);
    if (stream >= n_streams) return;                 // warp-uniform; the kernel has no block-level barrier
    unsigned char *smem = smem_all + (size_t)(threadIdx.x >> 5) * kEncSmemPerWarp;
    uint4 *tab = reinterpret_cast<uint4 *>(smem);                                   // EncSym of every symbol
    // staged per symbol of the block, indexed [b][lane] (symbol b of lane's group): conflict-free for the lanes
    uint4 *st_a = tab + 256;                                                        // {x_lim, rcp, cmpl, sh | cum << 8 | flags}
    uint32_t *st_x = reinterpret_cast<uint32_t *>(st_a + kEncBlock);                // state before the step of each symbol
    uint32_t *grp = st_x + kEncBlock;                                               // per group of 16 symbols: kGrpSmall | kGrpGeneric
    uint8_t *ring = reinterpret_cast<uint8_t *>(grp + 32);                          // emitted bytes of the block, filled from the top down
    uint8_t *st_sym = ring + kEncRing;                                              // the symbols themselves (generic path)
    const int lane = threadIdx.x & 31;
    const bool lane0 = lane == 0;
    {
        const uint4 *src = reinterpret_cast<const uint4 *>(enc_all + (size_t)stream * 256);
        for (int i = lane; i < 256; i += 32) tab[i] = src[i];
    }
    __syncwarp();
    const RansEncJob job = jobs[stream];
    const uint8_t *sym = job.symbols;
    uint8_t *wp = job.out + job.cap;        // the stream ends at out + cap and grows downwards
    uint32_t x = kRansL;                    // rans.rs:244
    uint32_t sp = kEncRing;                 // next byte goes to ring[--sp]
    uint32_t status = 0;                    // 1 overflow, 2 zero-frequency symbol
    auto room = [&](uint32_t need) { return (unsigned long long)(wp - job.out) >= need; };

    // generic step, any frequency (rans.rs:269-285 literally)
    auto step_generic = [&](const uint4 e) {
        if (e.w & kEncZero) { status |= 2u; return; }
        while (x > e.x) {                   // while x >= freq << 19 (limit saturated for freq >= 8192: never)
            --sp;
            ring[sp] = (uint8_t)x;          // every lane stores the same byte (see the note at the state loop)
            x >>= 8;
        }
        const uint32_t f = kProbScale - e.z;
        const uint32_t q = x / f;
        x = x + ((e.w >> 8) & 0xffffu) + q * e.z;  // (q << 12) + x % f + cum
    };
    // move ring[sp, kEncRing) to the stream (which grows towards lower addresses) and reset the ring
    auto flush = [&]() {
        __syncwarp();
        const uint32_t n = (uint32_t)kEncRing - sp;
        uint8_t *dst = wp - n;
        for (uint32_t i = lane; i < n; i += 32) dst[i] = ring[sp + i];
        wp = dst;
        sp = kEncRing;
        __syncwarp();
    };

    long long i = (long long)job.n;  // symbols [0, i) remain; encode from the back (rans.rs:288-294)
    // ragged tail until the read pointer is 16-byte aligned
    if (!room(64)) status |= 1u;
    while (i > 0 && ((reinterpret_cast<uintptr_t>(sym + i)) & 15) != 0 && status == 0) {
        step_generic(tab[__ldg(sym + i - 1)]);
        i--;
    }
    flush();
    // full 512-symbol blocks: one coalesced 16-byte load per lane
    uint4 cur = make_uint4(0, 0, 0, 0);
    if (i >= kEncBlock) cur = __ldg(reinterpret_cast<const uint4 *>(sym + i - kEncBlock) + lane);
    while (i >= kEncBlock && status == 0) {
        if (!room(2 * kEncBlock)) { status |= 1u; break; }
        uint4 nxt = make_uint4(0, 0, 0, 0);
        if (i >= 2 * kEncBlock) nxt = __ldg(reinterpret_cast<const uint4 *>(sym + i - 2 * kEncBlock) + lane);
        // ---- all lanes: expand this lane's 16 symbols into ready-to-use table entries
        {
            const uint32_t wd[4] = {cur.x, cur.y, cur.z, cur.w};
            uint32_t fl = 0;
#pragma unroll
            for (int b = 0; b < 16; b++) {
                const uint32_t sy = (wd[b >> 2] >> (8 * (b & 3))) & 0xff;
                const uint4 t = tab[sy];
                st_sym[b * 32 + lane] = (uint8_t)sy;
                st_a[b * 32 + lane] = t;
                fl |= t.w >> 24;
            }
            grp[lane] = ((fl & (kEncSmall >> 24)) ? kGrpSmall : 0u) |
                        ((fl & ((kEncWide | kEncZero | kEncOne) >> 24)) ? kGrpGeneric : 0u);
        }
        __syncwarp();
        // ---- lane 0 only: the state recurrence, last symbol first.  It records the state before each step in
        // st_x; which bytes that step emitted is recomputed from (state, limit) by all lanes afterwards, so the
        // serial code has no stream pointer to maintain.  (One active lane also makes every 16-byte shared load a
        // single wavefront.)  Entries of the next group are loaded into each register slot as soon as the
        // current group has used it, so the loads issue in the shadow of the dependent arithmetic.
        if (lane0) {
            uint4 ea[16];
#pragma unroll
            for (int b = 0; b < 16; b++) ea[b] = st_a[b * 32 + 31];
            uint32_t g = grp[31];
            for (int c = 31; c >= 0; c--) {
                const int cn = c > 0 ? c - 1 : 0;
                const uint32_t gn = grp[cn];
                if (g == 0) {
                    // every freq in (16, 4096]: at most one renormalisation byte per symbol.  Both outcomes are
                    // computed and selected at the end, so the comparison is off the critical path.
                    // (Round 2: dividing by 2^sh with a multiply-high instead of the register-count shifts, which show
                    //  dispatch stalls in the ncu source page, measured 42 instead of 55 Msym/s per lane and was dropped.)
#pragma unroll
                    for (int b = 15; b >= 0; b--) {
                        st_x[b * 32 + c] = x;
                        const bool k = x > ea[b].x;
                        const uint32_t hi = __umulhi(x, ea[b].y);       // floor(x / freq) << sh
                        const uint32_t w = ea[b].w;                     // sh | cum << 8 (no flags in this group)
                        const uint32_t cum = w >> 8;
                        const uint32_t xa = __funnelshift_r(hi, 0u, w) * ea[b].z + (x + cum);     // the shift wraps: sh = w & 31
                        // floor(floor(x/f) / 256) == floor((x >> 8) / f)
                        const uint32_t xb = __funnelshift_r(hi, 0u, w + 8u) * ea[b].z + ((x >> 8) + cum);
                        x = k ? xb : xa;
                        ea[b] = st_a[b * 32 + cn];
                    }
                } else if (!(g & kGrpGeneric)) {
                    // some freq in [2, 16]: up to two renormalisation bytes
#pragma unroll
                    for (int b = 15; b >= 0; b--) {
                        st_x[b * 32 + c] = x;
                        const uint32_t lim = ea[b].x;
                        const uint32_t w = ea[b].w;
                        const uint32_t lim2 = (w & kEncSmall) ? ((lim << 8) | 0xffu) : 0xffffffffu;
                        const uint32_t sh = w & 31u;
                        const bool k1 = x > lim, k2 = x > lim2;
                        const uint32_t hi = __umulhi(x, ea[b].y);
                        uint32_t sx = k1 ? 8u : 0u;
                        sx = k2 ? 16u : sx;
                        x = (hi >> (sh + sx)) * ea[b].z + ((x >> sx) + ((w >> 8) & 0xffffu));
                        ea[b] = st_a[b * 32 + cn];
                    }
                } else {
                    for (int b = 15; b >= 0; b--) {
                        const uint4 e = tab[st_sym[b * 32 + c]];
                        st_x[b * 32 + c] = x;
                        if (e.w & kEncZero) { status |= 2u; continue; }
                        while (x > e.x) x >>= 8;       // rans.rs:275-279; the bytes are emitted below
                        const uint32_t f = kProbScale - e.z;
                        const uint32_t q = x / f;
                        x = x + ((e.w >> 8) & 0xffffu) + q * e.z;
                    }
#pragma unroll
                    for (int b = 0; b < 16; b++) ea[b] = st_a[b * 32 + cn];
                }
                g = gn;
            }
        }
        __syncwarp();
        x = __shfl_sync(kFullMask, x, 0);
        status = __shfl_sync(kFullMask, status, 0);
        if (status) break;
        // ---- all lanes: lane c emits the bytes of group c.  A step that started in state s with limit L emitted
        // s & 0xff if s > L and then (s >> 8) & 0xff if (s >> 8) > L (at most two bytes, rans.rs:275-279).
        {
            uint32_t kb1 = 0, kb2 = 0;   // bit b: symbol b of my group emitted a first / second byte
#pragma unroll
            for (int b = 0; b < 16; b++) {
                const uint32_t sx = st_x[b * 32 + lane], lim = st_a[b * 32 + lane].x;
                kb1 |= (sx > lim ? 1u : 0u) << b;
                kb2 |= ((sx > lim) && ((sx >> 8) > lim) ? 1u : 0u) << b;
            }
            const uint32_t mine = (uint32_t)(__popc(kb1) + __popc(kb2));
            // bytes emitted before mine = those of the groups processed earlier = lanes above me
            uint32_t incl = mine;
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) {
                const uint32_t o = __shfl_down_sync(kFullMask, incl, d);
                if (lane + d < 32) incl += o;
            }
            const uint32_t total = __shfl_sync(kFullMask, incl, 0);
            uint32_t pos = sp - (incl - mine);          // my first byte goes to ring[pos - 1]
#pragma unroll
            for (int b = 15; b >= 0; b--) {
                const uint32_t sx = st_x[b * 32 + lane];
                if (kb1 & (1u << b)) ring[--pos] = (uint8_t)sx;
                if (kb2 & (1u << b)) ring[--pos] = (uint8_t)(sx >> 8);
            }
            sp -= total;
        }
        flush();
        cur = nxt;
        i -= kEncBlock;
    }
    if (status == 0 && !room(2 * kEncBlock + 8)) status |= 1u;
    while (i > 0 && status == 0) {
        step_generic(tab[__ldg(sym + i - 1)]);
        i--;
    }
    // finish (rans.rs:298-308): 4 state bytes, low byte first, then the whole vector is reversed
    if (status == 0) {
        ring[sp - 1] = (uint8_t)x;
        ring[sp - 2] = (uint8_t)(x >> 8);
        ring[sp - 3] = (uint8_t)(x >> 16);
        ring[sp - 4] = (uint8_t)(x >> 24);
        sp -= 4;
        flush();
    }
    if (lane0) {
        results[2 * stream] = (unsigned long long)((job.out + job.cap) - wp);
        results[2 * stream + 1] = status;
    }
}

void rans_encode(const RansEncJob *d_jobs, const EncSym *d_enc, const unsigned *, unsigned long long *d_results,
                 int n_streams, cudaStream_t st, bool shared_gpu) {
    if (n_streams <= 0) return;
    launch_lanes(n_streams, shared_gpu, [&](auto lpb) {
        constexpr int LPB = decltype(lpb)::value;
        // Four-warp blocks take the shared memory they need (63 KB): up to three per SM, so the blocks of several batches
        // in flight share SMs with two or three streams per scheduler, like the decoder's (105 KB per four-warp block, two
        // per SM).  Round 1 padded the block to 116 KB to keep an SM to one block -- per-stream speed over throughput --
        // which left room for only 148 encoder blocks per GPU and queued the launches of the other batches.
        const int smem = LPB * kEncSmemPerWarp;
#ifndef ALICE_EMUL
        static unsigned long long attr_done = 0;
        ensure_dyn_smem(k_rans_encode<LPB>, LPB * kEncSmemPerWarp, attr_done);
#endif
        auto k = k_rans_encode<LPB>;
        ALICE_LAUNCH(k, dim3((n_streams + LPB - 1) / LPB), dim3(32 * LPB), smem, st, d_jobs, d_enc, d_results, n_streams);
    });
}

// --------------------------------------------------------------------------------- decode
constexpr int kDecBlock = 128;                   // symbols per fast block (one 4-byte store per lane)
constexpr int kWinPos = 512;                     // byte positions held by the window ring
constexpr int kWinMirror = 2 * kDecBlock + 16;   // positions mirrored past the end: a block reads linearly
constexpr int kWinFill = 128;                    // bytes converted per refill (4 per lane)
// window entry of position p: {bytes p..p+3, bytes p+4..p+7} as two big-endian words; 8 bytes per position makes
// the renormalisation shift (8 bits per byte) equal to the address increment.
// Tables: {freq} and {slot - cum} as two u16 arrays (the two 2-byte loads zero-extend for free, so the dependent
// chain LDS -> IMAD is that of one 8-byte entry).  26.4 KB per stream: eight streams per SM = two per warp scheduler.
// Measured (profiles/r02_rans_occupancy.md): one stream per scheduler decodes 33-36 Msym/s, two sharing a scheduler
// 28.8 Msym/s each (the step is latency bound, so the second stream is almost free); the 8-byte-entry layout of round 1
// (48.9 KB, four streams per SM, 36.2 Msym/s per lane) gave 145 Msym/s per SM against 173+ for this one.
// Tried in round 2 and dropped (profiles/r02_rans_twelve_per_sm.md): a 17.7 KB layout (64-symbol blocks, 4-byte window
// entries, slot -> symbol map read from global memory one block late) that fits TWELVE streams per SM: 270 Msym/s per SM
// at twelve against 232 here at eight, but 208 at eight and 28.8 instead of 32.4 Msym/s for a stream alone -- and a chunk
// in flight costs 3 B/px of symbol planes whatever the plan, so HBM holds eight streams per SM of 1080p chunks, not twelve.
constexpr int kDecSmemBytes = kDecLutEntries * 4 + (kWinPos + kWinMirror) * 8 + kDecLutEntries + kDecBlock * 2;
static_assert(kDecSmemBytes % 16 == 0, "per-warp shared memory must keep 16-byte alignment");
static_assert(kWinPos >= 2 * kDecBlock + 12 + kWinFill + 16, "a refill must not overwrite unread positions");

struct DecState {
    uint32_t x;
    unsigned long long pos, len;
    const uint8_t *in;
};

// generic step (rans.rs:351-371 literally), reading stream bytes from global memory
ALICE_D uint32_t dec_step_generic(DecState &s, const void *tab, const uint8_t *symt, uint32_t wide_sym,
                                  uint32_t wide_freq) {
    const uint32_t slot = s.x & (kProbScale - 1);
    const uint16_t *f16 = reinterpret_cast<const uint16_t *>(tab);
    const uint2 e = make_uint2(f16[slot], f16[kDecLutEntries + slot]);
    const uint32_t sym = symt[slot];
    const uint32_t f = (sym == wide_sym) ? wide_freq : e.x;
    s.x = f * (s.x >> kProbBits) + e.y;          // low 32 bits of the reference's u64 expression
    while (s.x < kRansL && s.pos < s.len) {
        s.x = (s.x << 8) | (uint32_t)__ldg(s.in + s.pos);
        s.pos++;
    }
    return sym;
}

template <int LPB>
__global__ void ALICE_LAUNCH_BOUNDS(32 * LPB, 1)
k_rans_decode(const RansDecJob *__restrict__ jobs, const uint32_t *__restrict__ lut_all,
              const DecAux *__restrict__ aux_all, int n_streams) {
    ALICE_DYN_SMEM(smem_all);
    const int stream = blockIdx.x * LPB + (threadIdx.x >> 5);
    if (stream >= n_streams) return;                 // warp-uniform; the kernel has no block-level barrier
    constexpr int kTabBytes = kDecLutEntries * 4;
    constexpr int SH = 1;                            // log2 of the table stride in bytes: slot << SH addresses the tables
    unsigned char *smem = smem_all + (size_t)(threadIdx.x >> 5) * kDecSmemBytes;
    uint16_t *f16 = reinterpret_cast<uint16_t *>(smem);                         // slot -> freq ...
    uint16_t *b16 = f16 + kDecLutEntries;                                       // ... and slot -> slot - cum
    uint2 *win = reinterpret_cast<uint2 *>(smem + kTabBytes);                   // position -> next 8 bytes, big-endian
    uint8_t *symt = smem + kTabBytes + (kWinPos + kWinMirror) * 8;              // slot -> symbol
    uint16_t *slots = reinterpret_cast<uint16_t *>(symt + kDecLutEntries);      // slots decoded in this block
    const int lane = threadIdx.x & 31;
    const bool lane0 = lane == 0;
    {
        const uint32_t *src = lut_all + (size_t)stream * kDecLutEntries;
        for (int i = lane; i < kDecLutEntries; i += 32) {
            const uint32_t p = src[i];
            f16[i] = (uint16_t)(((p >> 8) & 0xfffu) + 1u);
            b16[i] = (uint16_t)(p >> 20);
            symt[i] = (uint8_t)p;
        }
    }
    __syncwarp();
    const RansDecJob job = jobs[stream];
    const DecAux aux = aux_all[stream];
    DecState s;
    s.in = job.in;
    s.len = job.len;
    s.x = 0;
    s.pos = 0;
    if (s.len >= 4) {  // rans.rs:341-347 big-endian initial state
        s.x = ((uint32_t)__ldg(s.in) << 24) | ((uint32_t)__ldg(s.in + 1) << 16) | ((uint32_t)__ldg(s.in + 2) << 8) |
              (uint32_t)__ldg(s.in + 3);
        s.pos = 4;
    }
    const bool fast_ok = aux.wide_reachable == 0;
    // window ring over byte offsets relative to the 16-byte aligned address below job.in
    const uintptr_t in_addr = reinterpret_cast<uintptr_t>(job.in);
    const uint8_t *ga = reinterpret_cast<const uint8_t *>(in_addr & ~(uintptr_t)15);
    const unsigned long long skew = in_addr & 15;             // offset of stream byte 0 from ga
    const unsigned long long end_off = skew + s.len;          // offsets >= end_off are not stream bytes
    unsigned long long filled = 0;                            // window valid for offsets [.., filled)
    bool win_started = false;
    // the three words a lane converts in a refill starting at offset `at` (whole words may reach past the end of the
    // stream: the payload arena leaves 16 bytes of slack, Engine::decode_chunks)
    auto load_words = [&](unsigned long long at, uint32_t (&d)[3]) {
        const unsigned long long base = at + 4ull * lane;
#pragma unroll
        for (int k = 0; k < 3; k++)
            d[k] = (base + 4 * k < end_off) ? __ldg(reinterpret_cast<const uint32_t *>(ga + base + 4 * k)) : 0u;
    };
    unsigned long long pf_at = ~0ull;                         // offset the prefetched words belong to
    uint32_t pf_d[3] = {0, 0, 0};

    uint8_t *out = job.symbols;
    unsigned long long i = 0;
    const unsigned long long n = job.n;

    auto careful = [&](unsigned long long upto) {   // generic steps for symbols [i, upto); true if the rest was filled
        for (; i < upto; i++) {
            const uint32_t xb = s.x;
            const uint32_t sy = dec_step_generic(s, smem, symt, aux.wide_sym, aux.wide_freq);
            if (lane0) out[i] = (uint8_t)sy;
            if (s.pos >= s.len && s.x == xb) {
                // exhausted stream and a fixed point of the state map: every further symbol is `sy`
                for (unsigned long long j = i + 1 + lane; j < n; j += 32) out[j] = (uint8_t)sy;
                i = n;
                return true;
            }
        }
        return false;
    };

    // peel until the output pointer is 16-byte aligned
    {
        unsigned long long peel = (16 - (reinterpret_cast<uintptr_t>(out) & 15)) & 15;
        if (peel > n) peel = n;
        careful(peel);
    }
    while (i < n) {
        const bool fast = fast_ok && (n - i) >= (unsigned long long)kDecBlock && s.x >= kRansL &&
                          s.pos + 2ull * kDecBlock <= s.len;
        if (!fast) {
            unsigned long long upto = i + kDecBlock;
            if (upto > n) upto = n;
            if (careful(upto)) break;
            continue;
        }
        // ---- make the window cover offsets [o, o + 2*kDecBlock + 12)
        const unsigned long long o = skew + s.pos;
        if (!win_started || o >= filled) { filled = o & ~(unsigned long long)15; win_started = true; }
        while (filled < o + 2ull * kDecBlock + 12) {
            __syncwarp();
            {
                const unsigned long long base = filled + 4ull * lane;   // this lane converts positions base .. base+3
                uint32_t d[3];                                          // stream bytes base .. base+11
                if (pf_at == filled) { d[0] = pf_d[0]; d[1] = pf_d[1]; d[2] = pf_d[2]; }   // requested one refill ago
                else load_words(filled, d);
                uint32_t be[8];    // be[k] = big-endian word of bytes base+k .. base+k+3
#pragma unroll
                for (int k = 0; k < 8; k++)
                    be[k] = __byte_perm(__funnelshift_r(d[k >> 2], d[(k >> 2) + 1 > 2 ? 2 : (k >> 2) + 1], 8 * (k & 3)), 0, 0x0123);
#pragma unroll
                for (int k = 0; k < 4; k++) {
                    const uint32_t idx = (uint32_t)((base + k) & (kWinPos - 1));
                    const uint2 e = make_uint2(be[k], be[k + 4]);
                    win[idx] = e;
                    if (idx < (uint32_t)kWinMirror) win[kWinPos + idx] = e;
                }
            }
            filled += kWinFill;
            __syncwarp();
        }
        // request the bytes of the next refill now: they arrive while lane 0 runs the recurrence
        if (pf_at != filled) { load_words(filled, pf_d); pf_at = filled; }
        // ---- kDecBlock symbols, state recurrence only
        uint32_t x = s.x;
        const uint32_t wi0 = (uint32_t)(o & (kWinPos - 1));   // window index of the next stream byte
        const smem_addr_t wa0 = smem_addr_of(win) + 8 * wi0;
        smem_addr_t wa = wa0;                                 // running window address: 8 bytes per stream byte
        // ---- lane 0 only (one active lane: every shared access is a single wavefront)
        // (Tried in round 2 and dropped, profiles/r02_rans_decoder_chain_variants.jsonl: reading the table entries of both
        //  likely next states speculatively -- with and without one renormalisation byte -- so that the comparison only
        //  selects between loaded entries.  Shared-memory loads return in order, so the select waits for the last of five
        //  or seven loads per symbol: 22-26 Msym/s per lane branch-free, 16-17 with a branch for the two-byte case,
        //  against 28-32 for this chain.)
        if (lane0) {
            uint32_t v = win[wi0].x;                          // the next four stream bytes, big-endian
            // The loop keeps the state only in its shifted form x3 = x << SH (its low bits address the tables, its high
            // bits are x >> 12): nine instead of twelve instructions per symbol on the integer pipe, which two streams
            // on one warp scheduler share (27.9 -> 29.1 Msym/s per lane at eight streams per SM).
            uint32_t x3 = x << SH;
            for (int g = 0; g < kDecBlock / 16; g++) {
#pragma unroll
                for (int b = 0; b < 16; b++) {
                    const uint32_t slot8 = x3 & ((kProbScale - 1) << SH);          // byte offset of the slot's entry
                    const uint32_t xs = x3 >> (kProbBits + SH);
                    uint2 e;
                    e.x = *reinterpret_cast<const uint16_t *>(reinterpret_cast<const uint8_t *>(f16) + slot8);
                    e.y = *reinterpret_cast<const uint16_t *>(reinterpret_cast<const uint8_t *>(b16) + slot8);
                    const uint32_t lo = smem_ld_u32<4>(wa);   // the four bytes after v; address known one symbol early
                    slots[g * 16 + b] = (uint16_t)slot8;
                    const uint32_t xn = e.x * xs + e.y;
                    // xn >= 2^11 here, so at most two bytes bring it back to [2^23, 2^31)
                    const bool ka = xn < kRansL, kb = xn < (1u << 15);
                    uint32_t sa3 = ka ? 8u + SH : (uint32_t)SH;
                    sa3 = kb ? 16u + SH : sa3;
                    const uint32_t sa = sa3 - SH;
                    x3 = __funnelshift_l(v, xn, sa3);         // (renormalised x) << SH, without waiting for it
                    v = __funnelshift_l(lo, v, sa);
                    wa += sa;                                 // 8 address bytes per consumed stream byte
                }
            }
            x = x3 >> SH;
        }
        __syncwarp();
        x = __shfl_sync(kFullMask, x, 0);
        wa = wa0 + __shfl_sync(kFullMask, (uint32_t)(wa - wa0), 0);
        s.x = x;
        s.pos += (unsigned long long)(wa - wa0) / 8;
        __syncwarp();
        // ---- all lanes: slot -> symbol for 4 symbols each, one 4-byte store per lane
        {
            const uint2 sv = *reinterpret_cast<const uint2 *>(slots + 4 * lane);
            const uint32_t a = symt[(sv.x & 0xffffu) >> SH], b2 = symt[sv.x >> (16 + SH)];
            const uint32_t c2 = symt[(sv.y & 0xffffu) >> SH], d2 = symt[sv.y >> (16 + SH)];
            *reinterpret_cast<uint32_t *>(out + i + 4 * lane) = a | (b2 << 8) | (c2 << 16) | (d2 << 24);
        }
        __syncwarp();
        i += kDecBlock;
    }
}

void rans_decode(const RansDecJob *d_jobs, const uint32_t *d_dec_lut, const DecAux *d_aux, int n_streams,
                 cudaStream_t st, bool shared_gpu) {
    if (n_streams <= 0) return;
    launch_lanes(n_streams, shared_gpu, [&](auto lpb) {
        constexpr int LPB = decltype(lpb)::value;
        const int smem = LPB * kDecSmemBytes;      // four-warp blocks: 105.6 KB, two per SM
#ifndef ALICE_EMUL
        static unsigned long long attr_done = 0;
        ensure_dyn_smem(k_rans_decode<LPB>, smem, attr_done);
#endif
        auto k = k_rans_decode<LPB>;
        ALICE_LAUNCH(k, dim3((n_streams + LPB - 1) / LPB), dim3(32 * LPB), smem, st, d_jobs, d_dec_lut, d_aux, n_streams);
    });
}

}  // namespace alice
