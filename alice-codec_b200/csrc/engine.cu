// engine.cu — host orchestration of the encode / decode pipeline on one CUDA device.
// See engine.h for the mapping to src/pipeline.rs.
#include "engine.h"

#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <memory>
#include <mutex>

namespace alice {

// ------------------------------------------------------------------------------- errors
static thread_local int t_err_code = 0;
static thread_local std::string t_err_msg;
void set_error(int code, const std::string &msg) { t_err_code = code; t_err_msg = msg; }
int last_error_code() { return t_err_code; }
const char *last_error_msg() { return t_err_msg.c_str(); }

#define CU_TRY(expr)                                                                                  \
    do {                                                                                              \
        cudaError_t _e = (expr);                                                                      \
        if (_e != cudaSuccess) {                                                                      \
            set_error(kErrCuda, std::string(#expr) + ": " + cudaGetErrorString(_e));                  \
            return kErrCuda;                                                                          \
        }                                                                                             \
    } while (0)

bool cuda_ready() {
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n <= 0) {
        set_error(kErrCuda, std::string("no usable CUDA device: ") +
                                (e != cudaSuccess ? cudaGetErrorString(e) : "device count is 0") +
                                " (libalice_codec has no CPU fallback)");
        cudaGetLastError();
        return false;
    }
    return true;
}

// ------------------------------------------------------------------------------ ByteBuf
namespace {
struct PoolEntry2 { uint8_t *p; size_t cap; };
std::mutex g_buf_mu;
std::vector<PoolEntry2> g_buf_pool;
size_t g_buf_pool_bytes = 0;
size_t buf_pool_limit() {
    static size_t lim = [] {
        const char *e = getenv("ALICE_CODEC_PINNED_POOL_MB");
        long long mb = e ? atoll(e) : 1024;   // idle page-locked memory kept for reuse; raise it for sustained batch traffic
        return (size_t)(mb < 0 ? 0 : mb) << 20;
    }();
    return lim;
}
}  // namespace

bool ByteBuf::assign(const uint8_t *src, size_t n) {
    release();
    p_ = (uint8_t *)malloc(n ? n : 1);
    if (!p_) return false;
    if (n) memcpy(p_, src, n);
    n_ = cap_ = n;
    pinned_ = false;
    return true;
}

bool ByteBuf::acquire_pinned(size_t n) {
    release();
    {
        std::lock_guard<std::mutex> lk(g_buf_mu);
        size_t best = g_buf_pool.size();
        for (size_t i = 0; i < g_buf_pool.size(); i++)
            if (g_buf_pool[i].cap >= n && g_buf_pool[i].cap <= 2 * n + 65536 &&   // never hand a small chunk a huge buffer
                (best == g_buf_pool.size() || g_buf_pool[i].cap < g_buf_pool[best].cap)) best = i;
        if (best != g_buf_pool.size()) {
            p_ = g_buf_pool[best].p;
            cap_ = g_buf_pool[best].cap;
            g_buf_pool_bytes -= cap_;
            g_buf_pool.erase(g_buf_pool.begin() + (long)best);
            n_ = n;
            pinned_ = true;
            return true;
        }
    }
    const size_t cap = (n + n / 8 + 4095) / 4096 * 4096 + 4096;   // head-room so similar chunks share buffers
    void *q = nullptr;
    if (posix_memalign(&q, 4096, cap) != 0) return false;
    if (cudaHostRegister(q, cap, cudaHostRegisterPortable) != cudaSuccess) {
        cudaGetLastError();
        free(q);
        return false;
    }
    p_ = (uint8_t *)q;
    cap_ = cap;
    n_ = n;
    pinned_ = true;
    return true;
}

void ByteBuf::release() {
    if (!p_) return;
    if (pinned_) {
        std::unique_lock<std::mutex> lk(g_buf_mu);
        if (g_buf_pool_bytes + cap_ <= buf_pool_limit()) {
            g_buf_pool.push_back({p_, cap_});
            g_buf_pool_bytes += cap_;
        } else {
            lk.unlock();
            cudaHostUnregister(p_);
            cudaGetLastError();
            free(p_);
        }
    } else {
        free(p_);
    }
    p_ = nullptr;
    n_ = cap_ = 0;
    pinned_ = false;
}

void trim_pinned_pool() {
    std::vector<PoolEntry2> drop;
    {
        std::lock_guard<std::mutex> lk(g_buf_mu);
        drop.swap(g_buf_pool);
        g_buf_pool_bytes = 0;
    }
    for (PoolEntry2 &e : drop) {
        cudaHostUnregister(e.p);
        cudaGetLastError();
        free(e.p);
    }
}

// ------------------------------------------------------------------------- .alc container
static void put_u32(std::vector<uint8_t> &b, uint32_t v) {
    b.push_back((uint8_t)v); b.push_back((uint8_t)(v >> 8)); b.push_back((uint8_t)(v >> 16)); b.push_back((uint8_t)(v >> 24));
}
static uint32_t get_u32(const uint8_t *p) {
    return (uint32_t)p[0] | ((uint32_t)p[1] << 8) | ((uint32_t)p[2] << 16) | ((uint32_t)p[3] << 24);
}

std::vector<uint8_t> Chunk::to_bytes() const {
    std::vector<uint8_t> buf;
    buf.reserve(kFixedHeaderBytes + 3 * kChannelHeaderBytes + data.size());
    buf.push_back('A'); buf.push_back('L'); buf.push_back('C'); buf.push_back('C');
    buf.push_back(1);  // FORMAT_VERSION, pipeline.rs:145
    buf.push_back(wavelet);
    put_u32(buf, width);
    put_u32(buf, height);
    put_u32(buf, frames);
    for (const ChannelHeader &c : ch) {
        put_u32(buf, c.compressed_len);
        put_u32(buf, (uint32_t)c.quant_step);
        put_u32(buf, (uint32_t)c.quant_dead_zone);
        put_u32(buf, c.num_symbols);
        for (uint32_t v : c.histogram) put_u32(buf, v);
    }
    buf.insert(buf.end(), data.data(), data.data() + data.size());
    return buf;
}

int Chunk::from_bytes(const uint8_t *p, size_t len, Chunk &out) {
    const size_t min_len = kFixedHeaderBytes + 3 * kChannelHeaderBytes;
    if (len < min_len) { set_error(kErrBitstream, "data too short"); return kErrBitstream; }
    if (memcmp(p, "ALCC", 4) != 0) { set_error(kErrBitstream, "bad magic (expected ALCC)"); return kErrBitstream; }
    if (p[4] != 1) { set_error(kErrBitstream, "unsupported version"); return kErrBitstream; }
    if (p[5] > 2) { set_error(kErrBitstream, "unknown wavelet type byte"); return kErrBitstream; }
    out.wavelet = p[5];
    out.width = get_u32(p + 6);
    out.height = get_u32(p + 10);
    out.frames = get_u32(p + 14);
    size_t off = kFixedHeaderBytes;
    size_t total = 0;
    for (ChannelHeader &c : out.ch) {
        c.compressed_len = get_u32(p + off); off += 4;
        c.quant_step = (int32_t)get_u32(p + off); off += 4;
        c.quant_dead_zone = (int32_t)get_u32(p + off); off += 4;
        c.num_symbols = get_u32(p + off); off += 4;
        for (uint32_t &v : c.histogram) { v = get_u32(p + off); off += 4; }
        total += c.compressed_len;
    }
    if (len < off + total) { set_error(kErrBitstream, "truncated payload"); return kErrBitstream; }
    if (!out.data.assign(p + off, total)) { set_error(kErrCuda, "host allocation failed"); return kErrCuda; }  // trailing bytes are ignored, pipeline.rs:303
    return kOk;
}

int make_dims(uint32_t w, uint32_t h, uint32_t f, Dims &d) {
    unsigned __int128 p = (unsigned __int128)w * h;
    p *= f;
    if (p > (unsigned __int128)UINT64_MAX) { set_error(kErrOverflow, "dimensions overflow usize"); return kErrOverflow; }
    d.w = w; d.h = h; d.f = f;
    d.n_pixels = (uint64_t)p;
    d.pw = w + (w & 1);
    d.ph = h + (h & 1);
    d.pf = (f == 1) ? 2 : f + (f & 1);
    unsigned __int128 pp = (unsigned __int128)d.pw * d.ph * d.pf;
    d.padded = pp > (unsigned __int128)UINT64_MAX ? UINT64_MAX : (uint64_t)pp;
    return kOk;
}

int quality_to_step(uint8_t quality) {
    int q = quality > 100 ? 100 : quality;
    int s = 64 - (q * 63) / 100;
    return s < 1 ? 1 : s;
}

// -------------------------------------------------------------------------------- Engine
template <class T> static bool dev_alloc(T *&p, size_t bytes, uint64_t &acc) {
    void *q = nullptr;
    if (cudaMalloc(&q, bytes ? bytes : 16) != cudaSuccess) { cudaGetLastError(); p = nullptr; return false; }
    p = reinterpret_cast<T *>(q);
    acc += bytes;
    return true;
}
static size_t round_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

Engine::Engine(const Dims &d, uint32_t cap_chunks, uint64_t payload_cap, cudaStream_t user_stream, bool own_stream,
               bool shared_workspace, bool well_formed_tables)
    : d_(d), cap_(cap_chunks), own_stream_(own_stream), shared_ws_(shared_workspace), well_formed_(well_formed_tables) {
    const size_t N = (size_t)d_.padded;
    const size_t vol = (size_t)d_.f * d_.ph * d_.pw;
    pay_cap_ = payload_cap ? round_up((size_t)payload_cap, 16) : rans_enc_worst_case(N);
    const size_t S = (size_t)cap_ * 3;
    if (own_stream_) {
        if (cudaStreamCreateWithFlags(&st_, cudaStreamNonBlocking) != cudaSuccess) { cudaGetLastError(); return; }
    } else st_ = user_stream;
    bool a = true;
    a = a && dev_alloc(d_scratch_, vol * 3 * 4, dev_bytes_);
    if (!shared_ws_) a = a && dev_alloc(d_symbols_, S * N, dev_bytes_);
    a = a && dev_alloc(d_hist_, S * 256 * sizeof(unsigned), dev_bytes_);
    if (well_formed_) a = a && dev_alloc(d_wf_hist_, S * 256 * sizeof(unsigned), dev_bytes_);
    d_tab_hist_ = well_formed_ ? d_wf_hist_ : d_hist_;
    a = a && dev_alloc(d_enc_, S * 256 * sizeof(EncSym), dev_bytes_);
    a = a && dev_alloc(d_dec_lut_, S * kDecLutEntries * sizeof(uint32_t), dev_bytes_);
    a = a && dev_alloc(d_aux_, S * sizeof(DecAux), dev_bytes_);
    a = a && dev_alloc(d_payload_, S * pay_cap_, dev_bytes_);
    a = a && dev_alloc(d_enc_jobs_, S * sizeof(RansEncJob), dev_bytes_);
    a = a && dev_alloc(d_dec_jobs_, S * sizeof(RansDecJob), dev_bytes_);
    a = a && dev_alloc(d_fwd_jobs_, (size_t)cap_ * sizeof(FwdFusedJob), dev_bytes_);
    a = a && dev_alloc(d_inv_jobs_, (size_t)cap_ * sizeof(InvFusedJob), dev_bytes_);
    a = a && cudaMallocHost((void **)&h_inv_jobs_, (size_t)cap_ * sizeof(InvFusedJob)) == cudaSuccess;
    a = a && cudaMallocHost((void **)&h_fwd_jobs_, (size_t)cap_ * sizeof(FwdFusedJob)) == cudaSuccess;
    a = a && dev_alloc(d_results_, S * 2 * sizeof(unsigned long long), dev_bytes_);
    a = a && cudaMallocHost((void **)&h_results_, S * 2 * sizeof(unsigned long long)) == cudaSuccess;
    a = a && cudaMallocHost((void **)&h_hist_, S * 256 * sizeof(unsigned)) == cudaSuccess;
    a = a && cudaMallocHost((void **)&h_enc_jobs_, S * sizeof(RansEncJob)) == cudaSuccess;
    a = a && cudaMallocHost((void **)&h_dec_jobs_, S * sizeof(RansDecJob)) == cudaSuccess;
    for (auto &e : ev_) a = a && cudaEventCreate(&e) == cudaSuccess;
    if (!a) { cudaGetLastError(); set_error(kErrCuda, "device or pinned memory allocation failed"); return; }
    overflow_bufs_.assign(S, nullptr);
    sym_ptr_.assign(cap_, nullptr);
    if (!shared_ws_)
        for (uint32_t c = 0; c < cap_; c++) sym_ptr_[c] = d_symbols_ + (size_t)c * 3 * N;
    stream_off_.assign(S, 0);
    stream_len_.assign(S, 0);
    stream_base_.assign(S, nullptr);
    chunk_step_.assign(cap_, 1);
    ok_ = true;
}

Engine::~Engine() {
    if (st_ && own_stream_) cudaStreamSynchronize(st_);
    cudaFree(d_scratch_); cudaFree(d_symbols_); cudaFree(d_hist_); cudaFree(d_wf_hist_); cudaFree(d_enc_); cudaFree(d_dec_lut_);
    cudaFree(d_aux_); cudaFree(d_payload_); cudaFree(d_enc_jobs_); cudaFree(d_dec_jobs_); cudaFree(d_results_);
    for (uint8_t *p : rgb_stage_) cudaFree(p);
    for (uint8_t *p : overflow_bufs_) if (p) cudaFree(p);
    if (h_pay_) cudaFreeHost(h_pay_);
    if (h_results_) cudaFreeHost(h_results_);
    if (h_hist_) cudaFreeHost(h_hist_);
    if (h_enc_jobs_) cudaFreeHost(h_enc_jobs_);
    if (h_dec_jobs_) cudaFreeHost(h_dec_jobs_);
    if (h_fwd_jobs_) cudaFreeHost(h_fwd_jobs_);
    if (h_inv_jobs_) cudaFreeHost(h_inv_jobs_);
    cudaFree(d_fwd_jobs_);
    cudaFree(d_inv_jobs_);
    cudaFree(d_coef_); cudaFree(d_vhist_); cudaFree(d_rate_hist_); cudaFree(d_rate_wf_hist_); cudaFree(d_rate_enc_);
    cudaFree(d_rate_lut_); cudaFree(d_rate_aux_); cudaFree(d_rate_est_); cudaFree(d_rate_out_);
    if (h_rate_out_) cudaFreeHost(h_rate_out_);
    for (auto &e : ev_) if (e) cudaEventDestroy(e);
    if (st_ && own_stream_) cudaStreamDestroy(st_);
    cudaGetLastError();
}

bool Engine::ensure_pinned_payload(size_t bytes) {
    if (bytes <= h_pay_cap_) return true;
    if (h_pay_) { cudaFreeHost(h_pay_); h_pay_ = nullptr; h_pay_cap_ = 0; }
    const size_t want = round_up(bytes + bytes / 4 + 4096, 4096);
    if (cudaMallocHost((void **)&h_pay_, want) != cudaSuccess) {
        cudaGetLastError();
        set_error(kErrCuda, "pinned host allocation failed (payload staging)");
        return false;
    }
    h_pay_cap_ = want;
    return true;
}

uint8_t *Engine::rgb_stage(uint32_t slot) {
    while (rgb_stage_.size() <= slot) {
        uint8_t *p = nullptr;
        if (!dev_alloc(p, std::max((size_t)d_.n_pixels * 3, shared_ws_ ? (size_t)d_.padded * 3 : (size_t)0), dev_bytes_)) {
            set_error(kErrCuda, "device memory allocation failed (rgb staging)");
            return nullptr;
        }
        rgb_stage_.push_back(p);
    }
    return rgb_stage_[slot];
}

int Engine::run_rans_encode(uint32_t n) {
    const size_t N = (size_t)d_.padded;
    const uint32_t S = n * 3;
    // Payload placement: the streams go back to back into the engine's payload arena (cap_ * 3 * pay_cap_ bytes), each with
    // the upper bound that its histogram and table give (k_estimate_stream_bytes) instead of a fixed slot, so the arena
    // only has to hold what the batch really produces (+ 0.03 %).  A stream that does not fit any more gets no room at all
    // and goes through the overflow path below.  The estimate takes the symbol counts, whatever table they are coded with.
    estimate_stream_bytes(d_hist_, d_enc_, (int)S, N, d_results_, st_);
    CU_TRY(cudaMemcpyAsync(h_results_, d_results_, S * sizeof(unsigned long long), cudaMemcpyDeviceToHost, st_));
    CU_TRY(cudaStreamSynchronize(st_));
    const size_t arena = (size_t)cap_ * 3 * pay_cap_;
    size_t used = 0;
    for (uint32_t s = 0; s < S; s++) {
        const size_t want = (size_t)h_results_[s];
        const bool fits = used + want <= arena;
        h_enc_jobs_[s].symbols = sym_ptr_[s / 3] + (size_t)(s % 3) * N;
        h_enc_jobs_[s].n = N;
        h_enc_jobs_[s].out = d_payload_ + used;
        h_enc_jobs_[s].cap = fits ? want : 0;
        stream_base_[s] = h_enc_jobs_[s].out;
        if (fits) used += want;
    }
    CU_TRY(cudaMemcpyAsync(d_enc_jobs_, h_enc_jobs_, S * sizeof(RansEncJob), cudaMemcpyHostToDevice, st_));
    rans_encode(d_enc_jobs_, d_enc_, d_hist_, d_results_, (int)S, st_, small_smem_);
    CU_TRY(cudaEventRecord(ev_[3], st_));
    CU_TRY(cudaMemcpyAsync(h_results_, d_results_, S * 2 * sizeof(unsigned long long), cudaMemcpyDeviceToHost, st_));
    CU_TRY(cudaMemcpyAsync(h_hist_, d_tab_hist_, (size_t)S * 256 * sizeof(unsigned), cudaMemcpyDeviceToHost, st_));
    CU_TRY(cudaStreamSynchronize(st_));
    CU_TRY(cudaGetLastError());
    for (uint32_t s = 0; s < S; s++) {
        unsigned long long status = h_results_[2 * s + 1];
        if (status & 2) {
            set_error(kErrPanic, "symbol with zero frequency in use: the reference aborts on this input");
            return kErrPanic;
        }
        if (status & 1) {
            // payload did not fit the per-stream capacity: redo this stream into a worst-case buffer
            const size_t full = rans_enc_worst_case(N);
            if (!overflow_bufs_[s]) {
                if (!dev_alloc(overflow_bufs_[s], full, dev_bytes_)) {
                    set_error(kErrCuda, "device memory allocation failed (rANS overflow buffer)");
                    return kErrCuda;
                }
            }
            h_enc_jobs_[s].out = overflow_bufs_[s];
            h_enc_jobs_[s].cap = full;
            stream_base_[s] = overflow_bufs_[s];
            CU_TRY(cudaMemcpyAsync(d_enc_jobs_ + s, h_enc_jobs_ + s, sizeof(RansEncJob), cudaMemcpyHostToDevice, st_));
            rans_encode(d_enc_jobs_ + s, d_enc_ + (size_t)s * 256, d_hist_, d_results_ + 2 * s, 1, st_);
            CU_TRY(cudaMemcpyAsync(h_results_ + 2 * s, d_results_ + 2 * s, 2 * sizeof(unsigned long long),
                                   cudaMemcpyDeviceToHost, st_));
            CU_TRY(cudaStreamSynchronize(st_));
            if (h_results_[2 * s + 1] != 0) { set_error(kErrCuda, "rANS retry failed"); return kErrCuda; }
        }
        stream_len_[s] = h_results_[2 * s];
        stream_off_[s] = h_enc_jobs_[s].cap - stream_len_[s];
    }
    return kOk;
}

// symbol counts of n chunks -> the headers' histograms (well-formed engines) -> the rANS tables
void Engine::build_encode_tables(uint32_t n) {
    if (well_formed_) well_formed_hists(d_hist_, (int)n * 3, d_wf_hist_, st_);
    build_tables(d_tab_hist_, (int)n * 3, 256, d_enc_, d_dec_lut_, d_aux_, nullptr, nullptr, nullptr, st_);
}

// whether a chunk's symbol planes [3][N] and an RGB buffer of one chunk share bytes
bool Engine::overlaps(const uint8_t *sym, const uint8_t *rgb) const {
    return sym < rgb + 3 * (size_t)d_.n_pixels && rgb < sym + 3 * (size_t)d_.padded;
}

// The fused front-end (k_fwd_fused.cu) takes 64-frame chunks of even height and a width that is a multiple of 16.  It
// reads RGB and writes symbols in the same launch, so a chunk whose symbol planes overlap its own RGB takes the
// two-kernel path, which finishes reading the RGB before the first symbol is written.
bool Engine::fused_frontend_ok(const uint8_t *d_rgb, const uint8_t *sym) const {
    return !small_smem_ && forward_fused_eligible(d_rgb, (int)d_.w, (int)d_.h, (int)d_.f) &&
           (reinterpret_cast<uintptr_t>(sym) & 3) == 0 && !overlaps(sym, d_rgb);
}

// One chunk's front-end on the stream (no synchronisation) into the symbol planes `sym` and chunk slot c's histogram, which
// the caller has zeroed.  coef_dump: optional device i32 [3][N], the coefficients of the padded volume [3][pf][ph][pw]
// (pf = f + 1 for odd f, 2 for f == 1).
int Engine::frontend_one(uint32_t c, uint8_t wavelet, const uint8_t *d_rgb, uint8_t *sym, int step, int32_t *coef_dump) {
    unsigned *hist = d_hist_ + (size_t)c * 3 * 256;
    if (fused_frontend_ok(d_rgb, sym)) {
        h_fwd_jobs_[c] = FwdFusedJob{d_rgb, sym, hist, coef_dump};
        CU_TRY(cudaMemcpyAsync(d_fwd_jobs_ + c, h_fwd_jobs_ + c, sizeof(FwdFusedJob), cudaMemcpyHostToDevice, st_));
        forward_frontend_fused(wavelet, d_fwd_jobs_ + c, 1, coef_dump != nullptr, hist, (int)d_.w, (int)d_.h, step,
                               device_sm_count(), st_);
    } else {
        forward_frontend(wavelet, d_rgb, reinterpret_cast<int16_t *>(d_scratch_), sym, hist, (int)d_.w, (int)d_.h,
                         (int)d_.f, (int)d_.pw, (int)d_.ph, (int)d_.pf, step, coef_dump, st_);
    }
    return kOk;
}

int Engine::encode_device(uint8_t quality, uint8_t wavelet, const uint8_t *const *d_rgb, uint32_t n,
                          int32_t *d_coef_dump, uint8_t *const *d_work) {
    if (n > cap_) { set_error(kErrBufferSize, "batch larger than engine capacity"); return kErrBufferSize; }
    int rc = encode_begin(quality, wavelet);
    if (rc) return rc;
    if (shared_ws_) {
        if (!d_work) { set_error(kErrNull, "shared-workspace batch: workspace pointers required"); return kErrNull; }
        for (uint32_t c = 0; c < n; c++) {
            if (!d_work[c]) { set_error(kErrNull, "null workspace pointer"); return kErrNull; }
            sym_ptr_[c] = d_work[c];
        }
    }
    const int step = begin_step_;
    CU_TRY(cudaMemsetAsync(d_hist_, 0, (size_t)n * 3 * 256 * sizeof(unsigned), st_));
    // Engine-owned symbol planes: one fused launch for the whole batch.  Caller-provided workspaces (shared-workspace
    // batches): one launch per chunk, in index order, so workspace i may be the RGB buffer of any chunk j < i (already
    // consumed).
    bool batch_fused = !shared_ws_;
    for (uint32_t c = 0; c < n; c++) {
        chunk_step_[c] = step;
        batch_fused = batch_fused && fused_frontend_ok(d_rgb[c], sym_ptr_[c]);
    }
    if (batch_fused) {
        for (uint32_t c = 0; c < n; c++)
            h_fwd_jobs_[c] = FwdFusedJob{d_rgb[c], sym_ptr_[c], d_hist_ + (size_t)c * 3 * 256, c == 0 ? d_coef_dump : nullptr};
        CU_TRY(cudaMemcpyAsync(d_fwd_jobs_, h_fwd_jobs_, n * sizeof(FwdFusedJob), cudaMemcpyHostToDevice, st_));
        const uint32_t m = (d_coef_dump && n) ? 1 : 0;   // chunk 0 alone when its coefficients are dumped (parity tests)
        if (m) forward_frontend_fused(wavelet, d_fwd_jobs_, 1, true, d_hist_, (int)d_.w, (int)d_.h, step, device_sm_count(), st_);
        forward_frontend_fused(wavelet, d_fwd_jobs_ + m, (int)(n - m), false, d_hist_ + (size_t)m * 3 * 256, (int)d_.w,
                               (int)d_.h, step, device_sm_count(), st_);
    } else {
        for (uint32_t c = 0; c < n && !rc; c++)
            rc = frontend_one(c, wavelet, d_rgb[c], sym_ptr_[c], step, c == 0 ? d_coef_dump : nullptr);
        if (rc) return rc;
    }
    submitted_ = n;
    return encode_finish(n);
}

// ---- chunk-at-a-time encode: encode_begin, then encode_submit(c) for c = 0, 1, ... in order (each enqueues the front-end of
// one chunk and returns at once), then encode_finish(n): tables, all 3n rANS streams, one synchronisation.
int Engine::encode_begin(uint8_t quality, uint8_t wavelet) {
    last_wavelet = wavelet;
    begin_step_ = quality_to_step(quality);
    last_n = 0;
    submitted_ = 0;
    resident_decoded_ = 0;
    CU_TRY(cudaEventRecord(ev_[0], st_));
    return kOk;
}
int Engine::encode_submit(uint32_t c, const uint8_t *d_rgb, uint8_t *d_work, int step) {
    if (c >= cap_ || c != submitted_) { set_error(kErrBufferSize, "chunks must be submitted in index order, below the batch capacity"); return kErrBufferSize; }
    if (shared_ws_) {
        if (!d_work) { set_error(kErrNull, "shared-workspace batch: workspace pointer required"); return kErrNull; }
        sym_ptr_[c] = d_work;
    }
    if (step <= 0) step = begin_step_;
    chunk_step_[c] = step;
    CU_TRY(cudaMemsetAsync(d_hist_ + (size_t)c * 3 * 256, 0, 3 * 256 * sizeof(unsigned), st_));
    int rc = frontend_one(c, last_wavelet, d_rgb, sym_ptr_[c], step, nullptr);
    if (rc) return rc;
    submitted_ = c + 1;
    return kOk;
}
int Engine::encode_finish(uint32_t n) {
    if (n != submitted_) { set_error(kErrBufferSize, "collect: chunk count differs from the chunks submitted"); return kErrBufferSize; }
    last_n = n;
    CU_TRY(cudaEventRecord(ev_[1], st_));
    build_encode_tables(n);
    CU_TRY(cudaEventRecord(ev_[2], st_));
    int rc = run_rans_encode(n);
    if (rc) { last_n = 0; return rc; }
    cudaEventElapsedTime(&timings.ms[0], ev_[0], ev_[1]);   // includes the host copies enqueued between the submits
    cudaEventElapsedTime(&timings.ms[1], ev_[1], ev_[2]);
    cudaEventElapsedTime(&timings.ms[2], ev_[2], ev_[3]);
    return kOk;
}

// headers of chunk i + the device->host copies of its payload, enqueued on the engine's stream (no synchronisation)
int Engine::fetch_enqueue(uint32_t i, Chunk &out, bool &direct) {
    if (i >= last_n) { set_error(kErrBufferSize, "chunk index out of range"); return kErrBufferSize; }
    out.width = d_.w; out.height = d_.h; out.frames = d_.f;
    out.wavelet = last_wavelet;
    size_t total = 0;
    for (int c = 0; c < 3; c++) {
        const uint32_t s = i * 3 + c;
        ChannelHeader &h = out.ch[c];
        h.compressed_len = (uint32_t)stream_len_[s];
        h.quant_step = chunk_step_[i];
        h.quant_dead_zone = chunk_step_[i];     // Quantizer::new: dead_zone = step (quant.rs:70-75)
        h.num_symbols = (uint32_t)d_.padded;    // `as u32`, pipeline.rs:492
        memcpy(h.histogram, h_hist_ + (size_t)s * 256, 256 * sizeof(uint32_t));
        total += stream_len_[s];
    }
    // payload: the device writes straight into the chunk's page-locked buffer (pooled, see ByteBuf)
    uint8_t *dst = nullptr;
    direct = out.data.acquire_pinned(total);
    if (direct) dst = out.data.data();
    else {
        if (!ensure_pinned_payload(total)) return kErrCuda;
        dst = h_pay_;
    }
    size_t off = 0;
    for (int c = 0; c < 3; c++) {
        const uint32_t s = i * 3 + c;
        if (stream_len_[s])
            CU_TRY(cudaMemcpyAsync(dst + off, stream_base_[s] + stream_off_[s], stream_len_[s],
                                   cudaMemcpyDeviceToHost, st_));
        off += stream_len_[s];
    }
    return kOk;
}

int Engine::fetch_chunk(uint32_t i, Chunk &out) {
    bool direct = false;
    int rc = fetch_enqueue(i, out, direct);
    if (rc) return rc;
    CU_TRY(cudaStreamSynchronize(st_));
    if (!direct) {
        size_t total = 0;
        for (int c = 0; c < 3; c++) total += out.ch[c].compressed_len;
        if (!out.data.assign(h_pay_, total)) { set_error(kErrCuda, "host allocation failed"); return kErrCuda; }
    }
    return kOk;
}

// All n chunks of the last encode: every payload copy is enqueued first, ONE synchronisation at the end (a chunk whose
// page-locked buffer cannot be had goes through the single staging buffer and synchronises on its own).
int Engine::fetch_chunks(uint32_t n, Chunk *const *out) {
    for (uint32_t i = 0; i < n; i++) {
        bool direct = false;
        int rc = fetch_enqueue(i, *out[i], direct);
        if (rc) return rc;
        if (!direct) {
            CU_TRY(cudaStreamSynchronize(st_));
            size_t total = 0;
            for (int c = 0; c < 3; c++) total += out[i]->ch[c].compressed_len;
            if (!out[i]->data.assign(h_pay_, total)) { set_error(kErrCuda, "host allocation failed"); return kErrCuda; }
        }
    }
    CU_TRY(cudaStreamSynchronize(st_));
    return kOk;
}

// The fused back-end (k_inv_fused.cu) takes chunks of the fused front-end's shape whose headers stay within its arithmetic
// bound.  It reads symbols and writes RGB in the same launch, so an output that overlaps its own chunk's symbol planes
// takes the two-kernel path, which finishes reading the planes before it writes RGB.
bool Engine::fused_backend_ok(const uint8_t *sym, const uint8_t *d_rgb, const BackendHeader &hdr) const {
    return !small_smem_ && inverse_fused_eligible(sym, d_rgb, (int)d_.w, (int)d_.h, (int)d_.f, hdr.steps) &&
           !overlaps(sym, d_rgb);
}

// Back-end of n chunks whose symbol planes are in sym_ptr_[c]: RGB into d_rgb_out[c].
//   * engine-owned symbol planes, every chunk fused with one header: one launch;
//   * otherwise one chunk at a time (backend_one); caller-provided workspaces (shared-workspace batches) in DESCENDING
//     index order, so the output of chunk i may be the workspace of any chunk j > i (already consumed).  The host
//     staging layout of the batch calls (host_stage in capi.cu) relies on this order.
int Engine::run_backend(uint32_t n, const BackendHeader *hdr, uint8_t *const *d_rgb_out) {
    bool uniform = !shared_ws_ && n > 0;
    for (uint32_t c = 0; c < n && uniform; c++)
        uniform = fused_backend_ok(sym_ptr_[c], d_rgb_out[c], hdr[c]) && hdr[c].wavelet == hdr[0].wavelet &&
                  hdr[c].steps[0] == hdr[0].steps[0] && hdr[c].steps[1] == hdr[0].steps[1] && hdr[c].steps[2] == hdr[0].steps[2];
    if (uniform) {
        for (uint32_t c = 0; c < n; c++) h_inv_jobs_[c] = InvFusedJob{sym_ptr_[c], d_rgb_out[c]};
        CU_TRY(cudaMemcpyAsync(d_inv_jobs_, h_inv_jobs_, n * sizeof(InvFusedJob), cudaMemcpyHostToDevice, st_));
        inverse_backend_fused(hdr[0].wavelet, d_inv_jobs_, (int)n, (int)d_.w, (int)d_.h, hdr[0].steps, device_sm_count(), st_);
        return kOk;
    }
    int rc = kOk;
    for (uint32_t k = 0; k < n && !rc; k++) {
        const uint32_t c = shared_ws_ ? n - 1 - k : k;
        rc = backend_one(c, hdr[c], d_rgb_out[c]);
    }
    return rc;
}

// One chunk's back-end on the stream (no synchronisation).
int Engine::backend_one(uint32_t c, const BackendHeader &hdr, uint8_t *d_rgb_out) {
    if (fused_backend_ok(sym_ptr_[c], d_rgb_out, hdr)) {
        h_inv_jobs_[c] = InvFusedJob{sym_ptr_[c], d_rgb_out};
        CU_TRY(cudaMemcpyAsync(d_inv_jobs_ + c, h_inv_jobs_ + c, sizeof(InvFusedJob), cudaMemcpyHostToDevice, st_));
        inverse_backend_fused(hdr.wavelet, d_inv_jobs_ + c, 1, (int)d_.w, (int)d_.h, hdr.steps, device_sm_count(), st_);
    } else {
        inverse_backend(hdr.wavelet, sym_ptr_[c], reinterpret_cast<int32_t *>(d_scratch_), d_rgb_out, (int)d_.w, (int)d_.h,
                        (int)d_.f, (int)d_.pw, (int)d_.ph, (int)d_.pf, hdr.steps, st_);
    }
    return kOk;
}

int Engine::decode_resident_begin(uint32_t n) {
    if (n > last_n) { set_error(kErrBufferSize, "decode: more chunks than the last encode"); return kErrBufferSize; }
    const size_t N = (size_t)d_.padded;
    const uint32_t S = n * 3;
    resident_decoded_ = 0;
    CU_TRY(cudaEventRecord(ev_[4], st_));
    build_tables(d_tab_hist_, (int)S, 256, d_enc_, d_dec_lut_, d_aux_, nullptr, nullptr, nullptr, st_);
    CU_TRY(cudaEventRecord(ev_[5], st_));
    for (uint32_t s = 0; s < S; s++) {
        h_dec_jobs_[s].in = stream_base_[s] + stream_off_[s];
        h_dec_jobs_[s].len = stream_len_[s];
        h_dec_jobs_[s].symbols = sym_ptr_[s / 3] + (size_t)(s % 3) * N;
        h_dec_jobs_[s].n = N;
    }
    CU_TRY(cudaMemcpyAsync(d_dec_jobs_, h_dec_jobs_, S * sizeof(RansDecJob), cudaMemcpyHostToDevice, st_));
    rans_decode(d_dec_jobs_, d_dec_lut_, d_aux_, (int)S, st_, small_smem_);
    CU_TRY(cudaEventRecord(ev_[6], st_));
    CU_TRY(cudaGetLastError());
    resident_decoded_ = n;
    return kOk;
}

int Engine::decode_resident_next(uint32_t c, uint8_t *d_rgb_out) {
    if (c >= resident_decoded_) { set_error(kErrBufferSize, "decode_next: chunk index beyond the last decode_begin"); return kErrBufferSize; }
    if (!d_rgb_out) { set_error(kErrNull, "null output pointer"); return kErrNull; }
    const int step = chunk_step_[c];
    int rc = backend_one(c, BackendHeader{last_wavelet, {step, step, step}}, d_rgb_out);
    if (rc) return rc;
    CU_TRY(cudaGetLastError());
    return kOk;
}

int Engine::decode_resident_end() {
    CU_TRY(cudaEventRecord(ev_[7], st_));
    CU_TRY(cudaStreamSynchronize(st_));
    CU_TRY(cudaGetLastError());
    if (resident_decoded_) {
        cudaEventElapsedTime(&timings.ms[3], ev_[4], ev_[5]);
        cudaEventElapsedTime(&timings.ms[4], ev_[5], ev_[6]);
        cudaEventElapsedTime(&timings.ms[5], ev_[6], ev_[7]);
    }
    return kOk;
}

int Engine::decode_device_resident(uint8_t *const *d_rgb_out, uint32_t n) {
    int rc = decode_resident_begin(n);
    if (rc) return rc;
    std::vector<BackendHeader> hdr(n);
    for (uint32_t c = 0; c < n; c++) hdr[c] = BackendHeader{last_wavelet, {chunk_step_[c], chunk_step_[c], chunk_step_[c]}};
    rc = run_backend(n, hdr.data(), d_rgb_out);
    return rc ? rc : decode_resident_end();
}

int Engine::decode_chunks(const Chunk *const *chunks, uint32_t n, uint8_t *const *d_rgb_out, uint8_t *const *d_work,
                          uint8_t *const *h_rgb_out) {
    if (n > cap_) { set_error(kErrBufferSize, "batch larger than engine capacity"); return kErrBufferSize; }
    if (h_rgb_out && shared_ws_) { set_error(kErrDimensions, "interleaved host copies need engine-owned symbol planes"); return kErrDimensions; }
    // This call reuses the histogram, table, payload and overflow buffers of the last encode: whatever encode_device left
    // resident is gone afterwards (fetch_chunk / decode_device_resident then report "out of range" instead of returning
    // another batch's data).
    last_n = 0;
    resident_decoded_ = 0;
    for (size_t s = 0; s < stream_base_.size(); s++) { stream_base_[s] = nullptr; stream_len_[s] = 0; stream_off_[s] = 0; }
    if (shared_ws_)   // the symbol planes of chunk i live in its workspace, by default its output buffer (>= workspace_bytes())
        for (uint32_t i = 0; i < n; i++) sym_ptr_[i] = d_work ? d_work[i] : d_rgb_out[i];
    const size_t N = (size_t)d_.padded;
    const uint32_t S = n * 3;
    // validation, in the reference's order (pipeline.rs:562-579)
    for (uint32_t i = 0; i < n; i++) {
        const Chunk &ck = *chunks[i];
        if (ck.width != d_.w || ck.height != d_.h || ck.frames != d_.f) {
            set_error(kErrDimensions, "chunk shape differs from the engine's");
            return kErrDimensions;
        }
        size_t off = 0;
        for (int c = 0; c < 3; c++) {
            if ((uint64_t)ck.ch[c].num_symbols != d_.padded) {
                set_error(kErrBitstream, "num_symbols != padded_pixels");
                return kErrBitstream;
            }
            if (off + ck.ch[c].compressed_len > ck.data.size()) {
                set_error(kErrBitstream, "compressed data overrun");
                return kErrBitstream;
            }
            off += ck.ch[c].compressed_len;
        }
    }
    const size_t arena = (size_t)cap_ * 3 * pay_cap_;
    size_t arena_used = 0;
    for (uint32_t i = 0; i < n; i++) {
        const Chunk &ck = *chunks[i];
        size_t off = 0;
        const bool direct = ck.data.pinned();     // page-locked buffer: the device reads it directly
        if (!direct) {
            CU_TRY(cudaStreamSynchronize(st_));   // the previous chunk's copies out of the staging buffer have landed
            if (!ensure_pinned_payload(ck.data.size())) return kErrCuda;
        }
        for (int c = 0; c < 3; c++) {
            const uint32_t s = i * 3 + c;
            memcpy(h_hist_ + (size_t)s * 256, ck.ch[c].histogram, 256 * sizeof(uint32_t));
            const size_t len = ck.ch[c].compressed_len;
            uint8_t *dst = d_payload_ + arena_used;
            if (arena_used + round_up(len, 16) + 16 > arena) {
                const size_t full = std::max(round_up(len, 16), rans_enc_worst_case(N));
                if (overflow_bufs_[s]) { cudaFree(overflow_bufs_[s]); overflow_bufs_[s] = nullptr; }
                if (!dev_alloc(overflow_bufs_[s], full, dev_bytes_)) {
                    set_error(kErrCuda, "device memory allocation failed (payload)");
                    return kErrCuda;
                }
                dst = overflow_bufs_[s];
            } else arena_used += round_up(len, 16) + 16;   // (the decoder's window refill reads whole words past the end)
            if (len) {
                // host vector -> pinned staging -> device; the staging buffer is reused once the copy has landed
                const uint8_t *src = ck.data.data() + off;
                if (!direct) { memcpy(h_pay_ + off, src, len); src = h_pay_ + off; }
                CU_TRY(cudaMemcpyAsync(dst, src, len, cudaMemcpyHostToDevice, st_));
            }
            off += len;
            h_dec_jobs_[s].in = dst;
            h_dec_jobs_[s].len = len;
            h_dec_jobs_[s].symbols = sym_ptr_[i] + (size_t)c * N;
            h_dec_jobs_[s].n = N;
        }
    }
    CU_TRY(cudaMemcpyAsync(d_hist_, h_hist_, (size_t)S * 256 * sizeof(unsigned), cudaMemcpyHostToDevice, st_));
    CU_TRY(cudaMemcpyAsync(d_dec_jobs_, h_dec_jobs_, S * sizeof(RansDecJob), cudaMemcpyHostToDevice, st_));
    CU_TRY(cudaEventRecord(ev_[4], st_));
    build_tables(d_hist_, (int)S, 256, d_enc_, d_dec_lut_, d_aux_, nullptr, nullptr, nullptr, st_);
    CU_TRY(cudaEventRecord(ev_[5], st_));
    rans_decode(d_dec_jobs_, d_dec_lut_, d_aux_, (int)S, st_, small_smem_);
    CU_TRY(cudaEventRecord(ev_[6], st_));
    {
        std::vector<BackendHeader> hdr(n);
        for (uint32_t i = 0; i < n; i++) {
            const Chunk &ck = *chunks[i];
            hdr[i] = BackendHeader{ck.wavelet, {ck.ch[0].quant_step, ck.ch[1].quant_step, ck.ch[2].quant_step}};
        }
        if (h_rgb_out) {
            // chunk by chunk: back-end, then the copy to the host, so that every chunk may use the same device buffer
            const size_t bytes = (size_t)d_.n_pixels * 3;
            for (uint32_t i = 0; i < n; i++) {
                int rc = backend_one(i, hdr[i], d_rgb_out[i]);
                if (rc) return rc;
                CU_TRY(cudaMemcpyAsync(h_rgb_out[i], d_rgb_out[i], bytes, cudaMemcpyDeviceToHost, st_));
            }
        } else {
            int rc = run_backend(n, hdr.data(), d_rgb_out);
            if (rc) return rc;
        }
    }
    CU_TRY(cudaEventRecord(ev_[7], st_));
    CU_TRY(cudaStreamSynchronize(st_));
    CU_TRY(cudaGetLastError());
    cudaEventElapsedTime(&timings.ms[3], ev_[4], ev_[5]);
    cudaEventElapsedTime(&timings.ms[4], ev_[5], ev_[6]);
    cudaEventElapsedTime(&timings.ms[5], ev_[6], ev_[7]);
    return kOk;
}

// ------------------------------------------------------------------------------ rate curve
bool Engine::ensure_rate_buffers() {
    if (d_coef_) return true;
    const size_t N = (size_t)d_.padded;
    const size_t S = (size_t)kRateSteps * 3;
    int bound = 0;
    for (int wv = 0; wv < 3; wv++) bound = std::max(bound, rate_value_bound(wv));
    bool a = true;
    a = a && dev_alloc(d_coef_, 3 * N * sizeof(int32_t), dev_bytes_);
    a = a && dev_alloc(d_vhist_, 3 * (2 * (size_t)bound + 1) * sizeof(unsigned), dev_bytes_);
    a = a && dev_alloc(d_rate_hist_, S * 256 * sizeof(unsigned), dev_bytes_);
    if (well_formed_) a = a && dev_alloc(d_rate_wf_hist_, S * 256 * sizeof(unsigned), dev_bytes_);
    a = a && dev_alloc(d_rate_enc_, S * 256 * sizeof(EncSym), dev_bytes_);
    a = a && dev_alloc(d_rate_lut_, S * kDecLutEntries * sizeof(uint32_t), dev_bytes_);
    a = a && dev_alloc(d_rate_aux_, S * sizeof(DecAux), dev_bytes_);
    a = a && dev_alloc(d_rate_est_, S * sizeof(unsigned long long), dev_bytes_);
    a = a && dev_alloc(d_rate_out_, (kRateSteps + 1) * sizeof(unsigned long long), dev_bytes_);
    a = a && cudaMallocHost((void **)&h_rate_out_, (kRateSteps + 1) * sizeof(unsigned long long)) == cudaSuccess;
    if (!a) {
        cudaGetLastError();
        // leave the engine as it was: a later call retries
        cudaFree(d_coef_); cudaFree(d_vhist_); cudaFree(d_rate_hist_); cudaFree(d_rate_wf_hist_); cudaFree(d_rate_enc_);
        cudaFree(d_rate_lut_); cudaFree(d_rate_aux_); cudaFree(d_rate_est_); cudaFree(d_rate_out_);
        if (h_rate_out_) cudaFreeHost(h_rate_out_);
        d_coef_ = nullptr; d_vhist_ = nullptr; d_rate_hist_ = nullptr; d_rate_wf_hist_ = nullptr; d_rate_enc_ = nullptr;
        d_rate_lut_ = nullptr; d_rate_aux_ = nullptr; d_rate_est_ = nullptr; d_rate_out_ = nullptr; h_rate_out_ = nullptr;
        set_error(kErrCuda, "device or pinned memory allocation failed (rate curve)");
        return false;
    }
    return true;
}

int Engine::rate_curve(uint8_t wavelet, const uint8_t *d_rgb, uint64_t bytes[kRateSteps], unsigned *h_hist_out,
                       uint32_t slot, uint8_t *d_work) {
    if (slot >= cap_) { set_error(kErrBufferSize, "rate curve: chunk slot beyond the engine capacity"); return kErrBufferSize; }
    uint8_t *sym = d_work ? d_work : sym_ptr_[slot];
    if (!sym) { set_error(kErrNull, "shared-workspace engine: workspace pointer required"); return kErrNull; }
    const uint64_t dev_before = dev_bytes_;
    if (!ensure_rate_buffers()) { dev_bytes_ = dev_before; return kErrCuda; }
    const size_t N = (size_t)d_.padded;
    CU_TRY(cudaMemsetAsync(d_hist_ + (size_t)slot * 3 * 256, 0, 3 * 256 * sizeof(unsigned), st_));
    int rc = frontend_one(slot, wavelet, d_rgb, sym, 1, d_coef_);   // at any step (1): only the coefficient dump is used
    if (rc) return rc;
    const int bound = rate_value_bound(wavelet);
    CU_TRY(cudaMemsetAsync(d_vhist_, 0, 3 * (2 * (size_t)bound + 1) * sizeof(unsigned), st_));
    CU_TRY(cudaMemsetAsync(d_rate_out_ + kRateSteps, 0, sizeof(unsigned long long), st_));
    coef_value_hist(d_coef_, N, bound, d_vhist_, d_rate_out_ + kRateSteps, st_);
    step_hists(d_vhist_, bound, N, d_rate_hist_, st_);
    // the tables the encode at each step would use; the estimate and the zero-frequency check take the symbol counts
    if (well_formed_) well_formed_hists(d_rate_hist_, kRateSteps * 3, d_rate_wf_hist_, st_);
    build_tables(well_formed_ ? d_rate_wf_hist_ : d_rate_hist_, kRateSteps * 3, 256, d_rate_enc_, d_rate_lut_, d_rate_aux_,
                 nullptr, nullptr, nullptr, st_);
    estimate_stream_bytes(d_rate_hist_, d_rate_enc_, kRateSteps * 3, N, d_rate_est_, st_);
    rate_sizes(d_rate_hist_, d_rate_enc_, d_rate_est_, N, kFixedHeaderBytes + 3 * kChannelHeaderBytes, d_rate_out_, st_);
    CU_TRY(cudaMemcpyAsync(h_rate_out_, d_rate_out_, (kRateSteps + 1) * sizeof(unsigned long long), cudaMemcpyDeviceToHost, st_));
    if (h_hist_out)
        CU_TRY(cudaMemcpyAsync(h_hist_out, d_rate_hist_, (size_t)kRateSteps * 3 * 256 * sizeof(unsigned), cudaMemcpyDeviceToHost, st_));
    CU_TRY(cudaStreamSynchronize(st_));
    CU_TRY(cudaGetLastError());
    if (h_rate_out_[kRateSteps]) {
        set_error(kErrPanic, "rate curve: " + std::to_string(h_rate_out_[kRateSteps]) +
                                 " coefficients outside the derived value range");
        return kErrPanic;
    }
    for (int i = 0; i < kRateSteps; i++) bytes[i] = h_rate_out_[i];
    return kOk;
}

// ------------------------------------------------------------------------------ the pool
namespace {
struct PoolEntry {
    std::unique_ptr<Engine> eng;
    int device = 0;
    bool busy = false;
    uint64_t stamp = 0;
};
std::mutex g_pool_mu;
std::vector<PoolEntry> g_pool;
uint64_t g_stamp = 0;
constexpr size_t kMaxIdleEngines = 2;
}  // namespace

Engine *acquire_engine(const Dims &d, bool well_formed_tables) {
    int dev = 0;
    cudaGetDevice(&dev);
    std::lock_guard<std::mutex> lk(g_pool_mu);
    for (PoolEntry &p : g_pool)
        if (!p.busy && p.device == dev && p.eng->dims().w == d.w && p.eng->dims().h == d.h && p.eng->dims().f == d.f &&
            p.eng->well_formed_tables() == well_formed_tables) {
            p.busy = true;
            p.stamp = ++g_stamp;
            return p.eng.get();
        }
    // drop idle engines of other shapes beyond the cap (oldest first) before allocating a new one
    for (;;) {
        size_t idle = 0, oldest = g_pool.size();
        for (size_t i = 0; i < g_pool.size(); i++)
            if (!g_pool[i].busy) {
                idle++;
                if (oldest == g_pool.size() || g_pool[i].stamp < g_pool[oldest].stamp) oldest = i;
            }
        if (idle < kMaxIdleEngines || oldest == g_pool.size()) break;
        g_pool.erase(g_pool.begin() + (long)oldest);
    }
    std::unique_ptr<Engine> e(new Engine(d, 1, 0, nullptr, true, false, well_formed_tables));
    if (!e->ok()) {
        // out of memory: release every idle engine and retry once
        for (size_t i = g_pool.size(); i-- > 0;)
            if (!g_pool[i].busy) g_pool.erase(g_pool.begin() + (long)i);
        e.reset(new Engine(d, 1, 0, nullptr, true, false, well_formed_tables));
        if (!e->ok()) return nullptr;
    }
    PoolEntry p;
    p.eng = std::move(e);
    p.device = dev;
    p.busy = true;
    p.stamp = ++g_stamp;
    g_pool.push_back(std::move(p));
    return g_pool.back().eng.get();
}

void release_engine(Engine *e) {
    std::lock_guard<std::mutex> lk(g_pool_mu);
    for (PoolEntry &p : g_pool)
        if (p.eng.get() == e) p.busy = false;
}

}  // namespace alice
