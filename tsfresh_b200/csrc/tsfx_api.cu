// tsfx_api.cu -- the C ABI of libtsfx.so (include/tsfx.h): context, plan, extraction entry points, and the native
// runtime around the kernels: pinned host pool, threaded pageable->pinned staging ring, the row-block pipeline of the
// long-frame path (stage (a) + kernels + result transfer on three streams), multi-GPU result placement.
#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <condition_variable>
#include <functional>
#include <map>
#include <mutex>
#include <new>
#include <string>
#include <thread>
#include <unordered_map>
#include <vector>

#include "tsfx_common.cuh"
#include "tsfx_kernels.h"
#include "tsfx_csr.h"
#include "tsfx_impute.h"
#include "tsfx_select.h"

using namespace tsfx;

static std::string g_create_error;

struct DevBuf {
    void* p = nullptr;
    size_t cap = 0;
    cudaError_t reserve(size_t bytes) {
        if (bytes <= cap) return cudaSuccess;
        if (p) cudaFree(p);
        p = nullptr;
        cap = 0;
        cudaError_t e = cudaMalloc(&p, bytes);
        if (e == cudaSuccess) cap = bytes;
        return e;
    }
    void release() { if (p) cudaFree(p); p = nullptr; cap = 0; }
};

// ---------------------------------------------------------------------------------- pinned host memory pool
// Page-locking is slow (a few GB/s), so blocks handed back with tsfx_host_free are cached and reused.
struct HostPool {
    std::mutex mu;
    std::multimap<size_t, void*> idle;
    std::unordered_map<void*, size_t> live;
    void* alloc(size_t bytes) {
        if (bytes == 0) bytes = 1;
        const size_t want = (bytes + ((size_t)2 << 20) - 1) & ~(((size_t)2 << 20) - 1);
        {
            std::lock_guard<std::mutex> g(mu);
            auto it = idle.lower_bound(want);
            if (it != idle.end() && it->first <= want + want / 2 + ((size_t)64 << 20)) {
                void* p = it->second;
                live[p] = it->first;
                idle.erase(it);
                return p;
            }
        }
        void* p = nullptr;
        if (cudaHostAlloc(&p, want, cudaHostAllocPortable) != cudaSuccess) {
            cudaGetLastError();
            trim();                                  // give cached blocks back and retry once
            if (cudaHostAlloc(&p, want, cudaHostAllocPortable) != cudaSuccess) { cudaGetLastError(); return nullptr; }
        }
        std::lock_guard<std::mutex> g(mu);
        live[p] = want;
        return p;
    }
    bool free(void* p) {
        std::lock_guard<std::mutex> g(mu);
        auto it = live.find(p);
        if (it == live.end()) return false;
        idle.emplace(it->second, p);
        live.erase(it);
        return true;
    }
    void trim() {
        std::lock_guard<std::mutex> g(mu);
        for (auto& kv : idle) cudaFreeHost(kv.second);
        idle.clear();
    }
    void release_all() {
        // blocks still handed out (a DataFrame may live on one) are deliberately NOT freed when the context goes away:
        // they stay valid until the process exits
        trim();
        std::lock_guard<std::mutex> g(mu);
        live.clear();
    }
};

// ---------------------------------------------------------------------------------- pageable -> device staging
// Host buffers that are not page-locked (numpy / pandas columns) are copied chunk by chunk into a ring of pinned
// slots by a few worker threads (one memcpy thread cannot feed PCIe gen5) and sent with cudaMemcpyAsync, so the
// transfer overlaps both the next chunk's memcpy and the kernels already queued.
struct Stager {
    static const int SLOTS = 3;
    size_t slot_bytes = (size_t)32 << 20;
    void* slot[SLOTS] = {nullptr, nullptr, nullptr};
    cudaEvent_t ev[SLOTS] = {nullptr, nullptr, nullptr};
    bool busy[SLOTS] = {false, false, false};
    int next = 0;
    // worker pool
    std::vector<std::thread> workers;
    std::mutex mu;
    std::condition_variable cv, cv_done;
    const char* src = nullptr;
    char* dst = nullptr;
    size_t total = 0, piece = 0;
    int next_piece = 0, n_pieces = 0, pending = 0;
    uint64_t generation = 0;
    bool stop = false;

    void worker() {
        uint64_t seen = 0;
        for (;;) {
            std::unique_lock<std::mutex> lk(mu);
            cv.wait(lk, [&] { return stop || (generation != seen && next_piece < n_pieces); });
            if (stop) return;
            while (next_piece < n_pieces) {
                const int k = next_piece++;
                lk.unlock();
                const size_t off = (size_t)k * piece;
                memcpy(dst + off, src + off, std::min(piece, total - off));
                lk.lock();
                if (--pending == 0) cv_done.notify_all();
            }
            seen = generation;
        }
    }
    void start(int n) {
        if (!workers.empty()) return;
        for (int i = 0; i < n; ++i) workers.emplace_back([this] { worker(); });
    }
    void parallel_copy(void* d, const void* s_, size_t bytes) {
        if (workers.empty() || bytes < ((size_t)1 << 20)) { memcpy(d, s_, bytes); return; }
        std::unique_lock<std::mutex> lk(mu);
        src = (const char*)s_; dst = (char*)d; total = bytes;
        n_pieces = (int)std::min<size_t>(workers.size() * 2, (bytes + ((size_t)1 << 20) - 1) >> 20);
        piece = ((bytes + n_pieces - 1) / n_pieces + 63) & ~(size_t)63;
        n_pieces = (int)((bytes + piece - 1) / piece);
        next_piece = 0; pending = n_pieces; ++generation;
        cv.notify_all();
        cv_done.wait(lk, [&] { return pending == 0; });
    }
    cudaError_t init() {
        if (slot[0]) return cudaSuccess;
        for (int i = 0; i < SLOTS; ++i) {
            cudaError_t e = cudaHostAlloc(&slot[i], slot_bytes, cudaHostAllocDefault);
            if (e != cudaSuccess) return e;
            e = cudaEventCreateWithFlags(&ev[i], cudaEventDisableTiming);
            if (e != cudaSuccess) return e;
        }
        const int n = std::min(8, std::max(1, (int)std::thread::hardware_concurrency() / 2));
        if (n > 1) start(n);
        return cudaSuccess;
    }
    void release() {
        {
            std::lock_guard<std::mutex> g(mu);
            stop = true;
        }
        cv.notify_all();
        for (auto& t : workers) t.join();
        workers.clear();
        for (int i = 0; i < SLOTS; ++i) { if (slot[i]) cudaFreeHost(slot[i]); if (ev[i]) cudaEventDestroy(ev[i]); slot[i] = nullptr; ev[i] = nullptr; }
    }
    // host (pageable or pinned) -> device, asynchronous with respect to the device; returns when the LAST chunk's
    // cudaMemcpyAsync has been issued (pageable source: the source buffer is no longer needed by then)
    cudaError_t h2d(void* d, const void* h, size_t bytes, cudaStream_t st) {
        if (bytes == 0) return cudaSuccess;
        cudaPointerAttributes at;
        bool pinned = false;
        if (cudaPointerGetAttributes(&at, h) == cudaSuccess) pinned = (at.type == cudaMemoryTypeHost || at.type == cudaMemoryTypeManaged);
        else cudaGetLastError();
        if (pinned) return cudaMemcpyAsync(d, h, bytes, cudaMemcpyHostToDevice, st);
        cudaError_t e = init();
        if (e != cudaSuccess) return e;
        for (size_t off = 0; off < bytes; off += slot_bytes) {
            const size_t cnt = std::min(slot_bytes, bytes - off);
            const int k = next;
            next = (next + 1) % SLOTS;
            if (busy[k]) { e = cudaEventSynchronize(ev[k]); if (e != cudaSuccess) return e; }
            parallel_copy(slot[k], (const char*)h + off, cnt);
            e = cudaMemcpyAsync((char*)d + off, slot[k], cnt, cudaMemcpyHostToDevice, st);
            if (e != cudaSuccess) return e;
            e = cudaEventRecord(ev[k], st);
            if (e != cudaSuccess) return e;
            busy[k] = true;
        }
        return cudaSuccess;
    }
};

static const char* kGroupNames[G_EVENTS] = {"basic", "sorted", "spectral", "la", "entropy", "seq", "peaks", "assemble"};

struct tsfx_ctx {
    int device = 0;
    cudaStream_t stream = nullptr;
    bool own_stream = false;
    int sm_count = 148;
    std::string err;
    DevBuf values, begin, len, out, misc, stage;
    double* d_dec = nullptr;
    double2* d_tw = nullptr;
    int tw_n = 0;
    cudaEvent_t ev[G_EVENTS][2];
    bool ev_used[G_EVENTS];
    float ms[G_EVENTS];
    int launches = 0;
    CsrWorkspace csr;
    ImputeWorkspace imp;
    SelectWorkspace sel;
    DevBuf sel_x, sel_y, sel_out;
    int64_t held_series = -1;    // CSR kept on the device by the last stage-(a) call (-1: none)
    int held_max_len = 0;
    bool used_moments = false;   // the last pass ran k_moments in place of k_basic (reported as "moments")
    DevBuf kvals, kvals_sorted;  // value columns of kinds 1 .. K-1 of a wide frame (input order / CSR order)
    DevBuf times, times_sorted;  // tsfx_set_row_times: row timestamps of the next extract call (linear_trend_timewise)
    const int64_t* times_ptr = nullptr;
    int64_t times_rows = -1;
    int max_len_hint = 0;        // tsfx_set_max_len_hint: longest series of the coming device-pointer CSR calls
    HostPool pool;
    Stager stager;
    // multi-GPU result placement (tsfx_set_peer_outputs): peers' mapped result matrices
    std::vector<uint64_t> peer_out;
    int peer_self = -1, peer_mode = 0;
    uint64_t peer_mc = 0;
    cudaStream_t s_peer = nullptr;
    cudaEvent_t ev_peer = nullptr;
    cudaStream_t s_in = nullptr, s_out = nullptr;   // copy streams of the pipelined host path
    cudaEvent_t ev_in[2] = {nullptr, nullptr}, ev_done[2] = {nullptr, nullptr};
};

struct tsfx_plan {
    tsfx_ctx* ctx = nullptr;
    std::vector<Desc> host[G_COUNT];
    Desc* dev[G_COUNT] = {nullptr};
    int32_t* d_final_col = nullptr;   // final column of every staged column, groups concatenated
    bool basic_moments_only = false;  // the BASIC group is reductions only: k_moments replaces k_basic
    int moments_need_high = 0;
    int n_groups_used = 0;
    int basic_nfin = 0;               // leading "finisher" descriptors of the BASIC group
    int sorted_nfin = 0;              // same for the SORTED group
    int spectral_nfft = 0;            // leading fft_coefficient descriptors of the SPECTRAL group
    int cum[G_COUNT + 1] = {0};
    int ncols = 0;
    int lag_needed = 0, pacf_want = -1;
    int basic_bins = 0, fourier_bins = 0;
    int need_fft = 0, need_welch = 0;
    int max_ar_k = 0, need_adf = 0;
    int max_lz_bins = 0, max_perm_dim = 0, max_cwt_peaks_n = 0, n_lz = 0;
    int need_times = 0;               // linear_trend_timewise columns: the extract call needs tsfx_set_row_times
    int friedrich_r = 0;
    double* d_tables = nullptr;
    int64_t* d_toff = nullptr;
    int32_t* d_thalf = nullptr;
    int n_tables = 0;
    std::vector<int64_t> toff;
    std::vector<int32_t> thalf;
};

static int fail(tsfx_ctx* c, int code, const std::string& msg) {
    if (c) c->err = msg; else g_create_error = msg;
    return code;
}
#define CK(call)                                                                                  \
    do {                                                                                          \
        cudaError_t e__ = (call);                                                                 \
        if (e__ != cudaSuccess)                                                                   \
            return fail(ctx, TSFX_E_CUDA, std::string(#call) + ": " + cudaGetErrorString(e__));  \
    } while (0)

static int group_of(int calc) {
    switch (calc) {
        case TSFX_SYMMETRY_LOOKING: case TSFX_HAS_DUPLICATE: case TSFX_MEDIAN:
        case TSFX_PERCENTAGE_OF_REOCCURRING_VALUES_TO_ALL_VALUES:
        case TSFX_PERCENTAGE_OF_REOCCURRING_DATAPOINTS_TO_ALL_DATAPOINTS:
        case TSFX_SUM_OF_REOCCURRING_VALUES: case TSFX_SUM_OF_REOCCURRING_DATA_POINTS:
        case TSFX_RATIO_VALUE_NUMBER_TO_TIME_SERIES_LENGTH: case TSFX_QUANTILE:
        case TSFX_MEAN_N_ABSOLUTE_MAX: case TSFX_CHANGE_QUANTILES: case TSFX_FRIEDRICH_COEFFICIENTS:
        case TSFX_MAX_LANGEVIN_FIXED_POINT:
            return G_SORTED;
        case TSFX_FFT_COEFFICIENT: case TSFX_FFT_AGGREGATED: case TSFX_SPKT_WELCH_DENSITY:
        case TSFX_FOURIER_ENTROPY: case TSFX_CWT_COEFFICIENTS:
            return G_SPECTRAL;
        case TSFX_AR_COEFFICIENT: case TSFX_AUGMENTED_DICKEY_FULLER:
            return G_LA;
        case TSFX_SAMPLE_ENTROPY: case TSFX_APPROXIMATE_ENTROPY:
            return G_ENTROPY;
        case TSFX_LEMPEL_ZIV_COMPLEXITY: case TSFX_PERMUTATION_ENTROPY:
            return G_SEQ;
        case TSFX_NUMBER_CWT_PEAKS:
            return G_PEAKS;
        default:
            return G_BASIC;
    }
}

extern "C" int tsfx_version(void) { return TSFX_VERSION; }

extern "C" int tsfx_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
    return n;
}

extern "C" const char* tsfx_last_error(const tsfx_ctx* ctx) { return ctx ? ctx->err.c_str() : g_create_error.c_str(); }

extern "C" int tsfx_ctx_create(int device, void* cuda_stream, tsfx_ctx** out) {
    if (!out) return fail(nullptr, TSFX_E_INVALID, "out is NULL");
    *out = nullptr;
    tsfx_ctx* ctx = nullptr;
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0)
        return fail(nullptr, TSFX_E_CUDA, std::string("no CUDA device: ") + cudaGetErrorString(e));
    if (device < 0 || device >= ndev) return fail(nullptr, TSFX_E_INVALID, "device index out of range");
    ctx = new (std::nothrow) tsfx_ctx();
    if (!ctx) return fail(nullptr, TSFX_E_NOMEM, "out of host memory");
    ctx->device = device;
    for (int g = 0; g < G_EVENTS; ++g) { ctx->ev_used[g] = false; ctx->ms[g] = 0.f; ctx->ev[g][0] = ctx->ev[g][1] = nullptr; }
#define CKC(call)                                                                                     \
    do {                                                                                              \
        cudaError_t e__ = (call);                                                                     \
        if (e__ != cudaSuccess) {                                                                     \
            std::string m = std::string(#call) + ": " + cudaGetErrorString(e__);                     \
            delete ctx;                                                                               \
            return fail(nullptr, TSFX_E_CUDA, m);                                                     \
        }                                                                                             \
    } while (0)
    CKC(cudaSetDevice(device));
    cudaDeviceProp prop;
    CKC(cudaGetDeviceProperties(&prop, device));
    ctx->sm_count = prop.multiProcessorCount;
    if (cuda_stream) { ctx->stream = (cudaStream_t)cuda_stream; ctx->own_stream = false; }
    else { CKC(cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking)); ctx->own_stream = true; }
    for (int g = 0; g < G_EVENTS; ++g) { CKC(cudaEventCreate(&ctx->ev[g][0])); CKC(cudaEventCreate(&ctx->ev[g][1])); }
    CKC(cudaStreamCreateWithFlags(&ctx->s_in, cudaStreamNonBlocking));
    CKC(cudaStreamCreateWithFlags(&ctx->s_out, cudaStreamNonBlocking));
    CKC(cudaStreamCreateWithFlags(&ctx->s_peer, cudaStreamNonBlocking));
    CKC(cudaEventCreateWithFlags(&ctx->ev_peer, cudaEventDisableTiming));
    for (int i = 0; i < 2; ++i) { CKC(cudaEventCreateWithFlags(&ctx->ev_in[i], cudaEventDisableTiming)); CKC(cudaEventCreateWithFlags(&ctx->ev_done[i], cudaEventDisableTiming)); }
    // decimal threshold table d * 10^k (correctly rounded literals via strtod)
    {
        std::vector<double> dec((TSFX_DEC_MAX - TSFX_DEC_MIN + 1) * 9);
        for (int k = TSFX_DEC_MIN; k <= TSFX_DEC_MAX; ++k)
            for (int d = 1; d <= 9; ++d) {
                char buf[32];
                snprintf(buf, sizeof buf, "%de%d", d, k);
                dec[(k - TSFX_DEC_MIN) * 9 + (d - 1)] = strtod(buf, nullptr);
            }
        CKC(cudaMalloc(&ctx->d_dec, dec.size() * sizeof(double)));
        CKC(cudaMemcpy(ctx->d_dec, dec.data(), dec.size() * sizeof(double), cudaMemcpyHostToDevice));
    }
#undef CKC
    *out = ctx;
    return TSFX_OK;
}

extern "C" void tsfx_ctx_destroy(tsfx_ctx* ctx) {
    if (!ctx) return;
    cudaSetDevice(ctx->device);
    cudaStreamSynchronize(ctx->stream);
    ctx->values.release(); ctx->begin.release(); ctx->len.release(); ctx->out.release(); ctx->misc.release(); ctx->stage.release();
    ctx->times.release(); ctx->times_sorted.release(); ctx->kvals.release(); ctx->kvals_sorted.release();
    ctx->csr.release();
    ctx->imp.release();
    ctx->sel.release();
    ctx->sel_x.release(); ctx->sel_y.release(); ctx->sel_out.release();
    ctx->stager.release();
    ctx->pool.release_all();
    if (ctx->s_peer) cudaStreamDestroy(ctx->s_peer);
    if (ctx->ev_peer) cudaEventDestroy(ctx->ev_peer);
    if (ctx->d_dec) cudaFree(ctx->d_dec);
    if (ctx->d_tw) cudaFree(ctx->d_tw);
    for (int g = 0; g < G_EVENTS; ++g) { if (ctx->ev[g][0]) cudaEventDestroy(ctx->ev[g][0]); if (ctx->ev[g][1]) cudaEventDestroy(ctx->ev[g][1]); }
    if (ctx->s_in) cudaStreamDestroy(ctx->s_in);
    if (ctx->s_out) cudaStreamDestroy(ctx->s_out);
    for (int i = 0; i < 2; ++i) { if (ctx->ev_in[i]) cudaEventDestroy(ctx->ev_in[i]); if (ctx->ev_done[i]) cudaEventDestroy(ctx->ev_done[i]); }
    if (ctx->own_stream && ctx->stream) cudaStreamDestroy(ctx->stream);
    delete ctx;
}

extern "C" int tsfx_sync(tsfx_ctx* ctx) {
    if (!ctx) return TSFX_E_INVALID;
    CK(cudaSetDevice(ctx->device));
    CK(cudaStreamSynchronize(ctx->stream));
    return TSFX_OK;
}

// ------------------------------------------------------------------------------------------ plan
extern "C" int tsfx_plan_create(tsfx_ctx* ctx, const tsfx_feature_desc* descs, int32_t n_descs, int32_t n_cols,
                                const double* tables, const int64_t* table_off, const int32_t* table_half,
                                int32_t n_tables, tsfx_plan** out) {
    if (!ctx) return TSFX_E_INVALID;
    if (!out || (!descs && n_descs > 0) || n_descs < 0 || n_cols < 0)
        return fail(ctx, TSFX_E_INVALID, "tsfx_plan_create: bad arguments");
    *out = nullptr;
    CK(cudaSetDevice(ctx->device));
    tsfx_plan* P = new (std::nothrow) tsfx_plan();
    if (!P) return fail(ctx, TSFX_E_NOMEM, "out of host memory");
    P->ctx = ctx;
    P->ncols = n_cols;
    for (int i = 0; i < n_descs; ++i) {
        const Desc& d = descs[i];
        if (d.calc < 0 || d.calc >= TSFX_N_CALCS || d.col < 0 || d.col >= n_cols) {
            delete P;
            return fail(ctx, TSFX_E_INVALID, "tsfx_plan_create: descriptor " + std::to_string(i) + " out of range");
        }
        P->host[group_of(d.calc)].push_back(d);
        switch (d.calc) {
            case TSFX_AUTOCORRELATION: P->lag_needed = std::max(P->lag_needed, d.i0); break;
            case TSFX_AGG_AUTOCORRELATION: P->lag_needed = std::max(P->lag_needed, d.i0); break;
            case TSFX_PARTIAL_AUTOCORRELATION:
                P->lag_needed = std::max(P->lag_needed, d.i1);
                P->pacf_want = std::max(P->pacf_want, d.i1);
                break;
            case TSFX_BINNED_ENTROPY: P->basic_bins = std::max(P->basic_bins, d.i0); break;
            case TSFX_FOURIER_ENTROPY: P->fourier_bins = std::max(P->fourier_bins, d.i0); P->need_welch = 1; break;
            case TSFX_SPKT_WELCH_DENSITY: P->need_welch = 1; break;
            case TSFX_FFT_COEFFICIENT: case TSFX_FFT_AGGREGATED: P->need_fft = 1; break;
            case TSFX_CWT_COEFFICIENTS:
                if (d.i1 < 0 || d.i1 >= n_tables) { delete P; return fail(ctx, TSFX_E_INVALID, "cwt table index out of range"); }
                break;
            case TSFX_AR_COEFFICIENT:
                if (d.i1 < 1 || d.i1 > 32) { delete P; return fail(ctx, TSFX_E_UNSUPPORTED, "ar_coefficient: k must be in 1..32"); }
                P->max_ar_k = std::max(P->max_ar_k, d.i1);
                break;
            case TSFX_AUGMENTED_DICKEY_FULLER: P->need_adf = 1; break;
            case TSFX_LINEAR_TREND_TIMEWISE: P->need_times = 1; break;
            case TSFX_APPROXIMATE_ENTROPY:
                if (d.i0 != 2) { delete P; return fail(ctx, TSFX_E_UNSUPPORTED, "approximate_entropy: only m=2"); }
                break;
            case TSFX_LEMPEL_ZIV_COMPLEXITY: P->max_lz_bins = std::max(P->max_lz_bins, d.i0); P->n_lz += 1; break;
            case TSFX_PERMUTATION_ENTROPY:
                if (d.i1 < 2 || d.i1 > 8 || d.i0 < 1) { delete P; return fail(ctx, TSFX_E_UNSUPPORTED, "permutation_entropy: dimension 2..8, tau >= 1"); }
                P->max_perm_dim = std::max(P->max_perm_dim, d.i1);
                break;
            case TSFX_NUMBER_CWT_PEAKS:
                if (d.i0 < 1 || d.i0 > 16) { delete P; return fail(ctx, TSFX_E_UNSUPPORTED, "number_cwt_peaks: n must be in 1..16"); }
                P->max_cwt_peaks_n = std::max(P->max_cwt_peaks_n, d.i0);
                break;
            case TSFX_FRIEDRICH_COEFFICIENTS: case TSFX_MAX_LANGEVIN_FIXED_POINT:
                if (d.i1 != 3 || d.i2 < 1 || d.i2 > 256) { delete P; return fail(ctx, TSFX_E_UNSUPPORTED, "friedrich: only m=3, r in 1..256"); }
                P->friedrich_r = std::max(P->friedrich_r, d.i2);
                break;
            default: break;
        }
    }
    if (P->lag_needed > 4096) { delete P; return fail(ctx, TSFX_E_UNSUPPORTED, "lag > 4096"); }
    std::vector<int32_t> final_col;
    for (int g = 0; g < G_COUNT; ++g) {
        std::stable_sort(P->host[g].begin(), P->host[g].end(), [g](const Desc& a, const Desc& b) {
            if (g == G_BASIC) {               // O(1) finishers first (evaluated lane-parallel)
                const bool fa = basic_finisher_calc(a.calc), fb = basic_finisher_calc(b.calc);
                if (fa != fb) return fa;
            }
            if (g == G_SORTED) {
                const bool fa = sorted_finisher_calc(a.calc), fb = sorted_finisher_calc(b.calc);
                if (fa != fb) return fa;
            }
            if (g == G_SPECTRAL) {            // fft_coefficient first, grouped by attribute
                const bool fa = a.calc == TSFX_FFT_COEFFICIENT, fb = b.calc == TSFX_FFT_COEFFICIENT;
                if (fa != fb) return fa;
                if (fa && a.attr != b.attr) return a.attr < b.attr;
            }
            if (a.calc != b.calc) return a.calc < b.calc;
            if (a.i1 != b.i1) return a.i1 < b.i1;
            if (a.i2 != b.i2) return a.i2 < b.i2;
            if (a.p0 != b.p0) return a.p0 < b.p0;
            if (a.p1 != b.p1) return a.p1 < b.p1;
            if (a.i0 != b.i0) return a.i0 < b.i0;
            return a.col < b.col;
        });
        if (g == G_BASIC)
            for (const Desc& d : P->host[g]) P->basic_nfin += basic_finisher_calc(d.calc) ? 1 : 0;
        if (g == G_SORTED)
            for (const Desc& d : P->host[g]) P->sorted_nfin += sorted_finisher_calc(d.calc) ? 1 : 0;
        if (g == G_SPECTRAL)
            for (const Desc& d : P->host[g]) P->spectral_nfft += (d.calc == TSFX_FFT_COEFFICIENT) ? 1 : 0;
        P->cum[g + 1] = P->cum[g] + (int)P->host[g].size();
        for (size_t j = 0; j < P->host[g].size(); ++j) {      // col becomes the index inside the group's staging row
            final_col.push_back(P->host[g][j].col);
            P->host[g][j].col = (int32_t)j;
        }
        if (!P->host[g].empty()) {
            size_t bytes = P->host[g].size() * sizeof(Desc);
            cudaError_t e = cudaMalloc(&P->dev[g], bytes);
            if (e == cudaSuccess) e = cudaMemcpy(P->dev[g], P->host[g].data(), bytes, cudaMemcpyHostToDevice);
            if (e != cudaSuccess) { tsfx_plan_destroy(P); return fail(ctx, TSFX_E_CUDA, cudaGetErrorString(e)); }
        }
    }
    P->basic_moments_only = !P->host[G_BASIC].empty();
    for (const Desc& d : P->host[G_BASIC]) {
        if (!moments_only_calc(d.calc)) P->basic_moments_only = false;
        if (d.calc == TSFX_SKEWNESS || d.calc == TSFX_KURTOSIS) P->moments_need_high = 1;
    }
    for (int g = 0; g < G_COUNT; ++g) P->n_groups_used += P->host[g].empty() ? 0 : 1;
    if (!final_col.empty()) {
        cudaError_t e = cudaMalloc(&P->d_final_col, final_col.size() * sizeof(int32_t));
        if (e == cudaSuccess) e = cudaMemcpy(P->d_final_col, final_col.data(), final_col.size() * sizeof(int32_t), cudaMemcpyHostToDevice);
        if (e != cudaSuccess) { tsfx_plan_destroy(P); return fail(ctx, TSFX_E_CUDA, cudaGetErrorString(e)); }
    }
    if (n_tables > 0) {
        if (!tables || !table_off || !table_half) { tsfx_plan_destroy(P); return fail(ctx, TSFX_E_INVALID, "cwt tables missing"); }
        P->n_tables = n_tables;
        P->toff.assign(table_off, table_off + n_tables + 1);
        P->thalf.assign(table_half, table_half + n_tables);
        size_t tb = (size_t)table_off[n_tables] * sizeof(double);
        cudaError_t e = cudaMalloc(&P->d_tables, std::max<size_t>(tb, 8));
        if (e == cudaSuccess) e = cudaMemcpy(P->d_tables, tables, tb, cudaMemcpyHostToDevice);
        if (e == cudaSuccess) e = cudaMalloc(&P->d_toff, (n_tables + 1) * sizeof(int64_t));
        if (e == cudaSuccess) e = cudaMemcpy(P->d_toff, table_off, (n_tables + 1) * sizeof(int64_t), cudaMemcpyHostToDevice);
        if (e == cudaSuccess) e = cudaMalloc(&P->d_thalf, n_tables * sizeof(int32_t));
        if (e == cudaSuccess) e = cudaMemcpy(P->d_thalf, table_half, n_tables * sizeof(int32_t), cudaMemcpyHostToDevice);
        if (e != cudaSuccess) { tsfx_plan_destroy(P); return fail(ctx, TSFX_E_CUDA, cudaGetErrorString(e)); }
    }
    *out = P;
    return TSFX_OK;
}

extern "C" void tsfx_plan_destroy(tsfx_plan* P) {
    if (!P) return;
    if (P->ctx) cudaSetDevice(P->ctx->device);
    for (int g = 0; g < G_COUNT; ++g) if (P->dev[g]) cudaFree(P->dev[g]);
    if (P->d_final_col) cudaFree(P->d_final_col);
    if (P->d_tables) cudaFree(P->d_tables);
    if (P->d_toff) cudaFree(P->d_toff);
    if (P->d_thalf) cudaFree(P->d_thalf);
    delete P;
}

// ------------------------------------------------------------------------------------------ launch all groups
static int even(int v) { return (v + 1) & ~1; }

static int ensure_twiddle(tsfx_ctx* ctx, int n_pow2) {
    if (n_pow2 <= ctx->tw_n) return TSFX_OK;
    if (ctx->d_tw) { cudaStreamSynchronize(ctx->stream); cudaFree(ctx->d_tw); ctx->d_tw = nullptr; ctx->tw_n = 0; }
    CK(cudaMalloc(&ctx->d_tw, (size_t)(n_pow2 / 2 + 1) * sizeof(double2)));
    CK(launch_fill_twiddle(ctx->d_tw, n_pow2, ctx->stream));
    ctx->tw_n = n_pow2;
    return TSFX_OK;
}

// row timestamps handed over with tsfx_set_row_times for a call whose `values` array has `rows` rows (consumed)
static int take_times(tsfx_ctx* ctx, const tsfx_plan* P, int64_t rows, const int64_t** out) {
    *out = nullptr;
    const bool have = ctx->times_rows >= 0;
    const int64_t got = ctx->times_rows;
    const int64_t* p = ctx->times_ptr;
    ctx->times_rows = -1;
    ctx->times_ptr = nullptr;
    if (!P->need_times) return TSFX_OK;
    if (!have) return fail(ctx, TSFX_E_INVALID, "linear_trend_timewise needs the row timestamps (tsfx_set_row_times)");
    if (got != rows) return fail(ctx, TSFX_E_INVALID, "tsfx_set_row_times: " + std::to_string(got) + " timestamps for " + std::to_string(rows) + " rows");
    *out = p;
    return TSFX_OK;
}

extern "C" int tsfx_set_row_times(tsfx_ctx* ctx, const int64_t* row_time_ns, int64_t n_rows, uint32_t flags) {
    if (!ctx) return TSFX_E_INVALID;
    if (n_rows < 0 || (n_rows > 0 && !row_time_ns)) return fail(ctx, TSFX_E_INVALID, "tsfx_set_row_times: bad arguments");
    CK(cudaSetDevice(ctx->device));
    if (flags & TSFX_FLAG_DEVICE_PTRS) ctx->times_ptr = row_time_ns;
    else {
        CK(ctx->times.reserve(std::max<size_t>((size_t)n_rows * 8, 8)));
        CK(ctx->stager.h2d(ctx->times.p, row_time_ns, (size_t)n_rows * 8, ctx->stream));
        ctx->times_ptr = (const int64_t*)ctx->times.p;
    }
    ctx->times_rows = n_rows;
    return TSFX_OK;
}

static int run_groups(tsfx_ctx* ctx, const tsfx_plan* P, const SeriesRef& R, int max_len, double* d_final, uint32_t flags, int ld = 0) {
    if (ld <= 0) ld = P->ncols;          // row stride of the caller's matrix
    const bool timing = (flags & TSFX_FLAG_TIMING) != 0;
    for (int g = 0; g < G_EVENTS; ++g) ctx->ev_used[g] = false;
    ctx->launches = 0;
    if (R.n_series == 0) return TSFX_OK;
    const int staged = P->cum[G_COUNT];
    if (staged == 0) return TSFX_OK;
    CK(ctx->stage.reserve((size_t)R.n_series * staged * sizeof(double)));
    CK(ctx->misc.reserve(max_len > 1024 ? ((size_t)1 << 30) : ((size_t)256 << 20)));      // global working regions for series too long for shared memory
    // the groups run back to back on ctx->stream, so each may use the whole working region
    unsigned char* const gscratch = (unsigned char*)ctx->misc.p;
    const size_t gscratch_bytes = ctx->misc.cap;
    if (!P->host[G_SPECTRAL].empty()) {      // FFT twiddle table (filled once)
        int p2 = 1;
        while (p2 < max_len) p2 <<= 1;
        if (p2 > max_len) p2 >>= 1;            // largest power of two <= max_len
        p2 = std::max(p2, 256);
        int rc = ensure_twiddle(ctx, p2);
        if (rc) return rc;
    }
    bool direct = false;          // the only group wrote the final matrix itself
    ctx->used_moments = false;
    if (max_len < 1) return fail(ctx, TSFX_E_INVALID, "series of length < 1");
    auto too_long = [&](const char* g) {
        return fail(ctx, TSFX_E_TOO_LONG, std::string("series length ") + std::to_string(max_len) +
                                              " exceeds the shared-memory staging of kernel group " + g);
    };
    for (int g = 0; g < G_COUNT; ++g) {
        if (P->host[g].empty()) continue;
        if (timing) { CK(cudaEventRecord(ctx->ev[g][0], ctx->stream)); }
        cudaError_t e = cudaSuccess;
        double* d_stage = (double*)ctx->stage.p + (size_t)R.n_series * P->cum[g];      // this group's staging matrix
        const int g_ncols = (int)P->host[g].size();
        switch (g) {
            case G_BASIC: {
                if (P->basic_moments_only) {
                    // reductions only: stream the series from HBM; with no other group in the plan the rows go
                    // straight into the caller's matrix (no staging, no assemble pass)
                    MomentsArgs M;
                    M.R = R; M.descs = P->dev[g]; M.nd = g_ncols; M.need_high = P->moments_need_high;
                    direct = (P->n_groups_used == 1) && ctx->peer_out.empty() && (P->ncols == g_ncols);
                    M.out = direct ? d_final : d_stage;
                    M.ncols = direct ? ld : g_ncols;
                    M.colmap = direct ? P->d_final_col + P->cum[g] : nullptr;
                    e = launch_moments(M, ctx->stream, ctx->sm_count);
                    ctx->used_moments = true;
                    break;
                }
                BasicArgs A;
                A.R = R; A.gscratch = gscratch; A.gscratch_bytes = gscratch_bytes; A.descs = P->dev[g]; A.nd = (int)P->host[g].size(); A.out = d_stage; A.ncols = g_ncols;
                A.lag_needed = P->lag_needed;
                A.nfin = P->basic_nfin;
                int pac = P->pacf_want >= 0 ? 4 * (P->pacf_want + 1) : 0;
                A.pacf_off = P->lag_needed + 1;
                A.nlag = even(P->lag_needed + 1 + pac);
                A.nscr = even(std::max(std::max(max_len, 64), (P->basic_bins + 1) / 2));
                A.nalt = 0;
                {
                    int prev = -1;
                    for (const Desc& q : P->host[g])
                        if (q.calc == TSFX_AGG_LINEAR_TREND) {
                            const int key = (q.i0 << 4) | q.i1;
                            if (key != prev) { ++A.nalt; prev = key; }
                        }
                }
                A.dec = ctx->d_dec;
                e = launch_basic(A, max_len, ctx->stream, ctx->sm_count);
                break;
            }
            case G_SORTED: {
                SortedArgs A;
                A.R = R; A.gscratch = gscratch; A.gscratch_bytes = gscratch_bytes; A.descs = P->dev[g]; A.nd = (int)P->host[g].size(); A.out = d_stage; A.ncols = g_ncols;
                A.nscr = even(4 * (P->friedrich_r + 2) + 16);
                A.nfin = P->sorted_nfin;
                A.ncq = 0;
                {
                    double pl = -1.0, ph = -1.0;
                    for (const Desc& q : P->host[g])
                        if (q.calc == TSFX_CHANGE_QUANTILES && !(q.p0 == pl && q.p1 == ph)) { ++A.ncq; pl = q.p0; ph = q.p1; }
                }
                e = launch_sorted(A, max_len, ctx->stream, ctx->sm_count);
                break;
            }
            case G_SPECTRAL: {
                SpectralArgs A;
                A.R = R; A.gscratch = gscratch; A.gscratch_bytes = gscratch_bytes; A.descs = P->dev[g]; A.nd = (int)P->host[g].size(); A.out = d_stage; A.ncols = g_ncols;
                A.twiddle = ctx->d_tw; A.tw_n = ctx->tw_n;
                A.tables = P->d_tables; A.table_off = P->d_toff; A.table_half = P->d_thalf;
                A.need_fft = P->need_fft; A.need_welch = P->need_welch;
                A.max_hist = P->fourier_bins;
                A.nfft = P->spectral_nfft;
                e = launch_spectral(A, max_len, ctx->stream, ctx->sm_count);
                break;
            }
            case G_LA: {
                LaArgs A;
                A.R = R; A.gscratch = gscratch; A.gscratch_bytes = gscratch_bytes; A.descs = P->dev[g]; A.nd = (int)P->host[g].size(); A.out = d_stage; A.ncols = g_ncols;
                A.nscr = P->max_ar_k;
                e = launch_la(A, max_len, ctx->stream, ctx->sm_count);
                break;
            }
            case G_ENTROPY: {
                EntropyArgs A;
                A.R = R; A.gscratch = gscratch; A.gscratch_bytes = gscratch_bytes; A.descs = P->dev[g]; A.nd = (int)P->host[g].size(); A.out = d_stage; A.ncols = g_ncols;
                e = launch_entropy(A, max_len, ctx->stream, ctx->sm_count);
                break;
            }
            case G_SEQ: {
                SeqArgs A;
                A.R = R; A.gscratch = gscratch; A.gscratch_bytes = gscratch_bytes; A.descs = P->dev[g]; A.nd = (int)P->host[g].size(); A.out = d_stage; A.ncols = g_ncols;
                A.nscr = (P->max_lz_bins > 0 ? 1 : 0) | (P->max_perm_dim > 0 ? 2 : 0) | (P->max_cwt_peaks_n << 8) |
                         (std::min(P->n_lz, 255) << 16) | (std::min(P->max_lz_bins, 255) << 24);
                e = launch_seq(A, max_len, ctx->stream, ctx->sm_count);
                break;
            }
            case G_PEAKS: {
                SeqArgs A;
                A.R = R; A.gscratch = gscratch; A.gscratch_bytes = gscratch_bytes; A.descs = P->dev[g]; A.nd = (int)P->host[g].size(); A.out = d_stage; A.ncols = g_ncols;
                A.nscr = (P->max_cwt_peaks_n << 8);
                e = launch_peaks(A, max_len, ctx->stream, ctx->sm_count);
                break;
            }
        }
        if (e == cudaErrorInvalidConfiguration) return too_long(kGroupNames[g]);
        if (e != cudaSuccess) return fail(ctx, TSFX_E_CUDA, std::string("launch ") + kGroupNames[g] + ": " + cudaGetErrorString(e));
        ctx->launches += 1;
        if (timing) { CK(cudaEventRecord(ctx->ev[g][1], ctx->stream)); ctx->ev_used[g] = true; }
    }
    if (!direct) {   // scatter the staging matrices into the caller's [n_series x ncols] matrix
        if (timing) { CK(cudaEventRecord(ctx->ev[G_COUNT][0], ctx->stream)); }
        AssembleArgs A;
        A.stage = (const double*)ctx->stage.p; A.out = d_final; A.n_series = R.n_series; A.ncols = P->ncols; A.ld = ld;
        if (ld != P->ncols && !ctx->peer_out.empty()) return fail(ctx, TSFX_E_UNSUPPORTED, "peer placement of a strided matrix");
        A.n_groups = G_COUNT;
        for (int g = 0; g <= G_COUNT; ++g) A.cum[g] = P->cum[g];
        A.final_col = P->d_final_col;
        A.n_extra = 0;
        A.out_mc = nullptr;
        // multi-GPU placement: where does this row block live inside the peers' copies of the result matrix?
        int64_t peer_off = -1;                 // byte offset of d_final inside this rank's mapped matrix
        if (!ctx->peer_out.empty()) {
            const uint64_t self = ctx->peer_out[ctx->peer_self];
            if ((uint64_t)d_final < self) return fail(ctx, TSFX_E_INVALID, "out is not inside the matrix registered with tsfx_set_peer_outputs");
            peer_off = (int64_t)((uint64_t)d_final - self);
            if (ctx->peer_mode == TSFX_PEER_MULTICAST) A.out_mc = (double*)(ctx->peer_mc + (uint64_t)peer_off);
            else if (ctx->peer_mode == TSFX_PEER_STORE)
                for (size_t p = 0; p < ctx->peer_out.size(); ++p)
                    if ((int)p != ctx->peer_self) A.extra[A.n_extra++] = (double*)(ctx->peer_out[p] + (uint64_t)peer_off);
        }
        cudaError_t e = launch_assemble(A, ctx->stream, ctx->sm_count);
        if (e != cudaSuccess) return fail(ctx, TSFX_E_CUDA, std::string("launch assemble: ") + cudaGetErrorString(e));
        ctx->launches += 1;
        if (timing) { CK(cudaEventRecord(ctx->ev[G_COUNT][1], ctx->stream)); ctx->ev_used[G_COUNT] = true; }
        if (peer_off >= 0 && ctx->peer_mode == TSFX_PEER_COPY) {
            // copy engines push the finished row block to every peer while the next block's kernels run
            const size_t bytes = (size_t)R.n_series * P->ncols * sizeof(double);
            CK(cudaEventRecord(ctx->ev_peer, ctx->stream));
            CK(cudaStreamWaitEvent(ctx->s_peer, ctx->ev_peer, 0));
            const size_t np = ctx->peer_out.size();
            for (size_t k = 1; k < np; ++k) {          // start with the next rank so the ranks do not all hit one peer
                const size_t p = ((size_t)ctx->peer_self + k) % np;
                CK(cudaMemcpyAsync((void*)(ctx->peer_out[p] + (uint64_t)peer_off), d_final, bytes, cudaMemcpyDeviceToDevice, ctx->s_peer));
            }
        }
    }
    return TSFX_OK;
}

static int impute_after_extract(tsfx_ctx* ctx, double* d_out, int64_t rows, int cols);
static int nan_error(tsfx_ctx* ctx);

static int check_args(tsfx_ctx* ctx, const tsfx_plan* plan, const void* values, const void* out, int64_t n_series) {
    if (!ctx) return TSFX_E_INVALID;
    if (!plan || plan->ctx != ctx) return fail(ctx, TSFX_E_INVALID, "plan does not belong to this context");
    if (n_series < 0) return fail(ctx, TSFX_E_INVALID, "n_series < 0");
    if (n_series > 0 && (!values || !out)) return fail(ctx, TSFX_E_INVALID, "NULL values/out");
    return TSFX_OK;
}

extern "C" int tsfx_extract_csr(tsfx_ctx* ctx, const tsfx_plan* plan, const float* values, int64_t n_values,
                                const int64_t* begin, const int32_t* len, int64_t n_series, double* out,
                                uint32_t flags) {
    int rc = check_args(ctx, plan, values, out, n_series);
    if (rc) return rc;
    if (n_series == 0) return TSFX_OK;
    if (!begin || !len) return fail(ctx, TSFX_E_INVALID, "NULL begin/len");
    CK(cudaSetDevice(ctx->device));
    SeriesRef R;
    R.dense_len = 0;
    R.n_series = n_series;
    rc = take_times(ctx, plan, n_values, &R.times);
    if (rc) return rc;
    int max_len = 0;
    if (flags & TSFX_FLAG_DEVICE_PTRS) {
        R.values = values; R.begin = begin; R.len = len;
        if (ctx->max_len_hint > 0) max_len = ctx->max_len_hint;       // stays asynchronous
        else {
            int rc2 = csr_max_len(ctx->csr, len, n_series, ctx->stream, &max_len);
            if (rc2) return fail(ctx, TSFX_E_CUDA, "max-length reduction failed");
        }
        rc = run_groups(ctx, plan, R, max_len, out, flags);
        if (!rc && (flags & TSFX_FLAG_IMPUTE)) rc = impute_after_extract(ctx, out, n_series, plan->ncols);
        return rc;
    }
    for (int64_t s = 0; s < n_series; ++s) {
        if (len[s] < 1 || begin[s] < 0 || begin[s] + len[s] > n_values)
            return fail(ctx, TSFX_E_INVALID, "series " + std::to_string(s) + " has an invalid (begin, len)");
        max_len = std::max(max_len, (int)len[s]);
    }
    size_t ob = (size_t)n_series * plan->ncols * sizeof(double);
    CK(ctx->values.reserve((size_t)n_values * sizeof(float) + 16));
    CK(ctx->begin.reserve((size_t)n_series * sizeof(int64_t)));
    CK(ctx->len.reserve((size_t)n_series * sizeof(int32_t)));
    CK(ctx->out.reserve(std::max<size_t>(ob, 8)));
    CK(cudaMemcpyAsync(ctx->values.p, values, (size_t)n_values * sizeof(float), cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaMemcpyAsync(ctx->begin.p, begin, (size_t)n_series * sizeof(int64_t), cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaMemcpyAsync(ctx->len.p, len, (size_t)n_series * sizeof(int32_t), cudaMemcpyHostToDevice, ctx->stream));
    R.values = (const float*)ctx->values.p; R.begin = (const int64_t*)ctx->begin.p; R.len = (const int32_t*)ctx->len.p;
    const bool check_nan = !(flags & TSFX_FLAG_NO_NAN_CHECK);
    if (check_nan) {
        CK(ctx->csr.init_info());
        CK(cudaMemsetAsync(ctx->csr.d_info, 0, sizeof(CsrInfo), ctx->stream));
        csr_check_nan(ctx->csr, R.values, n_values, ctx->stream);
        CK(cudaMemcpyAsync(ctx->csr.h_info, ctx->csr.d_info, sizeof(CsrInfo), cudaMemcpyDeviceToHost, ctx->stream));
    }
    rc = run_groups(ctx, plan, R, max_len, (double*)ctx->out.p, flags);
    if (rc) return rc;
    if (flags & TSFX_FLAG_IMPUTE) { rc = impute_after_extract(ctx, (double*)ctx->out.p, n_series, plan->ncols); if (rc) return rc; }
    CK(cudaMemcpyAsync(out, ctx->out.p, ob, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    if (check_nan && ctx->csr.h_info->has_nan) return nan_error(ctx);
    return TSFX_OK;
}

extern "C" int tsfx_extract_dense(tsfx_ctx* ctx, const tsfx_plan* plan, const float* values, int64_t n_series,
                                  int32_t len, double* out, uint32_t flags) {
    int rc = check_args(ctx, plan, values, out, n_series);
    if (rc) return rc;
    if (n_series == 0) return TSFX_OK;
    if (len < 1) return fail(ctx, TSFX_E_INVALID, "len < 1");
    CK(cudaSetDevice(ctx->device));
    SeriesRef R;
    R.begin = nullptr; R.len = nullptr; R.dense_len = len; R.n_series = n_series;
    const int64_t* all_times = nullptr;
    rc = take_times(ctx, plan, n_series * (int64_t)len, &all_times);
    if (rc) return rc;
    R.times = all_times;
    if (flags & TSFX_FLAG_DEVICE_PTRS) {
        R.values = values;
        rc = run_groups(ctx, plan, R, len, out, flags);
        if (!rc && (flags & TSFX_FLAG_IMPUTE)) rc = impute_after_extract(ctx, out, n_series, plan->ncols);
        return rc;
    }
    // host path: pipelined over row blocks -- the H2D copy of block b+1 and the D2H copy of block b-1 run on
    // their own streams while the kernels of block b execute (pinned host buffers make the copies truly async)
    const size_t ncols = (size_t)plan->ncols;
    const size_t vb = (size_t)n_series * len * sizeof(float), ob = (size_t)n_series * ncols * sizeof(double);
    CK(ctx->values.reserve(vb + 16));
    CK(ctx->out.reserve(std::max<size_t>(ob, 8)));
    int64_t block = std::max<int64_t>(16384, (n_series + 15) / 16);
    if (flags & TSFX_FLAG_TIMING) block = n_series;            // per-group events describe one whole pass
    float* dv = (float*)ctx->values.p;
    double* dout = (double*)ctx->out.p;
    const bool check_nan = !(flags & TSFX_FLAG_NO_NAN_CHECK);
    if (check_nan) { CK(ctx->csr.init_info()); CK(cudaMemsetAsync(ctx->csr.d_info, 0, sizeof(CsrInfo), ctx->stream)); }
    int nb = 0;
    for (int64_t lo = 0; lo < n_series; lo += block, ++nb) {
        const int64_t cnt = std::min<int64_t>(block, n_series - lo);
        const int slot = nb & 1;
        CK(ctx->stager.h2d(dv + (size_t)lo * len, values + (size_t)lo * len, (size_t)cnt * len * sizeof(float), ctx->s_in));
        CK(cudaEventRecord(ctx->ev_in[slot], ctx->s_in));
        CK(cudaStreamWaitEvent(ctx->stream, ctx->ev_in[slot], 0));
        if (check_nan) csr_check_nan(ctx->csr, dv + (size_t)lo * len, cnt * len, ctx->stream);
        R.values = dv + (size_t)lo * len;
        R.times = all_times ? all_times + (size_t)lo * len : nullptr;
        R.n_series = cnt;
        rc = run_groups(ctx, plan, R, len, dout + (size_t)lo * ncols, flags);
        if (rc) return rc;
        if (flags & TSFX_FLAG_IMPUTE) continue;         // column statistics need every row: one copy at the end
        CK(cudaEventRecord(ctx->ev_done[slot], ctx->stream));
        CK(cudaStreamWaitEvent(ctx->s_out, ctx->ev_done[slot], 0));
        CK(cudaMemcpyAsync(out + (size_t)lo * ncols, dout + (size_t)lo * ncols, (size_t)cnt * ncols * sizeof(double),
                           cudaMemcpyDeviceToHost, ctx->s_out));
    }
    if (flags & TSFX_FLAG_IMPUTE) {
        rc = impute_after_extract(ctx, dout, n_series, plan->ncols);
        if (rc) return rc;
        CK(cudaMemcpyAsync(out, dout, ob, cudaMemcpyDeviceToHost, ctx->stream));
    }
    if (check_nan) CK(cudaMemcpyAsync(ctx->csr.h_info, ctx->csr.d_info, sizeof(CsrInfo), cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->s_out));
    CK(cudaStreamSynchronize(ctx->stream));
    if (check_nan && ctx->csr.h_info->has_nan) return nan_error(ctx);
    return TSFX_OK;
}

// impute the device matrix of the extract call that just ran (TSFX_FLAG_IMPUTE)
static int impute_after_extract(tsfx_ctx* ctx, double* d_out, int64_t rows, int cols) {
    int n = 0;
    cudaError_t e = impute_device(ctx->imp, d_out, rows, cols, TSFX_IMPUTE_RANGE, false, nullptr, ctx->sm_count, ctx->stream, &n);
    if (e != cudaSuccess) return fail(ctx, TSFX_E_CUDA, std::string("impute: ") + cudaGetErrorString(e));
    ctx->launches += n;
    return TSFX_OK;
}

extern "C" int tsfx_impute(tsfx_ctx* ctx, double* matrix, int64_t n_rows, int32_t n_cols, int32_t mode, double* col_stats,
                           uint32_t flags) {
    if (!ctx) return TSFX_E_INVALID;
    if (n_rows < 0 || n_cols < 0 || mode < TSFX_IMPUTE_RANGE || mode > TSFX_IMPUTE_STATS)
        return fail(ctx, TSFX_E_INVALID, "tsfx_impute: bad arguments");
    if (n_rows == 0 || n_cols == 0) return TSFX_OK;
    if (!matrix) return fail(ctx, TSFX_E_INVALID, "tsfx_impute: NULL matrix");
    if ((mode == TSFX_IMPUTE_GIVEN || mode == TSFX_IMPUTE_STATS) && !col_stats)
        return fail(ctx, TSFX_E_INVALID, "tsfx_impute: col_stats is required for this mode");
    if (mode == TSFX_IMPUTE_GIVEN)
        for (int64_t i = 0; i < (int64_t)3 * n_cols; ++i)
            if (!std::isfinite(col_stats[i]))       // dataframe_functions.py:147-156 raises ValueError
                return fail(ctx, TSFX_E_INVALID, "tsfx_impute: non-finite replacement value");
    CK(cudaSetDevice(ctx->device));
    const size_t bytes = (size_t)n_rows * n_cols * sizeof(double);
    double* d_m = matrix;
    const bool host = !(flags & TSFX_FLAG_DEVICE_PTRS);
    if (host) {
        CK(ctx->out.reserve(bytes));
        d_m = (double*)ctx->out.p;
        CK(cudaMemcpyAsync(d_m, matrix, bytes, cudaMemcpyHostToDevice, ctx->stream));
    }
    int n = 0;
    cudaError_t e = impute_device(ctx->imp, d_m, n_rows, n_cols, mode, (flags & TSFX_FLAG_ALL_MEDIANS) != 0 || mode == TSFX_IMPUTE_STATS,
                                  col_stats, ctx->sm_count, ctx->stream, &n);
    if (e != cudaSuccess) return fail(ctx, TSFX_E_CUDA, std::string("impute: ") + cudaGetErrorString(e));
    ctx->launches = n;
    if (host) {
        if (mode != TSFX_IMPUTE_STATS) CK(cudaMemcpyAsync(matrix, d_m, bytes, cudaMemcpyDeviceToHost, ctx->stream));
        CK(cudaStreamSynchronize(ctx->stream));
    }
    return TSFX_OK;
}

extern "C" int tsfx_get_timings(tsfx_ctx* ctx, float* ms_out, const char** names_out, int32_t cap) {
    if (!ctx) return TSFX_E_INVALID;
    CK(cudaSetDevice(ctx->device));
    CK(cudaStreamSynchronize(ctx->stream));
    int k = 0;
    for (int g = 0; g < G_EVENTS && k < cap; ++g) {
        if (!ctx->ev_used[g]) continue;
        float ms = 0.f;
        CK(cudaEventElapsedTime(&ms, ctx->ev[g][0], ctx->ev[g][1]));
        if (ms_out) ms_out[k] = ms;
        if (names_out) names_out[k] = (g == G_BASIC && ctx->used_moments) ? "moments" : kGroupNames[g];
        ++k;
    }
    return k;
}

extern "C" int tsfx_last_launch_count(const tsfx_ctx* ctx) { return ctx ? ctx->launches : 0; }

// ------------------------------------------------------------------------------------------ stage (a)
// Long frame -> device CSR -> kernels, pipelined.  See tsfx_csr.h for the two paths.  `in` columns are host pointers
// (copied through Stager::h2d: pinned sources go straight to cudaMemcpyAsync, pageable ones through the pinned ring)
// or, with TSFX_FLAG_DEVICE_PTRS, device pointers that are used in place.
struct LongIn {
    const int64_t* ids;
    const void* keys;
    int is_f64;
    const float* values;           // value column of kind 0
    int64_t n;
    bool device;
    const float* const* more = nullptr;   // value columns of kinds 1 .. n_kinds-1 (wide format: the kinds share ids and sort keys)
    int n_kinds = 1;
    const float* col(int k) const { return k == 0 ? values : more[k - 1]; }
};

static inline size_t kind_stride(int64_t n) { return ((size_t)n + 3) & ~(size_t)3; }   // floats between the kinds' device columns

static int nan_error(tsfx_ctx* ctx) { return fail(ctx, TSFX_E_NAN, "the value column contains NaN"); }

// Brings the frame into CSR form on the device (sizes in *info).  When the rows arrive ordered and the input is on
// the host, only the id column has been copied on return (*streamed = true): the caller streams the other columns.
static int stage_a(tsfx_ctx* ctx, const LongIn& in, int max_blocks, bool check_nan, CsrInfo* info, bool* streamed,
                   const int64_t** d_ids_out, const uint64_t** d_keys_out, const float** d_vals_out) {
    CsrWorkspace& W = ctx->csr;
    std::string msg;
    const int64_t n = in.n;
    const int64_t* d_ids = in.ids;
    const uint64_t* d_keys = (const uint64_t*)in.keys;
    const float* d_vals = in.values;
    if (!in.device) {
        CK(W.reserve(0, (size_t)n * 8));
        CK(W.reserve(2, (size_t)n * 4 + 16));
        if (in.keys) CK(W.reserve(1, (size_t)n * 8));
        CK(ctx->stager.h2d(W.ids(), in.ids, (size_t)n * 8, ctx->stream));
        d_ids = W.ids();
        d_keys = in.keys ? W.keys() : nullptr;
        d_vals = W.vals();
    }
    int rc = csr_ids_pass(W, d_ids, n, 16384, max_blocks, ctx->stream, &msg);
    if (rc) return fail(ctx, rc, msg);
    CK(cudaStreamSynchronize(ctx->stream));
    *info = *W.h_info;
    *streamed = false;
    if (!info->unsorted_ids) {
        W.d_values = const_cast<float*>(d_vals);
        if (!in.device) *streamed = true;
        else csr_check_rows(W, d_ids, d_keys, in.is_f64, d_vals, 0, n, check_nan, ctx->stream);   // result read by the caller
    }
    *d_ids_out = d_ids; *d_keys_out = d_keys; *d_vals_out = d_vals;
    return TSFX_OK;
}

// rows in arbitrary order: (copy the remaining columns,) sort, rebuild the CSR
static int stage_a_sort(tsfx_ctx* ctx, const LongIn& in, int max_blocks, bool check_nan, CsrInfo* info,
                        const int64_t* d_ids, const uint64_t* d_keys, const float* d_vals) {
    CsrWorkspace& W = ctx->csr;
    std::string msg;
    if (!in.device) {
        if (in.keys) CK(ctx->stager.h2d(W.keys(), in.keys, (size_t)in.n * 8, ctx->stream));
        CK(ctx->stager.h2d(W.vals(), in.values, (size_t)in.n * 4, ctx->stream));
    }
    int rc = csr_sort_pass(W, d_ids, d_keys, in.is_f64, d_vals, in.n, 16384, max_blocks, check_nan, ctx->stream, &msg);
    if (rc) return fail(ctx, rc, msg);
    CK(cudaStreamSynchronize(ctx->stream));
    *info = *W.h_info;
    return TSFX_OK;
}

extern "C" int tsfx_build_csr(tsfx_ctx* ctx, const int64_t* ids, const void* sort_keys, int32_t sort_key_is_f64,
                              const float* values, int64_t n_rows, int64_t* out_ids, int64_t* out_begin,
                              int32_t* out_len, float* sorted_values, int64_t out_capacity, int64_t* n_series_out) {
    if (!ctx) return TSFX_E_INVALID;
    if (n_rows < 0 || !n_series_out || (n_rows > 0 && (!ids || !values)))
        return fail(ctx, TSFX_E_INVALID, "tsfx_build_csr: bad arguments");
    CK(cudaSetDevice(ctx->device));
    *n_series_out = 0;
    if (n_rows == 0) return TSFX_OK;
    ctx->held_series = -1;
    LongIn in{ids, sort_keys, sort_key_is_f64, values, n_rows, false};
    CsrInfo info;
    bool streamed = false;
    const int64_t* d_ids; const uint64_t* d_keys; const float* d_vals;
    int rc = stage_a(ctx, in, 1, true, &info, &streamed, &d_ids, &d_keys, &d_vals);
    if (rc) return rc;
    CsrWorkspace& W = ctx->csr;
    bool need_sort = info.unsorted_ids != 0;
    if (!need_sort) {        // ids ascending: bring the other columns over and look inside the ids
        if (sort_keys) CK(ctx->stager.h2d(W.keys(), sort_keys, (size_t)n_rows * 8, ctx->stream));
        CK(ctx->stager.h2d(W.vals(), values, (size_t)n_rows * 4, ctx->stream));
        csr_check_rows(W, d_ids, d_keys, sort_key_is_f64, d_vals, 0, n_rows, true, ctx->stream);
        CK(cudaMemcpyAsync(W.h_info, W.d_info, sizeof(CsrInfo), cudaMemcpyDeviceToHost, ctx->stream));
        CK(cudaStreamSynchronize(ctx->stream));
        info = *W.h_info;
        need_sort = info.unsorted_keys != 0;
        if (need_sort) {     // columns are resident now: sort in place
            LongIn dev{d_ids, d_keys, sort_key_is_f64, d_vals, n_rows, true};
            rc = stage_a_sort(ctx, dev, 1, true, &info, d_ids, d_keys, d_vals);
            if (rc) return rc;
        }
    } else {
        rc = stage_a_sort(ctx, in, 1, true, &info, d_ids, d_keys, d_vals);
        if (rc) return rc;
    }
    if (info.has_nan) return nan_error(ctx);
    const int64_t ns = info.n_series;
    ctx->held_series = ns;
    ctx->held_max_len = info.max_len;
    *n_series_out = ns;
    if (!out_ids && !out_begin && !out_len && !sorted_values) return TSFX_OK;      // count + keep on device
    if (ns > out_capacity) return fail(ctx, TSFX_E_INVALID, "out_capacity too small: " + std::to_string(ns) + " series");
    if (out_ids) CK(cudaMemcpyAsync(out_ids, W.d_uid, ns * sizeof(int64_t), cudaMemcpyDeviceToHost, ctx->stream));
    if (out_begin) CK(cudaMemcpyAsync(out_begin, W.d_begin, ns * sizeof(int64_t), cudaMemcpyDeviceToHost, ctx->stream));
    if (out_len) CK(cudaMemcpyAsync(out_len, W.d_len, ns * sizeof(int32_t), cudaMemcpyDeviceToHost, ctx->stream));
    if (sorted_values) CK(cudaMemcpyAsync(sorted_values, W.d_values, n_rows * sizeof(float), cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    return TSFX_OK;
}

// the kinds of one call: plan, device value column (CSR order) and first output column of each
#define TSFX_MAX_KINDS 64
struct KindSet {
    int n = 1;
    const tsfx_plan* plan[TSFX_MAX_KINDS];
    const float* dvals[TSFX_MAX_KINDS];
    int col0[TSFX_MAX_KINDS];
    int total_cols = 0;
};

// kernels + result transfer over the row blocks of a device CSR.  stream_in: the key / value rows of a block are
// copied from the host right before the block's kernels (fast path); d_out == nullptr: results go through ctx->out
// and are copied to `out` (host) block by block on the D2H stream.  Several kinds (wide format) share the CSR: every
// block runs each kind's plan on that kind's value column and writes its own column block of the one result matrix.
static int run_blocks(tsfx_ctx* ctx, const KindSet& K, const CsrInfo& info, const LongIn* stream_in,
                      const int64_t* d_ids, const uint64_t* d_keys, bool check_rows, bool check_nan,
                      double* out, bool out_is_device, uint32_t flags, const int64_t* row_times = nullptr) {
    CsrWorkspace& W = ctx->csr;
    const size_t ncols = (size_t)K.total_cols;
    const int64_t ns = info.n_series;
    double* dout = out;
    if (!out_is_device) {
        CK(ctx->out.reserve(std::max<size_t>((size_t)ns * ncols * sizeof(double), 8)));
        dout = (double*)ctx->out.p;
    }
    const bool impute = (flags & TSFX_FLAG_IMPUTE) != 0;
    for (int b = 0; b < info.n_blocks; ++b) {
        const int64_t s0 = info.series_lo[b], s1 = info.series_lo[b + 1];
        const int64_t r0 = info.row_lo[b], r1 = info.row_lo[b + 1];
        const int slot = b & 1;
        if (stream_in) {
            if (stream_in->keys) CK(ctx->stager.h2d(W.keys() + r0, (const uint64_t*)stream_in->keys + r0, (size_t)(r1 - r0) * 8, ctx->s_in));
            for (int k = 0; k < K.n; ++k)
                CK(ctx->stager.h2d(const_cast<float*>(K.dvals[k]) + r0, stream_in->col(k) + r0, (size_t)(r1 - r0) * 4, ctx->s_in));
            CK(cudaEventRecord(ctx->ev_in[slot], ctx->s_in));
            CK(cudaStreamWaitEvent(ctx->stream, ctx->ev_in[slot], 0));
        }
        if (check_rows) {
            csr_check_rows(W, d_ids, d_keys, stream_in ? stream_in->is_f64 : 0, K.dvals[0], r0, r1, check_nan, ctx->stream);
            if (check_nan) for (int k = 1; k < K.n; ++k) csr_check_nan(W, K.dvals[k] + r0, r1 - r0, ctx->stream);
        }
        for (int k = 0; k < K.n; ++k) {
            if (K.plan[k]->ncols == 0) continue;
            SeriesRef R;
            R.values = K.dvals[k]; R.begin = W.d_begin + s0; R.len = W.d_len + s0; R.dense_len = 0; R.n_series = s1 - s0;
            R.times = row_times;
            int rc = run_groups(ctx, K.plan[k], R, info.max_len, dout + (size_t)s0 * ncols + K.col0[k], flags, K.total_cols);
            if (rc) return rc;
        }
        if (impute || out_is_device) continue;
        CK(cudaEventRecord(ctx->ev_done[slot], ctx->stream));
        CK(cudaStreamWaitEvent(ctx->s_out, ctx->ev_done[slot], 0));
        CK(cudaMemcpyAsync(out + (size_t)s0 * ncols, dout + (size_t)s0 * ncols, (size_t)(s1 - s0) * ncols * sizeof(double),
                           cudaMemcpyDeviceToHost, ctx->s_out));
    }
    if (impute) {
        int rc = impute_after_extract(ctx, dout, ns, K.total_cols);
        if (rc) return rc;
        if (!out_is_device) CK(cudaMemcpyAsync(out, dout, (size_t)ns * ncols * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    }
    return TSFX_OK;
}

static int extract_long_impl(tsfx_ctx* ctx, const tsfx_plan* const* plans, const LongIn& in, int64_t* out_ids, double* out,
                             int64_t out_capacity, int64_t** out_ids_alloc, double** out_alloc, int64_t* n_series_out,
                             uint32_t flags) {
    CsrWorkspace& W = ctx->csr;
    const tsfx_plan* plan = plans[0];
    KindSet K;
    K.n = in.n_kinds;
    if (K.n < 1 || K.n > TSFX_MAX_KINDS) return fail(ctx, TSFX_E_INVALID, "between 1 and 64 kinds per call");
    for (int k = 0; k < K.n; ++k) {
        if (!plans[k] || plans[k]->ctx != ctx) return fail(ctx, TSFX_E_INVALID, "plan does not belong to this context");
        K.plan[k] = plans[k];
        K.col0[k] = K.total_cols;
        K.total_cols += plans[k]->ncols;
    }
    for (int k = 0; k < K.n; ++k) if (plans[k]->need_times) plan = plans[k];      // take_times looks at one plan's flag
    const size_t kstride = kind_stride(in.n);
    if (K.n > 1 && !in.device) CK(ctx->kvals.reserve((size_t)(K.n - 1) * kstride * 4 + 16));
    const bool check_nan = !(flags & TSFX_FLAG_NO_NAN_CHECK);
    const int max_blocks = (flags & TSFX_FLAG_TIMING) ? 1 : 16;
    ctx->held_series = -1;
    const int64_t* times_in = nullptr;           // row timestamps (input row order), device
    int rc = take_times(ctx, plan, in.n, &times_in);
    if (rc) return rc;
    CsrInfo info;
    bool streamed = false;
    const int64_t* d_ids; const uint64_t* d_keys; const float* d_vals;
    rc = stage_a(ctx, in, max_blocks, check_nan, &info, &streamed, &d_ids, &d_keys, &d_vals);
    if (rc) return rc;
    bool sorted = !info.unsorted_ids;
    bool extra_resident = in.device;              // value columns of kinds 1.. are on the device in input order
    auto extra_in = [&](int k) -> const float* {  // device column of kind k >= 1, input row order
        return in.device ? in.col(k) : (const float*)ctx->kvals.p + (size_t)(k - 1) * kstride;
    };
    if (sorted && in.device && check_nan)
        for (int k = 1; k < K.n; ++k) csr_check_nan(W, in.col(k), in.n, ctx->stream);
    for (int attempt = 0; attempt < 2; ++attempt) {
        if (!sorted) {
            rc = stage_a_sort(ctx, in, max_blocks, check_nan, &info, d_ids, d_keys, d_vals);
            if (rc) return rc;
            if (info.has_nan) return nan_error(ctx);
        }
        // device value column of every kind in CSR order
        K.dvals[0] = W.d_values;
        if (K.n > 1) {
            if (W.d_perm) {                       // rows were sorted on the device: the other kinds follow the permutation
                CK(ctx->kvals_sorted.reserve((size_t)(K.n - 1) * kstride * 4 + 16));
                for (int k = 1; k < K.n; ++k) {
                    if (!extra_resident) CK(ctx->stager.h2d(const_cast<float*>(extra_in(k)), in.col(k), (size_t)in.n * 4, ctx->stream));
                    if (check_nan) csr_check_nan(W, extra_in(k), in.n, ctx->stream);
                    float* dst = (float*)ctx->kvals_sorted.p + (size_t)(k - 1) * kstride;
                    csr_gather_f32(W, extra_in(k), dst, in.n, ctx->stream);
                    K.dvals[k] = dst;
                }
                extra_resident = true;
            } else {
                for (int k = 1; k < K.n; ++k) K.dvals[k] = extra_in(k);
            }
        }
        const int64_t ns = info.n_series;
        *n_series_out = ns;
        const size_t ob = (size_t)ns * K.total_cols * sizeof(double);
        if (out_alloc) {                         // library-sized result from the pinned pool
            if (!*out_alloc) {
                *out_alloc = (double*)ctx->pool.alloc(std::max<size_t>(ob, 8));
                *out_ids_alloc = (int64_t*)ctx->pool.alloc(std::max<size_t>((size_t)ns * 8, 8));
                if (!*out_alloc || !*out_ids_alloc) return fail(ctx, TSFX_E_NOMEM, "pinned host allocation failed");
            }
            out = *out_alloc;
            out_ids = *out_ids_alloc;
        } else if (ns > out_capacity) {
            return fail(ctx, TSFX_E_INVALID, "out_capacity too small: " + std::to_string(ns) + " series");
        }
        if (info.max_len < 1 && ns > 0) return fail(ctx, TSFX_E_INVALID, "empty series");
        const bool first_sorted_try = sorted && attempt == 0;
        const int64_t* row_times = times_in;
        if (times_in && W.d_perm) {               // the rows were sorted on the device: the timestamps follow
            CK(ctx->times_sorted.reserve((size_t)in.n * 8));
            csr_gather_i64(W, times_in, (int64_t*)ctx->times_sorted.p, in.n, ctx->stream);
            row_times = (const int64_t*)ctx->times_sorted.p;
        }
        rc = run_blocks(ctx, K, info, (first_sorted_try && streamed) ? &in : nullptr, d_ids, d_keys,
                        /*check_rows=*/first_sorted_try && streamed, check_nan, out, in.device, flags, row_times);
        if (first_sorted_try && streamed) extra_resident = true;
        if (rc) return rc;
        if (out_ids) CK(cudaMemcpyAsync(out_ids, W.d_uid, (size_t)ns * sizeof(int64_t), in.device ? cudaMemcpyDeviceToDevice : cudaMemcpyDeviceToHost, ctx->stream));
        if (in.device && !first_sorted_try) break;                       // asynchronous contract: nothing to wait for
        // the NaN scans of the other kinds' columns were queued after the sort pass read its flags: read them again
        const bool late_nan_flags = !first_sorted_try && K.n > 1 && check_nan;
        if (first_sorted_try || late_nan_flags) CK(cudaMemcpyAsync(W.h_info, W.d_info, sizeof(CsrInfo), cudaMemcpyDeviceToHost, ctx->stream));
        CK(cudaStreamSynchronize(ctx->s_out));
        CK(cudaStreamSynchronize(ctx->stream));
        if (late_nan_flags && W.h_info->has_nan) return nan_error(ctx);
        if (!first_sorted_try) break;
        if (W.h_info->has_nan) return nan_error(ctx);
        if (!W.h_info->unsorted_keys) break;
        // ids ascending but some sort key decreases inside an id: the columns are resident now, sort and run again
        sorted = false;
        if (!in.device) {
            LongIn dev{d_ids, d_keys, in.is_f64, d_vals, in.n, true};
            rc = stage_a_sort(ctx, dev, max_blocks, check_nan, &info, d_ids, d_keys, d_vals);
            if (rc) return rc;
            if (info.has_nan) return nan_error(ctx);
            sorted = true;                        // CSR rebuilt: second trip only runs the kernels
            streamed = false;
        }
    }
    ctx->held_series = info.n_series;
    ctx->held_max_len = info.max_len;
    return TSFX_OK;
}

extern "C" int tsfx_extract_long(tsfx_ctx* ctx, const tsfx_plan* plan, const int64_t* ids, const void* sort_keys,
                                 int32_t sort_key_is_f64, const float* values, int64_t n_rows, int64_t* out_ids,
                                 double* out, int64_t out_capacity, int64_t* n_series_out, uint32_t flags) {
    if (!ctx) return TSFX_E_INVALID;
    if (!plan || plan->ctx != ctx) return fail(ctx, TSFX_E_INVALID, "plan does not belong to this context");
    const bool reuse = (ids == nullptr && values == nullptr);     // run on the CSR held from tsfx_build_csr
    if (n_rows < 0 || !n_series_out || (!reuse && n_rows > 0 && (!ids || !values)) || !out)
        return fail(ctx, TSFX_E_INVALID, "tsfx_extract_long: bad arguments");
    CK(cudaSetDevice(ctx->device));
    *n_series_out = 0;
    if (reuse) {
        if (flags & TSFX_FLAG_DEVICE_PTRS) return fail(ctx, TSFX_E_INVALID, "the held CSR is extracted into host buffers");
        if (ctx->held_series < 0) return fail(ctx, TSFX_E_INVALID, "tsfx_extract_long: no CSR is held by this context");
        if (plan->need_times) return fail(ctx, TSFX_E_UNSUPPORTED, "linear_trend_timewise: use the one-call form of tsfx_extract_long");
        const int64_t ns = ctx->held_series;
        *n_series_out = ns;
        if (ns == 0) return TSFX_OK;
        if (ns > out_capacity) return fail(ctx, TSFX_E_INVALID, "out_capacity too small: " + std::to_string(ns) + " series");
        CsrInfo info = {};
        info.n_series = ns; info.max_len = ctx->held_max_len; info.n_blocks = 1;
        info.series_lo[0] = 0; info.series_lo[1] = ns; info.row_lo[0] = 0; info.row_lo[1] = 0;
        KindSet K1;
        K1.plan[0] = plan; K1.dvals[0] = ctx->csr.d_values; K1.col0[0] = 0; K1.total_cols = plan->ncols;
        int rc = run_blocks(ctx, K1, info, nullptr, nullptr, nullptr, false, false, out, false, flags);
        if (rc) return rc;
        if (out_ids) CK(cudaMemcpyAsync(out_ids, ctx->csr.d_uid, ns * sizeof(int64_t), cudaMemcpyDeviceToHost, ctx->stream));
        CK(cudaStreamSynchronize(ctx->s_out));
        CK(cudaStreamSynchronize(ctx->stream));
        return TSFX_OK;
    }
    if (n_rows == 0) return TSFX_OK;
    LongIn in{ids, sort_keys, sort_key_is_f64, values, n_rows, (flags & TSFX_FLAG_DEVICE_PTRS) != 0};
    return extract_long_impl(ctx, &plan, in, out_ids, out, out_capacity, nullptr, nullptr, n_series_out, flags);
}

extern "C" int tsfx_extract_long_alloc(tsfx_ctx* ctx, const tsfx_plan* plan, const int64_t* ids, const void* sort_keys,
                                       int32_t sort_key_is_f64, const float* values, int64_t n_rows, int64_t** out_ids,
                                       double** out, int64_t* n_series_out, uint32_t flags) {
    if (!ctx) return TSFX_E_INVALID;
    if (!plan || plan->ctx != ctx) return fail(ctx, TSFX_E_INVALID, "plan does not belong to this context");
    if (flags & TSFX_FLAG_DEVICE_PTRS) return fail(ctx, TSFX_E_INVALID, "tsfx_extract_long_alloc takes host pointers");
    if (n_rows < 0 || !n_series_out || !out || !out_ids || (n_rows > 0 && (!ids || !values)))
        return fail(ctx, TSFX_E_INVALID, "tsfx_extract_long_alloc: bad arguments");
    CK(cudaSetDevice(ctx->device));
    *n_series_out = 0;
    *out = nullptr;
    *out_ids = nullptr;
    if (n_rows == 0) return TSFX_OK;
    LongIn in{ids, sort_keys, sort_key_is_f64, values, n_rows, false};
    int rc = extract_long_impl(ctx, &plan, in, nullptr, nullptr, 0, out_ids, out, n_series_out, flags);
    if (rc) {
        if (*out) ctx->pool.free(*out);
        if (*out_ids) ctx->pool.free(*out_ids);
        *out = nullptr; *out_ids = nullptr;
    }
    return rc;
}

extern "C" int tsfx_extract_long_kinds(tsfx_ctx* ctx, const tsfx_plan* const* plans, const int64_t* ids, const void* sort_keys,
                                       int32_t sort_key_is_f64, const float* const* values, int32_t n_kinds, int64_t n_rows,
                                       int64_t** out_ids, double** out, int64_t* n_series_out, uint32_t flags) {
    if (!ctx) return TSFX_E_INVALID;
    if (flags & TSFX_FLAG_DEVICE_PTRS) return fail(ctx, TSFX_E_INVALID, "tsfx_extract_long_kinds takes host pointers");
    if (n_kinds < 1 || n_kinds > TSFX_MAX_KINDS || !plans || !values || n_rows < 0 || !n_series_out || !out || !out_ids ||
        (n_rows > 0 && !ids))
        return fail(ctx, TSFX_E_INVALID, "tsfx_extract_long_kinds: bad arguments");
    for (int k = 0; k < n_kinds; ++k)
        if (!plans[k] || (n_rows > 0 && !values[k])) return fail(ctx, TSFX_E_INVALID, "tsfx_extract_long_kinds: NULL plan / column");
    CK(cudaSetDevice(ctx->device));
    *n_series_out = 0;
    *out = nullptr;
    *out_ids = nullptr;
    if (n_rows == 0) return TSFX_OK;
    LongIn in{ids, sort_keys, sort_key_is_f64, values[0], n_rows, false};
    in.more = values + 1;
    in.n_kinds = n_kinds;
    int rc = extract_long_impl(ctx, plans, in, nullptr, nullptr, 0, out_ids, out, n_series_out, flags);
    if (rc) {
        if (*out) ctx->pool.free(*out);
        if (*out_ids) ctx->pool.free(*out_ids);
        *out = nullptr; *out_ids = nullptr;
    }
    return rc;
}

extern "C" void* tsfx_host_alloc(tsfx_ctx* ctx, size_t bytes) {
    if (!ctx) return nullptr;
    cudaSetDevice(ctx->device);
    return ctx->pool.alloc(bytes);
}
extern "C" void tsfx_host_free(tsfx_ctx* ctx, void* p) {
    if (ctx && p) ctx->pool.free(p);
}

// ------------------------------------------------------------------------------------------ feature selection
extern "C" int tsfx_select_classification(tsfx_ctx* ctx, const double* X, int64_t n_rows, int32_t n_cols, const int32_t* y_codes,
                                          int32_t n_classes, double* out, uint32_t flags) {
    if (!ctx) return TSFX_E_INVALID;
    if (n_rows < 1 || n_cols < 0 || n_classes < 1 || !y_codes || !out || (n_cols > 0 && !X))
        return fail(ctx, TSFX_E_INVALID, "tsfx_select_classification: bad arguments");
    if (n_cols == 0) return TSFX_OK;
    CK(cudaSetDevice(ctx->device));
    std::vector<int64_t> counts(n_classes, 0);
    for (int64_t i = 0; i < n_rows; ++i) {
        if (y_codes[i] < 0 || y_codes[i] >= n_classes) return fail(ctx, TSFX_E_INVALID, "class code out of range");
        counts[y_codes[i]] += 1;
    }
    const double* d_X = X;
    if (!(flags & TSFX_FLAG_DEVICE_PTRS)) {
        CK(ctx->sel_x.reserve((size_t)n_rows * n_cols * 8));
        CK(ctx->stager.h2d(ctx->sel_x.p, X, (size_t)n_rows * n_cols * 8, ctx->stream));
        d_X = (const double*)ctx->sel_x.p;
    }
    CK(ctx->sel_y.reserve((size_t)n_rows * 4));
    CK(ctx->stager.h2d(ctx->sel_y.p, y_codes, (size_t)n_rows * 4, ctx->stream));
    const size_t ob = (size_t)n_classes * n_cols * TSFX_SEL_NSTAT * sizeof(double);
    CK(ctx->sel_out.reserve(ob));
    std::string msg;
    int has_nan = 0;
    int rc = select_class_stats(ctx->sel, d_X, n_rows, n_cols, (const int32_t*)ctx->sel_y.p, n_classes, counts.data(),
                                (double*)ctx->sel_out.p, &has_nan, ctx->stream, &msg);
    if (rc) return fail(ctx, rc, msg);
    CK(cudaMemcpyAsync(out, ctx->sel_out.p, ob, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    if (has_nan) return fail(ctx, TSFX_E_NAN, "the feature matrix contains NaN");
    return TSFX_OK;
}

extern "C" int tsfx_select_regression(tsfx_ctx* ctx, const double* X, int64_t n_rows, int32_t n_cols, const double* y, double* out,
                                      uint32_t flags) {
    if (!ctx) return TSFX_E_INVALID;
    if (n_rows < 1 || n_cols < 0 || !y || !out || (n_cols > 0 && !X))
        return fail(ctx, TSFX_E_INVALID, "tsfx_select_regression: bad arguments");
    if (n_cols == 0) return TSFX_OK;
    CK(cudaSetDevice(ctx->device));
    const double* d_X = X;
    if (!(flags & TSFX_FLAG_DEVICE_PTRS)) {
        CK(ctx->sel_x.reserve((size_t)n_rows * n_cols * 8));
        CK(ctx->stager.h2d(ctx->sel_x.p, X, (size_t)n_rows * n_cols * 8, ctx->stream));
        d_X = (const double*)ctx->sel_x.p;
    }
    CK(ctx->sel_y.reserve((size_t)n_rows * 8));
    CK(ctx->stager.h2d(ctx->sel_y.p, y, (size_t)n_rows * 8, ctx->stream));
    const size_t ob = ((size_t)n_cols * TSFX_SEL_NSTAT + 4) * sizeof(double);
    CK(ctx->sel_out.reserve(ob));
    std::string msg;
    int has_nan = 0;
    int rc = select_regression_stats(ctx->sel, d_X, n_rows, n_cols, (const double*)ctx->sel_y.p, (double*)ctx->sel_out.p, &has_nan,
                                     ctx->stream, &msg);
    if (rc) return fail(ctx, rc, msg);
    CK(cudaMemcpyAsync(out, ctx->sel_out.p, ob, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    if (has_nan) return fail(ctx, TSFX_E_NAN, "the feature matrix or the target contains NaN");
    return TSFX_OK;
}

// ------------------------------------------------------------------------------------------ multi-GPU placement
extern "C" int tsfx_set_peer_outputs(tsfx_ctx* ctx, const uint64_t* peer_out, int32_t n_peers, int32_t self_index,
                                     uint64_t multicast_out, int32_t mode) {
    if (!ctx) return TSFX_E_INVALID;
    CK(cudaSetDevice(ctx->device));
    CK(cudaStreamSynchronize(ctx->s_peer));
    ctx->peer_out.clear();
    ctx->peer_self = -1;
    ctx->peer_mc = 0;
    if (n_peers <= 0) return TSFX_OK;
    if (!peer_out || self_index < 0 || self_index >= n_peers || n_peers > 8 || mode < TSFX_PEER_AUTO || mode > TSFX_PEER_MULTICAST)
        return fail(ctx, TSFX_E_INVALID, "tsfx_set_peer_outputs: bad arguments (at most 8 ranks)");
    if (mode == TSFX_PEER_AUTO) mode = TSFX_PEER_COPY;      // measured on 2 x B200: copy engines 204 ms, P2P stores 209, multicast stores 218 per step
    if (mode == TSFX_PEER_MULTICAST && !multicast_out) return fail(ctx, TSFX_E_INVALID, "no multicast mapping was supplied");
    ctx->peer_out.assign(peer_out, peer_out + n_peers);
    ctx->peer_self = self_index;
    ctx->peer_mc = multicast_out;
    ctx->peer_mode = mode;
    return TSFX_OK;
}

extern "C" int tsfx_set_max_len_hint(tsfx_ctx* ctx, int32_t max_len) {
    if (!ctx || max_len < 0) return TSFX_E_INVALID;
    ctx->max_len_hint = max_len;
    return TSFX_OK;
}

extern "C" int tsfx_peer_flush(tsfx_ctx* ctx) {
    if (!ctx) return TSFX_E_INVALID;
    CK(cudaSetDevice(ctx->device));
    CK(cudaEventRecord(ctx->ev_peer, ctx->s_peer));
    CK(cudaStreamWaitEvent(ctx->stream, ctx->ev_peer, 0));
    return TSFX_OK;
}

// ------------------------------------------------------------------------------------------ roll_time_series views
extern "C" int64_t tsfx_roll_windows(const int64_t* begin, const int32_t* len, int64_t n_series,
                                     int32_t rolling_direction, int32_t max_timeshift, int32_t min_timeshift,
                                     int64_t* win_begin, int32_t* win_len, int64_t* win_parent,
                                     int32_t* win_end_index, int64_t capacity) {
    // dataframe_functions.py:340-373, 548-562.  rolling_direction > 0: the shifts are
    // reversed(range(Lmax, 0, -rolling_direction)) where Lmax is the LONGEST series of the frame (:555-560), so
    // window ends are anchored to Lmax for every series; shift t applies to a series of length L when t <= L,
    // the window is rows [max(t-max_timeshift-1, 0), t), kept when it has at least min_timeshift+1 rows, and
    // its id is (parent id, time of row t-1).
    // rolling_direction < 0 (:351-356, 365-366): shifts range(1, Lmax+1, |rolling_direction|), the window is rows
    // [t-1, min(t+max_timeshift, L)), same minimum length, id = (parent id, time of row t-1) -- the window's FIRST row.
    // win_end_index is therefore "the row whose sort value names the window": last row (positive) / first row (negative).
    if (!begin || !len || n_series < 0 || rolling_direction == 0 || max_timeshift < 0 || min_timeshift < 0)
        return TSFX_E_INVALID;
    int32_t Lmax = 0;
    for (int64_t s = 0; s < n_series; ++s) { if (len[s] < 1) return TSFX_E_INVALID; Lmax = std::max(Lmax, len[s]); }
    const int32_t amount = rolling_direction > 0 ? rolling_direction : -rolling_direction;
    const int32_t first = rolling_direction > 0 ? (Lmax > 0 ? Lmax - ((Lmax - 1) / amount) * amount : 1) : 1;   // smallest shift
    int64_t k = 0;
    for (int64_t s = 0; s < n_series; ++s) {
        const int32_t L = len[s];
        for (int32_t t = first; t <= L; t += amount) {
            int32_t lo, wl;
            if (rolling_direction > 0) {
                lo = t - max_timeshift - 1;
                if (lo < 0) lo = 0;
                wl = t - lo;
            } else {
                lo = t - 1;
                const int64_t hi = std::min<int64_t>((int64_t)lo + max_timeshift + 1, L);
                wl = (int32_t)(hi - lo);
            }
            if (wl < min_timeshift + 1) continue;
            if (win_begin) {
                if (k >= capacity) return TSFX_E_INVALID;
                win_begin[k] = begin[s] + lo;
                win_len[k] = wl;
                if (win_parent) win_parent[k] = s;
                if (win_end_index) win_end_index[k] = t - 1;
            }
            ++k;
        }
    }
    return k;
}
