// gate_host.cu -- C ABI (include/b200gate.h) and host planner of libb200gate.
//
// The planner turns the reference's chunk loop (noisereduce/spectralgate/base.py:167-226) into a
// table of independent (chunk, channel) units, sizes the device workspace, and launches
// k1_analyze -> k_rowfloor -> k_smooth -> k2c_synthesize per batch of units on the caller's stream.
#include "../../include/b200gate.h"
#include "gate_kernels_2k.cuh"
#include "gate_synth.cuh"
#include "gate_synth_2k.cuh"
#include "gate_dual.cuh"
#include "gate_peer.cuh"
#include "gate_generic.cuh"

#include <math.h>
#include <cmath>
#include <stdarg.h>
#include <stdio.h>
#include <string.h>

#include <algorithm>
#include <condition_variable>
#include <functional>
#include <future>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

using namespace b200;

namespace {

const double kEps64 = 2.220446049250313e-16;       // np.finfo(np.float64).eps (spectralgate/utils.py:11)
const double kEps32 = 5.9604644775390625e-08;      // 2^-24, FP32 unit roundoff
const double kKappa = 16.0;                        // guard band: |dX| <= kappa * eps32 * ||frame pair||_2
thread_local std::string g_create_error;          // one handle per thread: a failed create reports through the calling thread

}  // namespace

struct b200gate_handle {
    b200gate_params p{};
    std::string err;
    int num_sm = 148;
    int device = 0;
    int F = kF;
    // device tables
    float *d_wa = nullptr, *d_ws = nullptr, *d_invn = nullptr, *d_thr4 = nullptr, *d_gco = nullptr,
          *d_floor4 = nullptr, *d_ef = nullptr;
    float2* d_tw = nullptr;
    double *d_thr2_64 = nullptr, *d_wa64 = nullptr;
    double2* d_cs64 = nullptr;
    float ws_to_w = 0.f;
    float wa_max = 0.f;                            // max of the scaled analysis window (frame-energy bounds, gate_dual.cuh)
    unsigned* d_need_rowmax = nullptr;             // device flag raised by k1d_analyze when the top_db floor is reachable
    float2 *d_wa2 = nullptr, *d_ws2 = nullptr, *d_w2k = nullptr, *d_invn2 = nullptr;   // n_fft = 2048 family
    double sum_w = 0.0;
    std::vector<float> user_window;                // torch surface: torch.hann_window values
    float* d_tthr = nullptr;                       // torch surface: thresholds from xn, [tthr_units][FPad]
    int tthr_units = 0;
    bool have_thresh = false;
    double min_floor_amp = 0.0;                    // min_f 10^((thresh+top_db)/20): smallest |X| that lifts a row
    int range_mode = 0;                            // b200gate_set_range
    long long range_a = 0, range_b = 0;
    std::vector<double> thr, mean, sd;
    // general-geometry family (gate_generic.cuh)
    bool generic = false;
    int g_logN = 0;
    int g_M = 0, g_logM = 0;                       // Bluestein length for a non-power-of-two n_fft (0: radix-2 directly)
    double2 *d_gchirp = nullptr, *d_gbbr = nullptr;
    int g_W = 0;                                   // frame length: win_length (numpy surface) / n_fft (torch surface)
    double* d_gtthr = nullptr;                     // torch surface: thresholds from xn, [tthr_units][F]
    double *d_gwa = nullptr, *d_gws = nullptr, *d_gw2 = nullptr, *d_gthr = nullptr;
    double2* d_gcs = nullptr;
    // workspace
    char* d_ws_buf = nullptr;
    size_t ws_bytes = 0;
    void *d_in = nullptr, *d_out = nullptr;        // staging for host callers (kernel dtype)
    size_t in_bytes = 0, out_bytes = 0;
    void* d_raw = nullptr;                         // raw-dtype staging
    size_t raw_bytes = 0;
    Counters* d_cnt = nullptr;
    Counters* h_cnt = nullptr;                     // pinned: the run's exactness counters land here (stream-ordered copy)
    cudaEvent_t ev0 = nullptr, ev1 = nullptr, ev_done = nullptr;
    // statistics of a device-pointer run are resolved lazily (b200gate_get_stats): the run itself never blocks the host
    // torch surface: the masks of the last forward stay in the workspace so that the adjoint (= the same synthesis
    // with the same masks, TorchGate.backward) can reuse them -- b200gate_torch_apply_masks
    bool masks_valid = false, reuse_masks = false;
    long long masks_C = 0, masks_N = 0;
    bool stats_pending = false;
    size_t pend_batches = 0;
    std::vector<cudaEvent_t> group_ev;             // b200gate_run_sharded: one per channel group + 1
    std::vector<cudaEvent_t> stage_ev;             // 4 per batch: analysis start, analysis end, smoothing end, synthesis end
    std::vector<cudaEvent_t> pipe_ev;              // 4 per batch: input landed, compute done, output landed, seam copied
    cudaStream_t s_h2d = nullptr, s_d2h = nullptr; // pipelined host path
    void* hp_in[2] = {nullptr, nullptr};           // pinned staging slabs for pageable host rows (pipelined path)
    void* hp_out[2] = {nullptr, nullptr};
    size_t hp_in_bytes[2] = {0, 0}, hp_out_bytes[2] = {0, 0};
    int host_threads = 24;
    void* d_slab_in[2] = {nullptr, nullptr};       // caller-dtype slabs
    void* d_slab_out[2] = {nullptr, nullptr};
    size_t slab_in_bytes[2] = {0, 0}, slab_out_bytes[2] = {0, 0};
    b200gate_stats stats{};
    // debug taps
    long long dbg_chunk = -1, dbg_channel = -1;
    long long dbg_T = 0;
    float *d_dbg_spec = nullptr, *d_dbg_mask = nullptr;
    unsigned* d_dbg_bits = nullptr;
    size_t dbg_T_alloc = 0;
};

namespace {

int fail(b200gate_handle* h, int code, const char* fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof(buf), fmt, ap);
    va_end(ap);
    if (h) h->err = buf; else g_create_error = buf;
    return code;
}

#define CK(h, call)                                                                            \
    do {                                                                                       \
        cudaError_t e_ = (call);                                                               \
        if (e_ != cudaSuccess)                                                                 \
            return fail((h), B200GATE_ERR_CUDA, "%s failed: %s (%s:%d)", #call,               \
                        cudaGetErrorString(e_), __FILE__, __LINE__);                           \
    } while (0)

template <class T>
int upload(b200gate_handle* h, T** dptr, const std::vector<T>& v) {
    if (!*dptr) CK(h, cudaMalloc((void**)dptr, v.size() * sizeof(T)));
    CK(h, cudaMemcpy(*dptr, v.data(), v.size() * sizeof(T), cudaMemcpyHostToDevice));
    return B200GATE_OK;
}

// one-call device scratch: freed on every return path
struct Scratch {
    void* p = nullptr;
    ~Scratch() { if (p) cudaFree(p); }
    Scratch() = default;
    Scratch(const Scratch&) = delete;
    Scratch& operator=(const Scratch&) = delete;
    cudaError_t alloc(size_t bytes) { return cudaMalloc(&p, bytes ? bytes : 1); }
    template <class T> T* as() const { return (T*)p; }
};

// A reduce_noise() call creates a handle, runs once and destroys it: its large device buffers (workspace, slabs, staging)
// would be cudaMalloc'ed and cudaFree'd every call (~15 ms together at config-2 sizes).  Destroyed handles leave them in a
// small process-wide cache instead (per device; bounded: B200GATE_DEVICE_CACHE_MB, default 4096, 0 disables), and ensure()
// looks there first.  Buffers enter the cache only after the device is idle (b200gate_destroy synchronises).
struct DevicePool {
    struct Item { void* p; size_t bytes; int dev; };
    std::mutex mu;
    std::vector<Item> items;
    size_t cached = 0;
    static size_t cap() {
        static const size_t c = [] {
            const char* e = getenv("B200GATE_DEVICE_CACHE_MB");
            return (size_t)(e ? std::max(0LL, atoll(e)) : 4096LL) << 20;
        }();
        return c;
    }
    void* take(size_t bytes, int dev, size_t* got) {
        std::lock_guard<std::mutex> lk(mu);
        size_t best = items.size();
        for (size_t i = 0; i < items.size(); ++i)
            if (items[i].dev == dev && items[i].bytes >= bytes && items[i].bytes <= bytes + bytes / 4 + (1 << 20) &&
                (best == items.size() || items[i].bytes < items[best].bytes))
                best = i;
        if (best == items.size()) return nullptr;
        void* p = items[best].p;
        *got = items[best].bytes;
        cached -= items[best].bytes;
        items.erase(items.begin() + (long)best);
        return p;
    }
    void give(void* p, size_t bytes, int dev) {            // the device must be idle with respect to p
        if (!p) return;
        {
            std::lock_guard<std::mutex> lk(mu);
            if (bytes >= (1 << 20) && cached + bytes <= cap() && items.size() < 16) {
                items.push_back(Item{p, bytes, dev});
                cached += bytes;
                return;
            }
        }
        cudaFree(p);
    }
    void drop_all(int dev) {                               // out of memory: give everything cached on this device back
        std::lock_guard<std::mutex> lk(mu);
        for (size_t i = items.size(); i-- > 0;)
            if (items[i].dev == dev) { cudaFree(items[i].p); cached -= items[i].bytes; items.erase(items.begin() + (long)i); }
    }
};
DevicePool g_device_pool;

int ensure(b200gate_handle* h, void** p, size_t* have, size_t need) {
    if (*have >= need) return B200GATE_OK;
    if (*p) cudaFree(*p);                                   // (synchronises: work still using the old buffer has finished)
    *p = nullptr;
    *have = 0;
    size_t got = 0;
    if (void* c = g_device_pool.take(need, h->device, &got)) {
        *p = c;
        *have = got;
        return B200GATE_OK;
    }
    cudaError_t e = cudaMalloc(p, need);
    if (e != cudaSuccess) {
        cudaGetLastError();
        g_device_pool.drop_all(h->device);
        e = cudaMalloc(p, need);
    }
    if (e != cudaSuccess) return fail(h, B200GATE_ERR_NOMEM, "cudaMalloc(%zu bytes) failed: %s", need, cudaGetErrorString(e));
    *have = need;
    return B200GATE_OK;
}

// Tables that depend only on the geometry: windows, twiddles, overlap-add norm, edge factors.
int build_static_tables_2k(b200gate_handle* h) {
    const int N = kN2, H = h->p.hop_length;
    std::vector<double> w(N);
    double sw = 0.0;
    for (int n = 0; n < N; ++n) {
        w[n] = 0.5 - 0.5 * cos(2.0 * M_PI * (double)n / (double)N);
        sw += w[n];
    }
    h->sum_w = sw;
    h->ws_to_w = (float)(1024.0 / sw);
    std::vector<float2> wa2(1024), ws2(1024), w2k(kF2), invn2(256), tw(32 * 32);
    for (int m = 0; m < 1024; ++m) {
        wa2[m] = make_float2((float)(w[2 * m] / sw), (float)(w[2 * m + 1] / sw));
        ws2[m] = make_float2((float)(w[2 * m] * sw / 1024.0), (float)(w[2 * m + 1] * sw / 1024.0));
    }
    for (int k = 0; k < kF2; ++k) {
        const long double th = M_PIl * (long double)k / 1024.0L;
        w2k[k] = make_float2((float)cosl(th), (float)(-sinl(th)));
    }
    for (int r = 0; r < H; ++r) {
        double sacc = 0.0;
        for (int i = 0; i * H + r < N; ++i) sacc += w[i * H + r] * w[i * H + r];
        const float v = (float)(sacc > 1e-10 ? 1.0 / sacc : 1.0);
        if (r & 1) invn2[r >> 1].y = v; else invn2[r >> 1].x = v;
    }
    for (int q = 0; q < 32; ++q)
        for (int l = 0; l < 32; ++l) {
            const long double th = 2.0L * M_PIl * (long double)(l * q) / 1024.0L;
            tw[q * 32 + l] = make_float2((float)cosl(th), (float)(-sinl(th)));
        }
    int rc;
    if ((rc = upload(h, &h->d_wa2, wa2))) return rc;
    if ((rc = upload(h, &h->d_ws2, ws2))) return rc;
    if ((rc = upload(h, &h->d_w2k, w2k))) return rc;
    if ((rc = upload(h, &h->d_invn2, invn2))) return rc;
    if ((rc = upload(h, &h->d_tw, tw))) return rc;
    return B200GATE_OK;
}

int build_static_tables(b200gate_handle* h) {
    if (h->p.n_fft == kN2) return build_static_tables_2k(h);
    const int N = h->p.n_fft, H = h->p.hop_length;
    std::vector<double> w(N);
    double sw = 0.0;
    for (int n = 0; n < N; ++n) {
        if ((int)h->user_window.size() == N) w[n] = (double)h->user_window[n];   // torch.hann_window (float32)
        else w[n] = 0.5 - 0.5 * cos(2.0 * M_PI * (double)n / (double)N);         // periodic Hann (scipy 'hann', fftbins)
        sw += w[n];
    }
    h->sum_w = sw;
    std::vector<float> wa(N), ws(N), invn(H);
    std::vector<double> wa64(N);
    for (int n = 0; n < N; ++n) {
        wa64[n] = w[n] / sw;
        wa[n] = (float)(w[n] / sw);
        ws[n] = (float)(w[n] * sw / (double)N);
    }
    h->ws_to_w = (float)((double)N / sw);
    h->wa_max = 0.f;
    for (int n = 0; n < N; ++n) h->wa_max = std::max(h->wa_max, (float)fabs(w[n] / sw) * (1.0f + 1e-6f));
    for (int r = 0; r < H; ++r) {
        double s = 0.0;
        for (int i = 0; i * H + r < N; ++i) s += w[i * H + r] * w[i * H + r];
        invn[r] = (float)(s > 1e-10 ? 1.0 / s : 1.0);
    }
    std::vector<float2> tw(32 * 32);
    for (int q = 0; q < 32; ++q)
        for (int l = 0; l < 32; ++l) {
            const long double th = 2.0L * M_PIl * (long double)(l * q) / 1024.0L;
            tw[q * 32 + l] = make_float2((float)cosl(th), (float)(-sinl(th)));
        }
    std::vector<double2> cs(N);
    for (int m = 0; m < N; ++m) {
        const long double th = 2.0L * M_PIl * (long double)m / (long double)N;
        cs[m] = make_double2((double)cosl(th), (double)sinl(th));
    }
    const int nf = h->p.n_grad_freq;
    std::vector<float> ef(kFPad, 0.f);
    for (int f = 0; f < kF; ++f) {
        long s = 0;
        for (int d = -nf; d <= nf; ++d)
            if (f - d >= 0 && f - d < kF) s += nf + 1 - abs(d);
        ef[f] = (float)((double)s / (double)((nf + 1) * (nf + 1)));
    }
    int rc;
    if ((rc = upload(h, &h->d_wa, wa))) return rc;
    if ((rc = upload(h, &h->d_ws, ws))) return rc;
    if ((rc = upload(h, &h->d_invn, invn))) return rc;
    if ((rc = upload(h, &h->d_tw, tw))) return rc;
    if ((rc = upload(h, &h->d_cs64, cs))) return rc;
    if ((rc = upload(h, &h->d_wa64, wa64))) return rc;
    if ((rc = upload(h, &h->d_ef, ef))) return rc;
    return B200GATE_OK;
}

// Tables that depend on the noise threshold (stationary.py:79-81), in the linear power domain:
// dB > thresh  <=>  |X| + eps > 10^(thresh/20)  <=>  |X|^2 > T_amp^2.
int build_threshold_tables(b200gate_handle* h) {
    std::vector<float> thr4(kFPad, INFINITY), gco(kFPad, 0.f), floor4(kFPad, INFINITY);
    std::vector<double> t2(kF);
    for (int f = 0; f < kF; ++f) {
        double T = pow(10.0, h->thr[f] / 20.0) - kEps64;
        if (!(T > 0.0)) T = 0.0;
        double Tf = pow(10.0, (h->thr[f] + h->p.top_db) / 20.0) - kEps64;
        if (!(Tf > 0.0)) Tf = 0.0;
        t2[f] = T * T;
        if (f == 0 || Tf < h->min_floor_amp) h->min_floor_amp = Tf;
        thr4[f] = (float)(4.0 * T * T);
        gco[f] = (float)(8.0 * T * kKappa * kEps32 * (h->p.debug_guard_scale > 0 ? h->p.debug_guard_scale : 1));
        floor4[f] = (float)(4.0 * Tf * Tf);
    }
    int rc;
    if ((rc = upload(h, &h->d_thr4, thr4))) return rc;
    if ((rc = upload(h, &h->d_gco, gco))) return rc;
    if ((rc = upload(h, &h->d_floor4, floor4))) return rc;
    if ((rc = upload(h, &h->d_thr2_64, t2))) return rc;
    h->have_thresh = true;
    return B200GATE_OK;
}

Tables device_tables(const b200gate_handle* h) {
    Tables tb{};
    tb.wa = h->d_wa; tb.ws = h->d_ws; tb.tw = h->d_tw; tb.invn = h->d_invn;
    tb.thr4 = h->d_thr4; tb.gco = h->d_gco; tb.floor4 = h->d_floor4; tb.ef = h->d_ef;
    tb.thr2_64 = h->d_thr2_64; tb.wa64 = h->d_wa64; tb.cs64 = h->d_cs64;
    tb.ws_to_w = h->ws_to_w;
    return tb;
}

size_t dtype_size(int dtype) { return dtype == B200GATE_F32 ? 4 : dtype == B200GATE_I16 ? 2 : dtype == B200GATE_F64 ? 8 : 0; }

int grid_1d(long long n, int block, int cap) {
    long long g = (n + block - 1) / block;
    return (int)std::max(1LL, std::min<long long>(g, cap));
}

int generic_noise_stats_from_mean(b200gate_handle* h, const double* d_yn, long long n, cudaStream_t st);

// collapsed noise clip (float64, device) -> thresholds
int noise_stats_from_mean(b200gate_handle* h, const double* d_yn, long long n, cudaStream_t st) {
    if (h->generic) return generic_noise_stats_from_mean(h, d_yn, n, st);
    const int H = h->p.hop_length;
    const int Tn = (int)(n / H) + 1;                     // scipy: (n + 2*(W/2) - W)/H + 1
    Scratch s_db, s_res;
    CK(h, s_db.alloc((size_t)Tn * kF * sizeof(double)));
    CK(h, s_res.alloc(3 * kF * sizeof(double)));
    double *d_db = s_db.as<double>(), *d_res = s_res.as<double>();
    K0Args a{};
    a.yn = d_yn; a.n = n; a.H = H; a.Tn = Tn; a.wa64 = h->d_wa64; a.cs64 = h->d_cs64; a.eps = kEps64; a.db = d_db;
    B200_LAUNCH(k0_stft_db, dim3(Tn), dim3(256), kN * sizeof(double2), st, a);
    B200_LAUNCH(k0_stats, dim3(kF), dim3(256), 0, st, d_db, Tn, kF, h->p.top_db, h->p.std_ddof, h->p.n_std_thresh,
                d_res, d_res + kF, d_res + 2 * kF);
    CK(h, cudaGetLastError());
    std::vector<double> res(3 * kF);
    CK(h, cudaMemcpyAsync(res.data(), d_res, res.size() * sizeof(double), cudaMemcpyDeviceToHost, st));
    CK(h, cudaStreamSynchronize(st));
    h->mean.assign(res.begin(), res.begin() + kF);
    h->sd.assign(res.begin() + kF, res.begin() + 2 * kF);
    h->thr.assign(res.begin() + 2 * kF, res.end());
    return build_threshold_tables(h);
}

// ---- general-geometry family: tables, noise statistics ----------------------------------------------------------
int build_generic_tables(b200gate_handle* h) {
    const int N = h->p.n_fft, W = h->p.win_length;
    const bool torch_sem = h->p.surface == B200GATE_SURFACE_TORCH;
    std::vector<double> w(W);
    double sw = 0.0;
    for (int n = 0; n < W; ++n) {
        if ((int)h->user_window.size() == W) w[n] = (double)h->user_window[n];             // torch.hann_window (float32)
        else if (torch_sem) w[n] = (double)(cosf((float)n * (float)(M_PI * 2.0 / W)) * -0.5f + 0.5f);
        else w[n] = 0.5 - 0.5 * cos(2.0 * M_PI * (double)n / (double)W);                  // scipy get_window('hann', W): periodic
        sw += w[n];
    }
    h->sum_w = sw;
    // numpy surface: frames of win_length samples, spectrum scaled by 1 / sum(w) (scaling='spectrum'), rfft pads at
    // the END.  torch surface (torch.stft, center=True): frames of n_fft samples under the window centre-padded
    // to n_fft, no scaling (torchgate.py:223-232).
    const int Wf = torch_sem ? N : W, left = torch_sem ? (N - W) / 2 : 0;
    h->g_W = Wf;
    std::vector<double> wa(Wf, 0.0), ws(Wf, 0.0), w2(Wf, 0.0);
    for (int n = 0; n < W; ++n) {
        wa[left + n] = torch_sem ? w[n] : w[n] / sw;
        ws[left + n] = torch_sem ? w[n] / (double)N : w[n] * sw / (double)N;               // irfft's 1/N (* sum(w) in scipy's istft)
        w2[left + n] = w[n] * w[n];
    }
    // transform tables: radix-2 twiddles of n_fft itself, or -- n_fft not a power of two -- Bluestein's chirp-z
    // through two length-M radix-2 transforms (M = 2^k >= 2 n_fft - 1)
    const int L = h->g_M ? h->g_M : N;
    std::vector<double2> cs(L);
    for (int m = 0; m < L; ++m) {
        const long double th = 2.0L * M_PIl * (long double)m / (long double)L;
        cs[m] = make_double2((double)cosl(th), (double)sinl(th));
    }
    int rc;
    if (h->g_M) {
        const int M = h->g_M, logM = h->g_logM;
        std::vector<double2> chirp(N);
        std::vector<long double> br(M, 0.0L), bi(M, 0.0L);
        for (int n = 0; n < N; ++n) {
            const long long q = ((long long)n * n) % (2LL * N);                  // n^2 mod 2N keeps the angle small
            const long double th = M_PIl * (long double)q / (long double)N;
            chirp[n] = make_double2((double)cosl(th), (double)(-sinl(th)));      // exp(-i pi n^2 / N)
            br[n] = cosl(th); bi[n] = sinl(th);                                  // conjugate chirp, circular
            if (n) { br[M - n] = br[n]; bi[M - n] = bi[n]; }
        }
        // forward FFT_M of the kernel in long double (iterative radix-2 DIT)
        for (int i = 0; i < M; ++i) {
            int r = 0;
            for (int b = 0; b < logM; ++b) r |= ((i >> b) & 1) << (logM - 1 - b);
            if (r > i) { std::swap(br[i], br[r]); std::swap(bi[i], bi[r]); }
        }
        for (int len = 2; len <= M; len <<= 1) {
            const int half = len >> 1;
            for (int blk = 0; blk < M; blk += len)
                for (int o = 0; o < half; ++o) {
                    const long double th = -2.0L * M_PIl * (long double)o / (long double)len;
                    const long double wr = cosl(th), wi = sinl(th);
                    const long double xr = br[blk + o], xi = bi[blk + o];
                    const long double yr = br[blk + o + half] * wr - bi[blk + o + half] * wi;
                    const long double yi = br[blk + o + half] * wi + bi[blk + o + half] * wr;
                    br[blk + o] = xr + yr; bi[blk + o] = xi + yi;
                    br[blk + o + half] = xr - yr; bi[blk + o + half] = xi - yi;
                }
        }
        std::vector<double2> bbr(M);
        for (int i = 0; i < M; ++i) {
            int r = 0;
            for (int b = 0; b < logM; ++b) r |= ((i >> b) & 1) << (logM - 1 - b);
            bbr[i] = make_double2((double)(br[r] / (long double)M), (double)(bi[r] / (long double)M));   // bit-reversed, 1/M folded in
        }
        if (h->d_gchirp) { cudaFree(h->d_gchirp); h->d_gchirp = nullptr; }
        if ((rc = upload(h, &h->d_gchirp, chirp))) return rc;
        if ((rc = upload(h, &h->d_gbbr, bbr))) return rc;
    }
    if ((rc = upload(h, &h->d_gwa, wa))) return rc;
    if ((rc = upload(h, &h->d_gws, ws))) return rc;
    if ((rc = upload(h, &h->d_gw2, w2))) return rc;
    if ((rc = upload(h, &h->d_gcs, cs))) return rc;
    return B200GATE_OK;
}

GTables generic_tables(const b200gate_handle* h) {
    GTables t{};
    t.wa = h->d_gwa; t.ws = h->d_gws; t.w2 = h->d_gw2; t.cs = h->d_gcs; t.chirp = h->d_gchirp; t.bbr = h->d_gbbr;
    return t;
}

GGeom generic_geom(const b200gate_handle* h, const Geom& g) {
    GGeom gg{};
    gg.g = g; gg.N = h->p.n_fft; gg.logN = h->g_logN; gg.W = h->g_W; gg.F = h->F; gg.out_len = 0;
    gg.M = h->g_M; gg.logM = h->g_logM;
    return gg;
}

int generic_threads(int N) { return N >= 512 ? 256 : std::max(32, (N / 2 + 31) / 32 * 32); }
int generic_fft_len(const b200gate_handle* h) { return h->g_M ? h->g_M : h->p.n_fft; }

int generic_noise_stats_from_mean(b200gate_handle* h, const double* d_yn, long long n, cudaStream_t st) {
    const int H = h->p.hop_length, W = h->p.win_length, N = h->p.n_fft, F = h->F;
    const long long Tn = (n + 2 * (W / 2) - W) / H + 1;
    if (Tn < 1 || Tn > 0x7fffffffLL) return fail(h, B200GATE_ERR_ARG, "noise clip length %lld unusable", n);
    Scratch s_X, s_db, s_res;
    CK(h, s_X.alloc((size_t)Tn * F * sizeof(double2)));
    CK(h, s_db.alloc((size_t)Tn * F * sizeof(double)));
    CK(h, s_res.alloc(3 * (size_t)F * sizeof(double)));
    double2* d_X = s_X.as<double2>();
    double *d_db = s_db.as<double>(), *d_res = s_res.as<double>();
    Geom g{};
    g.H = H; g.C = 1; g.T = (int)Tn; g.n_chunks = 1; g.n_total = n; g.step = n; g.pad = 0; g.Lp = n;
    g.in_stride = n; g.out_stride = n; g.u0 = 0; g.n_units = 1;
    GStftArgs<double> a{};
    a.gg = generic_geom(h, g); a.tb = generic_tables(h); a.x = d_yn; a.X = d_X;
    { auto kern_ = gk_stft<double>; B200_LAUNCH(kern_, dim3((unsigned)Tn, 1), dim3(generic_threads(generic_fft_len(h))), (size_t)generic_fft_len(h) * sizeof(double2), st, a); }
    B200_LAUNCH(gk_noise_db, dim3(grid_1d(Tn * F, 256, 1 << 16)), dim3(256), 0, st, (const double2*)d_X, (long long)Tn * F, kEps64, d_db);
    B200_LAUNCH(k0_stats, dim3(F), dim3(256), 0, st, d_db, (int)Tn, F, h->p.top_db, h->p.std_ddof, h->p.n_std_thresh,
                d_res, d_res + F, d_res + 2 * F);
    CK(h, cudaGetLastError());
    std::vector<double> res(3 * (size_t)F);
    CK(h, cudaMemcpyAsync(res.data(), d_res, res.size() * sizeof(double), cudaMemcpyDeviceToHost, st));
    CK(h, cudaStreamSynchronize(st));
    h->mean.assign(res.begin(), res.begin() + F);
    h->sd.assign(res.begin() + F, res.begin() + 2 * F);
    h->thr.assign(res.begin() + 2 * F, res.end());
    int rc = upload(h, &h->d_gthr, h->thr);
    if (rc) return rc;
    h->have_thresh = true;
    return B200GATE_OK;
}

template <typename Tin, typename Tacc>
void launch_channel_sum(const void* y, long long C, long long n, long long stride, void* acc, int init, cudaStream_t st) {
    auto kern = k0_channel_sum<Tin, Tacc>;
    B200_LAUNCH(kern, dim3(grid_1d(n, 256, 4096)), dim3(256), 0, st, (const Tin*)y, C, n, stride, (Tacc*)acc, init);
}

// Persistent host workers for the staging copies: a slab pipeline of ~50 slabs would otherwise create and join ~15 threads
// per slab and direction (~1 ms of a ~3 ms slab).  Workers sleep on a condition variable between jobs; one job at a time.
class HostWorkers {
public:
    // run work(id) for id in [0, nt) on nt - 1 pooled threads plus the caller
    void run(int nt, const std::function<void(int)>& work) {
        if (nt <= 1) { work(0); return; }
        std::unique_lock<std::mutex> job_lock(job_mu_);               // one job at a time (handles on several threads share the pool)
        {
            std::lock_guard<std::mutex> lk(mu_);
            while ((int)threads_.size() < nt - 1) {
                const int id = (int)threads_.size() + 1;
                threads_.emplace_back([this, id] { loop(id); });
            }
            work_ = &work;
            nt_ = nt;
            pending_ = nt - 1;
            ++generation_;
        }
        cv_.notify_all();
        work(0);
        std::unique_lock<std::mutex> lk(mu_);
        done_cv_.wait(lk, [this] { return pending_ == 0; });
        work_ = nullptr;
    }
    ~HostWorkers() {
        {
            std::lock_guard<std::mutex> lk(mu_);
            stop_ = true;
        }
        cv_.notify_all();
        for (auto& t : threads_) t.join();
    }

private:
    void loop(int id) {
        unsigned long long seen = 0;
        for (;;) {
            const std::function<void(int)>* w = nullptr;
            {
                std::unique_lock<std::mutex> lk(mu_);
                cv_.wait(lk, [&] { return stop_ || (generation_ != seen && id < nt_); });
                if (stop_) return;
                seen = generation_;
                w = work_;
            }
            (*w)(id);
            {
                std::lock_guard<std::mutex> lk(mu_);
                if (--pending_ == 0) done_cv_.notify_one();
            }
        }
    }
    std::mutex mu_, job_mu_;
    std::condition_variable cv_, done_cv_;
    std::vector<std::thread> threads_;
    const std::function<void(int)>* work_ = nullptr;
    int nt_ = 0, pending_ = 0;
    unsigned long long generation_ = 0;
    bool stop_ = false;
};
// pool 0: staging of pageable input rows; pool 1: copy-out of results into pageable rows (the two overlap in the slab pipeline)
HostWorkers& host_workers(int pool) {
    static HostWorkers* w[2] = {new HostWorkers(), new HostWorkers()};   // (never destroyed: no joins from static destructors at exit)
    return *w[pool & 1];
}

// device-resident (or staged) y -> running channel-order sum in acc
int channel_sum_impl(b200gate_handle* h, const void* y, int dtype, long long C, long long n, long long stride,
                     int is_device, void* acc, int init, cudaStream_t st) {
    const size_t es = dtype_size(dtype);
    const void* src = y;
    long long sstride = stride;
    Scratch tmp;
    if (!is_device && init) {
        // host rows: the channel-order sum is taken by the host workers (the same sequential additions in the same type, so
        // the same bits as k0_channel_sum) and only the n sums cross PCIe -- not C rows of pageable memory (64 x 600000 float32
        // through the driver's bounce buffer cost ~15 ms per reduce_noise() call)
        const size_t as = (dtype == B200GATE_F32) ? 4 : 8;
        std::vector<unsigned char> hacc((size_t)n * as);
        const long long blk = 8192;
        const long long n_blk = (n + blk - 1) / blk;
        const int nt = (int)std::max<long long>(1, std::min<long long>(std::min(h->host_threads, 32), n_blk));
        std::function<void(int)> work = [&](int id) {
            for (long long bix = id; bix < n_blk; bix += nt) {
                const long long i0 = bix * blk, i1 = std::min(n, i0 + blk);
                if (dtype == B200GATE_F32) {
                    float* a = (float*)hacc.data();
                    for (long long i = i0; i < i1; ++i) a[i] = 0.f;
                    for (long long c = 0; c < C; ++c) {
                        const float* r = (const float*)y + c * stride;
                        for (long long i = i0; i < i1; ++i) a[i] = a[i] + r[i];
                    }
                } else if (dtype == B200GATE_I16) {
                    double* a = (double*)hacc.data();
                    for (long long i = i0; i < i1; ++i) a[i] = 0.0;
                    for (long long c = 0; c < C; ++c) {
                        const short* r = (const short*)y + c * stride;
                        for (long long i = i0; i < i1; ++i) a[i] = a[i] + (double)r[i];
                    }
                } else {
                    double* a = (double*)hacc.data();
                    for (long long i = i0; i < i1; ++i) a[i] = 0.0;
                    for (long long c = 0; c < C; ++c) {
                        const double* r = (const double*)y + c * stride;
                        for (long long i = i0; i < i1; ++i) a[i] = a[i] + r[i];
                    }
                }
            }
        };
        host_workers(0).run(nt, work);
        CK(h, cudaMemcpyAsync(acc, hacc.data(), (size_t)n * as, cudaMemcpyHostToDevice, st));
        CK(h, cudaStreamSynchronize(st));                      // (hacc is freed on return)
        return B200GATE_OK;
    }
    if (!is_device) {
        CK(h, tmp.alloc((size_t)C * n * es));
        CK(h, cudaMemcpy2DAsync(tmp.p, (size_t)n * es, y, (size_t)stride * es, (size_t)n * es, (size_t)C,
                                cudaMemcpyHostToDevice, st));
        src = tmp.p;
        sstride = n;
    }
    if (dtype == B200GATE_F32) launch_channel_sum<float, float>(src, C, n, sstride, acc, init, st);
    else if (dtype == B200GATE_I16) launch_channel_sum<short, double>(src, C, n, sstride, acc, init, st);
    else launch_channel_sum<double, double>(src, C, n, sstride, acc, init, st);
    CK(h, cudaGetLastError());
    if (tmp.p) CK(h, cudaStreamSynchronize(st));          // the staging copy is freed on return
    return B200GATE_OK;
}

// run `stmt` with T bound to the kernels' sample type
#define B200_WITH_DTYPE(dt, ...)                                           \
    do {                                                                   \
        if ((dt) == B200GATE_I16) { using T = short; __VA_ARGS__; }        \
        else if ((dt) == B200GATE_F64) { using T = double; __VA_ARGS__; }  \
        else { using T = float; __VA_ARGS__; }                             \
    } while (0)

void launch_k1n(const Geom& g, const Tables& tb, const void* x, int kdt, float* mag, const DebugTap& dbg, int resident,
                cudaStream_t st, float2* zc = nullptr, int z_lo = 0, int z_hi = 0x7fffffff) {
    K1nArgs a1{};
    a1.g = g; a1.tb = tb; a1.x = x; a1.mag = mag; a1.dbg = dbg; a1.zcache = zc; a1.zpairs = (g.T + 1) / 2;
    a1.z_lo = z_lo; a1.z_hi = z_hi;
    long long want = (long long)resident * kWarps * 4;
    long long run = ((long long)g.n_units * g.T + want - 1) / want;
    run = std::max(8LL, std::min(64LL, run));
    run += run & 1;
    a1.run = (int)run;
    a1.n_runs = (g.T + a1.run - 1) / a1.run;
    B200_WITH_DTYPE(kdt, { auto kern_ = k1n_magnitude<8, T>;
        B200_LAUNCH(kern_, dim3(grid_1d((long long)g.n_units * a1.n_runs, kWarps, resident)), dim3(kThreads),
                    k1n_smem_floats() * 4, st, a1); });
}

// Float-mask smoothing (non-stationary gate, TorchGate moving-mean gate): the box form for 1 <= nf <= 12 (k_smooth_box,
// compiled per nf), else the tap-loop streaming kernel, else (ring too large for shared memory) the tile kernel.
#define B200_SMOOTH_BOX_CASE(NF_) case NF_: { auto kern_ = k_smooth_box<NF_>; \
        if (set_attr) cudaFuncSetAttribute(kern_, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024); \
        else B200_LAUNCH(kern_, grid, dim3(sa.FPad / 4), smem, st, sa); } break;
static void smooth_box_dispatch(const SmoothFArgs& sa, int nf, dim3 grid, size_t smem, cudaStream_t st, bool set_attr) {
    switch (nf) {
        B200_SMOOTH_BOX_CASE(1) B200_SMOOTH_BOX_CASE(2) B200_SMOOTH_BOX_CASE(3) B200_SMOOTH_BOX_CASE(4)
        B200_SMOOTH_BOX_CASE(5) B200_SMOOTH_BOX_CASE(6) B200_SMOOTH_BOX_CASE(7) B200_SMOOTH_BOX_CASE(8)
        B200_SMOOTH_BOX_CASE(9) B200_SMOOTH_BOX_CASE(10) B200_SMOOTH_BOX_CASE(11) B200_SMOOTH_BOX_CASE(12)
        default: break;
    }
}
static void launch_smooth_float(SmoothFArgs sa, int nf, int nt, int tf_lo, int tf_hi, int nu, int path_flags, cudaStream_t st) {
    const bool box_ok = nf >= 1 && nf <= 12 && sa.FPad - sa.F >= 12 && smoothb_smem_bytes(sa.FPad, nt) <= 200 * 1024 &&
                        !(path_flags & 32) && !(path_flags & 128);
    if (box_ok) {
        sa.TT = 256;                        // frames per strip (2 nt warm-up rows each)
        const int strips = (tf_hi - tf_lo + sa.TT - 1) / sa.TT;
        smooth_box_dispatch(sa, nf, dim3(strips, nu), smoothb_smem_bytes(sa.FPad, nt), st, false);
    } else if (smooths_smem_bytes(sa.FPad, nf, nt) <= 200 * 1024 && !(path_flags & 32)) {
        sa.TT = 256;
        const int strips = (tf_hi - tf_lo + sa.TT - 1) / sa.TT;
        B200_LAUNCH(k_smooth_stream, dim3(strips, nu), dim3(sa.FPad / 4), smooths_smem_bytes(sa.FPad, nf, nt), st, sa);
    } else {
        const int tiles = (tf_hi - tf_lo + sa.TT - 1) / sa.TT;
        B200_LAUNCH(k_smooth_f, dim3(tiles, nu), dim3(256), smoothf_smem_bytes(sa.TT, sa.FPad, nf), st, sa);
    }
}

// Pageable host memory: cudaMemcpyAsync from / to it is neither asynchronous nor fast (the driver bounces it through a small
// pinned buffer at ~10 GB/s), and pinning a caller's 7 GB array in place costs a second (measured: cudaHostRegister 8.5 GB/s).
// The slab pipeline therefore stages pageable rows through its own pinned slabs with a handful of host threads
// (measured 60-70 GB/s with 8-16 threads), which keeps PCIe busy.
bool host_pointer_is_pinned(const void* p) {
#ifdef B200_CUSIM_BUILD
    (void)p;
    return false;                                  // simulator: exercise the staging path
#else
    cudaPointerAttributes at{};
    if (cudaPointerGetAttributes(&at, p) != cudaSuccess) { cudaGetLastError(); return false; }
    return at.type == cudaMemoryTypeHost || at.type == cudaMemoryTypeManaged;
#endif
}
void parallel_rows_copy(void* dst, size_t dpitch, const void* src, size_t spitch, size_t width, size_t rows, int nthreads,
                        int pool = 0) {
    if (rows == 0 || width == 0) return;
    // split every row into pieces of >= 1 MB so that few long rows still spread over all threads
    const size_t piece = std::max<size_t>(1 << 20, (width * rows / (size_t)std::max(1, nthreads) + 4095) / 4096 * 4096);
    const size_t per_row = (width + piece - 1) / piece;
    const size_t n_pieces = per_row * rows;
    const int nt = (int)std::min<size_t>((size_t)std::max(1, std::min(nthreads, 64)), n_pieces);
    std::function<void(int)> work = [&](int id) {
        for (size_t k = (size_t)id; k < n_pieces; k += (size_t)nt) {
            const size_t r = k / per_row, off = (k - r * per_row) * piece;
            memcpy((char*)dst + r * dpitch + off, (const char*)src + r * spitch + off, std::min(piece, width - off));
        }
    };
    host_workers(pool).run(nt, work);
}

// Pinned staging slabs are expensive to create (cudaMallocHost of 1 GB: ~0.2 s) and independent of the handle's parameters:
// they live in a small process-wide pool, borrowed for one run and returned (a handle is created per reduce_noise() call).
struct PinnedPool {
    std::mutex mu;
    std::vector<std::pair<void*, size_t>> free_list;
    std::vector<std::pair<void*, size_t>> leased;          // b200gate_host_alloc: sizes of the buffers callers hold
    // best fit, and never a buffer more than twice the request (a 7 GB result buffer must not end up as a 256 MB slab)
    void* take(size_t bytes, size_t* got) {
        {
            std::lock_guard<std::mutex> lk(mu);
            size_t best = free_list.size();
            for (size_t i = 0; i < free_list.size(); ++i)
                if (free_list[i].second >= bytes && free_list[i].second <= 2 * bytes + (1 << 20) &&
                    (best == free_list.size() || free_list[i].second < free_list[best].second))
                    best = i;
            if (best < free_list.size()) {
                void* p = free_list[best].first;
                *got = free_list[best].second;
                free_list.erase(free_list.begin() + (long)best);
                return p;
            }
        }
        void* p = nullptr;
        if (cudaMallocHost(&p, bytes) != cudaSuccess) { cudaGetLastError(); return nullptr; }
        *got = bytes;
        return p;
    }
    void give(void* p, size_t bytes) {
        if (!p) return;
        std::lock_guard<std::mutex> lk(mu);
        if (free_list.size() >= 8) {                       // keep the 8 largest
            size_t smallest = 0;
            for (size_t i = 1; i < free_list.size(); ++i)
                if (free_list[i].second < free_list[smallest].second) smallest = i;
            if (free_list[smallest].second >= bytes) { cudaFreeHost(p); return; }
            cudaFreeHost(free_list[smallest].first);
            free_list.erase(free_list.begin() + (long)smallest);
        }
        free_list.emplace_back(p, bytes);
    }
    void* lease(size_t bytes) {
        size_t got = 0;
        void* p = take(bytes, &got);
        if (!p) return nullptr;
        std::lock_guard<std::mutex> lk(mu);
        leased.emplace_back(p, got);
        return p;
    }
    void release(void* p) {
        size_t bytes = 0;
        {
            std::lock_guard<std::mutex> lk(mu);
            for (size_t i = 0; i < leased.size(); ++i)
                if (leased[i].first == p) { bytes = leased[i].second; leased.erase(leased.begin() + (long)i); break; }
        }
        if (bytes) give(p, bytes);
    }
};
PinnedPool g_pinned_pool;

// Fill h->stats from the last run's stream-ordered counter copy and stage events (blocks until that run is done).
int resolve_stats(b200gate_handle* h) {
    if (!h->stats_pending) return B200GATE_OK;
    h->stats_pending = false;
    cudaError_t e = cudaEventSynchronize(h->ev_done);
    if (e != cudaSuccess) return fail(h, B200GATE_ERR_CUDA, "CUDA error: %s", cudaGetErrorString(e));
    const Counters cnt = *h->h_cnt;
    float ms = 0.f;
    cudaEventElapsedTime(&ms, h->ev0, h->ev1);
    h->stats.bins_rechecked_fp64 = (int64_t)cnt.rechecked;
    h->stats.bins_unresolved = (int64_t)cnt.unresolved;
    h->stats.rowfloor_flags = (int64_t)cnt.floor_flags;
    h->stats.rowfloor_ambiguous = (int64_t)cnt.floor_ambiguous;
    h->stats.last_run_ms = ms;
    for (size_t b = 0; b < h->pend_batches; ++b) {
        float t1 = 0.f, t2 = 0.f, t3 = 0.f;
        cudaEventElapsedTime(&t1, h->stage_ev[4 * b + 0], h->stage_ev[4 * b + 1]);
        cudaEventElapsedTime(&t2, h->stage_ev[4 * b + 1], h->stage_ev[4 * b + 2]);
        cudaEventElapsedTime(&t3, h->stage_ev[4 * b + 2], h->stage_ev[4 * b + 3]);
        h->stats.k1_ms += t1;
        h->stats.smooth_ms += t2;
        h->stats.k2_ms += t3;
    }
    return B200GATE_OK;
}

}  // namespace

// =============================================================================================
extern "C" {

int b200gate_create(const b200gate_params* p, b200gate_handle** out) {
    if (!p || !out) return fail(nullptr, B200GATE_ERR_ARG, "null argument");
    *out = nullptr;
    if (p->abi_version != B200GATE_ABI_VERSION)
        return fail(nullptr, B200GATE_ERR_ARG, "ABI version %d, library is %d", p->abi_version, B200GATE_ABI_VERSION);
    if (p->surface != B200GATE_SURFACE_NUMPY && p->surface != B200GATE_SURFACE_TORCH)
        return fail(nullptr, B200GATE_ERR_ARG, "unknown surface %d", p->surface);
    const bool geo1k = p->n_fft == kN && p->win_length == kN && p->hop_length == kN / 4;
    const bool geo2k = p->n_fft == kN2 && p->win_length == kN2 && p->hop_length == kN2 / 4 &&
                       p->surface == B200GATE_SURFACE_NUMPY && !p->stationary;
    // everything else the reference accepts on the numpy surface runs on the general-geometry family
    // (path_flags bit 2 forces it for the tuned geometries too: the float64 cross-check of the fast kernels)
    // ... and so does a smoothing filter beyond what the tuned integer kernels hold (16-bit mask numerators, 64 taps a side)
    const bool big_filter = p->n_grad_freq > 64 || p->n_grad_time > 64 ||
                            (long long)(p->n_grad_freq + 1) * (p->n_grad_freq + 1) * (p->n_grad_time + 1) * (p->n_grad_time + 1) > 65535;
    const bool want_generic = (!geo1k && !geo2k) || (p->path_flags & 4) || big_filter;
    int logN = 0;
    while ((1 << logN) < p->n_fft) ++logN;
    if (want_generic) {
        const bool pow2 = (1 << logN) == p->n_fft;
        const bool size_ok = p->n_fft >= 8 && p->n_fft <= (pow2 ? 8192 : 4096);
        if (!size_ok || p->win_length < 1 || p->win_length > p->n_fft || p->hop_length < 1 || p->hop_length > p->win_length)
            return fail(nullptr, B200GATE_ERR_ARG,
                        "unsupported STFT geometry n_fft=%d win_length=%d hop_length=%d (%s gate, %s surface): n_fft must "
                        "be in [8, 8192] if a power of two, else in [8, 4096], with 1 <= hop_length <= win_length <= n_fft",
                        p->n_fft, p->win_length, p->hop_length, p->stationary ? "stationary" : "non-stationary",
                        p->surface == B200GATE_SURFACE_NUMPY ? "numpy" : "torch");
    }
    if (p->n_grad_freq < 0 || p->n_grad_time < 0 || p->n_grad_freq > 65535 || p->n_grad_time > 65535)
        return fail(nullptr, B200GATE_ERR_ARG, "smoothing extents out of range (%d, %d)", p->n_grad_freq, p->n_grad_time);
    if (p->padding < 0) return fail(nullptr, B200GATE_ERR_ARG, "padding must be >= 0");
    // TorchGate asserts 0 <= prop_decrease <= 1 (torchgate.py:52); reduce_noise() takes any value (stationary.py:108)
    if (!std::isfinite(p->prop_decrease) ||
        (p->surface == B200GATE_SURFACE_TORCH && !(p->prop_decrease >= 0.0 && p->prop_decrease <= 1.0)))
        return fail(nullptr, B200GATE_ERR_ARG, "prop_decrease must be finite (and in [0, 1] on the torch surface)");
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0)
        return fail(nullptr, B200GATE_ERR_CUDA, "no CUDA device (%s); this library has no CPU fallback",
                    e == cudaSuccess ? "device count 0" : cudaGetErrorString(e));
    b200gate_handle* h = new b200gate_handle();
    h->p = *p;
    int dev = 0;
    cudaGetDevice(&dev);
    h->device = dev;
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, dev) == cudaSuccess) h->num_sm = prop.multiProcessorCount;
    if (p->reserve_sms > 0 && p->reserve_sms < h->num_sm) h->num_sm -= p->reserve_sms;   // leave room for NCCL
    h->generic = want_generic;
    h->g_logN = logN;
    if (want_generic && (1 << logN) != p->n_fft) {              // Bluestein: M = 2^k >= 2 n_fft - 1
        while ((1 << h->g_logM) < 2 * p->n_fft - 1) ++h->g_logM;
        h->g_M = 1 << h->g_logM;
    }
    h->F = want_generic ? p->n_fft / 2 + 1 : (p->n_fft == kN2 ? kF2 : kF);
    int rc = want_generic ? build_generic_tables(h) : build_static_tables(h);
    if (rc == B200GATE_OK) {
        e = cudaMalloc((void**)&h->d_cnt, sizeof(Counters));
        if (e == cudaSuccess) e = cudaMalloc((void**)&h->d_need_rowmax, sizeof(unsigned));
        if (e == cudaSuccess) e = cudaMallocHost((void**)&h->h_cnt, sizeof(Counters));
        if (e == cudaSuccess) e = cudaEventCreate(&h->ev0);
        if (e == cudaSuccess) e = cudaEventCreate(&h->ev1);
        if (e == cudaSuccess) e = cudaEventCreate(&h->ev_done);
        if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&h->s_h2d, cudaStreamNonBlocking);
        if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&h->s_d2h, cudaStreamNonBlocking);
        if (e != cudaSuccess) rc = fail(h, B200GATE_ERR_CUDA, "handle resources: %s", cudaGetErrorString(e));
    }
    if (rc == B200GATE_OK) {
#ifndef B200_CUSIM_BUILD
        for (int dt = 0; dt < 3; ++dt)
            B200_WITH_DTYPE(dt, {
                cudaFuncSetAttribute(k1_analyze<8, T>, cudaFuncAttributeMaxDynamicSharedMemorySize, k1_smem_floats() * 4);
                cudaFuncSetAttribute(k1n_magnitude<8, T>, cudaFuncAttributeMaxDynamicSharedMemorySize, k1n_smem_floats() * 4);
                cudaFuncSetAttribute(k1d_analyze<8, T>, cudaFuncAttributeMaxDynamicSharedMemorySize, k1d_smem_bytes());
                cudaFuncSetAttribute(k2d_synthesize<8, false, T>, cudaFuncAttributeMaxDynamicSharedMemorySize, k2d_smem_bytes());
                cudaFuncSetAttribute(k2d_synthesize<8, true, T>, cudaFuncAttributeMaxDynamicSharedMemorySize, k2d_smem_bytes());
                cudaFuncSetAttribute(k2c_synthesize<8, kMaskU16, T>, cudaFuncAttributeMaxDynamicSharedMemorySize, k2c_smem_bytes<kMaskU16>());
                cudaFuncSetAttribute(k2c_synthesize<8, kMaskU16Blend, T>, cudaFuncAttributeMaxDynamicSharedMemorySize, k2c_smem_bytes<kMaskU16Blend>());
                cudaFuncSetAttribute(k2c_synthesize<8, kMaskF32, T>, cudaFuncAttributeMaxDynamicSharedMemorySize, k2c_smem_bytes<kMaskF32>());
            });
        cudaFuncSetAttribute(k_smooth_f, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
        cudaFuncSetAttribute(k_smooth_stream, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
        for (int nfb = 1; nfb <= 12; ++nfb) smooth_box_dispatch(SmoothFArgs{}, nfb, dim3(1), 0, nullptr, true);
        cudaFuncSetAttribute(k1n_magnitude_2k, cudaFuncAttributeMaxDynamicSharedMemorySize, k1n2_smem_floats() * 4);
        cudaFuncSetAttribute(k2c_synthesize_2k, cudaFuncAttributeMaxDynamicSharedMemorySize, k2c2_smem_bytes());
        cudaFuncSetAttribute(k_smooth_generic, cudaFuncAttributeMaxDynamicSharedMemorySize, 160 * 1024);
        for (int dt = 0; dt < 3; ++dt)
            B200_WITH_DTYPE(dt, { cudaFuncSetAttribute(gk_stft<T>, cudaFuncAttributeMaxDynamicSharedMemorySize, 8192 * 16); });
        cudaFuncSetAttribute(gk_istft, cudaFuncAttributeMaxDynamicSharedMemorySize, 8192 * 16);
#endif
    }
    if (rc != B200GATE_OK) {
        g_create_error = h->err;
        b200gate_destroy(h);
        return rc;
    }
    *out = h;
    return B200GATE_OK;
}

void b200gate_destroy(b200gate_handle* h) {
    if (!h) return;
    int cur_dev = 0;
    cudaGetDevice(&cur_dev);
    if (cur_dev != h->device) cudaSetDevice(h->device);
    cudaDeviceSynchronize();                                 // nothing of this handle is in flight when its buffers change hands
    g_device_pool.give(h->d_ws_buf, h->ws_bytes, h->device);
    g_device_pool.give(h->d_in, h->in_bytes, h->device);
    g_device_pool.give(h->d_out, h->out_bytes, h->device);
    g_device_pool.give(h->d_raw, h->raw_bytes, h->device);
    void* ptrs[] = {h->d_wa, h->d_ws, h->d_invn, h->d_thr4, h->d_gco, h->d_floor4, h->d_ef, h->d_tw, h->d_thr2_64,
                    h->d_wa64, h->d_cs64, h->d_tthr, h->d_wa2, h->d_ws2, h->d_w2k, h->d_invn2, h->d_cnt, h->d_dbg_spec,
                    h->d_dbg_mask, h->d_dbg_bits, h->d_gwa, h->d_gws, h->d_gw2, h->d_gthr, h->d_gcs, h->d_gtthr, h->d_gchirp, h->d_gbbr};
    for (void* p : ptrs)
        if (p) cudaFree(p);
    if (h->ev0) cudaEventDestroy(h->ev0);
    if (h->ev1) cudaEventDestroy(h->ev1);
    if (h->ev_done) cudaEventDestroy(h->ev_done);
    for (cudaEvent_t e : h->group_ev) cudaEventDestroy(e);
    if (h->h_cnt) cudaFreeHost(h->h_cnt);
    for (int i = 0; i < 2; ++i) { g_pinned_pool.give(h->hp_in[i], h->hp_in_bytes[i]); g_pinned_pool.give(h->hp_out[i], h->hp_out_bytes[i]); }
    if (h->d_need_rowmax) cudaFree(h->d_need_rowmax);
    for (cudaEvent_t e : h->stage_ev) cudaEventDestroy(e);
    for (cudaEvent_t e : h->pipe_ev) cudaEventDestroy(e);
    if (h->s_h2d) cudaStreamDestroy(h->s_h2d);
    if (h->s_d2h) cudaStreamDestroy(h->s_d2h);
    for (int i = 0; i < 2; ++i) {
        g_device_pool.give(h->d_slab_in[i], h->slab_in_bytes[i], h->device);
        g_device_pool.give(h->d_slab_out[i], h->slab_out_bytes[i], h->device);
    }
    if (cur_dev != h->device) cudaSetDevice(cur_dev);
    delete h;
}

const char* b200gate_last_error(const b200gate_handle* h) { return h ? h->err.c_str() : g_create_error.c_str(); }

int b200gate_set_noise_threshold(b200gate_handle* h, const double* thresh_db, int32_t n_bins) {
    if (!h || !thresh_db) return B200GATE_ERR_ARG;
    const int F = h->generic ? h->F : kF;
    if (n_bins != F) return fail(h, B200GATE_ERR_ARG, "expected %d bins, got %d", F, n_bins);
    h->thr.assign(thresh_db, thresh_db + F);
    h->mean.assign(F, NAN);
    h->sd.assign(F, NAN);
    if (h->generic) {
        int rc = upload(h, &h->d_gthr, h->thr);
        if (rc == B200GATE_OK) h->have_thresh = true;
        return rc;
    }
    return build_threshold_tables(h);
}

int b200gate_get_noise_threshold(const b200gate_handle* h, double* thresh_db, int32_t n_bins) {
    if (!h || !thresh_db || n_bins != (h->generic ? h->F : kF) || !h->have_thresh) return B200GATE_ERR_STATE;
    memcpy(thresh_db, h->thr.data(), (size_t)n_bins * sizeof(double));
    return B200GATE_OK;
}

int b200gate_get_noise_mean_std(const b200gate_handle* h, double* mean_db, double* std_db, int32_t n_bins) {
    if (!h || n_bins != (h->generic ? h->F : kF) || !h->have_thresh) return B200GATE_ERR_STATE;
    if (mean_db) memcpy(mean_db, h->mean.data(), (size_t)n_bins * sizeof(double));
    if (std_db) memcpy(std_db, h->sd.data(), (size_t)n_bins * sizeof(double));
    return B200GATE_OK;
}

int b200gate_set_window(b200gate_handle* h, const float* window, int32_t win_length) {
    if (!h || !window) return B200GATE_ERR_ARG;
    if (h->generic) {
        if (win_length != h->p.win_length) return fail(h, B200GATE_ERR_ARG, "window length %d != win_length %d", win_length, h->p.win_length);
        h->user_window.assign(window, window + win_length);
        return build_generic_tables(h);
    }
    if (win_length != h->p.n_fft) return fail(h, B200GATE_ERR_ARG, "window length %d != n_fft %d", win_length, h->p.n_fft);
    h->user_window.assign(window, window + win_length);
    return build_static_tables(h);
}

int b200gate_channel_sum(b200gate_handle* h, const void* y, int dtype, int64_t C, int64_t n, int64_t stride,
                         int is_device, void* acc, int init, void* stream) {
    if (!h || !y || !acc || C <= 0 || n <= 0 || dtype_size(dtype) == 0) return fail(h, B200GATE_ERR_ARG, "bad argument");
    return channel_sum_impl(h, y, dtype, C, n, stride, is_device, acc, init, (cudaStream_t)stream);
}

void* b200gate_host_alloc(size_t bytes) {
    if (bytes == 0) return nullptr;
#ifdef B200_CUSIM_BUILD
    return malloc(bytes);
#else
    return g_pinned_pool.lease(bytes);
#endif
}
void b200gate_host_free(void* p) {
    if (!p) return;
#ifdef B200_CUSIM_BUILD
    free(p);
#else
    g_pinned_pool.release(p);
#endif
}

int b200gate_noise_stats_collapsed(b200gate_handle* h, const void* noise_mean, int dtype, int64_t n, int is_device,
                                   void* stream) {
    if (!h || !noise_mean || n <= 0) return fail(h, B200GATE_ERR_ARG, "bad argument");
    if (dtype != B200GATE_F32 && dtype != B200GATE_F64) return fail(h, B200GATE_ERR_ARG, "collapsed noise must be f32 or f64");
    cudaStream_t st = (cudaStream_t)stream;
    const size_t es = dtype_size(dtype);
    Scratch s_src, s_yn;
    CK(h, s_yn.alloc((size_t)n * sizeof(double)));
    double* d_yn = s_yn.as<double>();
    const void* src = noise_mean;
    if (!is_device) {
        CK(h, s_src.alloc((size_t)n * es));
        CK(h, cudaMemcpyAsync(s_src.p, noise_mean, (size_t)n * es, cudaMemcpyHostToDevice, st));
        src = s_src.p;
    }
    if (dtype == B200GATE_F32)
        { auto kern_ = k0_mean_to_f64<float>; B200_LAUNCH(kern_, dim3(grid_1d(n, 256, 4096)), dim3(256), 0, st, (const float*)src, (long long)n, 1LL, d_yn); }
    else
        { auto kern_ = k0_mean_to_f64<double>; B200_LAUNCH(kern_, dim3(grid_1d(n, 256, 4096)), dim3(256), 0, st, (const double*)src, (long long)n, 1LL, d_yn); }
    return noise_stats_from_mean(h, d_yn, n, st);          // synchronises the stream before the scratch is freed
}

int b200gate_noise_stats(b200gate_handle* h, const void* y_noise, int dtype, int64_t C, int64_t N, int64_t stride,
                         int is_device, void* stream) {
    if (!h || !y_noise || C <= 0 || N <= 0 || dtype_size(dtype) == 0) return fail(h, B200GATE_ERR_ARG, "bad argument");
    cudaStream_t st = (cudaStream_t)stream;
    long long n = N;
    if (h->p.clip_noise && h->p.chunk_size > 0 && n > h->p.chunk_size) n = h->p.chunk_size;   // stationary.py:63-64
    const bool f32 = (dtype == B200GATE_F32);
    Scratch s_acc, s_yn;
    CK(h, s_acc.alloc((size_t)n * (f32 ? 4 : 8)));
    CK(h, s_yn.alloc((size_t)n * sizeof(double)));
    void* d_acc = s_acc.p;
    double* d_yn = s_yn.as<double>();
    int rc = channel_sum_impl(h, y_noise, dtype, C, n, stride, is_device, d_acc, 1, st);
    if (rc == B200GATE_OK) {
        if (f32)
            { auto kern_ = k0_mean_to_f64<float>; B200_LAUNCH(kern_, dim3(grid_1d(n, 256, 4096)), dim3(256), 0, st, (const float*)d_acc, n, (long long)C, d_yn); }
        else
            { auto kern_ = k0_mean_to_f64<double>; B200_LAUNCH(kern_, dim3(grid_1d(n, 256, 4096)), dim3(256), 0, st, (const double*)d_acc, n, (long long)C, d_yn); }
        rc = noise_stats_from_mean(h, d_yn, n, st);
    }
    return rc;
}

int b200gate_debug_select_unit(b200gate_handle* h, int64_t chunk, int64_t channel) {
    if (!h) return B200GATE_ERR_ARG;
    h->dbg_chunk = chunk;
    h->dbg_channel = channel;
    return B200GATE_OK;
}

int b200gate_debug_dims(const b200gate_handle* h, int64_t* T, int32_t* F, int32_t* words) {
    if (!h) return B200GATE_ERR_ARG;
    if (T) *T = h->dbg_T;
    if (F) *F = h->generic ? h->F : (h->p.n_fft == kN2 ? kF2 : kF);
    if (words) *words = h->generic ? (h->F + 31) / 32 : (h->p.n_fft == kN2 ? kFW2 : kFW);
    return B200GATE_OK;
}

int b200gate_debug_read_bits(b200gate_handle* h, uint32_t* bits) {
    if (!h || !bits || !h->d_dbg_bits || h->dbg_T <= 0) return B200GATE_ERR_STATE;
    if (!h->generic && h->p.n_fft == kN2) { memset(bits, 0, (size_t)h->dbg_T * kFW2 * 4); return B200GATE_OK; }   // no binary mask in this family
    CK(h, cudaDeviceSynchronize());
    CK(h, cudaMemcpy(bits, h->d_dbg_bits, (size_t)h->dbg_T * (h->generic ? (h->F + 31) / 32 : kFW) * 4, cudaMemcpyDeviceToHost));
    return B200GATE_OK;
}
int b200gate_debug_read_mask(b200gate_handle* h, float* mask) {
    if (!h || !mask || !h->d_dbg_mask || h->dbg_T <= 0) return B200GATE_ERR_STATE;
    CK(h, cudaDeviceSynchronize());
    CK(h, cudaMemcpy(mask, h->d_dbg_mask, (size_t)h->dbg_T * (h->generic ? h->F : (h->p.n_fft == kN2 ? kF2 : kF)) * 4, cudaMemcpyDeviceToHost));
    return B200GATE_OK;
}
int b200gate_debug_read_spec(b200gate_handle* h, float* spec) {
    if (!h || !spec || !h->d_dbg_spec || h->dbg_T <= 0) return B200GATE_ERR_STATE;
    CK(h, cudaDeviceSynchronize());
    CK(h, cudaMemcpy(spec, h->d_dbg_spec, (size_t)h->dbg_T * (h->generic ? h->F : (h->p.n_fft == kN2 ? kF2 : kF)) * 8, cudaMemcpyDeviceToHost));
    return B200GATE_OK;
}

int b200gate_set_range(b200gate_handle* h, int32_t mode, int64_t a, int64_t b) {
    if (!h) return B200GATE_ERR_ARG;
    if (mode < 0 || mode > 2 || (mode == 1 && (a < 0 || b < a)) || (mode == 2 && a <= 0))
        return fail(h, B200GATE_ERR_ARG, "bad range (mode %d, %lld, %lld)", mode, (long long)a, (long long)b);
    h->range_mode = mode; h->range_a = a; h->range_b = b;
    return B200GATE_OK;
}

int b200gate_get_stats(const b200gate_handle* h, b200gate_stats* out) {
    if (!h || !out) return B200GATE_ERR_ARG;
    const int rc = resolve_stats(const_cast<b200gate_handle*>(h));
    if (rc) return rc;
    *out = h->stats;
    return B200GATE_OK;
}

int b200gate_torch_set_noise(b200gate_handle* h, const void* xn, int dtype, int64_t Bn, int64_t Ln, int64_t stride,
                             int is_device, void* stream) {
    if (!h) return B200GATE_ERR_ARG;
    if (h->p.surface != B200GATE_SURFACE_TORCH) return fail(h, B200GATE_ERR_STATE, "torch surface only");
    if (!xn) { h->tthr_units = 0; return B200GATE_OK; }
    const bool f64 = dtype == B200GATE_F64 && h->generic;            // float64 noise clips: general family only
    if (Bn <= 0 || Ln <= 0 || (dtype != B200GATE_F32 && !f64))
        return fail(h, B200GATE_ERR_ARG, "xn must be float32 [Bn][Ln] (float64 on the general-geometry family)");
    cudaStream_t st = (cudaStream_t)stream;
    const size_t xes = f64 ? 8 : 4;
    const float* x = (const float*)xn;
    Scratch s_tmp;
    long long xs = stride;
    if (!is_device) {
        CK(h, s_tmp.alloc((size_t)Bn * Ln * xes));
        CK(h, cudaMemcpy2DAsync(s_tmp.p, (size_t)Ln * xes, xn, (size_t)stride * xes, (size_t)Ln * xes, (size_t)Bn, cudaMemcpyHostToDevice, st));
        x = s_tmp.as<float>(); xs = Ln;
    }
    Geom g{};
    g.H = h->p.hop_length; g.C = (int)Bn; g.n_total = Ln; g.step = Ln; g.n_chunks = 1; g.pad = 0; g.Lp = Ln;
    g.T = (int)(Ln / g.H) + 1; g.in_stride = xs; g.out_stride = xs; g.u0 = 0; g.n_units = (int)Bn;
    if (h->generic) {                                  // general family: float64 statistics of xn's own frames
        const int F = h->F, N = h->p.n_fft;
        if (Bn > 65535) return fail(h, B200GATE_ERR_ARG, "xn has too many rows");
        Scratch s_gX, s_gD;
        CK(h, s_gX.alloc((size_t)Bn * g.T * F * sizeof(double2)));
        CK(h, s_gD.alloc((size_t)Bn * g.T * F * sizeof(double)));
        double2* gX = s_gX.as<double2>();
        double* gD = s_gD.as<double>();
        if (h->d_gtthr) cudaFree(h->d_gtthr);
        h->d_gtthr = nullptr;
        CK(h, cudaMalloc((void**)&h->d_gtthr, (size_t)Bn * F * sizeof(double)));
        if (f64) {
            GStftArgs<double> sa{};
            sa.gg = generic_geom(h, g); sa.tb = generic_tables(h); sa.x = (const double*)(const void*)x; sa.X = gX;
            auto kern_ = gk_stft<double>;
            B200_LAUNCH(kern_, dim3((unsigned)g.T, (unsigned)Bn), dim3(generic_threads(generic_fft_len(h))), (size_t)generic_fft_len(h) * sizeof(double2), st, sa);
        } else {
            GStftArgs<float> sa{};
            sa.gg = generic_geom(h, g); sa.tb = generic_tables(h); sa.x = x; sa.X = gX;
            auto kern_ = gk_stft<float>;
            B200_LAUNCH(kern_, dim3((unsigned)g.T, (unsigned)Bn), dim3(generic_threads(generic_fft_len(h))), (size_t)generic_fft_len(h) * sizeof(double2), st, sa);
        }
        GTStatArgs ta{};
        ta.n_units = (int)Bn; ta.T = g.T; ta.F = F; ta.ddof = h->p.std_ddof; ta.eps = kEps64; ta.top_db = h->p.top_db;
        ta.n_std = h->p.n_std_thresh; ta.X = gX; ta.scratch = gD; ta.thr = h->d_gtthr;
        B200_LAUNCH(gk_tstats, dim3((unsigned)(((long long)Bn * F + 127) / 128)), dim3(128), 0, st, ta);
        CK(h, cudaGetLastError());
        CK(h, cudaStreamSynchronize(st));
        h->tthr_units = (int)Bn;
        return B200GATE_OK;
    }
    Scratch s_mag, s_rowmax;
    CK(h, s_mag.alloc((size_t)Bn * g.T * kFPad * 4));
    CK(h, s_rowmax.alloc((size_t)Bn * kFPad * 4));
    float *mag = s_mag.as<float>(), *rowmax = s_rowmax.as<float>();
    if (h->d_tthr) cudaFree(h->d_tthr);
    h->d_tthr = nullptr;
    CK(h, cudaMalloc((void**)&h->d_tthr, (size_t)Bn * kFPad * 4));
    DebugTap dbg{}; dbg.ul = -1;
    launch_k1n(g, device_tables(h), x, B200GATE_F32, mag, dbg, h->num_sm * 3, st);
    TStatArgs ta{};
    ta.n_units = (int)Bn; ta.T = g.T; ta.in_scale = (float)h->sum_w; ta.eps = (float)kEps64; ta.top_db = (float)h->p.top_db;
    ta.n_std = (float)h->p.n_std_thresh; ta.ddof = h->p.std_ddof; ta.mag = mag; ta.rowmax = rowmax; ta.thr = h->d_tthr;
    B200_LAUNCH(k_tgate_stats, dim3((unsigned)(Bn * kFW)), dim3(kTgWarps * 32), 0, st, ta);
    CK(h, cudaGetLastError());
    CK(h, cudaStreamSynchronize(st));
    h->tthr_units = (int)Bn;
    return B200GATE_OK;
}

int b200gate_run(b200gate_handle* h, const void* in, void* out, int dtype, int64_t C, int64_t N, int64_t in_stride,
                 int64_t out_stride, int is_device, void* stream) {
    if (!h || !in || !out || C <= 0 || N <= 0 || dtype_size(dtype) == 0) return fail(h, B200GATE_ERR_ARG, "bad argument");
    const bool torch_sem = h->p.surface == B200GATE_SURFACE_TORCH;
    // torch.istft(center=True) length: n_fft + hop (T - 1) minus n_fft/2 at both ends (torchgate.py:255-262)
    const int64_t No = torch_sem ? (N / h->p.hop_length) * h->p.hop_length + (h->p.n_fft & 1) : N;
    // In a range mode only samples [o_lo, o_hi) of a row are addressed, so `out` may be a virtual base
    // (slab - o_lo) over rows as short as the range: the stride check below uses the range length.
    if (in_stride < N || (out_stride < No && (torch_sem || h->range_mode == 0)))
        return fail(h, B200GATE_ERR_ARG, "row strides too small");
    if (torch_sem && N < 2 * h->p.win_length) return fail(h, B200GATE_ERR_ARG, "x must be bigger than %d", 2 * h->p.win_length);
    if (torch_sem && h->tthr_units > 1 && h->tthr_units != C)
        return fail(h, B200GATE_ERR_ARG, "xn has %d rows, x has %lld", h->tthr_units, (long long)C);
    if (h->p.stationary && !torch_sem && !h->have_thresh)
        return fail(h, B200GATE_ERR_STATE, "stationary gate: call b200gate_noise_stats first");
    cudaStream_t st = (cudaStream_t)stream;
    const b200gate_params& p = h->p;
    const size_t es = dtype_size(dtype);
    h->stats = b200gate_stats{};
    long long launches = 0;
    if (!h->reuse_masks) h->masks_valid = false;

    // ---- which part of the recording (base.py:167-226; b200gate_set_range) -----------------------------
    // range_mode 2: the reference's single padded chunk [0, a) inside a longer recording (base.py:222)
    const bool single_to = !torch_sem && h->range_mode == 2;
    if (single_to && h->range_a > N) return fail(h, B200GATE_ERR_ARG, "range end %lld beyond the recording", h->range_a);
    const bool chunked = !torch_sem && !single_to && p.chunk_size > 0 && N > p.chunk_size;
    const long long step = chunked ? p.chunk_size : (single_to ? h->range_a : N);
    const long long n_chunks = chunked ? (N - 1) / p.chunk_size + 1 : 1;
    // range_mode 1: a sub-range of the chunk grid
    long long chunk_first = 0, chunk_count = n_chunks;
    if (!torch_sem && h->range_mode == 1) {
        if (!chunked || h->range_b >= n_chunks) return fail(h, B200GATE_ERR_ARG, "chunk range outside the chunk grid");
        chunk_first = h->range_a;
        chunk_count = h->range_b - h->range_a + 1;
    }
    // samples written [o_lo, o_hi) and samples read [w_lo, w_hi)
    const long long o_lo = chunk_first * step;
    const long long o_hi = torch_sem ? No : std::min<long long>(N, (chunk_first + chunk_count) * step);
    const long long rpad = torch_sem ? 0 : p.padding;
    const long long w_lo = torch_sem ? 0 : std::max(0LL, o_lo - rpad);
    const long long w_hi = torch_sem ? N : std::min<long long>(N, o_hi + rpad);
    const long long Wn = w_hi - w_lo, On = o_hi - o_lo;
    if (out_stride < On) return fail(h, B200GATE_ERR_ARG, "output row stride %lld shorter than the range (%lld samples)",
                                     (long long)out_stride, On);

    // ---- where the kernels read / write ---------------------------------------------------------------
    // The n_fft = 1024 numpy-surface kernels are templated on the sample dtype: they read the caller's
    // float32 / int16 / float64 rows directly and cast on store (base.py:140, :218-226).  The 2048 family and
    // the torch surface run on float32 rows (other dtypes are converted at the edge).
    const bool generic = h->generic;
    // (the general family is templated on the sample type on both surfaces: float64 TorchGate input stays float64)
    const bool native = (!torch_sem && p.n_fft == kN) || generic;
    const int kdt = native ? dtype : B200GATE_F32;            // dtype the kernels see
    const size_t kes = dtype_size(kdt);
    const void* x = nullptr;
    void* y = nullptr;
    long long xs = in_stride, ys = out_stride;
    const bool direct = is_device && kdt == dtype;
    // Host input that the reference would chunk: stream it through the GPU slab by slab (H2D of slab k+1,
    // kernels of slab k and D2H of slab k-1 overlap on three streams) instead of staging the whole
    // recording -- the role of _read_chunk + the memmap write-back (base.py:130-187).
    const bool pipelined = !is_device && kdt == dtype && chunked && h->p.padding >= h->p.hop_length;
    if (direct || pipelined) {
        x = in;
        y = out;
    } else {
        // stage the window that is read / written; the kernels keep absolute sample indices through virtual
        // row bases (x - w_lo, y - o_lo)
        int rc;
        if ((rc = ensure(h, (void**)&h->d_in, &h->in_bytes, (size_t)C * Wn * kes))) return rc;
        if ((rc = ensure(h, (void**)&h->d_out, &h->out_bytes, (size_t)C * On * kes))) return rc;
        x = (const char*)h->d_in - (size_t)w_lo * kes;
        y = (char*)h->d_out - (size_t)o_lo * kes;
        xs = Wn;
        ys = On;
        if (kdt == dtype) {                                   // host rows
            CK(h, cudaMemcpy2DAsync(h->d_in, (size_t)Wn * es, (const char*)in + (size_t)w_lo * es, (size_t)in_stride * es,
                                    (size_t)Wn * es, (size_t)C, cudaMemcpyHostToDevice, st));
        } else {                                              // float32-only kernel family: convert at the edge
            const void* raw = (const char*)in + (size_t)w_lo * es;
            long long rs = in_stride;
            if (!is_device) {
                if ((rc = ensure(h, &h->d_raw, &h->raw_bytes, (size_t)C * std::max(Wn, On) * es))) return rc;
                CK(h, cudaMemcpy2DAsync(h->d_raw, (size_t)Wn * es, raw, (size_t)in_stride * es, (size_t)Wn * es, (size_t)C,
                                        cudaMemcpyHostToDevice, st));
                raw = h->d_raw;
                rs = Wn;
            }
            const int gr = grid_1d((long long)C * Wn, 256, h->num_sm * 16);
            if (dtype == B200GATE_I16)
                { auto kern_ = k_to_f32<short>; B200_LAUNCH(kern_, dim3(gr), dim3(256), 0, st, (const short*)raw, (float*)h->d_in, (long long)C, (long long)Wn, rs, (long long)Wn); }
            else
                { auto kern_ = k_to_f32<double>; B200_LAUNCH(kern_, dim3(gr), dim3(256), 0, st, (const double*)raw, (float*)h->d_in, (long long)C, (long long)Wn, rs, (long long)Wn); }
            ++launches;
        }
    }
    float h2d_ms = 0.f;
    cudaEvent_t evk0 = h->ev0, evk1 = h->ev1;

    // ---- geometry (base.py:167-226) -----------------------------------------------------------
    Geom g{};
    g.H = p.hop_length;
    g.C = (int)C;
    g.n_total = N;
    g.step = step;
    g.n_chunks = (int)n_chunks;
    g.pad = torch_sem ? 0 : p.padding;                 // TorchGate filters the whole row, no chunk padding
    g.Lp = g.step + 2 * g.pad;
    g.T = generic ? (int)((g.Lp + 2 * (h->g_W / 2) - h->g_W) / g.H) + 1 : (int)(g.Lp / g.H) + 1;
    g.in_stride = xs;
    g.out_stride = ys;
    const long long U = chunk_count * C;
    const long long Ubase = chunk_first * C;               // first unit of the selected range
    if (Ubase + U > 0x7fffffffLL || g.Lp / g.H > 0x3fffffffLL) return fail(h, B200GATE_ERR_ARG, "problem too large");

    const int NFFT = p.n_fft;
    const bool two_k = NFFT == kN2 && !generic;
    const int FP = two_k ? kFPad2 : kFPad, FF = generic ? h->F : (two_k ? kF2 : kF);
    // frames whose masks k2 needs (same for every full chunk)
    const long long sig_len = (long long)(g.T - 1) * g.H + (generic ? (h->g_W & 1) : 0);
    long long jp_hi = std::min(g.pad + g.step, sig_len);
    int tf_lo = 0, tf_hi = 0;
    int h_lo = 0, h_hi = 0;
    if (jp_hi > g.pad) {
        h_lo = (int)((g.pad + NFFT / 2) / g.H);
        h_hi = (int)((jp_hi + NFFT / 2 + g.H - 1) / g.H);
        tf_lo = std::max(0, h_lo - 3) & ~1;          // even: k2 walks k1's (2j, 2j+1) frame pairs when spectra are cached
        tf_hi = std::min(h_hi, g.T);
    }
    const bool tail_zeros = !torch_sem && !generic && (g.pad + g.step > sig_len);   // (gk_ola writes the zeros itself)     // stationary.py:126 leaves the tail zero
    if (tail_zeros) {
        for (long long c = 0; c < C; ++c)
            CK(h, cudaMemsetAsync((char*)y + ((size_t)c * ys + (size_t)o_lo) * kes, 0, (size_t)On * kes, st));
    }

    // ---- workspace / batching ---------------------------------------------------------------------
    const bool stat = p.stationary != 0;
    const size_t per_unit_2pass = (stat ? (size_t)g.T * kFW * 4 + (size_t)kFPad * 4 + (size_t)kFW * 4 + (size_t)num_unit_stride(g.T) * 2 + 64
                                        : 2 * (size_t)g.T * FP * 4 + 64) +
                                  (stat && torch_sem ? (size_t)g.T * kFPad * 4 + 2 * (size_t)kFPad * 4 : 0) + 2048;
    // spectrum cache of the tuned geometries: k1 / k1n keep the packed spectrum of every frame pair so k2 does not re-transform
    // (n_fft 2048: one half-length spectrum per frame; n_fft 1024: one packed spectrum per frame pair)
    const int zpairs = (g.T + 1) / 2;
    const size_t zunit = generic ? 0 : (size_t)(two_k ? g.T : zpairs) * 1024 * sizeof(float2);
    // dual kernels (gate_dual.cuh): two channels of a chunk per warp -- stationary numpy-surface gate, even channel count
    const bool use_dual = !generic && stat && !torch_sem && native && (C % 2 == 0) && !(p.path_flags & 16);
    // general-geometry family: float64 spectrum, mask, scratch and synthesis frames of every unit
    const size_t g_tf = (size_t)g.T * (size_t)h->F, g_tw = (size_t)g.T * (size_t)h->g_W;
    const size_t per_unit_generic = g_tf * 16 + 2 * g_tf * 8 + g_tw * 8 + 2 * (size_t)h->F * 8 + 6 * 256;
    const size_t per_unit = generic ? per_unit_generic : per_unit_2pass + zunit;
    // default workspace: up to 24 GiB, never more than 70 % of what is free now (plus what this handle already holds)
    double limit = p.workspace_limit_bytes;
    if (!(limit > 0)) {
        limit = 24.0 * 1024 * 1024 * 1024;
        size_t free_b = 0, total_b = 0;
        if (cudaMemGetInfo(&free_b, &total_b) == cudaSuccess)
            limit = std::min(limit, 0.7 * ((double)free_b + (double)h->ws_bytes));
    }
    long long ub = (long long)std::max(1.0, floor(limit / (double)per_unit));
    ub = std::min(ub, U);
    if (use_dual) ub = std::max(2LL, ub & ~1LL);             // duals are units (2d, 2d+1) of a batch
    if (generic) ub = std::min(ub, 65535LL);                 // gk_* put the unit on gridDim.y
    // reserve the workspace now; if the device cannot give it (the caller's own tensors may fill HBM), halve the batch
    for (;;) {
        const size_t est = (size_t)ub * per_unit + ((size_t)8 << 20);
        if (ensure(h, (void**)&h->d_ws_buf, &h->ws_bytes, est) == B200GATE_OK) break;
        cudaGetLastError();
        long long nub = ub / 2;
        if (use_dual) nub &= ~1LL;
        if (nub < (use_dual ? 2 : 1)) return B200GATE_ERR_NOMEM;     // (message set by ensure)
        ub = nub;
    }
    if (!pipelined && ub < U) {
        // several batches: equal ones (a full batch followed by a small remainder would end every kernel of the remainder
        // in a partial wave); the slab pipeline sizes its batches itself below
        const long long nb = (U + ub - 1) / ub;
        long long eq = (U + nb - 1) / nb;
        if (use_dual) eq += eq & 1;
        ub = std::min(ub, std::max(eq, use_dual ? 2LL : 1LL));
    }
    long long slab_chunks = 0, slab_w = 0, slab_ow = 0;
    bool stage_in = false, stage_out = false;
    if (pipelined) {
        // ~256 MB of input per slab (measured on B200 + PCIe Gen5: 160-320 MB best, profiles/r01_e2e_slab_sweep.md), whole chunks, within the workspace limit
        long long slab_bytes = 256LL << 20;
        if (const char* e = getenv("B200GATE_SLAB_MB")) slab_bytes = std::max(1LL, atoll(e)) << 20;     // tuning knob
        slab_chunks = std::max(1LL, std::min<long long>(chunk_count, slab_bytes / std::max<long long>(1, C * g.step * (long long)es)));
        slab_chunks = std::max(1LL, std::min(slab_chunks, ub / C));
        if (ub < C) return fail(h, B200GATE_ERR_NOMEM, "workspace limit too small for one chunk of all channels");
        ub = slab_chunks * C;
        slab_w = slab_chunks * g.step + 2 * g.pad;
        slab_ow = slab_chunks * g.step;
        for (int i = 0; i < 2; ++i) {
            int rc;
            if ((rc = ensure(h, (void**)&h->d_slab_in[i], &h->slab_in_bytes[i], (size_t)C * slab_w * es))) return rc;
            if ((rc = ensure(h, (void**)&h->d_slab_out[i], &h->slab_out_bytes[i], (size_t)C * slab_ow * es))) return rc;
        }
        stage_in = !host_pointer_is_pinned(in);
        stage_out = !host_pointer_is_pinned(out);
        for (int i = 0; i < 2; ++i) {                  // pinned staging slabs for pageable caller memory (process-wide pool)
            if (stage_in && h->hp_in_bytes[i] < (size_t)C * slab_w * es) {
                g_pinned_pool.give(h->hp_in[i], h->hp_in_bytes[i]);
                h->hp_in[i] = g_pinned_pool.take((size_t)C * slab_w * es, &h->hp_in_bytes[i]);
                if (!h->hp_in[i]) { h->hp_in_bytes[i] = 0; return fail(h, B200GATE_ERR_NOMEM, "pinned staging slab (%zu bytes)", (size_t)C * slab_w * es); }
            }
            if (stage_out && h->hp_out_bytes[i] < (size_t)C * slab_ow * es) {
                g_pinned_pool.give(h->hp_out[i], h->hp_out_bytes[i]);
                h->hp_out[i] = g_pinned_pool.take((size_t)C * slab_ow * es, &h->hp_out_bytes[i]);
                if (!h->hp_out[i]) { h->hp_out_bytes[i] = 0; return fail(h, B200GATE_ERR_NOMEM, "pinned staging slab (%zu bytes)", (size_t)C * slab_ow * es); }
            }
        }
        if (const char* e = getenv("B200GATE_HOST_THREADS")) h->host_threads = std::max(1, atoi(e));
    }
    // carve the workspace into 256-byte aligned sub-buffers (vector stores need natural alignment)
    auto al = [](size_t v) { return (v + 255) / 256 * 256; };
    const size_t off_bits = 0;
    const size_t off_rowmax = off_bits + al((size_t)ub * g.T * kFW * 4);
    const size_t off_rowflag = off_rowmax + al((size_t)ub * kFPad * 4);
    const size_t off_num = off_rowflag + al((size_t)ub * kFW * 4);
    const size_t end_stat = off_num + al((size_t)ub * num_unit_stride(g.T) * 2);
    const size_t off_m0 = al((size_t)ub * g.T * FP * 4);
    const size_t end_nonstat = off_m0 + al((size_t)ub * g.T * FP * 4);
    // torch surface, stationary: the stationary buffers follow the dB spectrogram
    const size_t off_tdb = end_stat;
    const size_t off_trow = off_tdb + al((size_t)ub * g.T * kFPad * 4);
    const size_t off_tthr = off_trow + al((size_t)ub * kFPad * 4);
    const size_t end_tstat = off_tthr + al((size_t)ub * kFPad * 4);
    const size_t goff_M = al((size_t)ub * g_tf * 16);
    const size_t goff_tmp = goff_M + al((size_t)ub * g_tf * 8);
    const size_t goff_fr = goff_tmp + al((size_t)ub * g_tf * 8);
    const size_t goff_thr = goff_fr + al((size_t)ub * g_tw * 8);          // torch surface: per-row thresholds
    const size_t goff_rmax = goff_thr + al((size_t)ub * h->F * 8);         // per-(unit, bin) dB maxima (top_db floor)
    const size_t end_generic = goff_rmax + al((size_t)ub * h->F * 8);
    const size_t end_base = generic ? end_generic : (stat ? (torch_sem ? end_tstat : end_stat) : end_nonstat);
    const size_t off_z = al(end_base);
    const size_t end_all = off_z + al((size_t)ub * zunit);
    {
        int rc = ensure(h, (void**)&h->d_ws_buf, &h->ws_bytes, end_all);
        if (rc) return rc;
    }
    float* d_tdb = (float*)(h->d_ws_buf + off_tdb);
    float* d_trow = (float*)(h->d_ws_buf + off_trow);
    float* d_tthr_self = (float*)(h->d_ws_buf + off_tthr);
    float2* d_zcache = generic ? nullptr : (float2*)(h->d_ws_buf + off_z);
    unsigned* d_bits = (unsigned*)(h->d_ws_buf + off_bits);
    unsigned* d_rowmax = (unsigned*)(h->d_ws_buf + off_rowmax);
    unsigned* d_rowflag = (unsigned*)(h->d_ws_buf + off_rowflag);
    unsigned short* d_num = (unsigned short*)(h->d_ws_buf + off_num);
    float* d_mag = (float*)h->d_ws_buf;                        // non-stationary: |X|, later the final mask
    float* d_m0 = (float*)(h->d_ws_buf + off_m0);              //                 forward sweep / sigmoid mask

    CK(h, cudaMemsetAsync(h->d_cnt, 0, sizeof(Counters), st));
    const long long dbg_u = (h->dbg_chunk >= 0 && h->dbg_chunk < g.n_chunks && h->dbg_channel >= 0 && h->dbg_channel < C)
                                ? h->dbg_chunk * C + h->dbg_channel : -1;
    if (dbg_u >= 0) {
        if (h->dbg_T_alloc < (size_t)g.T) {
            if (h->d_dbg_spec) cudaFree(h->d_dbg_spec);
            if (h->d_dbg_mask) cudaFree(h->d_dbg_mask);
            if (h->d_dbg_bits) cudaFree(h->d_dbg_bits);
            const size_t fmax_ = (size_t)std::max(kF2, h->F);
            CK(h, cudaMalloc((void**)&h->d_dbg_spec, (size_t)g.T * fmax_ * 8));
            CK(h, cudaMalloc((void**)&h->d_dbg_mask, (size_t)g.T * fmax_ * 4));
            CK(h, cudaMalloc((void**)&h->d_dbg_bits, (size_t)g.T * std::max<size_t>(kFW, (fmax_ + 31) / 32) * 4));
            h->dbg_T_alloc = g.T;
        }
        CK(h, cudaMemsetAsync(h->d_dbg_spec, 0, (size_t)g.T * FF * 8, st));
        CK(h, cudaMemsetAsync(h->d_dbg_mask, 0, (size_t)g.T * FF * 4, st));
        h->dbg_T = g.T;
    } else {
        h->dbg_T = 0;
    }

    const Tables tb = device_tables(h);
    const int nf = p.n_grad_freq, nt = p.n_grad_time;
    const double D = (double)(nf + 1) * (nf + 1) * (nt + 1) * (nt + 1);
    const int resident = h->num_sm * 3;
    const size_t n_batches = (size_t)((U + ub - 1) / ub);
    while (h->stage_ev.size() < 4 * n_batches) {
        cudaEvent_t e;
        CK(h, cudaEventCreate(&e));
        h->stage_ev.push_back(e);
    }
    while (pipelined && h->pipe_ev.size() < 4 * n_batches) {
        cudaEvent_t e;
        CK(h, cudaEventCreate(&e));
        h->pipe_ev.push_back(e);
    }
    size_t bi = 0;
    int nu_prev = 0;
    long long prev_o0 = 0, prev_o1 = 0;
    std::future<void> out_task;
    cudaEventRecord(evk0, st);
    for (long long u0 = 0; u0 < U; u0 += ub, ++bi) {
        const int nu = (int)std::min(ub, U - u0);
        g.u0 = (int)(Ubase + u0);
        g.n_units = nu;
        const void* xb = x;
        void* yb = y;
        if (pipelined) {
            // slab = chunks [c0, c1): input window [w0, w1) of every channel, output [c0*step, o1)
            const long long c0 = (Ubase + u0) / C, c1 = c0 + nu / C;
            const long long w0 = std::max(0LL, c0 * g.step - g.pad), w1 = std::min<long long>(N, c1 * g.step + g.pad);
            const long long o0 = c0 * g.step, o1 = std::min<long long>(N, c1 * g.step);
            const int ib = (int)(bi & 1);
            // The head of this slab's window -- [w0, pw1), the 2*padding samples around the slab seam -- is already
            // on the device at the tail of the previous slab's buffer: copy it device-to-device and bring only
            // [pw1, w1) over PCIe, so every sample crosses the bus once.
            const long long pw1 = bi == 0 ? w0 : std::min<long long>(N, c0 * g.step + g.pad);
            if (bi >= 1) CK(h, cudaStreamWaitEvent(h->s_h2d, h->pipe_ev[4 * (bi - 1) + 3], 0));   // slab buffer free
            if (w1 > pw1) {
                const void* src = (const char*)in + (size_t)pw1 * es;
                size_t spitch = (size_t)in_stride * es;
                if (stage_in) {
                    // pageable rows: host threads copy them into this slab's pinned staging buffer (free once the H2D of
                    // slab bi-2 has completed), the copy engine takes them from there
                    if (bi >= 2) CK(h, cudaEventSynchronize(h->pipe_ev[4 * (bi - 2) + 0]));
                    parallel_rows_copy(h->hp_in[ib], (size_t)(w1 - pw1) * es, src, spitch, (size_t)(w1 - pw1) * es, (size_t)C,
                                       stage_out ? std::max(1, h->host_threads / 2) : h->host_threads);
                    src = h->hp_in[ib];
                    spitch = (size_t)(w1 - pw1) * es;
                }
                CK(h, cudaMemcpy2DAsync((char*)h->d_slab_in[ib] + (size_t)(pw1 - w0) * es, (size_t)slab_w * es, src, spitch,
                                        (size_t)(w1 - pw1) * es, (size_t)C, cudaMemcpyHostToDevice, h->s_h2d));
            }
            CK(h, cudaEventRecord(h->pipe_ev[4 * bi + 0], h->s_h2d));
            if (bi >= 1 && pw1 > w0) {
                const long long pw0 = std::max(0LL, (c0 - nu_prev / C) * g.step - g.pad);           // previous window start
                CK(h, cudaMemcpy2DAsync(h->d_slab_in[ib], (size_t)slab_w * es,
                                        (const char*)h->d_slab_in[ib ^ 1] + (size_t)(w0 - pw0) * es, (size_t)slab_w * es,
                                        (size_t)(pw1 - w0) * es, (size_t)C, cudaMemcpyDeviceToDevice, st));
            }
            CK(h, cudaEventRecord(h->pipe_ev[4 * bi + 3], st));     // previous buffer's tail consumed (and its kernels done)
            CK(h, cudaStreamWaitEvent(st, h->pipe_ev[4 * bi + 0], 0));
            if (bi >= 2) CK(h, cudaStreamWaitEvent(st, h->pipe_ev[4 * (bi - 2) + 2], 0));         // output buffer drained
            // virtual row bases so the kernels keep absolute sample indices
            xb = (const char*)h->d_slab_in[ib] - (size_t)w0 * es;
            yb = (char*)h->d_slab_out[ib] - (size_t)o0 * es;
            g.in_stride = slab_w;
            g.out_stride = slab_ow;
            (void)o1;
        }
        DebugTap dbg{};
        dbg.ul = (dbg_u >= Ubase + u0 && dbg_u < Ubase + u0 + nu) ? (int)(dbg_u - Ubase - u0) : -1;
        dbg.spec = h->d_dbg_spec;
        dbg.mask = h->d_dbg_mask;

        if (generic) {
            GGeom gg = generic_geom(h, g);
            if (torch_sem) gg.out_len = No;                 // torch.istft length (torchgate.py:255-262)
            const GTables gt = generic_tables(h);
            const int F = h->F, W = h->g_W, FW = (F + 31) / 32;
            double2* gX = (double2*)h->d_ws_buf;
            double* gM = (double*)(h->d_ws_buf + goff_M);
            double* gTmp = (double*)(h->d_ws_buf + goff_tmp);
            double* gFr = (double*)(h->d_ws_buf + goff_fr);
            const int thr_fft = generic_threads(generic_fft_len(h));
            const size_t smem_fft = (size_t)generic_fft_len(h) * sizeof(double2);
            const bool smooth = nf > 0 || nt > 0;
            if (dbg.ul >= 0) CK(h, cudaMemsetAsync(h->d_dbg_bits, 0, (size_t)g.T * FW * 4, st));
            cudaEventRecord(h->stage_ev[4 * bi + 0], st);
            B200_WITH_DTYPE(kdt, {
                GStftArgs<T> sa{};
                sa.gg = gg; sa.tb = gt; sa.x = (const T*)xb; sa.X = gX;
                auto kern_ = gk_stft<T>;
                B200_LAUNCH(kern_, dim3((unsigned)g.T, (unsigned)nu), dim3(thr_fft), smem_fft, st, sa); });
            const int gr_elem = grid_1d((long long)nu * g.T * F, 256, h->num_sm * 16);
            if (stat) {
                unsigned long long* gRmax = (unsigned long long*)(h->d_ws_buf + goff_rmax);
                CK(h, cudaMemsetAsync(gRmax, 0, (size_t)nu * F * 8, st));
                GDbArgs ba{};
                ba.n_units = nu; ba.T = g.T; ba.F = F; ba.eps = kEps64; ba.X = gX; ba.M = gM; ba.rowmax = gRmax;
                B200_LAUNCH(gk_db_rowmax, dim3((unsigned)((F + 63) / 64), (unsigned)((g.T + 63) / 64), (unsigned)nu), dim3(256), 0, st, ba);
                ++launches;
                GDecideArgs da{};
                da.n_units = nu; da.T = g.T; da.F = F; da.top_db = p.top_db; da.p = p.prop_decrease;
                da.thr = h->d_gthr; da.thr_units = 1; da.rowmax = gRmax;
                da.M = gM; da.dbg_ul = dbg.ul; da.FW = FW; da.dbg_bits = h->d_dbg_bits;
                if (torch_sem) {                        // torchgate.py:127-165: per-row statistics (own frames or xn's)
                    if (h->tthr_units > 0) {
                        da.thr = h->tthr_units == 1 ? h->d_gtthr : h->d_gtthr + (size_t)u0 * F;
                        da.thr_units = h->tthr_units == 1 ? 1 : nu;
                    } else {
                        double* gThr = (double*)(h->d_ws_buf + goff_thr);
                        GTStatArgs ta{};
                        ta.n_units = nu; ta.T = g.T; ta.F = F; ta.ddof = p.std_ddof; ta.eps = kEps64; ta.top_db = p.top_db;
                        ta.n_std = p.n_std_thresh; ta.X = gX; ta.scratch = gM; ta.thr = gThr;
                        B200_LAUNCH(gk_tstats, dim3((unsigned)(((long long)nu * F + 127) / 128)), dim3(128), 0, st, ta);
                        ++launches;
                        da.thr = gThr;
                        da.thr_units = nu;
                    }
                }
                B200_LAUNCH(gk_decide, dim3(gr_elem), dim3(256), 0, st, da);
            } else if (torch_sem) {                     // torchgate.py:168-198: moving-mean follower
                GMovArgs ma{};
                ma.n_units = nu; ma.T = g.T; ma.F = F; ma.n = std::max(1, p.n_movemean); ma.n_thresh = p.thresh_n_mult;
                ma.inv_temp = p.sigmoid_slope; ma.p = p.prop_decrease; ma.X = gX; ma.M = gM; ma.tmp = gTmp;
                B200_LAUNCH(gk_movmean, dim3((unsigned)(((long long)nu * F + 127) / 128)), dim3(128), 0, st, ma);
            } else {
                const double tfr = p.time_constant_s * p.sr / (double)p.hop_length;       // nonstationary.py:109-114
                B200_LAUNCH(gk_abs, dim3(gr_elem), dim3(256), 0, st, (const double2*)gX, (long long)nu * g.T * F, gM);
                GFollowArgs fa{};
                fa.n_units = nu; fa.T = g.T; fa.F = F; fa.b = (sqrt(1.0 + 4.0 * tfr * tfr) - 1.0) / (2.0 * tfr * tfr);
                fa.A = gM; fa.S = gTmp;
                B200_LAUNCH(gk_follow, dim3((unsigned)(((long long)nu * F + 127) / 128)), dim3(128), 0, st, fa);
                GSigmoidArgs ga{};
                ga.n = (long long)nu * g.T * F; ga.n_mult = p.thresh_n_mult; ga.slope = p.sigmoid_slope; ga.p = p.prop_decrease;
                ga.blend = smooth ? 0 : 1; ga.S = gTmp; ga.M = gM;
                B200_LAUNCH(gk_sigmoid, dim3(gr_elem), dim3(256), 0, st, ga);
                launches += 2;
            }
            cudaEventRecord(h->stage_ev[4 * bi + 1], st);
            launches += 2;
            if (smooth) {
                GSmoothArgs ga{};
                ga.n_units = nu; ga.T = g.T; ga.F = F; ga.nf = nf; ga.nt = nt; ga.inv_D = 1.0 / D; ga.p = p.prop_decrease;
                ga.blend = (stat || torch_sem) ? 0 : 1;                                  // stationary.py / torchgate.py blend before smoothing
                const int gr = grid_1d((long long)nu * g.T * F, 256, h->num_sm * 16);
                ga.src = gM; ga.dst = gTmp;
                B200_LAUNCH(gk_smooth_f, dim3(gr), dim3(256), 0, st, ga);
                ga.src = gTmp; ga.dst = gM;
                B200_LAUNCH(gk_smooth_t, dim3(gr), dim3(256), 0, st, ga);
                launches += 2;
            }
            cudaEventRecord(h->stage_ev[4 * bi + 2], st);
            {
                GIstftArgs ia{};
                ia.gg = gg; ia.tb = gt; ia.X = gX; ia.M = gM; ia.frames = gFr; ia.dbg_ul = dbg.ul;
                ia.dbg_spec = (float2*)h->d_dbg_spec; ia.dbg_mask = h->d_dbg_mask;
                B200_LAUNCH(gk_istft, dim3((unsigned)g.T, (unsigned)nu), dim3(thr_fft), smem_fft, st, ia);
                const long long out_max = torch_sem ? No : std::min<long long>(g.step, N);
                B200_WITH_DTYPE(kdt, {
                    GOlaArgs<T> oa{};
                    oa.gg = gg; oa.tb = gt; oa.frames = gFr; oa.y = (T*)yb;
                    auto kern_ = gk_ola<T>;
                    B200_LAUNCH(kern_, dim3((unsigned)grid_1d(out_max, 256, 1 << 16), (unsigned)nu), dim3(256), 0, st, oa); });
                (void)W;
                launches += 2;
            }
            cudaEventRecord(h->stage_ev[4 * bi + 3], st);
        } else if (stat) {
            if (torch_sem) {
                // TorchGate: |X| -> dB, per-row statistics over the row's own frames (or xn's), compare
                cudaEventRecord(h->stage_ev[4 * bi + 0], st);
                launch_k1n(g, tb, xb, kdt, h->reuse_masks ? nullptr : d_tdb, dbg, resident, st, d_zcache, tf_lo, tf_hi + 1);
                if (!h->reuse_masks) {
                TStatArgs ta{};
                ta.n_units = nu; ta.T = g.T; ta.in_scale = (float)h->sum_w; ta.eps = (float)kEps64;
                ta.top_db = (float)p.top_db; ta.n_std = (float)p.n_std_thresh; ta.ddof = p.std_ddof;
                ta.mag = d_tdb; ta.rowmax = d_trow; ta.thr = d_tthr_self;
                B200_LAUNCH(k_tgate_stats, dim3((unsigned)((long long)nu * kFW)), dim3(kTgWarps * 32), 0, st, ta);
                TBitsArgs ba{};
                ba.n_units = nu; ba.T = g.T; ba.top_db = (float)p.top_db; ba.db = d_tdb; ba.rowmax = d_trow; ba.bits = d_bits;
                if (h->tthr_units > 0) {
                    ba.thr = h->tthr_units == 1 ? h->d_tthr : h->d_tthr + (size_t)u0 * kFPad;
                    ba.thr_units = h->tthr_units == 1 ? 1 : nu;
                } else {
                    ba.thr = d_tthr_self;
                    ba.thr_units = nu;
                }
                B200_LAUNCH(k_tgate_bits, dim3((unsigned)((long long)nu * kFW)), dim3(kTgWarps * 32), 0, st, ba);
                CK(h, cudaMemsetAsync(d_rowflag, 0, (size_t)nu * kFW * 4, st));
                ++launches;
                }
            } else {
                CK(h, cudaMemsetAsync(d_rowmax, 0, (size_t)nu * kFPad * 4, st));
                cudaEventRecord(h->stage_ev[4 * bi + 0], st);
                // k1: frames per work item: enough items to fill the machine, runs long enough to amortise
                K1Args a1{};
                a1.g = g; a1.tb = tb; a1.x = xb; a1.bits = d_bits; a1.rowmax = d_rowmax; a1.cnt = h->d_cnt; a1.dbg = dbg;
                a1.zcache = d_zcache; a1.zpairs = zpairs;
                a1.z_lo = tf_lo; a1.z_hi = tf_hi + 1;           // k2 walks pairs (2j, 2j+1) of frames [tf_lo, tf_hi)
                {
                    long long want = (long long)h->num_sm * B200_K1_MINBLOCKS * kWarps * 4;
                    long long run = ((long long)nu * g.T + want - 1) / want;
                    run = std::max(8LL, std::min(64LL, run));
                    run += run & 1;
                    a1.run = (int)run;
                    a1.n_runs = (g.T + a1.run - 1) / a1.run;
                }
                const long long items1 = (long long)nu * a1.n_runs;
                if (use_dual) {
                    // two channels per warp (gate_dual.cuh); the single-unit kernel below runs only if a frame could
                    // reach the top_db floor (device flag), to supply the per-bin row maxima
                    CK(h, cudaMemsetAsync(h->d_need_rowmax, 0, sizeof(unsigned), st));
                    K1dArgs ad{};
                    ad.g = g; ad.tb = tb; ad.x = xb; ad.bits = d_bits; ad.zd = (float4*)d_zcache; ad.zpairs = zpairs;
                    ad.z_lo = tf_lo; ad.z_hi = tf_hi + 1; ad.cnt = h->d_cnt; ad.need_rowmax = h->d_need_rowmax;
                    ad.min_floor4 = (float)(4.0 * h->min_floor_amp * h->min_floor_amp);
                    ad.wa_max = h->wa_max; ad.dbg = dbg;
                    {
                        long long want = (long long)h->num_sm * kDualWarpsK1 * 4;
                        long long run = ((long long)(nu / 2) * g.T + want - 1) / want;
                        run = std::max(8LL, std::min(64LL, run));
                        run += run & 1;
                        ad.run = (int)run;
                        ad.n_runs = (g.T + ad.run - 1) / ad.run;
                    }
                    B200_WITH_DTYPE(kdt, { auto kern_ = k1d_analyze<8, T>;
                        B200_LAUNCH(kern_, dim3(grid_1d((long long)(nu / 2) * ad.n_runs, kDualWarpsK1, h->num_sm)),
                                    dim3(kDualWarpsK1 * 32), k1d_smem_bytes(), st, ad); });
                    ++launches;
                    a1.guard = h->d_need_rowmax;
                    a1.zcache = nullptr;
                }
                B200_WITH_DTYPE(kdt, { auto kern_ = k1_analyze<8, T>;
                    B200_LAUNCH(kern_, dim3(grid_1d(items1, kWarps, h->num_sm * B200_K1_MINBLOCKS)), dim3(kThreads),
                                k1_smem_floats() * 4, st, a1); });
                B200_LAUNCH(k_rowfloor, dim3(grid_1d((long long)nu * kFW, 256, 1 << 30)), dim3(256), 0, st, nu,
                            (const unsigned*)d_rowmax, (const float*)h->d_floor4, d_rowflag, h->d_cnt);
            }
            launches += 2;
            cudaEventRecord(h->stage_ev[4 * bi + 1], st);
            cudaEventRecord(h->stage_ev[4 * bi + 2], st);
            cudaEventRecord(h->stage_ev[4 * bi + 3], st);
            if (tf_hi > tf_lo) {
                SmoothArgs sa{};
                sa.n_units = nu; sa.T = g.T; sa.nf = nf; sa.nt = nt; sa.tf_lo = tf_lo; sa.tf_hi = tf_hi; sa.TT = 32;
                sa.bits = d_bits; sa.rowflag = d_rowflag; sa.num = d_num;
                const int ntaps = 2 * nf + 1;
                if (h->reuse_masks) {
                    // the numerators of the last forward are still in d_num
                } else if (nt + 1 <= 14 && ntaps <= 36) {
                    SmoothPArgs pa{};
                    pa.n_units = nu; pa.T = g.T; pa.nf = nf; pa.nt = nt; pa.tf_lo = tf_lo; pa.tf_hi = tf_hi;
                    pa.bits = d_bits; pa.rowflag = d_rowflag; pa.num = d_num;
                    unsigned char tb8[36] = {0};
                    for (int d = -nf; d <= nf; ++d) tb8[d + nf] = (unsigned char)(nf + 1 - abs(d));
                    memcpy(pa.taps, tb8, 36);
                    // strips: enough CTAs to fill the machine, long enough to amortise the 2 nt warm-up frames
                    const int groups = (nu + kSmoothUnits - 1) / kSmoothUnits;
                    int n_strips = std::max(1, std::min((tf_hi - tf_lo + 127) / 128, (h->num_sm * 4 + groups - 1) / groups));
                    pa.strip = (tf_hi - tf_lo + n_strips - 1) / n_strips;
                    pa.strip = (pa.strip + kSmoothBatch - 1) / kSmoothBatch * kSmoothBatch;     // frame pairs (2j, 2j+1) leave together
                    n_strips = (tf_hi - tf_lo + pa.strip - 1) / pa.strip;
                    const dim3 grid(n_strips, groups);
                    if (ntaps <= 12) {
                        B200_LAUNCH(k_smooth_packed<3>, grid, dim3(kSmoothThreads), smoothp_smem_bytes<3>(), st, pa);
                    } else if (ntaps <= 24) {
                        B200_LAUNCH(k_smooth_packed<6>, grid, dim3(kSmoothThreads), smoothp_smem_bytes<6>(), st, pa);
                    } else {
                        B200_LAUNCH(k_smooth_packed<9>, grid, dim3(kSmoothThreads), smoothp_smem_bytes<9>(), st, pa);
                    }
                } else {
                    const int tiles = (tf_hi - tf_lo + sa.TT - 1) / sa.TT;
                    B200_LAUNCH(k_smooth_generic, dim3(tiles, nu), dim3(256), smooth_smem_bytes(sa.TT, nf, nt), st, sa);
                }
                cudaEventRecord(h->stage_ev[4 * bi + 2], st);
                K2Args a2{};
                a2.g = g; a2.tb = tb; a2.y = yb; a2.num = d_num; a2.zcache = d_zcache; a2.zpairs = zpairs;
                a2.pD = (float)(p.prop_decrease / D);
                a2.one_minus_p = (float)(1.0 - p.prop_decrease);
                a2.nt = nt;
                a2.dbg = dbg;
                {
                    const long long hops = h_hi - h_lo;
                    long long want = (long long)resident * kWarps * 4;
                    long long run = ((long long)nu * hops + want - 1) / want;
                    run = std::max(16LL, std::min(128LL, run));
                    run += run & 1;
                    a2.run = (int)run;
                    a2.n_runs = (int)((hops + a2.run - 1) / a2.run);
                }
                const long long items2 = (long long)nu * a2.n_runs;
                if (use_dual) {
                    K2dArgs ad{};
                    ad.g = g; ad.tb = tb; ad.y = yb; ad.num = d_num; ad.zd = (const float4*)d_zcache; ad.zpairs = zpairs;
                    ad.pD = a2.pD; ad.one_minus_p = a2.one_minus_p; ad.nt = nt; ad.dbg = dbg;
                    {
                        const long long hops = h_hi - h_lo;
                        long long want = (long long)h->num_sm * kDualWarpsK2 * 4;
                        long long run = ((long long)(nu / 2) * hops + want - 1) / want;
                        run = std::max(16LL, std::min(128LL, run));
                        run += run & 1;
                        ad.run = (int)run;
                        ad.n_runs = (int)((hops + ad.run - 1) / ad.run);
                    }
                    const long long itemsd = (long long)(nu / 2) * ad.n_runs;
                    if (ad.one_minus_p != 0.f) {
                        B200_WITH_DTYPE(kdt, { auto kern2 = k2d_synthesize<8, true, T>;
                            B200_LAUNCH(kern2, dim3(grid_1d(itemsd, kDualWarpsK2, h->num_sm)), dim3(kDualWarpsK2 * 32),
                                        k2d_smem_bytes(), st, ad); });
                    } else {
                        B200_WITH_DTYPE(kdt, { auto kern2 = k2d_synthesize<8, false, T>;
                            B200_LAUNCH(kern2, dim3(grid_1d(itemsd, kDualWarpsK2, h->num_sm)), dim3(kDualWarpsK2 * 32),
                                        k2d_smem_bytes(), st, ad); });
                    }
                } else if (a2.one_minus_p != 0.f) {       // spectra kept by k1: bulk-staged synthesis (gate_synth.cuh)
                    B200_WITH_DTYPE(kdt, { auto kern2 = k2c_synthesize<8, kMaskU16Blend, T>;
                        B200_LAUNCH(kern2, dim3(grid_1d(items2, kWarps, resident)), dim3(kThreads),
                                    k2c_smem_bytes<kMaskU16Blend>(), st, a2); });
                } else {
                    B200_WITH_DTYPE(kdt, { auto kern2 = k2c_synthesize<8, kMaskU16, T>;
                        B200_LAUNCH(kern2, dim3(grid_1d(items2, kWarps, resident)), dim3(kThreads),
                                    k2c_smem_bytes<kMaskU16>(), st, a2); });
                }
                cudaEventRecord(h->stage_ev[4 * bi + 3], st);
                launches += 2;
            }
        } else {
            if (two_k) {
                Tables2 t2{};
                t2.wa2 = h->d_wa2; t2.ws2 = h->d_ws2; t2.tw = h->d_tw; t2.w2k = h->d_w2k; t2.invn2 = h->d_invn2;
                t2.ws_to_w = h->ws_to_w;
                cudaEventRecord(h->stage_ev[4 * bi + 0], st);
                K1n2Args a1{};
                a1.g = g; a1.tb = t2; a1.x = (const float*)xb; a1.mag = d_mag; a1.dbg = dbg;
                a1.zcache = d_zcache; a1.z_lo = tf_lo; a1.z_hi = tf_hi + 1;
                {
                    long long want = (long long)resident * kWarps * 4;
                    long long run = ((long long)nu * g.T + want - 1) / want;
                    a1.run = (int)std::max(4LL, std::min(64LL, run));
                    a1.n_runs = (g.T + a1.run - 1) / a1.run;
                }
                B200_LAUNCH(k1n_magnitude_2k, dim3(grid_1d((long long)nu * a1.n_runs, kWarps, resident)), dim3(kThreads),
                            k1n2_smem_floats() * 4, st, a1);
                cudaEventRecord(h->stage_ev[4 * bi + 1], st);
                IirArgs ia{};
                ia.n_units = nu; ia.T = g.T; ia.F = kF2; ia.FPad = kFPad2;
                {
                    const double tfr = p.time_constant_s * p.sr / (double)g.H;
                    ia.b = (sqrt(1.0 + 4.0 * tfr * tfr) - 1.0) / (2.0 * tfr * tfr);
                }
                ia.n_mult = (float)p.thresh_n_mult; ia.slope = (float)p.sigmoid_slope;
                ia.regen = (ia.b < 0.5 && (double)g.T * -log1p(-ia.b) < 20.0 && !(p.path_flags & 64)) ? 1 : 0;
                ia.mag = d_mag; ia.m0 = d_m0;
                B200_LAUNCH(k_iir_sigmoid<kFPad2>, dim3(grid_1d((long long)nu * kFPad2, 128, 1 << 30)), dim3(128), 0, st, ia);
                launches += 2;
                cudaEventRecord(h->stage_ev[4 * bi + 2], st);
                cudaEventRecord(h->stage_ev[4 * bi + 3], st);
                if (tf_hi > tf_lo) {
                    SmoothFArgs sa{};
                    sa.n_units = nu; sa.T = g.T; sa.nf = nf; sa.nt = nt; sa.tf_lo = tf_lo; sa.tf_hi = tf_hi; sa.TT = 16;
                    sa.F = kF2; sa.FPad = kFPad2;
                    sa.p = (float)p.prop_decrease; sa.one_minus_p = (float)(1.0 - p.prop_decrease);
                    sa.m0 = d_m0; sa.m2 = d_mag;
                    launch_smooth_float(sa, nf, nt, tf_lo, tf_hi, nu, p.path_flags, st);
                    cudaEventRecord(h->stage_ev[4 * bi + 2], st);
                    // spectra kept by k1n: bulk-staged synthesis (gate_synth_2k.cuh)
                    K2c2Args ac{};
                    ac.g = g; ac.tb = t2; ac.y = (float*)yb; ac.fmask = d_mag; ac.zcache = d_zcache; ac.dbg = dbg;
                    const long long hops = h_hi - h_lo;
                    long long want = (long long)h->num_sm * kK2c2Warps * 4;
                    long long run = ((long long)nu * hops + want - 1) / want;
                    ac.run = (int)std::max(16LL, std::min(128LL, run));
                    ac.n_runs = (int)((hops + ac.run - 1) / ac.run);
                    B200_LAUNCH(k2c_synthesize_2k, dim3(grid_1d((long long)nu * ac.n_runs, kK2c2Warps, h->num_sm)),
                                dim3(kK2c2Warps * 32), k2c2_smem_bytes(), st, ac);
                    cudaEventRecord(h->stage_ev[4 * bi + 3], st);
                    launches += 2;
                }
            } else {
                cudaEventRecord(h->stage_ev[4 * bi + 0], st);
                launch_k1n(g, tb, xb, kdt, h->reuse_masks ? nullptr : d_mag, dbg, resident, st, d_zcache, tf_lo, tf_hi + 1);
                cudaEventRecord(h->stage_ev[4 * bi + 1], st);
                if (h->reuse_masks) {
                    // the final masks of the last forward are still in d_mag
                } else if (torch_sem) {
                    TMovArgs ma{};
                    ma.n_units = nu; ma.T = g.T; ma.n_movemean = p.n_movemean; ma.n_thresh = (float)p.thresh_n_mult;
                    ma.inv_temp = (float)p.sigmoid_slope; ma.p = (float)p.prop_decrease; ma.mag = d_mag; ma.m0 = d_m0;
                    B200_LAUNCH(k_tgate_movmean, dim3(grid_1d((long long)nu * kFPad, 128, 1 << 30)), dim3(128), 0, st, ma);
                } else {
                    IirArgs ia{};
                    ia.n_units = nu; ia.T = g.T; ia.F = kF; ia.FPad = kFPad;
                    {
                        const double tfr = p.time_constant_s * p.sr / (double)g.H;        // nonstationary.py:109-114
                        ia.b = (sqrt(1.0 + 4.0 * tfr * tfr) - 1.0) / (2.0 * tfr * tfr);
                    }
                    ia.n_mult = (float)p.thresh_n_mult; ia.slope = (float)p.sigmoid_slope;
                ia.regen = (ia.b < 0.5 && (double)g.T * -log1p(-ia.b) < 20.0 && !(p.path_flags & 64)) ? 1 : 0;
                    ia.mag = d_mag; ia.m0 = d_m0;
                    B200_LAUNCH(k_iir_sigmoid<kFPad>, dim3(grid_1d((long long)nu * kFPad, 128, 1 << 30)), dim3(128), 0, st, ia);
                }
                launches += 2;
                cudaEventRecord(h->stage_ev[4 * bi + 2], st);
                cudaEventRecord(h->stage_ev[4 * bi + 3], st);
                if (tf_hi > tf_lo) {
                    SmoothFArgs sa{};
                    sa.n_units = nu; sa.T = g.T; sa.nf = nf; sa.nt = nt; sa.tf_lo = tf_lo; sa.tf_hi = tf_hi; sa.TT = 32;
                    sa.F = kF; sa.FPad = kFPad;
                    sa.p = torch_sem ? 1.0f : (float)p.prop_decrease;
                    sa.one_minus_p = torch_sem ? 0.0f : (float)(1.0 - p.prop_decrease);
                    sa.m0 = d_m0; sa.m2 = d_mag;
                    if (h->reuse_masks) {
                        // masks of the last forward
                    } else {
                        launch_smooth_float(sa, nf, nt, tf_lo, tf_hi, nu, p.path_flags, st);
                    }
                    cudaEventRecord(h->stage_ev[4 * bi + 2], st);
                    K2Args a2{};
                    a2.g = g; a2.tb = tb; a2.y = yb; a2.fmask = d_mag; a2.zcache = d_zcache; a2.zpairs = zpairs;
                    a2.nt = nt;
                    a2.dbg = dbg;
                    {
                        const long long hops = h_hi - h_lo;
                        long long want = (long long)resident * kWarps * 4;
                        long long run = ((long long)nu * hops + want - 1) / want;
                        run = std::max(16LL, std::min(128LL, run));
                        run += run & 1;
                        a2.run = (int)run;
                        a2.n_runs = (int)((hops + a2.run - 1) / a2.run);
                    }
                    B200_WITH_DTYPE(kdt, { auto kern2 = k2c_synthesize<8, kMaskF32, T>;
                        B200_LAUNCH(kern2, dim3(grid_1d((long long)nu * a2.n_runs, kWarps, resident)), dim3(kThreads),
                                    k2c_smem_bytes<kMaskF32>(), st, a2); });
                    cudaEventRecord(h->stage_ev[4 * bi + 3], st);
                    launches += 2;
                }
            }
        }
        if (dbg.ul >= 0 && stat && !generic) {
            // tapped mask words with the row floor folded in, as the smoothing kernel consumes them
            std::vector<unsigned> fl(kFW);
            CK(h, cudaStreamSynchronize(st));
            CK(h, cudaMemcpy(fl.data(), d_rowflag + (size_t)dbg.ul * kFW, kFW * 4, cudaMemcpyDeviceToHost));
            std::vector<unsigned> bb((size_t)g.T * kFW);
            CK(h, cudaMemcpy(bb.data(), d_bits + (size_t)dbg.ul * g.T * kFW, bb.size() * 4, cudaMemcpyDeviceToHost));
            for (size_t i = 0; i < bb.size(); ++i) bb[i] |= fl[i % kFW];
            CK(h, cudaMemcpy(h->d_dbg_bits, bb.data(), bb.size() * 4, cudaMemcpyHostToDevice));
        }
        CK(h, cudaGetLastError());
        if (pipelined) {
            const long long c0 = (Ubase + u0) / C, c1 = c0 + nu / C;
            const long long o0 = c0 * g.step, o1 = std::min<long long>(N, c1 * g.step);
            const int ib = (int)(bi & 1);
            const void* d2h_src = h->d_slab_out[ib];
            CK(h, cudaEventRecord(h->pipe_ev[4 * bi + 1], st));
            CK(h, cudaStreamWaitEvent(h->s_d2h, h->pipe_ev[4 * bi + 1], 0));
            if (stage_out) {
                if (out_task.valid()) out_task.get();       // slab bi-2 has left this staging buffer
                // pageable result rows: D2H into this slab's pinned staging buffer (its previous content, slab bi-2, was
                // copied out by the host below), then the host threads move slab bi-1 -- whose D2H has had a whole slab of
                // kernel time -- into the caller's array
                CK(h, cudaMemcpy2DAsync(h->hp_out[ib], (size_t)(o1 - o0) * es, d2h_src, (size_t)slab_ow * es,
                                        (size_t)(o1 - o0) * es, (size_t)C, cudaMemcpyDeviceToHost, h->s_d2h));
                CK(h, cudaEventRecord(h->pipe_ev[4 * bi + 2], h->s_d2h));
                if (bi >= 1) {
                    // runs beside the next slab's copy-in (joined before that slab's D2H is enqueued into this staging buffer's twin)
                    cudaEvent_t evd = h->pipe_ev[4 * (bi - 1) + 2];
                    void* dstp = (char*)out + (size_t)prev_o0 * es;
                    const void* srcp = h->hp_out[ib ^ 1];
                    const size_t wbytes = (size_t)(prev_o1 - prev_o0) * es, dp = (size_t)out_stride * es;
                    const int nth = std::max(1, h->host_threads / 2), dev_now = h->device;
                    out_task = std::async(std::launch::async, [evd, dstp, srcp, wbytes, dp, C, nth, dev_now]() {
                        cudaSetDevice(dev_now);
                        cudaEventSynchronize(evd);
                        parallel_rows_copy(dstp, dp, srcp, wbytes, wbytes, (size_t)C, nth, 1);
                    });
                }
                prev_o0 = o0; prev_o1 = o1;
            } else {
                CK(h, cudaMemcpy2DAsync((char*)out + (size_t)o0 * es, (size_t)out_stride * es, d2h_src, (size_t)slab_ow * es,
                                        (size_t)(o1 - o0) * es, (size_t)C, cudaMemcpyDeviceToHost, h->s_d2h));
                CK(h, cudaEventRecord(h->pipe_ev[4 * bi + 2], h->s_d2h));
            }
            nu_prev = nu;
        }
    }
    cudaEventRecord(evk1, st);
    if (pipelined) {
        CK(h, cudaStreamSynchronize(h->s_d2h));
        CK(h, cudaStreamSynchronize(h->s_h2d));
        if (out_task.valid()) out_task.get();
        if (stage_out && bi >= 1)                      // the last slab's rows
            parallel_rows_copy((char*)out + (size_t)prev_o0 * es, (size_t)out_stride * es, h->hp_out[(bi - 1) & 1],
                               (size_t)(prev_o1 - prev_o0) * es, (size_t)(prev_o1 - prev_o0) * es, (size_t)C, h->host_threads, 1);
        if (getenv("B200GATE_TRACE")) {                       // slab timeline (ms since the first launch) on stderr
            CK(h, cudaStreamSynchronize(st));
            for (size_t b = 0; b < n_batches; ++b) {
                float t[4] = {0, 0, 0, 0};
                for (int i = 0; i < 4; ++i) cudaEventElapsedTime(&t[i], evk0, h->pipe_ev[4 * b + i]);
                fprintf(stderr, "slab %3zu  h2d_done %8.3f  seam_done %8.3f  kernels_done %8.3f  d2h_done %8.3f\n", b, t[0],
                        t[3], t[1], t[2]);
            }
        }
    }

    // ---- results back -------------------------------------------------------------------------------
    if (!direct && !pipelined) {
        void* out_w = (char*)out + (size_t)o_lo * es;             // first written sample of row 0
        if (kdt == dtype) {
            CK(h, cudaMemcpy2DAsync(out_w, (size_t)out_stride * es, h->d_out, (size_t)On * es, (size_t)On * es, (size_t)C,
                                    cudaMemcpyDeviceToHost, st));
        } else {
            int rc;
            if ((rc = ensure(h, &h->d_raw, &h->raw_bytes, (size_t)C * std::max(Wn, On) * es))) return rc;
            const int gr = grid_1d((long long)C * On, 256, h->num_sm * 16);
            void* dst = is_device ? out_w : h->d_raw;
            const long long ds = is_device ? out_stride : On;
            if (dtype == B200GATE_I16)
                { auto kern_ = k_from_f32<short>; B200_LAUNCH(kern_, dim3(gr), dim3(256), 0, st, (const float*)h->d_out, (short*)dst, (long long)C, (long long)On, (long long)On, ds); }
            else
                { auto kern_ = k_from_f32<double>; B200_LAUNCH(kern_, dim3(gr), dim3(256), 0, st, (const float*)h->d_out, (double*)dst, (long long)C, (long long)On, (long long)On, ds); }
            ++launches;
            if (!is_device)
                CK(h, cudaMemcpy2DAsync(out_w, (size_t)out_stride * es, h->d_raw, (size_t)On * es, (size_t)On * es, (size_t)C,
                                        cudaMemcpyDeviceToHost, st));
        }
    }
    CK(h, cudaGetLastError());

    // ---- stats: the counters travel to pinned host memory behind the kernels; a device-pointer run returns
    // here with everything enqueued (b200gate_get_stats waits for it), host-pointer runs return finished -----
    CK(h, cudaMemcpyAsync(h->h_cnt, h->d_cnt, sizeof(Counters), cudaMemcpyDeviceToHost, st));
    CK(h, cudaEventRecord(h->ev_done, st));
    h->stats.units = U;
    h->stats.frames = U * g.T;
    h->stats.kernel_launches = launches;
    h->stats.fused_path = 0;
    h->stats_pending = true;
    if (torch_sem && !generic && !two_k && n_batches == 1 && !h->reuse_masks) {
        h->masks_valid = true; h->masks_C = C; h->masks_N = N;
    }
    h->pend_batches = n_batches;
    if (!direct) {                               // host buffers: the result must be in `out` on return
        const int rc = resolve_stats(h);
        if (rc) return rc;
    }
    h->stats.last_h2d_ms = h2d_ms;
    return B200GATE_OK;
}


int b200gate_torch_apply_masks(b200gate_handle* h, const void* in, void* out, int dtype, int64_t C, int64_t N, int64_t in_stride,
                               int64_t out_stride, int is_device, void* stream) {
    if (!h) return B200GATE_ERR_ARG;
    if (h->p.surface != B200GATE_SURFACE_TORCH) return fail(h, B200GATE_ERR_STATE, "torch surface only");
    if (!h->masks_valid || h->masks_C != C || h->masks_N != N)
        return fail(h, B200GATE_ERR_STATE, "no masks of a matching forward are kept (run b200gate_run on [%lld][%lld] first; "
                    "tuned n_fft=1024 geometry, one workspace batch)", (long long)C, (long long)N);
    h->reuse_masks = true;
    const int rc = b200gate_run(h, in, out, dtype, C, N, in_stride, out_stride, is_device, stream);
    h->reuse_masks = false;
    return rc;
}

// ---- multi-GPU: kernel-issued NVLink stores (gate_peer.cuh) ---------------------------------------------------------
int b200gate_peer_push(const void* src, void* const* peer_dst, int32_t n_peers, int64_t rows, int64_t row_bytes,
                       int64_t src_stride_bytes, int64_t dst_stride_bytes, int32_t n_ctas, void* stream) {
    if (!src || !peer_dst || n_peers < 0 || n_peers > kMaxPeers || rows < 0 || row_bytes < 0) return B200GATE_ERR_ARG;
    if (n_peers == 0 || rows == 0 || row_bytes == 0) return B200GATE_OK;
    if ((row_bytes | src_stride_bytes | dst_stride_bytes | (int64_t)(uintptr_t)src) & 15) return B200GATE_ERR_ARG;
    PushArgs a{};
    a.src = (const uint4*)src;
    for (int p = 0; p < n_peers; ++p) {
        if (!peer_dst[p] || ((uintptr_t)peer_dst[p] & 15)) return B200GATE_ERR_ARG;
        a.dst[p] = (uint4*)peer_dst[p];
    }
    a.n_dst = n_peers;
    a.rows = rows; a.vec_per_row = row_bytes / 16; a.src_stride = src_stride_bytes / 16; a.dst_stride = dst_stride_bytes / 16;
    const int ctas = n_ctas > 0 ? n_ctas : 12;
    static bool attr_set = false;
    if (!attr_set) { cudaFuncSetAttribute(k_peer_push, cudaFuncAttributeMaxDynamicSharedMemorySize, kPushSmemBytes); attr_set = true; }
    B200_LAUNCH(k_peer_push, dim3(ctas), dim3(kPushThreads), kPushSmemBytes, (cudaStream_t)stream, a);
    return cudaGetLastError() == cudaSuccess ? B200GATE_OK : B200GATE_ERR_CUDA;
}

int b200gate_peer_barrier(void* local_flags, void* const* peer_flags, int32_t rank, int32_t world, uint32_t epoch, void* stream) {
    if (!local_flags || !peer_flags || world < 1 || world > kMaxPeers || rank < 0 || rank >= world) return B200GATE_ERR_ARG;
    BarrierArgs a{};
    a.local_flags = (unsigned*)local_flags;
    for (int p = 0; p < world; ++p) a.peer_flags[p] = (unsigned*)peer_flags[p];
    a.rank = rank; a.world = world; a.epoch = epoch;
    B200_LAUNCH(k_peer_barrier, dim3(1), dim3(32), 0, (cudaStream_t)stream, a);
    return cudaGetLastError() == cudaSuccess ? B200GATE_OK : B200GATE_ERR_CUDA;
}

int b200gate_run_sharded(b200gate_handle* h, const void* in_local, int dtype, int64_t C_local, int64_t N, int64_t in_stride,
                         void* gathered_local, void* const* gathered_peers, void* flags_local, void* const* flags_peers,
                         uint32_t epoch, int32_t rank, int32_t world, int32_t groups, int32_t push_ctas,
                         void* compute_stream, void* comm_stream) {
    if (!h || !in_local || !gathered_local || world < 1 || world > kMaxPeers || rank < 0 || rank >= world || C_local <= 0)
        return fail(h, B200GATE_ERR_ARG, "bad argument");
    if (world > 1 && (!gathered_peers || !flags_local || !flags_peers || !comm_stream || comm_stream == compute_stream))
        return fail(h, B200GATE_ERR_ARG, "a sharded run needs peer mappings, flag arrays and a separate communication stream");
    const size_t es = dtype_size(dtype);
    if (es == 0) return fail(h, B200GATE_ERR_ARG, "bad dtype");
    cudaStream_t cs = (cudaStream_t)compute_stream, ms = (cudaStream_t)comm_stream;
    if (groups < 1) groups = 1;
    const int64_t gs = (C_local + groups - 1) / groups;
    while (h->group_ev.size() < (size_t)groups + 1) {
        cudaEvent_t e;
        CK(h, cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
        h->group_ev.push_back(e);
    }
    // the previous step's pushes (other ranks') may still be landing in OUR buffer only before their barrier; ours are
    // ordered by the communication stream itself.  Compute must not overwrite rows a previous push is still reading:
    CK(h, cudaEventRecord(h->group_ev[groups], ms));
    CK(h, cudaStreamWaitEvent(cs, h->group_ev[groups], 0));
    char* mine = (char*)gathered_local + (size_t)rank * C_local * N * es;
    int gi = 0;
    for (int64_t g0 = 0; g0 < C_local; g0 += gs, ++gi) {
        const int64_t g1 = std::min<int64_t>(C_local, g0 + gs);
        const int rc = b200gate_run(h, (const char*)in_local + (size_t)g0 * in_stride * es, mine + (size_t)g0 * N * es, dtype,
                                    g1 - g0, N, in_stride, N, 1, compute_stream);
        if (rc) return rc;
        if (world == 1) continue;
        CK(h, cudaEventRecord(h->group_ev[gi], cs));
        CK(h, cudaStreamWaitEvent(ms, h->group_ev[gi], 0));
        void* dst[kMaxPeers];
        int np = 0;
        for (int p = 0; p < world; ++p)
            if (p != rank) dst[np++] = (char*)gathered_peers[p] + ((size_t)rank * C_local + g0) * N * es;
        const int rc2 = b200gate_peer_push(mine + (size_t)g0 * N * es, dst, np, g1 - g0, (int64_t)(N * es), (int64_t)(N * es),
                                           (int64_t)(N * es), push_ctas, comm_stream);
        if (rc2) return fail(h, rc2, "peer push failed (rows must be 16-byte multiples)");
    }
    if (world > 1) {
        const int rc = b200gate_peer_barrier(flags_local, flags_peers, rank, world, epoch, comm_stream);
        if (rc) return fail(h, rc, "peer barrier failed");
        CK(h, cudaEventRecord(h->group_ev[groups], ms));
        CK(h, cudaStreamWaitEvent(cs, h->group_ev[groups], 0));
    }
    return B200GATE_OK;
}

}  // extern "C"
