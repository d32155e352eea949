// gate_kernels.cuh -- sm_100a kernels of the spectral-gating hot path (n_fft = 1024 family).
//
// Reference semantics restated by these kernels (paths relative to /root/reference):
//   framing / STFT          scipy.signal.stft as called at noisereduce/spectralgate/stationary.py:87-93
//   dB floor + threshold    spectralgate/utils.py:11-16, stationary.py:96-110
//   mask smoothing          base.py:7-29 filter, fftconvolve(..., "same") at stationary.py:114
//   apply + iSTFT           stationary.py:117-126 (scipy.signal.istft)
//   chunk geometry          base.py:130-156, :167-226
//
// Work decomposition.  A *unit* is one (chunk, channel) pair -- the reference's _do_filter runs them
// independently (stationary.py:86), so they are the grid.  Inside a unit every warp is an autonomous
// worker that owns a run of consecutive STFT frames; it transforms TWO real frames per 1024-point
// complex FFT (frame a in the real part, frame b = next frame in the imaginary part) held entirely in
// its registers (warp_fft.cuh).  No warp ever waits for another warp.
//
//   k1_analyze    frames -> FFT -> |X|^2 against per-bin power thresholds -> 1 bit/bin mask words
//                 (+ per-(unit,bin) running max for the top_db floor, + FP64 re-decision of bins
//                 whose FP32 margin is inside a proven guard band, so decisions equal the float64
//                 reference's)
//   k_rowfloor    top_db floor:  max_t dB - top_db > thresh  <=>  lift the whole row
//   k_smooth      separable triangular smoothing of the binary mask in exact integer arithmetic
//                 (the reference's FFT convolution approximates exactly these rationals)
//   k2c / k2d     synthesis (gate_synth.cuh, gate_dual.cuh): the spectra k1 kept -> mask apply on the packed
//                 spectrum -> inverse FFT -> window -> overlap-add in registers -> normalise -> store the chunk centre
#pragma once
#include "warp_fft.cuh"

namespace b200 {

constexpr int kN = 1024;            // n_fft handled by this kernel family
constexpr int kF = kN / 2 + 1;      // 513 bins
constexpr int kFW = (kF + 31) / 32; // 17 mask words per frame
constexpr int kFPad = kFW * 32;     // 544: padded bin count (tables, mask row pitch)
constexpr int kWarps = 4;           // warps per CTA for k1/k2 (each warp is independent)
constexpr int kThreads = kWarps * 32;
#ifndef B200_K1_MINBLOCKS
#define B200_K1_MINBLOCKS 4          // k1 fits 128 registers: 16 warps per SM
#endif

struct Geom {
    int H;                  // hop
    int C;                  // channels
    int T;                  // frames per padded chunk: Lp / H + 1
    int n_chunks;
    long long n_total;      // samples per channel
    long long step;         // chunk_size (or n_total when there is a single chunk)
    long long pad;          // padding
    long long Lp;           // padded chunk length: step + 2 pad
    long long in_stride, out_stride;   // elements between channel rows
    int u0, n_units;        // this batch: units [u0, u0 + n_units); u = chunk * C + channel
};

struct Tables {              // device pointers, built once per handle
    const float* wa;         // [N] analysis window / sum(w)
    const float* ws;         // [N] synthesis window * sum(w) / N
    const float2* tw;        // [32*32] radix-32 inter-pass twiddles
    const float* invn;       // [H] 1 / sum_i w^2[i H + r]  (interior overlap-add norm)
    const float* thr4;       // [FPad] 4 * T_amp^2, T_amp = 10^(thresh/20) - eps
    const float* gco;        // [FPad] guard-band coefficient: 4 * T_amp * kappa * eps32
    const float* floor4;     // [FPad] 4 * (10^((thresh + top_db)/20) - eps)^2
    const float* ef;         // [FPad] frequency edge factor of the smoothing filter
    const double* thr2_64;   // [F]  T_amp^2 in float64
    const double* wa64;      // [N]  analysis window / sum(w), float64
    const double2* cs64;     // [N]  (cos, sin)(2 pi m / N), float64
    float ws_to_w;           // raw window = ws * ws_to_w
};

struct Counters {
    unsigned long long rechecked, unresolved, floor_flags, floor_ambiguous;
};

struct DebugTap {
    int ul;                  // local unit index to tap, -1 = off
    float* spec;             // [T][F][2]
    float* mask;             // [T][F]
};

// Mask numerators are stored as uint16 pairs, element [pair j][bin k][frame 2j + {0, 1}], so that the synthesis
// kernel fetches both frames of a pair with one 32-bit access; a unit owns ceil(T/2) pair rows of 2*FPad values.
__host__ __device__ __forceinline__ long long num_index(int t, int k) {
    return (((long long)(t >> 1) * kFPad + k) << 1) + (t & 1);
}
__host__ __device__ __forceinline__ long long num_unit_stride(int T) { return (long long)((T + 1) / 2) * (2 * kFPad); }

// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// One sample of the zero-extended padded chunk (base.py:130-142 zeros outside [0, n_total);
// scipy boundary='zeros' outside [0, Lp)).  j: chunk-local index, i1: global index of j = 0.
// The kernels read the caller's samples in their own dtype (float32 / int16 / float64) and convert on
// load -- the device-side form of base.py:140's promotion -- and k2 casts on store (base.py:218-226).
// u16 halves of a packed word -> float without the (quarter-rate) I2F unit: 2^23 + n as a float bit pattern, minus 2^23
// (exact for n < 2^23): integer-pipe bit operations and one FADD instead.
__device__ __forceinline__ float u16lo_to_float(unsigned pk) {
    return __uint_as_float((pk & 0xFFFFu) | 0x4B000000u) - 8388608.0f;
}
__device__ __forceinline__ float u16hi_to_float(unsigned pk) {
    return __uint_as_float((pk >> 16) | 0x4B000000u) - 8388608.0f;      // (the compiler emits one PRMT / LOP3)
}

template <typename T>
__device__ __forceinline__ float ld_sample(const T* p) { return (float)__ldg(p); }
template <typename T>
__device__ __forceinline__ double ld_sample_f64(const T* p) { return (double)__ldg(p); }
template <typename T>
__device__ __forceinline__ T st_cast(float v);
template <> __device__ __forceinline__ float st_cast<float>(float v) { return v; }
template <> __device__ __forceinline__ double st_cast<double>(float v) { return (double)v; }
template <> __device__ __forceinline__ short st_cast<short>(float v) { return (short)(int)v; }   // numpy astype: truncate, wrap

template <typename T>
__device__ __forceinline__ float chunk_sample(const T* __restrict__ xrow, long long j, long long i1,
                                              long long Lp, long long n_total) {
    const long long g = i1 + j;
    return (j >= 0 && j < Lp && g >= 0 && g < n_total) ? ld_sample(xrow + g) : 0.0f;
}
template <typename T>
__device__ __forceinline__ double chunk_sample_f64(const T* __restrict__ xrow, long long j, long long i1,
                                                   long long Lp, long long n_total) {
    const long long g = i1 + j;
    return (j >= 0 && j < Lp && g >= 0 && g < n_total) ? ld_sample_f64(xrow + g) : 0.0;
}

// Rows of a frame pair: frame t is rows 0..31, frame t+1 rows HR..31+HR of the same 32+HR row window
// (row = 32 consecutive samples = one coalesced 128-byte access of the warp).
template <int HR>
__device__ __forceinline__ bool pair_window_interior(long long base, long long i1, long long Lp, long long n_total) {
    const long long g0 = i1 + base;
    const int span = 32 * (32 + HR);
    return base >= 0 && base + span <= Lp && g0 >= 0 && g0 + span <= n_total;
}

// Load the raw samples of the pair (coalesced 128-byte rows straight into FFT order), window them and pack
// the two frames as one complex signal.  Returns this lane's contribution to ||frame pair||^2.
// (Measured and dropped: prefetch.global.L1 of the next pair's rows -- no effect -- and a register pre-load
//  of them -- more bookkeeping than hidden latency; see profiles/r01_scaling_notes.md.)
template <int HR>
__device__ __forceinline__ float pack_frame_pair(float (&re)[32], float (&im)[32], const float (&xr)[32 + HR],
                                                 const float* __restrict__ s_wa, int lane, bool vb) {
    float e = 0.f;
#pragma unroll
    for (int r = 0; r < 32; ++r) {
        const float w = s_wa[lane + 32 * r];
        re[r] = xr[r] * w;
        im[r] = xr[r + HR] * w;
        e = fmaf(re[r], re[r], e);
    }
    if (vb) {
#pragma unroll
        for (int r = 0; r < 32; ++r) e = fmaf(im[r], im[r], e);
    } else {                                         // odd frame count: the pair's second frame does not exist
#pragma unroll
        for (int r = 0; r < 32; ++r) im[r] = 0.f;
    }
    return e;
}

template <int HR, typename T>
__device__ __forceinline__ float load_frame_pair(float (&re)[32], float (&im)[32], const T* __restrict__ xrow,
                                                 long long base, long long i1, long long Lp, long long n_total,
                                                 const float* __restrict__ s_wa, int lane, bool vb) {
    float xr[32 + HR];
    if (pair_window_interior<HR>(base, i1, Lp, n_total)) {
        const T* p = xrow + i1 + base + lane;
#pragma unroll
        for (int r = 0; r < 32 + HR; ++r) xr[r] = ld_sample(p + 32 * r);
    } else {                                         // chunk / recording edges: zero-extended samples
#pragma unroll
        for (int r = 0; r < 32 + HR; ++r) xr[r] = chunk_sample(xrow, base + lane + 32 * r, i1, Lp, n_total);
    }
    return pack_frame_pair<HR>(re, im, xr, s_wa, lane, vb);
}

#ifdef B200_CUSIM_BUILD
#define B200_NOINLINE __attribute__((noinline))
#else
#define B200_NOINLINE __noinline__
#endif

// Exact (float64) re-decision of one bin of one frame: direct DFT of the windowed samples.
// Warp-cooperative; every lane returns the same value.  2 = above threshold, 1 = not above,
// 0 = unresolved even in float64 (|P - T^2| <= 1e-12 T^2).
template <typename T>
__device__ B200_NOINLINE int recheck_bin_fp64(const T* __restrict__ xrow, long long base, long long i1,
                                              long long Lp, long long n_total, int k, const Tables& tb, int lane) {
    double sr = 0.0, si = 0.0;
    for (int n = lane; n < kN; n += 32) {
        const double x = chunk_sample_f64(xrow, base + n, i1, Lp, n_total) * tb.wa64[n];   // the caller's exact samples
        const double2 cs = tb.cs64[(k * n) & (kN - 1)];
        sr = fma(x, cs.x, sr);
        si = fma(-x, cs.y, si);
    }
    sr = warp_sum(sr);
    si = warp_sum(si);
    const double P = sr * sr + si * si;
    const double T2 = tb.thr2_64[k];
    if (fabs(P - T2) <= 1e-12 * T2) return 0;
    return P > T2 ? 2 : 1;
}

// =============================================================================================
// k1: analysis.  bits[(ul*T + t)*FW + w] bit b  <=>  raw |X[32w+b, t]| above the bin threshold.
// =============================================================================================
struct K1Args {
    Geom g;
    Tables tb;
    const void* x;             // [C][in_stride] samples in the caller's dtype (kernel template T)
    unsigned* bits;            // [n_units][T][FW]
    unsigned* rowmax;          // [n_units][FPad]  max_t 4|X|^2 as float bits (>= 0 so uint order works)
    Counters* cnt;
    DebugTap dbg;
    int run;                   // frames per work item (even)
    int n_runs;                // ceil(T / run)
    float2* zcache;            // optional [n_units][ceil(T/2)][32 slots][32 lanes]: the packed spectrum of every
                               // frame pair, kept so that k2 need not transform the frames a second time
    int zpairs;                // ceil(T/2)
    int z_lo, z_hi;            // only frames [z_lo, z_hi) are read back by k2 (chunk centre + halo): the rest is not stored
    const unsigned* guard;     // optional device flag: when given and zero the kernel returns at once (it is then the
                               // row-maximum fallback behind k1d_analyze, gate_dual.cuh)
};

constexpr int k1_smem_floats() { return kN + 2 * kN + 2 * kFPad + kWarps * kExchFloats + kWarps * 2 * kFW + 8; }

template <int HR, typename T>
__global__ void __launch_bounds__(kThreads, B200_K1_MINBLOCKS) k1_analyze(const K1Args a) {
    if (a.guard && *a.guard == 0u) return;
    B200_DYN_SMEM(float, smem);
    float* s_wa = smem;
    float2* s_tw = reinterpret_cast<float2*>(smem + kN);
    float* s_thr4 = smem + 3 * kN;
    float* s_gco = s_thr4 + kFPad;
    float* s_tiles = s_gco + kFPad;
    unsigned* s_amb_all = reinterpret_cast<unsigned*>(s_tiles + kWarps * kExchFloats);
    for (int i = threadIdx.x; i < kN; i += kThreads) {
        s_wa[i] = a.tb.wa[i];
        s_tw[i] = a.tb.tw[i];
    }
    for (int i = threadIdx.x; i < kFPad; i += kThreads) {
        s_thr4[i] = a.tb.thr4[i];
        s_gco[i] = a.tb.gco[i];
    }
    __syncthreads();

    const Geom& g = a.g;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    float* tile = s_tiles + warp * kExchFloats;
    unsigned* s_amb = s_amb_all + warp * 2 * kFW;
    const int H = g.H;
    const int pl = (32 - lane) & 31;                 // partner lane holding the mirrored bins
    const long long n_items = (long long)g.n_units * a.n_runs;

    for (long long item = (long long)blockIdx.x * kWarps + warp; item < n_items;
         item += (long long)gridDim.x * kWarps) {
        const int ul = (int)(item / a.n_runs);
        const int run = (int)(item - (long long)ul * a.n_runs);
        const int u = g.u0 + ul;
        const int ic = u / g.C, c = u - ic * g.C;
        const long long i1 = (long long)ic * g.step - g.pad;
        const T* xrow = static_cast<const T*>(a.x) + (long long)c * g.in_stride;
        const int t0 = run * a.run;
        const int t1 = min(t0 + a.run, g.T);
        float mx[kFW];
#pragma unroll
        for (int q = 0; q < kFW; ++q) mx[q] = 0.f;

        for (int t = t0; t < t1; t += 2) {
            const bool vb = (t + 1 < t1);
            const long long base = (long long)t * H - kN / 2;
            float re[32], im[32];
            const float e = load_frame_pair<HR>(re, im, xrow, base, i1, g.Lp, g.n_total, s_wa, lane, vb);
            const float S = sqrtf(warp_sum(e));
            warp_fft1024(re, im, tile, s_tw, lane);
            if (a.zcache && t >= a.z_lo && t < a.z_hi) {      // warp-uniform
                float2* zp = a.zcache + ((long long)ul * a.zpairs + (t >> 1)) * 1024 + lane;
#pragma unroll
                for (int q = 0; q < 32; ++q) zp[32 * q] = make_float2(re[brev5(q)], im[brev5(q)]);
            }

            unsigned wordA = 0u, wordB = 0u;
            unsigned anyamb = 0u;
#pragma unroll
            for (int q = 0; q < kFW; ++q) {
                const int sA = brev5(q), sP = brev5(31 - q), s0 = brev5((32 - q) & 31);
                const float zr = re[sA], zi = im[sA];
                float pr = __shfl_sync(0xffffffffu, re[sP], pl);
                float pi = __shfl_sync(0xffffffffu, im[sP], pl);
                if (lane == 0) { pr = re[s0]; pi = im[s0]; }
                // 2 X_a = Z + conj(Zp),  2 X_b = (Z - conj(Zp)) / i
                const float ar = zr + pr, ai = zi - pi;
                const float br = zi + pi, bi = pr - zr;
                const float PA = fmaf(ar, ar, ai * ai);
                const float PB = fmaf(br, br, bi * bi);
                const int k = lane + 32 * q;
                const bool valid = (q < 16) || (lane == 0);
                const float th = s_thr4[k];
                const float gg = fmaf(s_gco[k], S, th * 8.0e-7f);
                const float dA = PA - th, dB = PB - th;
                const unsigned wA = __ballot_sync(0xffffffffu, valid && (dA > 0.f));
                const unsigned wB = __ballot_sync(0xffffffffu, valid && vb && (dB > 0.f));
                const bool amA = valid && fabsf(dA) <= gg, amB = valid && vb && fabsf(dB) <= gg;
                if (lane == q) { wordA = wA; wordB = wB; }
                if (__any_sync(0xffffffffu, amA || amB)) {   // rare: remember the bins inside the guard band
                    const unsigned mA = __ballot_sync(0xffffffffu, amA);
                    const unsigned mB = __ballot_sync(0xffffffffu, amB);
                    anyamb |= 1u << q;
                    if (lane == 0) { s_amb[2 * q] = mA; s_amb[2 * q + 1] = mB; }
                }
                if (valid) mx[q] = fmaxf(mx[q], vb ? fmaxf(PA, PB) : PA);
            }
            if (a.dbg.ul == ul) {                            // parity tap (tests): the FP32 STFT itself
#pragma unroll 1
                for (int q = 0; q < kFW; ++q) {
                    float zr = 0.f, zi = 0.f, pr = 0.f, pi = 0.f;
#pragma unroll
                    for (int qq = 0; qq < kFW; ++qq)
                        if (qq == q) {
                            zr = re[brev5(qq)]; zi = im[brev5(qq)];
                            pr = __shfl_sync(0xffffffffu, re[brev5(31 - qq)], pl);
                            pi = __shfl_sync(0xffffffffu, im[brev5(31 - qq)], pl);
                            if (lane == 0) { pr = re[brev5((32 - qq) & 31)]; pi = im[brev5((32 - qq) & 31)]; }
                        }
                    const int k = lane + 32 * q;
                    if (((q < 16) || lane == 0) && k < kF) {
                        float* sp = a.dbg.spec + ((long long)t * kF + k) * 2;
                        sp[0] = 0.5f * (zr + pr); sp[1] = 0.5f * (zi - pi);
                        if (vb) { sp[2 * kF] = 0.5f * (zi + pi); sp[2 * kF + 1] = 0.5f * (pr - zr); }
                    }
                }
            }
            if (anyamb) {                             // warp-uniform, rare: redo those bins in float64
                __syncwarp();
                unsigned nre = 0, nun = 0;
                for (int q = 0; q < kFW; ++q) {
                    if (!((anyamb >> q) & 1u)) continue;
                    for (int fr = 0; fr < 2; ++fr) {
                        unsigned m = s_amb[2 * q + fr];
                        while (m) {
                            const int src = __ffs((int)m) - 1;
                            m &= m - 1;
                            const int r = recheck_bin_fp64(xrow, base + (long long)fr * H, i1, g.Lp, g.n_total,
                                                           src + 32 * q, a.tb, lane);
                            ++nre;
                            if (r == 0) { ++nun; continue; }
                            if (lane == q) {
                                unsigned& wd = fr ? wordB : wordA;
                                wd = (r == 2) ? (wd | (1u << src)) : (wd & ~(1u << src));
                            }
                        }
                    }
                }
                __syncwarp();
                if (lane == 0) {
                    atomicAdd(&a.cnt->rechecked, (unsigned long long)nre);
                    if (nun) atomicAdd(&a.cnt->unresolved, (unsigned long long)nun);
                }
            }
            if (lane < kFW) {
                unsigned* dst = a.bits + ((long long)ul * g.T + t) * kFW + lane;
                dst[0] = wordA;
                if (vb) dst[kFW] = wordB;
            }
        }
#pragma unroll
        for (int q = 0; q < kFW; ++q)
            if ((q < 16) || (lane == 0))
                atomicMax(a.rowmax + (long long)ul * kFPad + lane + 32 * q, __float_as_uint(mx[q]));
    }
}

// =============================================================================================
// top_db floor (spectralgate/utils.py:16): clamped dB > thresh  <=>  raw > thresh  OR
// (row max over the chunk's frames - top_db > thresh).  One thread per (unit, mask word).
// =============================================================================================
__global__ void k_rowfloor(int n_units, const unsigned* __restrict__ rowmax, const float* __restrict__ floor4,
                           unsigned* __restrict__ rowflag, Counters* cnt) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_units * kFW) return;
    const int ul = i / kFW, w = i - ul * kFW;
    unsigned word = 0u, nflag = 0u, namb = 0u;
    for (int b = 0; b < 32; ++b) {
        const int f = w * 32 + b;
        if (f >= kF) break;
        const float v = __uint_as_float(rowmax[(long long)ul * kFPad + f]);
        const float tf = floor4[f];
        if (v > tf) { word |= 1u << b; ++nflag; }
        if (fabsf(v - tf) <= tf * 1.0e-5f) ++namb;
    }
    rowflag[i] = word;
    if (nflag) atomicAdd(&cnt->floor_flags, (unsigned long long)nflag);
    if (namb) atomicAdd(&cnt->floor_ambiguous, (unsigned long long)namb);
}

// =============================================================================================
// Mask smoothing in integers.  K = tri_f (x) tri_t / ((nf+1)^2 (nt+1)^2) with tri_n[k] = n+1-|k|
// (base.py:14-28), so  smoothed = p * num / D + (1-p) * edge,  num = sum tri_f tri_t bit.
// Output: num as uint16 [n_units][T][FPad] for frames [tf_lo, tf_hi).
// Time direction: per-bin streaming second-difference recurrence (tri = box * box);
// frequency direction: direct taps from the shared-memory tile.
// =============================================================================================
struct SmoothArgs {
    int n_units, T;
    int nf, nt;
    int tf_lo, tf_hi;          // frames that need masks
    int TT;                    // output frames per tile
    const unsigned* bits;      // [n_units][T][FW]
    const unsigned* rowflag;   // [n_units][FW]
    unsigned short* num;       // [n_units][ceil(T/2)][FPad][2]  (num_index)
};

__host__ __device__ inline int smooth_rows(int TT, int nt) { return TT + 2 * nt + 2 * (nt + 1); }
__host__ __device__ inline int smooth_cpitch(int nf) { return (kFPad + 2 * nf + 2) | 1; }   // odd #shorts/2 not needed; keep simple
inline size_t smooth_smem_bytes(int TT, int nf, int nt) {
    return (size_t)smooth_rows(TT, nt) * kFW * 4 + (size_t)TT * smooth_cpitch(nf) * 2 + 16;
}

__global__ void __launch_bounds__(256) k_smooth_generic(const SmoothArgs a) {
    B200_DYN_SMEM(unsigned, smem);
    const int nt = a.nt, nf = a.nf, aa = nt + 1;
    const int rows = smooth_rows(a.TT, nt);
    const int cp = smooth_cpitch(nf);
    unsigned* s_bits = smem;                                                   // [rows][FW]
    unsigned short* s_c = reinterpret_cast<unsigned short*>(smem + rows * kFW);  // [TT][cp]
    const int ul = blockIdx.y;
    const int t0 = a.tf_lo + blockIdx.x * a.TT;
    if (t0 >= a.tf_hi) return;
    const int tt_n = min(a.TT, a.tf_hi - t0);
    // row rho <-> frame tau = t0 - nt - 2aa + rho ; the first 2aa rows are "before the stream" = 0
    const int tau0 = t0 - nt - 2 * aa;
    for (int i = threadIdx.x; i < rows * kFW; i += blockDim.x) {
        const int rho = i / kFW, w = i - rho * kFW;
        const int tau = tau0 + rho;
        unsigned v = 0u;
        if (rho >= 2 * aa && tau >= 0 && tau < a.T)
            v = a.bits[((long long)ul * a.T + tau) * kFW + w] | a.rowflag[ul * kFW + w];
        s_bits[i] = v;
    }
    for (int i = threadIdx.x; i < a.TT * cp; i += blockDim.x) s_c[i] = 0;
    __syncthreads();
    // time direction: c[f, t] = sum_b tri_t[b] m[f, t-b];  s2[tau] = c[., tau - nt]
    for (int f = threadIdx.x; f < kF; f += blockDim.x) {
        const int w = f >> 5, sh = f & 31;
        int d1 = 0, s2 = 0;
        const int steps = tt_n + 2 * nt;
        for (int s = 0; s < steps; ++s) {
            const int rho = 2 * aa + s;
            const int e = (int)((s_bits[rho * kFW + w] >> sh) & 1u)
                        - 2 * (int)((s_bits[(rho - aa) * kFW + w] >> sh) & 1u)
                        + (int)((s_bits[(rho - 2 * aa) * kFW + w] >> sh) & 1u);
            d1 += e;
            s2 += d1;
            const int tt = s - 2 * nt;
            if (tt >= 0) s_c[tt * cp + nf + f] = (unsigned short)s2;
        }
    }
    __syncthreads();
    // frequency direction
    for (int i = threadIdx.x; i < tt_n * kFPad; i += blockDim.x) {
        const int tt = i / kFPad, f = i - tt * kFPad;
        int acc = 0;
        if (f < kF) {
            const unsigned short* cr = s_c + tt * cp + f;      // cr[nf + d] = c[f + d]
            for (int d = -nf; d <= nf; ++d) acc += (nf + 1 - (d < 0 ? -d : d)) * (int)cr[nf + d];
        }
        a.num[(long long)ul * num_unit_stride(a.T) + num_index(t0 + tt, f)] = (unsigned short)acc;
    }
}

// ---------------------------------------------------------------------------------------------
// Packed variant (the one that normally runs).  A thread owns 4 consecutive bins as byte lanes of
// one register and streams over time: the time-direction recurrence costs ~4 ops/bin, and the
// frequency-direction triangle is NTW dp4a dot products per output against byte windows of the
// shared row.  Requirements: nt + 1 <= 14 (byte lanes: counts <= 196, biased first difference
// <= 31) and 2 nf + 1 <= 4 NTW; otherwise the host falls back to k_smooth_generic.
// CTA = 544 threads = 4 units x 136 bin-groups; one __syncthreads per frame.
// ---------------------------------------------------------------------------------------------
struct SmoothPArgs {
    int n_units, T;
    int nf, nt;
    int tf_lo, tf_hi;
    int strip;                 // output frames per CTA
    const unsigned* bits;
    const unsigned* rowflag;
    unsigned short* num;
    unsigned taps[9];          // triangle taps nf+1-|d|, d = -nf..nf, as packed bytes (zero padded)
};
constexpr int kSmoothGroups = kFPad / 4;          // 136 threads per unit
constexpr int kSmoothUnits = 4;
constexpr int kSmoothThreads = kSmoothGroups * kSmoothUnits;   // 544
constexpr int kSmoothBatch = 4;                    // frames per barrier
template <int NTW> __host__ __device__ constexpr int smoothp_rowbytes() { return kFPad + 4 * (NTW + 2) + 64; }
template <int NTW> __host__ __device__ constexpr int smoothp_smem_bytes() {
    return 2 * kSmoothBatch * kSmoothUnits * smoothp_rowbytes<NTW>();
}

__device__ __forceinline__ unsigned dp4a_u(unsigned a, unsigned b, unsigned c) {
#ifdef B200_CUSIM_BUILD
    for (int i = 0; i < 4; ++i) c += ((a >> (8 * i)) & 0xFFu) * ((b >> (8 * i)) & 0xFFu);
    return c;
#else
    return __dp4a(a, b, c);
#endif
}

template <int NTW>
__global__ void __launch_bounds__(kSmoothThreads, 3) k_smooth_packed(const SmoothPArgs a) {
    constexpr int RB = smoothp_rowbytes<NTW>();
    constexpr int NB = kSmoothBatch;
    B200_DYN_SMEM(unsigned char, s_raw);                      // [2][NB][4 units][RB]
    const int tid = threadIdx.x;
    const int ug = tid / kSmoothGroups, i = tid - ug * kSmoothGroups;
    const int ul = blockIdx.y * kSmoothUnits + ug;
    const bool active = ul < a.n_units;
    const int t_begin = a.tf_lo + blockIdx.x * a.strip;
    if (t_begin >= a.tf_hi) return;
    const int t_end = min(t_begin + a.strip, a.tf_hi);
    const int nt = a.nt, nf = a.nf, aa = nt + 1;
    for (int k = tid; k < 2 * NB * kSmoothUnits * RB / 4; k += kSmoothThreads) reinterpret_cast<unsigned*>(s_raw)[k] = 0u;
    __syncthreads();

    const int w = i >> 3, sh = (i & 7) * 4;
    const unsigned fl = active ? ((a.rowflag[ul * kFW + w] >> sh) & 0xFu) : 0u;
    const unsigned* bp = a.bits + (long long)(active ? ul : 0) * a.T * kFW + w;
    unsigned short* outp = a.num + (long long)(active ? ul : 0) * num_unit_stride(a.T) + 8 * i;
    unsigned taps[NTW];
#pragma unroll
    for (int m = 0; m < NTW; ++m) taps[m] = a.taps[m];

    const int tau_s = t_begin - nt;                 // first frame fed into the recurrence
    const int tau_e = t_end - 1 + nt;               // last one
    unsigned d1b = 0x10101010u, s2 = 0u;
    int par = 0;
    // warm-up: the first 2 nt frames only feed the recurrence (no output yet)
    auto nib = [&](int t) -> unsigned {
        return (active && t >= tau_s && t >= 0 && t < a.T) ? (((__ldg(bp + (long long)t * kFW) >> sh) & 0xFu) | fl) : 0u;
    };
    auto advance = [&](unsigned na, unsigned nb, unsigned nc) {
        const unsigned ea = (na * 0x00204081u) & 0x01010101u;
        const unsigned eb = (nb * 0x00204081u) & 0x01010101u;
        const unsigned ec = (nc * 0x00204081u) & 0x01010101u;
        d1b = d1b + ea + ec - 2u * eb;
        s2 = s2 + d1b - 0x10101010u;
    };
    int tau = tau_s;
    for (; tau < t_begin + nt; ++tau) advance(nib(tau), nib(tau - aa), nib(tau - 2 * aa));
    // steady state: NB output frames per barrier.  Of the three rows a frame needs, the two old ones (tau - aa,
    // tau - 2 aa) were read by this thread a few iterations ago and hit L1; the NEW row comes from L2 / HBM, and its
    // first use was where the kernel stalled (28 % of all stall samples, profiles/r01_r_sass_mix.txt).  The new rows
    // of the NEXT batch are therefore requested one whole batch -- two barriers -- before they are needed.
    auto in_range = [&](int t) -> bool { return active && t >= tau_s && t >= 0 && t < a.T; };
    unsigned pre[NB];
#pragma unroll
    for (int j = 0; j < NB; ++j) pre[j] = (tau + j <= tau_e && in_range(tau + j)) ? __ldg(bp + (long long)(tau + j) * kFW) : 0u;
    for (; tau <= tau_e; tau += NB) {
        unsigned na[NB], nb[NB], nc[NB];
#pragma unroll
        for (int j = 0; j < NB; ++j) {
            const int tj = tau + j;
            const bool live = tj <= tau_e;
            na[j] = (live && in_range(tj)) ? (((pre[j] >> sh) & 0xFu) | fl) : 0u;
            pre[j] = (tj + NB <= tau_e && in_range(tj + NB)) ? __ldg(bp + (long long)(tj + NB) * kFW) : 0u;
            nb[j] = live ? nib(tj - aa) : 0u;
            nc[j] = live ? nib(tj - 2 * aa) : 0u;
        }
#pragma unroll
        for (int j = 0; j < NB; ++j) {
            advance(na[j], nb[j], nc[j]);
            unsigned char* row = s_raw + ((par * NB + j) * kSmoothUnits + ug) * RB;
            row[nf + 4 * i + 0] = (unsigned char)(s2 & 0xFFu);
            row[nf + 4 * i + 1] = (unsigned char)((s2 >> 8) & 0xFFu);
            row[nf + 4 * i + 2] = (unsigned char)((s2 >> 16) & 0xFFu);
            row[nf + 4 * i + 3] = (unsigned char)(s2 >> 24);
        }
        __syncthreads();
        // frequency direction; frames (t, t+1) of a pair leave together as one 16-byte store (num_index layout)
        auto freq_taps = [&](int j, unsigned (&o)[4]) {
            const unsigned char* row = s_raw + ((par * NB + j) * kSmoothUnits + ug) * RB;
            const unsigned* rw = reinterpret_cast<const unsigned*>(row) + i;
            unsigned wv[NTW + 1];
#pragma unroll
            for (int m = 0; m <= NTW; ++m) wv[m] = rw[m];
#pragma unroll
            for (int jj = 0; jj < 4; ++jj) {
                unsigned acc = 0u;
#pragma unroll
                for (int m = 0; m < NTW; ++m) {
                    const unsigned win = (jj == 0) ? wv[m] : __funnelshift_r(wv[m], wv[m + 1], 8 * jj);
                    acc = dp4a_u(win, taps[m], acc);
                }
                o[jj] = acc;
            }
        };
#pragma unroll
        for (int j = 0; j < NB; j += 2) {
            const int t_out = tau + j - nt;                   // even: strips start on even frames, NB is even
            if (tau + j > tau_e) break;
            unsigned oa[4], ob[4] = {0u, 0u, 0u, 0u};
            freq_taps(j, oa);
            if (tau + j + 1 <= tau_e) freq_taps(j + 1, ob);
            if (active) {
                uint4 pk;
                pk.x = oa[0] | (ob[0] << 16);
                pk.y = oa[1] | (ob[1] << 16);
                pk.z = oa[2] | (ob[2] << 16);
                pk.w = oa[3] | (ob[3] << 16);
                *reinterpret_cast<uint4*>(outp + (long long)(t_out >> 1) * (2 * kFPad)) = pk;
            }
        }
        par ^= 1;
    }
}

// =============================================================================================
// k2: synthesis (k2c_synthesize, gate_synth.cuh).
// =============================================================================================
struct K2Args {
    Geom g;
    Tables tb;
    void* y;                       // [C][out_stride], caller dtype
    const unsigned short* num;     // [n_units][T][FPad] integer mask numerators (stationary)
    const float* fmask;            // [n_units][T][FPad] final float masks (non-stationary)
    float pD;                      // prop_decrease / D
    float one_minus_p;             // 1 - prop_decrease
    int nt;                        // time half-width (edge factor of the first/last frames)
    int run;                       // output hops per work item
    int n_runs;
    DebugTap dbg;
    const float2* zcache;          // packed spectra of the frame pairs, stored by k1 / k1n
    int zpairs;
};

// time edge factor of the zero-padded smoothing: sum of the triangle taps that stay inside [0, T)
__device__ __forceinline__ float time_edge(int t, int T, int nt) {
    int s = 0;
    for (int b = -nt; b <= nt; ++b)
        if (t - b >= 0 && t - b < T) s += nt + 1 - (b < 0 ? -b : b);
    return (float)s / (float)((nt + 1) * (nt + 1));
}

// =============================================================================================
// Non-stationary gate (nonstationary.py:47-97).
//   k1n_magnitude  frames -> FFT -> |X|                         [n_units][T][FPad] float32
//   k_iir_sigmoid  filtfilt([b],[1,b-1]) along time per bin (forward sweep started at x[0], backward
//                  sweep over the forward output started at its last value -- nonstationary.py:106-115),
//                  then sigmoid(((|X| - S)/S - n_mult) * slope)  (spectralgate/utils.py:4-8)
//   k_smooth_box   separable triangular smoothing (zero padded), then  m * p + (1 - p); k_smooth_stream (nf > 12)
//                  and k_smooth_f (time extent too long for shared memory) are its fallbacks
// =============================================================================================
struct K1nArgs {
    Geom g;
    Tables tb;
    const void* x;
    float* mag;                // [n_units][T][FPad]
    DebugTap dbg;
    int run, n_runs;
    float2* zcache;            // optional, as in K1Args
    int zpairs;
    int z_lo, z_hi;
};

constexpr int k1n_smem_floats() { return kN + 2 * kN + kWarps * kExchFloats; }

template <int HR, typename T>
__global__ void __launch_bounds__(kThreads, 3) k1n_magnitude(const K1nArgs a) {
    B200_DYN_SMEM(float, smem);
    float* s_wa = smem;
    float2* s_tw = reinterpret_cast<float2*>(smem + kN);
    float* s_tiles = smem + 3 * kN;
    for (int i = threadIdx.x; i < kN; i += kThreads) {
        s_wa[i] = a.tb.wa[i];
        s_tw[i] = a.tb.tw[i];
    }
    __syncthreads();
    const Geom& g = a.g;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    float* tile = s_tiles + warp * kExchFloats;
    const int H = g.H;
    const int pl = (32 - lane) & 31;
    const long long n_items = (long long)g.n_units * a.n_runs;
    for (long long item = (long long)blockIdx.x * kWarps + warp; item < n_items;
         item += (long long)gridDim.x * kWarps) {
        const int ul = (int)(item / a.n_runs);
        const int run = (int)(item - (long long)ul * a.n_runs);
        const int u = g.u0 + ul;
        const int ic = u / g.C, c = u - ic * g.C;
        const long long i1 = (long long)ic * g.step - g.pad;
        const T* xrow = static_cast<const T*>(a.x) + (long long)c * g.in_stride;
        const int t0 = run * a.run;
        const int t1 = min(t0 + a.run, g.T);
        for (int t = t0; t < t1; t += 2) {
            const bool vb = (t + 1 < t1);
            const long long base = (long long)t * H - kN / 2;
            float re[32], im[32];
            load_frame_pair<HR>(re, im, xrow, base, i1, g.Lp, g.n_total, s_wa, lane, vb);
            warp_fft1024(re, im, tile, s_tw, lane);
            if (a.zcache && t >= a.z_lo && t < a.z_hi) {
                float2* zp = a.zcache + ((long long)ul * a.zpairs + (t >> 1)) * 1024 + lane;
#pragma unroll
                for (int q = 0; q < 32; ++q) zp[32 * q] = make_float2(re[brev5(q)], im[brev5(q)]);
            }
            if (!a.mag && a.dbg.ul != ul) continue;        // spectra only
            float* dstA = a.mag + ((long long)ul * g.T + t) * kFPad;
#pragma unroll
            for (int q = 0; q < kFW; ++q) {
                const int sA = brev5(q), sP = brev5(31 - q), s0 = brev5((32 - q) & 31);
                const float zr = re[sA], zi = im[sA];
                float pr = __shfl_sync(0xffffffffu, re[sP], pl);
                float pi = __shfl_sync(0xffffffffu, im[sP], pl);
                if (lane == 0) { pr = re[s0]; pi = im[s0]; }
                const float ar = zr + pr, ai = zi - pi;
                const float br = zi + pi, bi = pr - zr;
                const int k = lane + 32 * q;
                const bool valid = (q < 16) || (lane == 0);
                const float ma = valid ? 0.5f * sqrtf(fmaf(ar, ar, ai * ai)) : 0.f;
                const float mb = valid ? 0.5f * sqrtf(fmaf(br, br, bi * bi)) : 0.f;
                if (a.mag) {                               // (null: spectra only -- b200gate_torch_apply_masks)
                    dstA[k] = ma;
                    if (vb) dstA[kFPad + k] = mb;
                }
                if (a.dbg.ul == ul && valid && k < kF) {
                    float* sp = a.dbg.spec + ((long long)t * kF + k) * 2;
                    sp[0] = 0.5f * ar; sp[1] = 0.5f * ai;
                    if (vb) { sp[2 * kF] = 0.5f * br; sp[2 * kF + 1] = 0.5f * bi; }
                }
            }
        }
    }
}

struct IirArgs {
    int n_units, T;
    int F, FPad;               // bins and padded row pitch (513/544 for n_fft 1024, 1025/1056 for 2048)
    double b;                  // nonstationary.py:114
    float n_mult, slope;       // thresh_n_mult_nonstationary, sigmoid_slope_nonstationary
    int regen;                 // 1: regenerate the forward sweep in the backward pass instead of storing it
    const float* mag;          // [n_units][T][FPad]
    float* m0;                 // [n_units][T][FPad]: forward sweep, then overwritten by the sigmoid mask
};

template <int FP>                                       // padded row pitch: 544 (n_fft 1024) or 1056 (n_fft 2048)
__global__ void __launch_bounds__(128) k_iir_sigmoid(const IirArgs a) {
    const int FF = a.F;
    const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= (long long)a.n_units * FP) return;
    const int ul = (int)(idx / FP), f = (int)(idx - (long long)ul * FP);
    const float* __restrict__ A = a.mag + (long long)ul * a.T * FP + f;
    float* M = a.m0 + (long long)ul * a.T * FP + f;
    if (f >= FF) {
        for (int t = 0; t < a.T; ++t) M[(long long)t * FP] = 0.f;
        return;
    }
    // The recurrence state stays in float64 (the filter pole 1 - b ~ 0.995 accumulates rounding over hundreds of
    // frames); the follower ratio, exponential and reciprocal run in float32 (the float64 exp / divide of the first
    // version made this kernel 3x longer than both FFT kernels together).  The sweeps are serial per (unit, bin), so
    // what bounds them is the latency of each step and the instructions around it: every recurrence is ONE fused
    // multiply-add on the carried value (the input term b x is formed off the chain); the |X| column is fetched in
    // batches of kB frames through a walking pointer with compile-time offsets (the row pitch is a template parameter),
    // the next batch requested before the current one is consumed, so no load sits between two steps of the chain;
    // the ratio is num * rcp(s) and the sigmoid a correctly rounded reciprocal (no division slow paths in the loop).
    constexpr int kB = 8;
    const double b = a.b, omb = 1.0 - a.b;
    const float n_mult = a.n_mult, slope = a.slope;
    const int T = a.T;
    auto sigmoid_mask = [&](double x, double sm) -> float {
        const float num = (float)(x - sm);                     // |X| - S without float32 cancellation
        const float r = num * __frcp_rn((float)sm);
        return __frcp_rn(1.0f + expf(-(r - n_mult) * slope));
    };
    // frames t0 + dir * j, j = 0..kB-1; `full`: all of them exist (compile-time offsets), else clamped (never used)
    auto fetch = [&](const float* src, float (&x)[kB], int t0, int dir) {
        const bool full = dir > 0 ? (t0 >= 0 && t0 + kB <= T) : (t0 < T && t0 - kB + 1 >= 0);
        if (full) {
            const float* p = src + (long long)t0 * FP;
            if (dir > 0) {
#pragma unroll
                for (int j = 0; j < kB; ++j) x[j] = p[j * FP];
            } else {
#pragma unroll
                for (int j = 0; j < kB; ++j) x[j] = p[-j * FP];
            }
        } else {
#pragma unroll
            for (int j = 0; j < kB; ++j) x[j] = src[(long long)min(max(t0 + dir * j, 0), T - 1) * FP];
        }
    };
    double s = (double)A[0];
    if (a.regen) {
        // The forward sweep is not stored: the backward sweep regenerates it by the inverse recurrence
        // fwd[t-1] = (fwd[t] - b x[t]) / (1 - b) in float64.  Its error grows by 1/(1 - b) per step; the host selects
        // this variant only when (1 - b)^-T * 2^-53 stays far below float32 resolution (T ln(1/(1-b)) < 20), which
        // holds for the reference's time constants (config 3: 6.9).  One read of |X| less, no forward write.
        {
            float cur[kB], nxt[kB];
            fetch(A, cur, 0, 1);
            int t0 = 0;
            for (; t0 + kB <= T; t0 += kB) {
                fetch(A, nxt, t0 + kB, 1);
#pragma unroll
                for (int j = 0; j < kB; ++j) s = fma(omb, s, b * (double)cur[j]);
#pragma unroll
                for (int j = 0; j < kB; ++j) cur[j] = nxt[j];
            }
#pragma unroll
            for (int j = 0; j < kB; ++j)
                if (t0 + j < T) s = fma(omb, s, b * (double)cur[j]);
        }
        const double inv_omb = 1.0 / omb, nb_inv = -b * inv_omb;
        double fw = s;                                         // fwd[T-1]
        float cur[kB], nxt[kB];
        fetch(A, cur, T - 1, -1);
        int t0 = T - 1;
        for (; t0 - kB + 1 >= 0; t0 -= kB) {
            fetch(A, nxt, t0 - kB, -1);
            float* mp = M + (long long)t0 * FP;
#pragma unroll
            for (int j = 0; j < kB; ++j) {
                const double x = (double)cur[j];
                s = fma(omb, s, b * fw);
                mp[-j * FP] = sigmoid_mask(x, s);
                fw = fma(inv_omb, fw, nb_inv * x);
            }
#pragma unroll
            for (int j = 0; j < kB; ++j) cur[j] = nxt[j];
        }
#pragma unroll
        for (int j = 0; j < kB; ++j) {
            if (t0 - j >= 0) {
                const double x = (double)cur[j];
                s = fma(omb, s, b * fw);
                M[(long long)(t0 - j) * FP] = sigmoid_mask(x, s);
                fw = fma(inv_omb, fw, nb_inv * x);
            }
        }
        return;
    }
    {
        float cur[kB], nxt[kB];
        fetch(A, cur, 0, 1);
        for (int t0 = 0; t0 < T; t0 += kB) {
            fetch(A, nxt, t0 + kB, 1);
#pragma unroll
            for (int j = 0; j < kB; ++j) {
                if (t0 + j < T) {
                    s = fma(omb, s, b * (double)cur[j]);
                    M[(long long)(t0 + j) * FP] = (float)s;
                }
            }
#pragma unroll
            for (int j = 0; j < kB; ++j) cur[j] = nxt[j];
        }
    }
    // (the stored forward sweep is read back through M itself -- each element before it is overwritten)
    const float* Mr = M;
    s = (double)Mr[(long long)(T - 1) * FP];
    for (int t0 = T - 1; t0 >= 0; t0 -= kB) {
        float fwv[kB], xx[kB];
        fetch(Mr, fwv, t0, -1);
        fetch(A, xx, t0, -1);
#pragma unroll
        for (int j = 0; j < kB; ++j) {
            if (t0 - j >= 0) {
                s = fma(omb, s, b * (double)fwv[j]);
                M[(long long)(t0 - j) * FP] = sigmoid_mask((double)xx[j], s);
            }
        }
    }
}

struct SmoothFArgs {
    int n_units, T;
    int F, FPad;
    int nf, nt;
    int tf_lo, tf_hi, TT;
    float p, one_minus_p;
    const float* m0;           // [n_units][T][FPad]
    float* m2;                 // [n_units][T][FPad]
};
__host__ __device__ inline int smoothf_cpitch(int FPad, int nf) { return FPad + 2 * nf + 1; }
inline size_t smoothf_smem_bytes(int TT, int FPad, int nf) { return (size_t)TT * smoothf_cpitch(FPad, nf) * 4; }

__global__ void __launch_bounds__(256) k_smooth_f(const SmoothFArgs a) {
    B200_DYN_SMEM(float, s_c);                         // [TT][cp]
    const int FP = a.FPad, FF = a.F;
    const int nt = a.nt, nf = a.nf, cp = smoothf_cpitch(a.FPad, nf);
    const int ul = blockIdx.y;
    const int t0 = a.tf_lo + blockIdx.x * a.TT;
    if (t0 >= a.tf_hi) return;
    const int tt_n = min(a.TT, a.tf_hi - t0);
    for (int i = threadIdx.x; i < a.TT * cp; i += blockDim.x) s_c[i] = 0.f;
    __syncthreads();
    const float* src = a.m0 + (long long)ul * a.T * FP;
    for (int i = threadIdx.x; i < tt_n * FP; i += blockDim.x) {
        const int tt = i / FP, f = i - tt * FP;
        if (f >= FF) continue;
        const int t = t0 + tt;
        float acc = 0.f;
        for (int bb = -nt; bb <= nt; ++bb) {
            const int tq = t - bb;
            if (tq >= 0 && tq < a.T) acc = fmaf((float)(nt + 1 - (bb < 0 ? -bb : bb)), src[(long long)tq * FP + f], acc);
        }
        s_c[tt * cp + nf + f] = acc;
    }
    __syncthreads();
    const float invD = 1.0f / ((float)((nf + 1) * (nf + 1)) * (float)((nt + 1) * (nt + 1)));
    float* dst = a.m2 + (long long)ul * a.T * FP;
    for (int i = threadIdx.x; i < tt_n * FP; i += blockDim.x) {
        const int tt = i / FP, f = i - tt * FP;
        float v = 0.f;
        if (f < FF) {
            const float* cr = s_c + tt * cp + f;
            float acc = 0.f;
            for (int d = -nf; d <= nf; ++d) acc = fmaf((float)(nf + 1 - (d < 0 ? -d : d)), cr[nf + d], acc);
            v = fmaf(acc * invD, a.p, a.one_minus_p);           // nonstationary.py:82-84
        }
        dst[(long long)(t0 + tt) * FP + f] = v;
    }
}

// Streaming form of the same smoothing (it runs where the box form below does not apply, e.g. nf > 12; k_smooth_f
// above serves rings too large for shared memory).  A CTA walks a strip of frames of one unit; thread i owns bins
// i, i+G, i+2G, i+3G (G = FPad/4, so every shared-memory access of a warp is 32 consecutive floats): the last
// 2 nt + 1 mask rows live in a ring of thread-private columns (no barrier needed to refill it), the time-direction
// triangle is taken straight from the ring, the
// frequency-direction triangle from one zero-haloed row -- two barriers per frame, every mask value read from HBM
// once per strip and written once.
inline size_t smooths_smem_bytes(int FPad, int nf, int nt) { return ((size_t)(2 * nt + 1) * FPad + FPad + 2 * nf + 8) * 4; }

__global__ void __launch_bounds__(288) k_smooth_stream(const SmoothFArgs a) {
    B200_DYN_SMEM(float, s_buf);
    const int FP = a.FPad, FF = a.F, nt = a.nt, nf = a.nf, R = 2 * nt + 1;
    const int G = blockDim.x, tid = threadIdx.x;
    float* ring = s_buf;                     // [R][FP]
    float* row = s_buf + (size_t)R * FP;     // [nf | FP | nf]
    const int ul = blockIdx.y;
    const int t_begin = a.tf_lo + blockIdx.x * a.TT;
    if (t_begin >= a.tf_hi) return;
    const int t_end = min(t_begin + a.TT, a.tf_hi);
    const float* src = a.m0 + (long long)ul * a.T * FP;
    float* dst = a.m2 + (long long)ul * a.T * FP;
    for (int i = tid; i < FP + 2 * nf; i += G) row[i] = 0.f;
    auto load_row = [&](int t, int slot) {
        const bool in = t >= 0 && t < a.T;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int bin = tid + j * G;
            ring[slot * FP + bin] = (in && bin < FF) ? src[(long long)t * FP + bin] : 0.f;
        }
    };
    // ring slot of frame t: (t - t_begin + nt) mod R, so the newest row t + nt of step t sits at slot (t - t_begin + 2 nt) mod R
    for (int k = 0; k < 2 * nt; ++k) load_row(t_begin - nt + k, k);
    int newest = (2 * nt) % R;
    const float invD = 1.0f / ((float)((nf + 1) * (nf + 1)) * (float)((nt + 1) * (nt + 1)));
    __syncthreads();
    for (int t = t_begin; t < t_end; ++t) {
        load_row(t + nt, newest);
        float c[4] = {0.f, 0.f, 0.f, 0.f};
        int slot = newest;                                  // frame t + nt; walking back to t - nt
        for (int b = -nt; b <= nt; ++b) {
            const float w = (float)(nt + 1 - (b < 0 ? -b : b));
#pragma unroll
            for (int j = 0; j < 4; ++j) c[j] = fmaf(w, ring[slot * FP + tid + j * G], c[j]);
            slot = slot == 0 ? R - 1 : slot - 1;
        }
        newest = newest + 1 == R ? 0 : newest + 1;
        __syncthreads();                                    // the previous frame's frequency pass has read `row`
#pragma unroll
        for (int j = 0; j < 4; ++j) row[nf + tid + j * G] = c[j];
        __syncthreads();
        float o[4] = {0.f, 0.f, 0.f, 0.f};
        for (int d = -nf; d <= nf; ++d) {
            const float w = (float)(nf + 1 - (d < 0 ? -d : d));
#pragma unroll
            for (int j = 0; j < 4; ++j) o[j] = fmaf(w, row[nf + tid + j * G + d], o[j]);
        }
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int bin = tid + j * G;
            dst[(long long)t * FP + bin] = bin < FF ? fmaf(o[j] * invD, a.p, a.one_minus_p) : 0.f;      // nonstationary.py:82-84
        }
    }
}

// Box form of the streaming smoothing (the one that normally runs for 1 <= nf <= 12).  The triangle taps
// (n + 1 - |d|) are the self-convolution of a length-(n + 1) box, so the frequency direction is two sliding box sums
// instead of 2 nf + 1 multiply-adds per bin: thread i owns the four CONSECUTIVE bins 4i..4i+3 (every shared-memory
// access is one aligned 128-bit vector), takes the first box sum of each pass directly and the other three by
// add-one / drop-one.  Per four bins and frame: ~17 vector loads and ~75 floating-point instructions against the
// tap loops' ~120 scalar loads and ~120 FMAs.  The box sums restart in every thread and every frame, so no rounding
// accumulates along a row or over time.  Row buffers: rowA = time-smoothed row c[] with 16 zero floats either side,
// rowB = first box sums b1[g] = sum_{j=0..nf} c[g + j] stored at index g + 12 (g runs from -12: the second pass
// out[f] = sum_{g=f-nf..f} b1[g] reaches nf bins to the left); bins >= F hold zeros, and FPad - F >= 12.
inline size_t smoothb_smem_bytes(int FPad, int nt) { return ((size_t)(2 * nt + 1) * FPad + (FPad + 32) + (FPad + 16)) * 4; }

template <int NF>
__global__ void __launch_bounds__(288) k_smooth_box(const SmoothFArgs a) {
    static_assert(NF >= 1 && NF <= 12, "box smoothing handles 1 <= nf <= 12");
    B200_DYN_SMEM(float, s_buf);
    const int FP = a.FPad, FF = a.F, nt = a.nt, R = 2 * nt + 1;
    const int G = blockDim.x, tid = threadIdx.x;           // G == FP / 4
    float* ring = s_buf;                                   // [R][FP]
    float* rowA = s_buf + (size_t)R * FP;                  // [16 | FP | 16]
    float* rowB = rowA + FP + 32;                          // [FP + 16]
    const int ul = blockIdx.y;
    const int t_begin = a.tf_lo + blockIdx.x * a.TT;
    if (t_begin >= a.tf_hi) return;
    const int t_end = min(t_begin + a.TT, a.tf_hi);
    const float* src = a.m0 + (long long)ul * a.T * FP;
    float* dst = a.m2 + (long long)ul * a.T * FP;
    for (int i = tid; i < 2 * FP + 48; i += G) rowA[i] = 0.f;          // rowA and rowB are contiguous
    const int b0 = 4 * tid;
    auto fetch_row = [&](int t) -> float4 {
        float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
        if (t >= 0 && t < a.T) {
            v = __ldg(reinterpret_cast<const float4*>(src + (long long)t * FP + b0));
            if (b0 + 0 >= FF) v.x = 0.f;
            if (b0 + 1 >= FF) v.y = 0.f;
            if (b0 + 2 >= FF) v.z = 0.f;
            if (b0 + 3 >= FF) v.w = 0.f;
        }
        return v;
    };
    for (int k = 0; k < 2 * nt; ++k) *reinterpret_cast<float4*>(ring + k * FP + b0) = fetch_row(t_begin - nt + k);
    int newest = (2 * nt) % R;
    const float invD = 1.0f / ((float)((NF + 1) * (NF + 1)) * (float)((nt + 1) * (nt + 1)));
    // the rows of the next two frames are requested while this frame is being smoothed: the only global load of the loop
    // otherwise sits right in front of its first use (long-scoreboard stalls were 3.8 cycles per issued instruction)
    float4 pre0 = fetch_row(t_begin + nt), pre1 = fetch_row(t_begin + nt + 1);
    __syncthreads();
    for (int t = t_begin; t < t_end; ++t) {
        *reinterpret_cast<float4*>(ring + newest * FP + b0) = pre0;
        pre0 = pre1;
        pre1 = (t + 2 < t_end) ? fetch_row(t + nt + 2) : make_float4(0.f, 0.f, 0.f, 0.f);
        float4 c = make_float4(0.f, 0.f, 0.f, 0.f);
        {
            // (measured and dropped: walking the ring in physical order with a rotating tap table -- fewer instructions per
            //  tap, 1 ms slower per config-3 step; profiles/r02_experiments.md)
            int slot = newest;                              // frame t + nt; walking back to t - nt
            for (int b = -nt; b <= nt; ++b) {
                const float w = (float)(nt + 1 - (b < 0 ? -b : b));
                const float4 r = *reinterpret_cast<const float4*>(ring + slot * FP + b0);
                c.x = fmaf(w, r.x, c.x); c.y = fmaf(w, r.y, c.y); c.z = fmaf(w, r.z, c.z); c.w = fmaf(w, r.w, c.w);
                slot = slot == 0 ? R - 1 : slot - 1;
            }
        }
        newest = newest + 1 == R ? 0 : newest + 1;
        *reinterpret_cast<float4*>(rowA + 16 + b0) = c;     // (the previous frame's first pass finished before its 2nd barrier)
        __syncthreads();
        {   // first box: b1[g], g = b0 - 12 + m, from c[g .. g + NF] = rowA[16 + g ..]
            constexpr int NV = (4 + NF + 3) / 4;
            float v[4 * NV];
#pragma unroll
            for (int k = 0; k < NV; ++k) {
                const float4 q = *reinterpret_cast<const float4*>(rowA + b0 + 4 + 4 * k);
                v[4 * k] = q.x; v[4 * k + 1] = q.y; v[4 * k + 2] = q.z; v[4 * k + 3] = q.w;
            }
            float s0 = v[0];
#pragma unroll
            for (int j = 1; j <= NF; ++j) s0 += v[j];
            const float s1 = s0 + v[NF + 1] - v[0];
            const float s2 = s1 + v[NF + 2] - v[1];
            const float s3 = s2 + v[NF + 3] - v[2];
            *reinterpret_cast<float4*>(rowB + b0) = make_float4(s0, s1, s2, s3);   // (the previous frame's second pass finished before this frame's 1st barrier)
        }
        __syncthreads();
        {   // second box: out[f], f = b0 + m, from b1[f - NF .. f] = rowB[f + 12 - NF .. f + 12]
            constexpr int A0 = (12 - NF) & ~3, O = (12 - NF) & 3, NV = (16 - A0) / 4;
            float u[4 * NV];
#pragma unroll
            for (int k = 0; k < NV; ++k) {
                const float4 q = *reinterpret_cast<const float4*>(rowB + b0 + A0 + 4 * k);
                u[4 * k] = q.x; u[4 * k + 1] = q.y; u[4 * k + 2] = q.z; u[4 * k + 3] = q.w;
            }
            float o0 = u[O];
#pragma unroll
            for (int e = 1; e <= NF; ++e) o0 += u[O + e];
            const float o1 = o0 + u[O + NF + 1] - u[O];
            const float o2 = o1 + u[O + NF + 2] - u[O + 1];
            const float o3 = o2 + u[O + NF + 3] - u[O + 2];
            float4 r;                                                               // nonstationary.py:82-84
            r.x = b0 + 0 < FF ? fmaf(o0 * invD, a.p, a.one_minus_p) : 0.f;
            r.y = b0 + 1 < FF ? fmaf(o1 * invD, a.p, a.one_minus_p) : 0.f;
            r.z = b0 + 2 < FF ? fmaf(o2 * invD, a.p, a.one_minus_p) : 0.f;
            r.w = b0 + 3 < FF ? fmaf(o3 * invD, a.p, a.one_minus_p) : 0.f;
            *reinterpret_cast<float4*>(dst + (long long)t * FP + b0) = r;
        }
    }
}

// =============================================================================================
// TorchGate surface (noisereduce/torchgate/torchgate.py:200-264).  Same analysis / synthesis kernels;
// what differs is the mask: statistics per (row, bin) over the row's own frames (or over xn's),
// top_db = 40, unbiased std (torchgate.py:127-165, torchgate/utils.py:6-23), and for the
// non-stationary variant a moving mean instead of the IIR (torchgate.py:168-198).
// =============================================================================================
struct TStatArgs {
    int n_units, T;
    float in_scale;            // sum(window): TorchGate's STFT is not normalised
    float eps;                 // torch.finfo(float64).eps added in float32
    float top_db;
    float n_std;
    int ddof;
    float* mag;                // in: |X| / sum(w);  out: dB (float32), unclamped
    float* rowmax;             // [n_units][FPad] max_t dB
    float* thr;                // [n_units][FPad] mean + n_std * std of the clamped dB
};

// One CTA per (unit, 32-bin group); its kTgWarps warps share the frames (warp w takes t = w, w + kTgWarps, ...), every access
// of a warp is one 128-byte row segment, and the per-bin max / sum / sum of squares are combined through shared memory in
// warp order (deterministic).  One thread per (unit, bin) walking all T frames -- the first form of these kernels -- left
// a 256-row batch with 139 k threads and the column walks latency-bound (0.38 + 0.29 ms of a 1.47 ms forward).
constexpr int kTgWarps = 8;

__global__ void __launch_bounds__(kTgWarps * 32) k_tgate_stats(const TStatArgs a) {
    __shared__ double s_red[kTgWarps][32];
    __shared__ float s_mx[kTgWarps][32];
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const int ul = blockIdx.x / kFW, grp = blockIdx.x - ul * kFW;
    const int f = grp * 32 + lane;
    const long long idx = (long long)ul * kFPad + f;
    float* D = a.mag + (long long)ul * a.T * kFPad + f;
    const bool live = f < kF;
    float mx = -INFINITY;
    if (live) {
#pragma unroll 4
        for (int t = w; t < a.T; t += kTgWarps) {
            const float db = 20.0f * log10f(D[(long long)t * kFPad] * a.in_scale + a.eps);
            D[(long long)t * kFPad] = db;
            mx = fmaxf(mx, db);
        }
    }
    s_mx[w][lane] = mx;
    __syncthreads();
#pragma unroll
    for (int k = 0; k < kTgWarps; ++k) mx = fmaxf(mx, s_mx[k][lane]);
    const float fl = mx - a.top_db;
    double sum = 0.0;
    if (live) {
#pragma unroll 4
        for (int t = w; t < a.T; t += kTgWarps) sum += (double)fmaxf(D[(long long)t * kFPad], fl);     // (this thread's own stores)
    }
    s_red[w][lane] = sum;
    __syncthreads();
    sum = 0.0;
#pragma unroll
    for (int k = 0; k < kTgWarps; ++k) sum += s_red[k][lane];
    const double mean = sum / a.T;
    __syncthreads();
    double ss = 0.0;
    if (live) {
#pragma unroll 4
        for (int t = w; t < a.T; t += kTgWarps) {
            const double d = (double)fmaxf(D[(long long)t * kFPad], fl) - mean;
            ss += d * d;
        }
    }
    s_red[w][lane] = ss;
    __syncthreads();
    if (w == 0) {
        ss = 0.0;
#pragma unroll
        for (int k = 0; k < kTgWarps; ++k) ss += s_red[k][lane];
        const double sd = sqrt(ss / (double)(a.T - a.ddof));
        a.rowmax[idx] = live ? mx : -INFINITY;
        a.thr[idx] = live ? (float)(mean + sd * (double)a.n_std) : INFINITY;
    }
}

struct TBitsArgs {
    int n_units, T;
    int thr_units;             // rows of thr: n_units (self / per-row xn) or 1 (broadcast)
    float top_db;
    const float* db;           // [n_units][T][FPad]
    const float* rowmax;       // [n_units][FPad]  (of x itself)
    const float* thr;          // [thr_units][FPad]
    unsigned* bits;            // [n_units][T][FW]
};

__global__ void __launch_bounds__(kTgWarps * 32) k_tgate_bits(const TBitsArgs a) {
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const int ul = blockIdx.x / kFW, grp = blockIdx.x - ul * kFW;
    const int f = grp * 32 + lane;
    const float* D = a.db + (long long)ul * a.T * kFPad + f;
    const float fl = a.rowmax[(long long)ul * kFPad + f] - a.top_db;
    const float th = a.thr[(long long)(a.thr_units == 1 ? 0 : ul) * kFPad + f];
    const bool live = f < kF;
    unsigned* brow = a.bits + (long long)ul * a.T * kFW + grp;
    constexpr int kU = 4;                                   // rows requested together, then voted on
    for (int t0 = w; t0 < a.T; t0 += kU * kTgWarps) {
        float v[kU];
#pragma unroll
        for (int j = 0; j < kU; ++j) {
            const int t = t0 + j * kTgWarps;
            v[j] = (t < a.T) ? D[(long long)t * kFPad] : -INFINITY;
        }
#pragma unroll
        for (int j = 0; j < kU; ++j) {
            const int t = t0 + j * kTgWarps;
            const unsigned word = __ballot_sync(0xffffffffu, live && (fmaxf(v[j], fl) > th));
            if (t < a.T && lane == 0) brow[(long long)t * kFW] = word;
        }
    }
}

struct TMovArgs {
    int n_units, T;
    int n_movemean;
    float n_thresh, inv_temp, p;
    const float* mag;
    float* m0;                 // blended sigmoid mask, prop_decrease * (m - 1) + 1 (torchgate.py:241)
};

__global__ void __launch_bounds__(128) k_tgate_movmean(const TMovArgs a) {
    const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= (long long)a.n_units * kFPad) return;
    const int ul = (int)(idx / kFPad), f = (int)(idx - (long long)ul * kFPad);
    const float* A = a.mag + (long long)ul * a.T * kFPad + f;
    float* M = a.m0 + (long long)ul * a.T * kFPad + f;
    if (f >= kF) {
        for (int t = 0; t < a.T; ++t) M[(long long)t * kFPad] = 0.f;
        return;
    }
    // conv1d(ones(n), padding="same"): window [t - left, t + right], zero padded, left = (n-1)/2
    const int n = a.n_movemean, left = (n - 1) / 2, right = n - 1 - left;
    double run = 0.0;
    for (int t = 0; t <= right && t < a.T; ++t) run += (double)A[(long long)t * kFPad];
    for (int t = 0; t < a.T; ++t) {
        const float Av = A[(long long)t * kFPad];
        const float S = (float)(run / (double)n);
        const float r = (Av - S) / S;
        const float m = 1.0f / (1.0f + expf(-(r - a.n_thresh) * a.inv_temp));
        M[(long long)t * kFPad] = a.p * (m - 1.0f) + 1.0f;
        const int tin = t + 1 + right, tout = t - left;
        if (tin < a.T) run += (double)A[(long long)tin * kFPad];
        if (tout >= 0) run -= (double)A[(long long)tout * kFPad];
    }
}

// =============================================================================================
// dtype conversion at the edges (base.py:140 promotes every chunk to float64; :218-226 casts back)
// =============================================================================================
template <typename Tin>
__global__ void k_to_f32(const Tin* __restrict__ src, float* __restrict__ dst, long long C, long long n,
                         long long sstride, long long dstride) {
    const long long total = C * n;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total;
         i += (long long)gridDim.x * blockDim.x) {
        const long long c = i / n, j = i - c * n;
        dst[c * dstride + j] = (float)src[c * sstride + j];
    }
}
template <typename Tout>
__device__ __forceinline__ Tout cast_out(float v);
template <> __device__ __forceinline__ double cast_out<double>(float v) { return (double)v; }
template <> __device__ __forceinline__ short cast_out<short>(float v) {
    // numpy float -> int16 astype: C truncation toward zero, wrapping the low 16 bits
    return (short)(int)v;
}
template <typename Tout>
__global__ void k_from_f32(const float* __restrict__ src, Tout* __restrict__ dst, long long C, long long n,
                           long long sstride, long long dstride) {
    const long long total = C * n;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total;
         i += (long long)gridDim.x * blockDim.x) {
        const long long c = i / n, j = i - c * n;
        dst[c * dstride + j] = cast_out<Tout>(src[c * sstride + j]);
    }
}

// =============================================================================================
// K0: one-time stationary noise statistics (stationary.py:61-81), float64.
// =============================================================================================
// sequential channel sum in channel order (np.mean(axis=0) adds rows in order; float32 stays float32)
template <typename Tin, typename Tacc>
__global__ void k0_channel_sum(const Tin* __restrict__ y, long long C, long long n, long long stride,
                               Tacc* __restrict__ acc, int init) {
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n;
         i += (long long)gridDim.x * blockDim.x) {
        Tacc s = init ? (Tacc)0 : acc[i];
        for (long long c = 0; c < C; ++c) s = s + (Tacc)y[c * stride + i];
        acc[i] = s;
    }
}
template <typename Tacc>
__global__ void k0_mean_to_f64(const Tacc* __restrict__ acc, long long n, long long C, double* __restrict__ out) {
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n;
         i += (long long)gridDim.x * blockDim.x)
        out[i] = (double)(acc[i] / (Tacc)C);          // division in the accumulation dtype, as numpy
}

// One CTA per frame: float64 radix-2 FFT in shared memory -> dB (utils.py:15), [Tn][F].
struct K0Args {
    const double* yn;      // [n] collapsed noise clip
    long long n;
    int H, Tn;
    const double* wa64;
    const double2* cs64;
    double eps;
    double* db;            // [Tn][F]
};
__global__ void __launch_bounds__(256) k0_stft_db(const K0Args a) {
    B200_DYN_SMEM(double2, s);                      // [N]
    const int t = blockIdx.x;
    const long long base = (long long)t * a.H - kN / 2;
    for (int n = threadIdx.x; n < kN; n += blockDim.x) {
        const long long j = base + n;
        const double v = (j >= 0 && j < a.n) ? a.yn[j] * a.wa64[n] : 0.0;
        int r = 0;
        for (int b = 0; b < 10; ++b) r |= ((n >> b) & 1) << (9 - b);
        s[r] = make_double2(v, 0.0);
    }
    __syncthreads();
    for (int len = 2; len <= kN; len <<= 1) {
        const int half = len >> 1, stride = kN / len;
        for (int i = threadIdx.x; i < kN / 2; i += blockDim.x) {
            const int blk = i / half, o = i - blk * half;
            const int ia = blk * len + o, ib = ia + half;
            const double2 w = a.cs64[o * stride];                 // exp(-i th) = cos - i sin
            const double2 x = s[ia], y = s[ib];
            const double yr = y.x * w.x + y.y * w.y, yi = y.y * w.x - y.x * w.y;
            s[ia] = make_double2(x.x + yr, x.y + yi);
            s[ib] = make_double2(x.x - yr, x.y - yi);
        }
        __syncthreads();
    }
    for (int f = threadIdx.x; f < kF; f += blockDim.x) {
        const double2 v = s[f];
        a.db[(long long)t * kF + f] = 20.0 * log10(sqrt(v.x * v.x + v.y * v.y) + a.eps);
    }
}

// One CTA per bin: top_db floor, mean, std (ddof), thresh.
__global__ void __launch_bounds__(256) k0_stats(const double* __restrict__ db, int Tn, int F, double top_db, int ddof,
                                                double n_std, double* __restrict__ mean_out,
                                                double* __restrict__ std_out, double* __restrict__ thr_out) {
    __shared__ double red[256];
    const int f = blockIdx.x;
    double m = -1.0e300;
    for (int t = threadIdx.x; t < Tn; t += blockDim.x) m = fmax(m, db[(long long)t * F + f]);
    red[threadIdx.x] = m;
    __syncthreads();
    for (int o = 128; o > 0; o >>= 1) {
        if ((int)threadIdx.x < o) red[threadIdx.x] = fmax(red[threadIdx.x], red[threadIdx.x + o]);
        __syncthreads();
    }
    const double fl = red[0] - top_db;
    __syncthreads();
    double sum = 0.0;
    for (int t = threadIdx.x; t < Tn; t += blockDim.x) sum += fmax(db[(long long)t * F + f], fl);
    red[threadIdx.x] = sum;
    __syncthreads();
    for (int o = 128; o > 0; o >>= 1) {
        if ((int)threadIdx.x < o) red[threadIdx.x] += red[threadIdx.x + o];
        __syncthreads();
    }
    const double mean = red[0] / Tn;
    __syncthreads();
    double ss = 0.0;
    for (int t = threadIdx.x; t < Tn; t += blockDim.x) {
        const double d = fmax(db[(long long)t * F + f], fl) - mean;
        ss += d * d;
    }
    red[threadIdx.x] = ss;
    __syncthreads();
    for (int o = 128; o > 0; o >>= 1) {
        if ((int)threadIdx.x < o) red[threadIdx.x] += red[threadIdx.x + o];
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        const double sd = sqrt(red[0] / (double)(Tn - ddof));
        mean_out[f] = mean;
        std_out[f] = sd;
        thr_out[f] = mean + sd * n_std;
    }
}

}  // namespace b200
