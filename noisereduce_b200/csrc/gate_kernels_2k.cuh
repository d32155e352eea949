// gate_kernels_2k.cuh -- n_fft = 2048 family (BASELINE.json config 3: non-stationary gate, hop 512).
//
// One real frame of 2048 samples rides in one 1024-point complex warp FFT (warp_fft.cuh) by the
// half-length trick:  z[m] = x[2m] + i x[2m+1],  Z = FFT_1024(z),
//     E[k] = (Z[k] + conj Z[1024-k]) / 2,   O[k] = (Z[k] - conj Z[1024-k]) / (2i),   W_k = exp(-i pi k / 1024)
//     X[k] = E[k] + W_k O[k],               X[1024-k] = conj(E[k] - W_k O[k]),       k = 0..512
// and back:  with P = X[k], Q = conj X[1024-k] after masking,
//     E' = (P + Q)/2,  T' = (P - Q)/2,  Z'[k] = E' + i conj(W_k) T',  Z'[1024-k] = conj(E') + i W_k conj(T').
// The mirrored element lives in lane 32-lane, slot 31-slot -- the same shuffle pattern as the 1024
// family.  A hop (512 samples) is 8 rows of 32 sample PAIRS, so the overlap-add again stays in
// registers (32 rows of even samples + 32 rows of odd samples).
#pragma once
#include "gate_kernels.cuh"

namespace b200 {

constexpr int kN2 = 2048;
constexpr int kF2 = kN2 / 2 + 1;        // 1025
constexpr int kFW2 = (kF2 + 31) / 32;   // 33
constexpr int kFPad2 = kFW2 * 32;       // 1056

struct Tables2 {
    const float2* wa2;      // [1024] analysis window pairs (w[2m], w[2m+1]) / sum(w)
    const float2* ws2;      // [1024] synthesis window pairs * sum(w) / 1024
    const float2* tw;       // [32*32] radix-32 inter-pass twiddles
    const float2* w2k;      // [1025] exp(-i pi k / 1024) as (cos, -sin)
    const float2* invn2;    // [256]  1 / overlap-add norm, pairs, interior hops
    float ws_to_w;
};

// |X| for the non-stationary follower: one MUFU.SQRT (relative error <= 2^-22) instead of the correctly rounded sqrtf
// (reciprocal square root + Newton step + slow path, ~10 instructions, 34 of them per frame).  The magnitudes only feed the
// follower's ratio and sigmoid -- a soft mask with tolerance 1e-5 -- never a binary decision.
__device__ __forceinline__ float sqrt_approx(float x) {
#if defined(B200_CUSIM_BUILD) || defined(B200_EXACT_SQRT_2K)
    return sqrtf(x);
#else
    float r;
    asm("sqrt.approx.f32 %0, %1;" : "=f"(r) : "f"(x));
    return r;
#endif
}

// frame samples -> packed complex input of the 1024-point FFT, windowed
__device__ __forceinline__ void load_frame_2k(float (&re)[32], float (&im)[32], const float* __restrict__ xrow,
                                              long long base, long long i1, long long Lp, long long n_total,
                                              const float2* __restrict__ s_wa2, int lane) {
    const long long g0 = i1 + base;
    const float* p0 = xrow + g0;
    if (base >= 0 && base + kN2 <= Lp && g0 >= 0 && g0 + kN2 <= n_total && ((reinterpret_cast<uintptr_t>(p0) & 7) == 0)) {
        const float2* p = reinterpret_cast<const float2*>(p0) + lane;
#pragma unroll
        for (int r = 0; r < 32; ++r) {
            const float2 v = __ldg(p + 32 * r);
            const float2 w = s_wa2[lane + 32 * r];
            re[r] = v.x * w.x;
            im[r] = v.y * w.y;
        }
    } else {
#pragma unroll
        for (int r = 0; r < 32; ++r) {
            const long long j = base + 2 * (lane + 32 * r);
            const float2 w = s_wa2[lane + 32 * r];
            re[r] = chunk_sample(xrow, j, i1, Lp, n_total) * w.x;
            im[r] = chunk_sample(xrow, j + 1, i1, Lp, n_total) * w.y;
        }
    }
}

struct K1n2Args {
    Geom g;
    Tables2 tb;
    const float* x;
    float* mag;                // [n_units][T][FPad2]
    DebugTap dbg;              // spec: [T][F2][2]
    int run, n_runs;
    float2* zcache;            // [n_units][T][1024] packed half-length spectra Z of frames [z_lo, z_hi), or null
    int z_lo, z_hi;
};

__host__ __device__ constexpr int k2k_table_floats() { return 2 * 1024 + 2 * 1024 + 2 * kFPad2; }   // wa2, tw, w2k
constexpr int k1n2_smem_floats() { return k2k_table_floats() + kWarps * kExchFloats; }

__global__ void __launch_bounds__(kThreads, 3) k1n_magnitude_2k(const K1n2Args a) {
    B200_DYN_SMEM(float, smem);
    float2* s_wa2 = reinterpret_cast<float2*>(smem);
    float2* s_tw = reinterpret_cast<float2*>(smem + 2048);
    float2* s_w2k = reinterpret_cast<float2*>(smem + 4096);
    float* s_tiles = smem + k2k_table_floats();
    for (int i = threadIdx.x; i < 1024; i += kThreads) {
        s_wa2[i] = a.tb.wa2[i];
        s_tw[i] = a.tb.tw[i];
    }
    for (int i = threadIdx.x; i < kFPad2; i += kThreads) s_w2k[i] = (i < kF2) ? a.tb.w2k[i] : make_float2(0.f, 0.f);
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
        const float* xrow = a.x + (long long)c * g.in_stride;
        const int t0 = run * a.run;
        const int t1 = min(t0 + a.run, g.T);
        for (int t = t0; t < t1; ++t) {
            const long long base = (long long)t * H - kN2 / 2;
            float re[32], im[32];
            load_frame_2k(re, im, xrow, base, i1, g.Lp, g.n_total, s_wa2, lane);
            warp_fft1024(re, im, tile, s_tw, lane);
            if (a.zcache && t >= a.z_lo && t < a.z_hi) {        // k2c_synthesize_2k loads Z instead of transforming the frame again
                float2* zp = a.zcache + ((long long)ul * g.T + t) * 1024 + lane;
#pragma unroll
                for (int q = 0; q < 32; ++q) zp[32 * q] = make_float2(re[brev5(q)], im[brev5(q)]);
            }
            float* dst = a.mag + ((long long)ul * g.T + t) * kFPad2;
#pragma unroll
            for (int q = 0; q < 17; ++q) {
                const int sA = brev5(q), sP = brev5(31 - q), s0 = brev5((32 - q) & 31);
                const float zr = re[sA], zi = im[sA];
                float pr = __shfl_sync(0xffffffffu, re[sP], pl);
                float pi = __shfl_sync(0xffffffffu, im[sP], pl);
                if (lane == 0) { pr = re[s0]; pi = im[s0]; }
                const int k = lane + 32 * q;
                const bool valid = (q < 16) || (lane == 0);
                const float Er = 0.5f * (zr + pr), Ei = 0.5f * (zi - pi);
                const float Or = 0.5f * (zi + pi), Oi = 0.5f * (pr - zr);
                const float2 W = s_w2k[k];
                const float Tr = fmaf(-Oi, W.y, Or * W.x), Ti = fmaf(Or, W.y, Oi * W.x);
                const float Xr = Er + Tr, Xi = Ei + Ti;              // X[k]
                const float Yr = Er - Tr, Yi = Ti - Ei;              // X[1024-k] = conj(E - T)
                if (valid) {
                    dst[k] = sqrt_approx(fmaf(Xr, Xr, Xi * Xi));
                    if (k != 512) dst[1024 - k] = sqrt_approx(fmaf(Yr, Yr, Yi * Yi));
                    if (a.dbg.ul == ul) {
                        float* sp = a.dbg.spec + ((long long)t * kF2) * 2;
                        sp[2 * k] = Xr; sp[2 * k + 1] = Xi;
                        sp[2 * (1024 - k)] = Yr; sp[2 * (1024 - k) + 1] = Yi;
                    }
                }
            }
        }
    }
}

}  // namespace b200
