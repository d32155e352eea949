// gate_synth_2k.cuh -- k2c_synthesize_2k: synthesis of the n_fft = 2048 family (BASELINE.json config 3) from the
// spectra k1n_magnitude_2k kept, so that no frame is transformed a second time.
//
// Reference semantics (paths relative to /root/reference): mask apply at noisereduce/spectralgate/nonstationary.py:87,
// scipy.signal.istft as called at nonstationary.py:90-96, chunk centre written back at base.py:150.
//
// One warp owns a run of output hops of one (chunk, channel) unit.  Per frame:
//   1. the frame's half-length spectrum Z = FFT_1024(x[2m] + i x[2m+1]) (8 KB) and its mask row (1025 floats) arrive
//      in this warp's shared-memory buffers by 1-D bulk asynchronous copies (cp.async.bulk -> TMA engine) signalled
//      on a per-warp mbarrier; the copies of frame t+1 are issued as soon as frame t has been read;
//   2. the masks are applied in the half-length domain (gate_kernels_2k.cuh, header): bins k and 1024-k are
//      rebuilt from Z[k] and Z[1024-k] -- the mirrored element is read from the same shared buffer by its FLAT index,
//      so lane 0 is an ordinary lane -- masked, and folded back into Z'[k], Z'[1024-k].  A lane computes both members of
//      its 16 lower pairs; the upper members travel to their owners through the (idle) FFT exchange tile;
//   3. ONE inverse 1024-point FFT (ifft(z) = swap(fft(swap z)): the apply step writes real / imaginary parts exchanged),
//      synthesis window, overlap-add in registers (even / odd samples), normalise, store the chunk centre.
#pragma once
#include "gate_synth.cuh"
#include "gate_kernels_2k.cuh"

namespace b200 {

struct K2c2Args {
    Geom g;
    Tables2 tb;
    float* y;
    const float* fmask;        // [n_units][T][FPad2] final multiplicative masks
    const float2* zcache;      // [n_units][T][1024]
    int run, n_runs;           // output hops per work item
    DebugTap dbg;              // mask: [T][F2]
};

#ifndef B200_K2C2_WARPS
#define B200_K2C2_WARPS 8
#endif
constexpr int kK2c2Warps = B200_K2C2_WARPS;                                          // one CTA per SM
constexpr int kK2c2TableBytes = 1024 * 8 + kFPad2 * 8 + 1024 * 8 + 256 * 8;         // tw, w2k, ws2, invn2
constexpr int kK2c2WarpBytes = 1024 * 8 + kFPad2 * 4 + kK2cTileBytes + 16;          // spectrum, mask row, tile, mbarrier
constexpr int k2c2_smem_bytes() { return kK2c2TableBytes + kK2c2Warps * kK2c2WarpBytes; }
static_assert(kK2cTileBytes >= 513 * 8, "mirror buffer must fit the exchange tile");

// masked half-length spectrum members of bins (k, 1024-k) from Z[k] = (zr, zi), Z[1024-k] = (pr, pi)
__device__ __forceinline__ void apply_pair_2k(float zr, float zi, float pr, float pi, float m, float mp, float2 W,
                                              float& own_r, float& own_i, float& oth_r, float& oth_i) {
    const float Er = 0.5f * (zr + pr), Ei = 0.5f * (zi - pi);
    const float Or = 0.5f * (zi + pi), Oi = 0.5f * (pr - zr);
    const float Tr = fmaf(-Oi, W.y, Or * W.x), Ti = fmaf(Or, W.y, Oi * W.x);
    // P = X[k] = E + T,  Q = conj X[1024-k] = E - T;  masks applied to X[k], X[1024-k]
    const float Pr = m * (Er + Tr), Pi = m * (Ei + Ti);
    const float Qr = mp * (Er - Tr), Qi = mp * (Ei - Ti);
    const float Epr = 0.5f * (Pr + Qr), Epi = 0.5f * (Pi + Qi);
    const float Tpr = 0.5f * (Pr - Qr), Tpi = 0.5f * (Pi - Qi);
    // V = conj(W) T'   (W = (W.x, W.y) with W.y = -sin)
    const float Vr = fmaf(Tpi, W.y, Tpr * W.x), Vi = fmaf(-Tpr, W.y, Tpi * W.x);
    own_r = Epr - Vi; own_i = Epi + Vr;          // Z'[k]      = E' + i V
    oth_r = Epr + Vi; oth_i = Vr - Epi;          // Z'[1024-k] = conj(E') + i conj(V)
}

__global__ void __launch_bounds__(kK2c2Warps * 32, 1) k2c_synthesize_2k(const K2c2Args a) {
    constexpr int HR = 8, NH = 4;
    constexpr int MB = kFPad2 * 4;
    B200_DYN_SMEM(unsigned char, smraw);
    float2* s_tw = reinterpret_cast<float2*>(smraw);
    float2* s_w2k = reinterpret_cast<float2*>(smraw + 1024 * 8);
    float2* s_ws2 = reinterpret_cast<float2*>(smraw + 1024 * 8 + kFPad2 * 8);
    float2* s_invn2 = s_ws2 + 1024;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    unsigned char* wbase = smraw + kK2c2TableBytes + warp * kK2c2WarpBytes;
    const float2* zbuf = reinterpret_cast<const float2*>(wbase);
    const float* mrow = reinterpret_cast<const float*>(wbase + 1024 * 8);
    float* tile = reinterpret_cast<float*>(wbase + 1024 * 8 + MB);
    float2* qbuf = reinterpret_cast<float2*>(tile);
    unsigned long long* bar = reinterpret_cast<unsigned long long*>(wbase + 1024 * 8 + MB + kK2cTileBytes);
    const int nthr = kK2c2Warps * 32;
    for (int i = threadIdx.x; i < 1024; i += nthr) {
        s_tw[i] = a.tb.tw[i];
        s_ws2[i] = a.tb.ws2[i];
    }
    for (int i = threadIdx.x; i < kFPad2; i += nthr) s_w2k[i] = (i < kF2) ? a.tb.w2k[i] : make_float2(0.f, 0.f);
    for (int i = threadIdx.x; i < 256; i += nthr) s_invn2[i] = a.tb.invn2[i];
    if (lane == 0) mbar_init(bar, 1);
    mbar_init_fence();
    __syncthreads();
    unsigned phase = 0;

    const Geom& g = a.g;
    const int H = g.H;                                   // 512
    const long long n_items = (long long)g.n_units * a.n_runs;
    for (long long item = (long long)blockIdx.x * kK2c2Warps + warp; item < n_items;
         item += (long long)gridDim.x * kK2c2Warps) {
        const int ul = (int)(item / a.n_runs);
        const int run = (int)(item - (long long)ul * a.n_runs);
        const int u = g.u0 + ul;
        const int ic = u / g.C, c = u - ic * g.C;
        const long long i1 = (long long)ic * g.step - g.pad;
        long long out_len = g.n_total - (long long)ic * g.step;
        if (out_len > g.step) out_len = g.step;
        long long jp_hi = g.pad + out_len;
        const long long sig_len = (long long)(g.T - 1) * H;
        if (jp_hi > sig_len) jp_hi = sig_len;
        if (jp_hi <= g.pad) continue;
        const long long jlo = g.pad + kN2 / 2, jhi = jp_hi + kN2 / 2;
        const int h_lo = (int)(jlo / H), h_hi = (int)((jhi + H - 1) / H);
        const int hs = h_lo + run * a.run;
        const int he = min(hs + a.run, h_hi);
        if (hs >= he) continue;
        const int t_start = max(0, hs - (NH - 1));
        const int t_last = min(he - 1, g.T - 1);
        float* yrow = a.y + (long long)c * g.out_stride;
        const float2* zunit = a.zcache + (long long)ul * g.T * 1024;
        const float* funit = a.fmask + (long long)ul * g.T * kFPad2;

        float acc_e[32], acc_o[32];                      // even / odd samples of the overlap-add window
#pragma unroll
        for (int r = 0; r < 32; ++r) { acc_e[r] = 0.f; acc_o[r] = 0.f; }

        // request frame tt: spectrum + mask row.  All lanes have finished reading the buffers.
        auto stage = [&](int tt) {
            fence_proxy_async_smem();
            __syncwarp();
            if (lane == 0) {
                mbar_expect_tx(bar, (unsigned)(1024 * 8 + MB));
                bulk_g2s(wbase, zunit + (long long)tt * 1024, 1024 * 8, bar);
                bulk_g2s(wbase + 1024 * 8, funit + (long long)tt * kFPad2, MB, bar);
            }
        };
        if (t_start <= t_last) stage(t_start);

        for (int t = t_start; t < he; ++t) {
            if (t <= t_last) {
                float re[32], im[32];                   // what the FFT call sees: re = Im Z', im = Re Z'
                mbar_wait(bar, phase);
                phase ^= 1u;
                if (a.dbg.ul == ul) {                   // parity tap (tests): the masks this frame applies
#pragma unroll 1
                    for (int k = lane; k < kF2; k += 32) a.dbg.mask[(long long)t * kF2 + k] = mrow[k];
                }
                // ---- lower pairs k = lane + 32 q < 512: both members -------------------------------------------
#pragma unroll
                for (int q = 0; q < 16; ++q) {
                    const int k = 32 * q + lane;
                    const float2 own = zbuf[k];
                    const float2 par = zbuf[q == 0 ? ((1024 - lane) & 1023) : (1024 - k)];
                    float own_r, own_i, oth_r, oth_i;
                    apply_pair_2k(own.x, own.y, par.x, par.y, mrow[k], mrow[1024 - k], s_w2k[k], own_r, own_i, oth_r, oth_i);
                    im[q] = own_r;
                    re[q] = own_i;
                    qbuf[512 - k] = make_float2(oth_i, oth_r);          // slot of index 1024 - k, stored (re, im) as the FFT wants them
                }
                {   // slot 16: indices 512 + lane = 1024 - kk with kk = 512 - lane, computed directly (lane 0: the self-mirrored 512)
                    const int kk = 512 - lane;
                    const float2 own = zbuf[kk];
                    const float2 par = zbuf[512 + lane];
                    float own_r, own_i, oth_r, oth_i;
                    apply_pair_2k(own.x, own.y, par.x, par.y, mrow[kk], mrow[512 + lane], s_w2k[kk], own_r, own_i, oth_r, oth_i);
                    im[16] = lane == 0 ? own_r : oth_r;
                    re[16] = lane == 0 ? own_i : oth_i;
                }
                __syncwarp();
#pragma unroll
                for (int q = 17; q < 32; ++q) {
                    const float2 v = qbuf[32 * (q - 16) + lane];
                    re[q] = v.x;
                    im[q] = v.y;
                }
                __syncwarp();
                if (t + 1 <= t_last) stage(t + 1);      // the next frame streams in behind this frame's transform
                warp_fft1024(re, im, tile, s_tw, lane);
                // now im = 1024 * y[2m], re = 1024 * y[2m+1]  (m = lane + 32 q) at slot brev5(q)
#pragma unroll
                for (int q = 0; q < 32; ++q) {
                    const float2 w = s_ws2[lane + 32 * q];
                    acc_e[q] = fmaf(im[brev5(q)], w.x, acc_e[q]);
                    acc_o[q] = fmaf(re[brev5(q)], w.y, acc_o[q]);
                }
            }
            // hop t is complete: rows 0..7 (pairs) = samples [t*512, (t+1)*512)
            if (t >= hs) {
                const long long jp0 = (long long)t * H - kN2 / 2;          // chunk-local index of row 0, pair 0
                float* d0 = yrow + i1 + jp0 + 2 * lane;
                if (t >= NH - 1 && t <= g.T - 1 && jp0 >= g.pad && jp0 + H <= jp_hi &&
                    ((reinterpret_cast<uintptr_t>(d0) & 7) == 0)) {
#pragma unroll
                    for (int r = 0; r < HR; ++r) {
                        const float2 inv = s_invn2[r * 32 + lane];
                        *reinterpret_cast<float2*>(d0 + 64 * r) = make_float2(acc_e[r] * inv.x, acc_o[r] * inv.y);
                    }
                } else {
#pragma unroll 1
                    for (int r = 0; r < HR; ++r) {
                        float ve = 0.f, vo = 0.f;
#pragma unroll
                        for (int rr = 0; rr < HR; ++rr)
                            if (rr == r) { ve = acc_e[rr]; vo = acc_o[rr]; }
                        for (int par = 0; par < 2; ++par) {
                            const int ro = r * 64 + 2 * lane + par;         // sample offset within the hop
                            const long long jp = jp0 + ro;
                            if (jp < g.pad || jp >= jp_hi) continue;
                            float nrm = 0.f;
                            for (int i = 0; i < NH; ++i) {
                                const int tf = t - i;
                                if (tf >= 0 && tf <= g.T - 1) {
                                    const int n = i * H + ro;               // window index of this sample in frame tf
                                    const float2 wp = s_ws2[n >> 1];
                                    const float w = ((n & 1) ? wp.y : wp.x) * a.tb.ws_to_w;
                                    nrm = fmaf(w, w, nrm);
                                }
                            }
                            const float inv = nrm > 1e-10f ? 1.0f / nrm : 1.0f;
                            yrow[i1 + jp] = (par ? vo : ve) * inv;
                        }
                    }
                }
            }
#pragma unroll
            for (int r = 0; r < 32 - HR; ++r) { acc_e[r] = acc_e[r + HR]; acc_o[r] = acc_o[r + HR]; }
#pragma unroll
            for (int r = 32 - HR; r < 32; ++r) { acc_e[r] = 0.f; acc_o[r] = 0.f; }
        }
    }
}

}  // namespace b200
