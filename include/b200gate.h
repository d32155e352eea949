/* b200gate.h -- C ABI of libb200gate.so, the B200-native spectral-gating operator.
 *
 * Drop-in boundary (SURVEY.md section 8b).  Each entry point replaces one piece of the reference
 * (timsainb/noisereduce @ 51c8534, paths relative to /root/reference):
 *
 *   b200gate_create            <- SpectralGate.__init__ geometry + smoothing-filter extents
 *                                 (noisereduce/spectralgate/base.py:33-128) and the TorchGate
 *                                 constructor (noisereduce/torchgate/torchgate.py:32-71)
 *   b200gate_noise_stats       <- the one-time noise statistics of SpectralGateStationary.__init__
 *                                 (noisereduce/spectralgate/stationary.py:47-81)
 *   b200gate_run               <- SpectralGate.get_traces() -> filter_chunk -> _do_filter over all
 *                                 chunks and channels (base.py:130-226; stationary.py:83-131;
 *                                 nonstationary.py:47-115), i.e. the body of reduce_noise()
 *                                 (noisereduce/noisereduce.py:185), and TorchGate.forward
 *                                 (torchgate.py:200-264) when params.surface == B200GATE_SURFACE_TORCH
 *
 * Conventions: plain pointers and sizes, no torch / numpy types.  All buffers are caller-owned; the
 * library owns only its handle and device workspace.  Every function returns B200GATE_OK (0) or a
 * negative error code; b200gate_last_error() gives the message.  A handle serialises its work on the
 * CUDA stream passed in (0 = legacy default stream); handles are independent, so one per thread /
 * per rank is the threading model.  There is no CPU fallback: without a CUDA device
 * b200gate_create fails with B200GATE_ERR_CUDA.
 */
#ifndef B200GATE_H
#define B200GATE_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define B200GATE_ABI_VERSION 1

enum {
    B200GATE_OK = 0,
    B200GATE_ERR_ARG = -1,          /* bad argument / unsupported geometry                       */
    B200GATE_ERR_CUDA = -2,         /* CUDA runtime error (message has the CUDA error string)    */
    B200GATE_ERR_STATE = -3,        /* call order (e.g. stationary run before noise statistics)  */
    B200GATE_ERR_NOMEM = -4
};

enum { B200GATE_F32 = 0, B200GATE_I16 = 1, B200GATE_F64 = 2 };     /* sample dtypes */
enum { B200GATE_SURFACE_NUMPY = 0, B200GATE_SURFACE_TORCH = 1 };   /* which reference semantics */

/* Resolved operator parameters.  The Python shims resolve defaults exactly as the reference does
 * (win_length = n_fft, hop_length = win_length // 4, n_grad_* from Hz / ms) and raise the
 * reference's own exceptions; the library re-validates and rejects what this build cannot run. */
typedef struct b200gate_params {
    int32_t abi_version;        /* B200GATE_ABI_VERSION                                          */
    int32_t surface;            /* B200GATE_SURFACE_*                                            */
    int32_t stationary;         /* 1: stationary gate, 0: non-stationary gate                    */
    int32_t n_fft;              /* [8, 8192] if a power of two, else [8, 4096] (Bluestein)         */
    int32_t win_length;         /* 1 <= win_length <= n_fft                                      */
    int32_t hop_length;         /* 1 <= hop_length <= win_length.  n_fft=1024/win=1024/hop=256 (both gates, both
                                 * surfaces) and 2048/2048/512 (numpy surface, non-stationary) run the tuned FP32 kernels; every other
                                 * geometry runs the float64 general family (gate_generic.cuh)    */
    int32_t n_grad_freq;        /* smoothing half-widths; 0,0 = mask smoothing disabled          */
    int32_t n_grad_time;
    int32_t std_ddof;           /* 0 numpy surface (np.std), 1 torch surface (std_mean)          */
    int32_t clip_noise;         /* clip_noise_stationary                                         */
    int32_t n_movemean;         /* torch surface, non-stationary                                 */
    int32_t debug_guard_scale;  /* tests only: multiplies the FP32 guard band (0 = 1x), forcing more
                                 * bins through the FP64 re-decision path                          */
    int32_t reserve_sms;        /* SMs the persistent grids leave free (for a concurrent NCCL collective) */
    int32_t path_flags;         /* force a path that some input needs onto any input (default 0).  bit 2: run the
                                 * float64 general-geometry family even for a tuned geometry; bit 4: one unit per warp in
                                 * the n_fft 1024 FFT kernels instead of the dual (packed f32x2) forms; bit 5: tile-based
                                 * float-mask smoothing; bit 6: the non-stationary follower stores its forward sweep
                                 * instead of regenerating it; bit 7: tap-loop float-mask smoothing instead of the
                                 * box-sum form.  Bits 0, 1 and 3 selected variants that were removed; they are ignored */
    int64_t chunk_size;         /* <= 0: never chunk (torch surface / chunk_size=None)           */
    int64_t padding;
    double sr;
    double prop_decrease;
    double n_std_thresh;        /* n_std_thresh_stationary                                       */
    double top_db;              /* 80 numpy surface, 40 torch surface                            */
    double time_constant_s;     /* numpy surface, non-stationary                                 */
    double thresh_n_mult;       /* thresh_n_mult_nonstationary / n_thresh_nonstationary          */
    double sigmoid_slope;       /* sigmoid_slope_nonstationary / 1 / temp_coeff_nonstationary    */
    double workspace_limit_bytes; /* 0: library default; bounds the per-batch device workspace   */
} b200gate_params;

typedef struct b200gate_handle b200gate_handle;

/* Counters of the last b200gate_run (device-side exactness bookkeeping and launch counts). */
typedef struct b200gate_stats {
    int64_t units;                  /* (chunk, channel) units processed                           */
    int64_t frames;                 /* STFT frames analysed                                       */
    int64_t kernel_launches;        /* kernels launched by the last run                           */
    int64_t bins_rechecked_fp64;    /* mask decisions inside the FP32 guard band, redone in FP64  */
    int64_t bins_unresolved;        /* ... still inside 1e-12 relative after FP64 (expected 0)    */
    int64_t rowfloor_flags;         /* (unit, bin) rows lifted by the top_db floor                */
    int64_t rowfloor_ambiguous;     /* ... whose FP32 decision was inside the guard band (exp. 0) */
    double last_run_ms;             /* device time of the last run, CUDA events on its stream     */
    double last_h2d_ms, last_d2h_ms;
    double k1_ms, smooth_ms, k2_ms; /* per-kernel device time summed over the run's batches       */
    double fused_ms;                /* single-pass kernel (k1/smooth/k2 are 0 when it ran)        */
    int64_t fused_path;             /* 1: the single-pass kernel produced the result              */
    int64_t fused_fallbacks;        /* 1: top_db floor could trigger -> redone on the two-pass path */
} b200gate_stats;

int b200gate_create(const b200gate_params* params, b200gate_handle** out);
void b200gate_destroy(b200gate_handle* h);
const char* b200gate_last_error(const b200gate_handle* h);   /* h == NULL: last create() error */

/* Stationary noise statistics (stationary.py:47-81): channel mean in the input dtype, clip to
 * chunk_size, STFT, dB with top_db floor, per-bin mean/std over time, thresh = mean + n_std*std.
 * y_noise: [C][N] samples, row stride `stride` elements, host or device memory. */
int b200gate_noise_stats(b200gate_handle* h, const void* y_noise, int dtype, int64_t C, int64_t N,
                         int64_t stride, int is_device, void* cuda_stream);
/* Same, from an already collapsed (channel-mean) noise clip of n samples in float64 or float32:
 * used by multi-GPU callers that build the channel mean across ranks themselves. */
int b200gate_noise_stats_collapsed(b200gate_handle* h, const void* noise_mean, int dtype, int64_t n,
                                   int is_device, void* cuda_stream);
/* Channel-order partial sum of the first `n` samples of `C` channels, continuing from *acc_inout
 * (device buffer of n elements: float32 for F32 input, float64 otherwise; ignored if init != 0).
 * Lets ranks chain the reference's sequential float32 channel sum exactly. */
int b200gate_channel_sum(b200gate_handle* h, const void* y, int dtype, int64_t C, int64_t n,
                         int64_t stride, int is_device, void* acc_inout_device, int init,
                         void* cuda_stream);
int b200gate_set_noise_threshold(b200gate_handle* h, const double* thresh_db, int32_t n_bins);
int b200gate_get_noise_threshold(const b200gate_handle* h, double* thresh_db, int32_t n_bins);
int b200gate_get_noise_mean_std(const b200gate_handle* h, double* mean_db, double* std_db, int32_t n_bins);

/* Torch surface only: install the analysis/synthesis window the caller built with
 * torch.hann_window (float32, win_length values), so tables match the reference bit for bit. */
int b200gate_set_window(b200gate_handle* h, const float* window, int32_t win_length);
/* Torch surface only: thresholds from a noise clip xn [Bn][Ln] (float32; Bn == 1 or Bn == batch), as
 * TorchGate.forward(x, xn) (torchgate.py:140-164).  xn == NULL returns to self-statistics. */
int b200gate_torch_set_noise(b200gate_handle* h, const void* xn, int dtype, int64_t Bn, int64_t Ln,
                             int64_t stride, int is_device, void* cuda_stream);

/* Torch surface only: apply the MASKS OF THE LAST b200gate_run (same [C][N]) to another signal: analysis of `in`, the
 * stored masks, synthesis.  The gate is linear in its input once the masks are fixed and its operator is
 * out = OLA(w B_mask(w frame(in))) / env with a symmetric B_mask, so this call on g / env, times env, is the adjoint:
 * the backward pass of TorchGate.forward (torchgate.py:223-262 builds the masks under no_grad and lets the gradient flow
 * through stft -> * mask -> istft).  Needs the tuned n_fft = 1024 geometry and a forward that fitted one workspace batch. */
int b200gate_torch_apply_masks(b200gate_handle* h, const void* in, void* out, int dtype, int64_t C, int64_t N,
                               int64_t in_stride, int64_t out_stride, int is_device, void* cuda_stream);

/* The operator.  in/out: [C][N] samples of `dtype` with row strides in elements; host or device
 * pointers (is_device).  out may not alias in.  For the torch surface out holds [C][(N/hop)*hop].
 * Returns after the work is enqueued for device pointers; for host pointers it returns after the
 * result is in `out`. */
int b200gate_run(b200gate_handle* h, const void* in, void* out, int dtype, int64_t C, int64_t N,
                 int64_t in_stride, int64_t out_stride, int is_device, void* cuda_stream);

/* Sub-range processing for the next b200gate_run calls (SpectralGate.get_traces(start_frame, end_frame),
 * base.py:167-226).  mode 0: the whole recording (default).  mode 1: only chunks [a, b] of the chunk grid
 * anchored at sample 0 (the reference's chunked branch); samples outside those chunks are not written.
 * mode 2: one padded chunk covering [0, a) whose padding is read from the recording itself (the reference's
 * `filter_chunk(0, end_frame)` branch, base.py:222); only out[:, 0:a] is written.
 * In modes 1 and 2 `out` is still the address of (row 0, sample 0), but only the range is addressed: a caller
 * may pass `slab - first_sample` with out_stride = the slab's row pitch (>= the range length) to have the range
 * written densely into a [C][range] slab (noisereduce_b200/parallel.py gathers such slabs across GPUs). */
int b200gate_set_range(b200gate_handle* h, int32_t mode, int64_t a, int64_t b);

int b200gate_get_stats(const b200gate_handle* h, b200gate_stats* out);

/* Page-locked host buffers from the library's process-wide pool (the same pool the slab pipeline stages pageable
 * caller memory through).  A result array the reference would np.empty() (base.py:181-187 uses a temp-file memmap)
 * can be leased here instead: b200gate_run then copies device -> host straight into it at PCIe speed, with no page
 * faults and no staging copy, and a freed buffer is handed to the next call of the same size without paying
 * cudaMallocHost (~0.1 s per GB) again.  b200gate_host_alloc returns NULL when the memory cannot be pinned (callers fall
 * back to ordinary memory); b200gate_host_free(NULL) is a no-op.  Thread-safe. */
void* b200gate_host_alloc(size_t bytes);
void b200gate_host_free(void* p);

/* ---- multi-GPU (one process per GPU; SURVEY.md section 8e) ---------------------------------------------------
 * The path's one collective -- the all-gather of the final waveform -- is done with NVLink stores issued by a kernel
 * into buffers every peer has mapped (cudaIpc / CUDA VMM / torch symmetric memory), not with a library collective:
 * the interface therefore takes plain device pointers (this rank's buffer and its mappings of the peers' buffers)
 * instead of the ncclComm_t the survey sketched; NCCL / torch.distributed stays the caller's business (rendezvous,
 * the chained channel mean of the stationary threshold -- b200gate_channel_sum).
 *
 * b200gate_run_sharded: denoise this rank's [C_local][N] channels (device pointers) group by group into rows
 * [rank*C_local, (rank+1)*C_local) of `gathered_local` ([world*C_local][N], this rank's copy of the result) on
 * `compute_stream`, and push every finished group into the same rows of each peer's copy on `comm_stream` while
 * the next group is computed; a device-side barrier over the flag arrays (world uint32 each, zero-initialised,
 * `epoch` strictly increasing per call) ends the step.  On return everything is enqueued; after `compute_stream`
 * reaches this point `gathered_local` holds every rank's rows.  gathered_peers[r] / flags_peers[r] are this rank's
 * mappings of rank r's buffers (entry [rank] is ignored / the local array).  push_ctas = the number of SMs the copy kernel
 * occupies (each of its CTAs fills one SM; create the handle with reserve_sms >= push_ctas); <= 0 picks 12. */
int b200gate_run_sharded(b200gate_handle* h, const void* in_local, int dtype, int64_t C_local, int64_t N,
                         int64_t in_stride, void* gathered_local, void* const* gathered_peers, void* flags_local,
                         void* const* flags_peers, uint32_t epoch, int32_t rank, int32_t world, int32_t groups,
                         int32_t push_ctas, void* compute_stream, void* comm_stream);
/* The two building blocks, for callers with their own schedule (e.g. the slab ring of config 5): copy `rows` rows of
 * `row_bytes` bytes (16-byte multiples, 16-byte aligned) from local memory into n_peers mapped buffers; and the
 * epoch barrier described above. */
int b200gate_peer_push(const void* src, void* const* peer_dst, int32_t n_peers, int64_t rows, int64_t row_bytes,
                       int64_t src_stride_bytes, int64_t dst_stride_bytes, int32_t n_ctas, void* cuda_stream);
int b200gate_peer_barrier(void* local_flags, void* const* peer_flags, int32_t rank, int32_t world, uint32_t epoch,
                          void* cuda_stream);

/* ---- parity-test taps (tests/ only; read back stage outputs of the last run) ---------------- */
/* Select the (chunk, channel) unit whose stages the next run keeps.  chunk < 0 disables. */
int b200gate_debug_select_unit(b200gate_handle* h, int64_t chunk, int64_t channel);
/* Frames of the tapped unit; bits: [T][words] packed mask decisions (bit f%32 of word f/32),
 * with the top_db row floor already folded in.  mask: [T][F] smoothed multiplicative mask.
 * spec: [T][F][2] float, the FP32 STFT (re, im) as the analysis kernel saw it. */
int b200gate_debug_dims(const b200gate_handle* h, int64_t* T, int32_t* F, int32_t* words);
int b200gate_debug_read_bits(b200gate_handle* h, uint32_t* bits);
int b200gate_debug_read_mask(b200gate_handle* h, float* mask);
int b200gate_debug_read_spec(b200gate_handle* h, float* spec);

#ifdef __cplusplus
}
#endif
#endif /* B200GATE_H */
