/* sot_b200.h -- C ABI of the B200-native Spectral Optimal Transport (SOT) loss.
 *
 * This is the drop-in boundary for ONE hot path of bernardo-torres/1d-spectral-optimal-transport:
 * `losses.Wasserstein1D.forward` -> `losses.wasserstein_1d` -> `losses.quantile_function`
 * (reference losses.py:129-313, utils.py:135-142) and its autograd backward.  The reference has no
 * native code; what a maintainer binds (ctypes, shown in INTEGRATION.md) are the entry points
 * below -- plain pointers and sizes, no torch types.  All `const float*` / `float*` arguments of
 * the *_device entry points are CUDA device pointers on the current device; `stream` is a
 * `cudaStream_t` passed as `void*` (NULL = default stream).  Calls are asynchronous on `stream`
 * unless stated otherwise.  Every function returns 0 on success, a negative SOT_E* code on a
 * rejected argument (nothing was launched) or a positive `cudaError_t`; `sot_last_error()`
 * gives the text.  There is no CPU fallback anywhere in this library.
 *
 * Layout: spectra are row-major contiguous [n_frames, bins] float32 -- exactly the memory of the
 * reference's (batch, time, freq) tensors after `reshape(-1, F)` (losses.py:158-165).  Argument
 * order follows the reference: `u` is the TARGET spectrum (first argument `x`, normalised to
 * unit mass), `v` the PREDICTION (`y`; in cutoff mode divided by the target's mass).
 */
#ifndef SOT_B200_H
#define SOT_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SOT_B200_ABI_VERSION 2

/* flags (bit-or) */
#define SOT_SQUARE 1    /* square_dist=True: weights = magnitude^2        losses.py:172-174 */
#define SOT_CUT_SCALE 2 /* dont_normalize=True: v / mass(u), not / mass(v) losses.py:180-182 */
#define SOT_LIMIT 4     /* limit_quantile_range=True: strict `qs > 1` mask losses.py:306-307 */
#define SOT_RAW_WEIGHTS 8 /* rows are weights used as given, no normalisation: the module-level
                            `wasserstein_1d(u_values, v_values, u_weights, v_weights)` losses.py:223 */

#define SOT_UNIFORM_GRID 16 /* the caller asserts: one support shared by all frames (strides 0) with
                             pos_u[i] = pos_u[0] + i*h and pos_v[j] = pos_v[0] + j*h EXACTLY in float32,
                             h = pos_u[1] - pos_u[0] (e.g. rfftfreq / max for power-of-two n_fft,
                             trainer.py:193-197).  Positions are then computed, not loaded: same bits,
                             fewer shared-memory accesses.  Ignored by sot_quantiles_device. */

#define SOT_COMPLEX_INPUT 32 /* fused STFT-magnitude prologue (features.py:104-110, 217-237): u, v are rows of
                              interleaved complex64 STFT bins [N, n_u] / [N, n_v] (2 floats per bin, e.g.
                              `torch.stft(..., return_complex=True)` transposed to frame-major), the
                              magnitude is formed in the kernel, and grad_u / grad_v are complex rows
                              (dL/dre, dL/dim) of the same layout.  Forward / forward+backward entries only. */

/* error codes */
#define SOT_OK 0
#define SOT_EINVAL (-1)   /* bad pointer / size / flag combination        */
#define SOT_ETOOBIG (-2)  /* row longer than the entry point accepts       */
#define SOT_EDOMAIN (-3)  /* p < 1 (reference: AssertionError, losses.py:271) */

/* One batch of frames.  Mirrors the arguments of `wasserstein_1d` (losses.py:223-232) plus the
 * prologue switches of `Wasserstein1D.forward` (losses.py:172-184). */
typedef struct sot_problem {
    int64_t n_frames;      /* N = batch * time                                              */
    int32_t n_u;           /* bins of u (n)                                                 */
    int32_t n_v;           /* bins of v (m); may differ from n_u                            */
    const float* u;        /* [N, n_u] target magnitudes                                    */
    const float* v;        /* [N, n_v] prediction magnitudes                                */
    const float* pos_u;    /* support positions of u, ASCENDING along the row: [n_u] when    */
    const float* pos_v;    /*   pos_*_stride == 0 (one grid shared by all frames), else rows */
    int64_t pos_u_stride;  /*   of a [N, n_*] array with this element stride                */
    int64_t pos_v_stride;
    float p;               /* order of the distance, >= 1 (result is W_p^p, no root)        */
    int32_t flags;         /* SOT_SQUARE | SOT_CUT_SCALE | SOT_LIMIT | SOT_RAW_WEIGHTS | SOT_UNIFORM_GRID | SOT_COMPLEX_INPUT */
} sot_problem;

/* ---- the hot path ------------------------------------------------------------------------- */

/* Forward: loss[N] = per-frame W_p^p.  Replaces losses.py:172-184 + 286-313 (one launch). */
int sot_forward_device(const sot_problem* prob, float* loss, void* stream);

/* Fused forward + backward: loss[N] (nullable) and
 *   grad_u[N, n_u] = upstream[n] * d loss_n / d u   (nullable),
 *   grad_v[N, n_v] = upstream[n] * d loss_n / d v   (nullable),
 * `upstream` = dL/dloss_n per frame, NULL meaning 1.  Replaces the autograd backward of
 * losses.py:172-313 (SURVEY.md section 3.3); tie attribution = stable sort order. */
int sot_forward_backward_device(const sot_problem* prob, const float* upstream, float* loss,
                                float* grad_u, float* grad_v, void* stream);

/* The reference ends with `torch.mean` over all frames (losses.py:211).  These two fold that mean
 * into the launches: the forward also accumulates *loss_sum += sum_n loss[n] (fp64, one atomic per
 * CTA; the caller zeroes it; `loss` may be NULL), and the backward takes the upstream gradient as
 * upstream[n] * (*upstream_scale) with both factors optional -- for a mean, upstream = NULL and
 * *upstream_scale = dL/dmean / N, a DEVICE scalar, so no host synchronisation is needed. */
int sot_forward_sum_device(const sot_problem* prob, float* loss, double* loss_sum, uint16_t* coranks_out,
                           int32_t coranks_per_frame, void* stream);
int sot_forward_backward_scaled_device(const sot_problem* prob, const float* upstream,
                                       const float* upstream_scale, const uint16_t* coranks_in,
                                       int32_t coranks_per_frame, float* loss, float* grad_u, float* grad_v,
                                       void* stream);
/* "Saved merge indices": the forward launch can write the merge-path co-rank of every chunk of every
 * frame into coranks_out[n_frames, sot_coranks_per_frame(n_u, n_v)] (nullable) and the backward launch
 * reuse them (coranks_in, nullable) instead of repeating the search -- the CDFs of the two launches are
 * bit-identical.  Co-ranks from another kernel configuration (other count) are ignored. */
int sot_coranks_per_frame(int32_t n_u, int32_t n_v);

/* ---- the training step in ONE launch ---------------------------------------------------------------
 * What `loss = Wasserstein1D(...)(x, y, x_pos, y_pos); loss.backward()` needs (trainer.py:209-221, 233-238) is the
 * mean over the frames (losses.py:211) and its gradient.  `sot_mean_step_device` makes one launch of the fused
 * forward+backward kernel: gradients come out already scaled by `grad_scale` (1/N for the mean of N frames; 1/N_global
 * when the frames are sharded over ranks), and the LAST CTA of the launch finishes the mean:
 *     *mean_out     = (float)(sum_n loss_n * mean_scale)                  (nullable)
 *     total_out[0]  = sum_n loss_n,  total_out[1] = count_value            (nullable; the two doubles a sharded
 *                                                                           caller all-reduces with NCCL)
 *     peer mailboxes: (sum, count_value, post_seq) stored into slot [post_rank] of every rank's mailbox over
 *                     NVLink (post_world > 0; layout and protocol of sot_p2p_*; `sot_p2p_wait_mean_device`
 *                     collects them) -- the compute kernel itself starts the one exchange of the sharded loss.
 * `workspace` = 2 doubles of device memory, zero before the first use; the kernel leaves them zero, so no memset,
 * division or cast kernels surround the launch.  One workspace per stream that launches concurrently.
 * grad_u / grad_v nullable (both NULL: the loss-only kernel runs); `loss` (per-frame values) nullable.
 * The backward of the step is then `sot_scale_inplace_device`: rows *= *scale in place, leaving at once when
 * *scale == 1 (the upstream gradient of a loss that is summed with weight 1). */
typedef struct sot_mean_plan {
    double* workspace;
    float* mean_out;
    double mean_scale;
    double* total_out;
    double count_value;
    void* const* post_mailboxes; /* [post_world] device pointers, rank order */
    int32_t post_world;          /* 0 = no peer exchange */
    int32_t post_rank;
    uint64_t post_seq;
    uint64_t* post_seq_device;   /* nullable; overrides post_seq: the call number is *post_seq_device + 1, stored back
                                    by the kernel -- a CUDA graph that contains the launch can then be replayed */
    float grad_scale;
    const float* grad_scale_device; /* nullable device scalar that also multiplies the gradients (an upstream
                                       gradient that is only known on the device) */
} sot_mean_plan;
int sot_mean_step_device(const sot_problem* prob, const sot_mean_plan* plan, float* loss, float* grad_u,
                         float* grad_v, void* stream);
int sot_scale_inplace_device(float* rows_a, int64_t count_a, float* rows_b, int64_t count_b, const float* scale,
                             void* stream);

/* out[r, :] = unit[r, :] * scale[r]  -- backward of the per-frame "fused" autograd mode, where the forward
 * launch already produced the unit gradients.  `out` may be `unit`. */
int sot_scale_rows_device(const float* unit, const float* scale, float* out, int64_t rows,
                          int32_t width, void* stream);

/* `return_quantiles=True` (losses.py:198-201, 299-300).  All outputs nullable:
 *   uq, vq, qs : [N, n_u + n_v]   quantile positions and merged quantile grid
 *   cu, cv     : [N, n_u], [N, n_v]  CDFs
 *   iu, iv     : [N, n_u + n_v] int32  un-clamped `searchsorted(c*, qs)` indices (losses.py:219) */
int sot_quantiles_device(const sot_problem* prob, float* uq, float* vq, float* qs, float* cu,
                         float* cv, int32_t* iu, int32_t* iv, void* stream);

/* `quantile_function(qs, cws, xs)` (losses.py:214-220) as a stand-alone op:
 * out[r, k] = xs[r, min(lower_bound(cws[r, :], qs[r, k]), n_bins - 1)]. */
int sot_quantile_lookup_device(const float* qs, const float* cws, const float* xs, float* out,
                               int64_t rows, int32_t n_levels, int32_t n_bins, void* stream);

/* ---- parity harness (same kernels, prologue skipped) ------------------------------------------ */

/* Treat prob->u / prob->v as already-computed CDF rows (e.g. the reference's own `cumsum`
 * outputs): merged grid + searchsorted indices.  Bit-exact gate P1 of SURVEY.md App. B. */
int sot_plan_from_cdf_device(const sot_problem* prob, float* uq, float* vq, float* qs, int32_t* iu,
                             int32_t* iv, void* stream);
/* Same inputs: per-frame loss and dL/dcu, dL/dcv (before the cumsum transpose).  Gate P2. */
int sot_loss_from_cdf_device(const sot_problem* prob, float* loss, float* g_cu, float* g_cv,
                             void* stream);

/* ---- host-buffer entry point (what a non-torch caller binds) ---------------------------------- */

/* Whole job with HOST buffers: copies u, v (and positions) to the device in chunks on two
 * streams, runs the fused kernel, copies loss and gradients back.  Blocking.  `upstream` and
 * each output are nullable host pointers.  Pinned host memory is used as-is; pageable memory
 * works but is slower.  `device` = CUDA ordinal.  Device staging buffers are cached per device
 * (see sot_host_release); concurrent calls are serialised.
 * SOT_HOST_ZEROCOPY=1 in the environment: when every buffer is pinned and mapped (cudaHostAlloc /
 * cudaHostRegister) and the supports are shared rows, ONE launch reads the spectra from and writes loss and
 * gradients to host memory itself -- no staging buffers on the device; measured at the same PCIe-bound rate
 * as the copy pipeline (4.54 vs 4.64 M frames/s), hence opt-in.  Anything else falls back to the pipeline. */
int sot_loss_grad_host(const sot_problem* host_prob, const float* upstream, float* loss, float* grad_u,
                       float* grad_v, int32_t device);

/* Frees the device buffers, streams and events `sot_loss_grad_host` keeps per device between calls. */
int sot_host_release(int32_t device);

/* ---- housekeeping ---------------------------------------------------------------------------- */
int sot_abi_version(void);
const char* sot_last_error(void);
/* Largest row length (max(n_u, n_v)) the loss / gradient entry points accept: 2^24 - 1.  Real rows longer than one
 * CTA's shared memory holds (more than 8448 bins) run on the split-frame path (global-memory scratch, allocated
 * stream-ordered on the call's stream: no host synchronisation, capturable in a CUDA graph), which needs u, v and the
 * positions in memory the device can reach (else SOT_ETOOBIG); co-ranks are not kept for them (sot_coranks_per_frame
 * returns 0).  Shared memory bounds the rest: sot_quantiles_device and the CDF
 * harness take up to 8448 bins, SOT_COMPLEX_INPUT rows up to 4352; longer rows there return SOT_ETOOBIG. */
int sot_max_bins(int32_t with_grad, int32_t shared_positions);
/* ---- Multi-scale spectral loss term (row f3; losses.py:365-425 `MSSLoss`, :7-36 `mean_difference`,
 * utils.py:145-151 `safe_log`) for ONE fft size, straight from the two complex64 spectrograms zt (target) and zv
 * (prediction) of `count` elements each, any layout:
 *     S = sum_i mag_weight * d(|zt_i|, |zv_i|) + logmag_weight * d(safe_log|zt_i|, safe_log|zv_i|),
 *     d(a, b) = |a - b| (SOT_MSS_L1) or (a - b)^2 (SOT_MSS_L2).
 * forward:  *sum_out += post_scale * S   (fp64, device memory; the caller zeroes it; post_scale = 1/count gives the
 *           reference's mean, and one accumulator can collect all fft sizes).
 * backward: grad_z* = (*scale) * post_scale * dS/dz* as complex64 (dL/dre, dL/dim); `scale` is a device scalar
 *           (NULL = 1); either gradient may be NULL. */
#define SOT_MSS_L1 0
#define SOT_MSS_L2 1
int sot_mss_forward_device(const float* zt, const float* zv, int64_t count, float mag_weight, float logmag_weight,
                           int32_t loss_type, float post_scale, double* sum_out, void* stream);
int sot_mss_backward_device(const float* zt, const float* zv, int64_t count, float mag_weight, float logmag_weight,
                            int32_t loss_type, float post_scale, const float* scale, float* grad_zt, float* grad_zv,
                            void* stream);

/* ---- The one exchange of the frame-sharded loss (SURVEY.md 8e): all-reduce (sum) of `count` <= 8 doubles over
 * NVLink / NVSwitch peer memory, one tiny kernel per call.  `mailboxes[r]` = rank r's mailbox as mapped into this
 * process (a symmetric allocation of sot_p2p_mailbox_doubles(world) doubles per rank, zero-initialised before the
 * first call; e.g. torch.distributed._symmetric_memory), `seq` = 1, 2, 3, ... the same on every rank.  Every rank
 * receives bit-identical sums.  A peer that has not arrived after SOT_P2P_TIMEOUT_MS (environment, default 600 000 ms -- NCCL's watchdog scale)
 * makes the kernel trap: the next CUDA call on the stream fails loudly (never a silent NaN). */
int sot_p2p_mailbox_doubles(int32_t world);
/* The form the sharded loss uses: exchanges (*local_sum, local_count) and writes the global mean sum / count and
 * 1 / count as floats (device memory) -- the forward value and the backward's scale, no scalar-sized kernels around
 * the exchange. */
int sot_p2p_global_mean_device(const double* local_sum, double local_count, float* mean_out, float* inv_count_out,
                               void* const* mailboxes, int32_t world, int32_t rank, uint64_t seq, void* stream);
int sot_p2p_allreduce_device(const double* in, double* out, int32_t count, void* const* mailboxes, int32_t world,
                             int32_t rank, uint64_t seq, void* stream);
/* Second half of an exchange whose first half (the stores into the peers' mailboxes) was done by the last CTA of
 * `sot_mean_step_device`: waits for call `seq` of every rank in this rank's mailbox, then
 *     *mean_out = (float)(sum of the sums / sum of the counts);
 * if the counts do not add up to `expected_count` (> 0) the mean is NaN and *status (nullable; e.g. mapped pinned
 * host memory) is set to 1; a peer that has not arrived after `timeout_ms` sets *status = 2 and traps. */
int sot_p2p_wait_mean_device(float* mean_out, double expected_count, int32_t* status, void* const* mailboxes,
                             int32_t world, int32_t rank, uint64_t seq, uint64_t* seq_device, uint32_t timeout_ms,
                             void* stream);
/* (`seq_device` nullable; overrides `seq` like `post_seq_device` above: call number = *seq_device + 1, stored back.) */

/* Tuning override for benchmarking: threads per frame (32/64/128/256), bins per thread (odd) and
 * merge chains per thread (1/2, 0 = any); 0, 0, 0 restores the built-in choice.  Returns SOT_EINVAL
 * if that combination is not compiled in.  -1, 0, 0 routes every real-row loss / gradient request through the
 * split-frame path, whatever the row length (tests and benchmarks compare it with the shared-memory kernels). */
int sot_set_tuning(int32_t threads_per_frame, int32_t bins_per_thread, int32_t chains_per_thread);
/* Number of kernel launches issued by this library in the calling process so far. */
int64_t sot_launch_count(void);

#ifdef __cplusplus
}
#endif
#endif /* SOT_B200_H */
