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

#define SOT_B200_ABI_VERSION 3

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

/* ---- pairwise distances (the `torch.cdist` of the loss) ------------------------------------------
 * dist[b, i, j] = per-frame W_p^p of the pair (u[b, i], v[b, j]), what sot_forward_device gives for that one pair
 * (u is the target: in SOT_CUT_SCALE mode v is divided by u's mass), without materialising the B*P*R pairs: each
 * row's CDF is built once.  Positions are one ascending grid per side.  Flags: SOT_SQUARE | SOT_CUT_SCALE | SOT_LIMIT
 * only (anything else: SOT_EINVAL); rows of at most 8448 bins (else SOT_ETOOBIG); B*P*R at most 2^31 - 1;
 * B*P*R == 0 launches nothing and returns 0.  Scratch is allocated stream-ordered on `stream` (capturable in a CUDA
 * graph). */
typedef struct sot_pairwise_problem {
    int64_t batch, rows_u, rows_v; /* B, P, R */
    int32_t n_u, n_v;              /* bins */
    const float *u, *v;            /* [B, P, n_u], [B, R, n_v] contiguous */
    const float *pos_u, *pos_v;    /* [n_u], [n_v], ascending */
    float p;
    int32_t flags;                 /* SOT_SQUARE | SOT_CUT_SCALE | SOT_LIMIT only */
} sot_pairwise_problem;
int sot_pairwise_device(const sot_pairwise_problem* prob, float* dist /* [B, P, R] */, void* stream);
/* grad_u[b, i, :] = sum_j upstream[b, i, j] * d dist[b, i, j] / d u[b, i, :], grad_v likewise over i; either output
 * nullable.  Deterministic: two calls give the same bits. */
int sot_pairwise_backward_device(const sot_pairwise_problem* prob, const float* upstream /* [B, P, R] */,
                                 float* grad_u, float* grad_v /* nullable */, void* stream);
/* Exact k nearest neighbours: for every u[b, i], the k smallest dist[b, i, :] of sot_pairwise_device, sorted ascending
 * (NaN after every number, the lower index first on equal values), as values[b, i, :k] (the same bits as the dist
 * entries) and their v row indices indices[b, i, :k] -- the first k columns of a stable sort of dist, without forming
 * it.  1 <= k <= min(rows_v, 128) (else SOT_EINVAL): 128 keeps 32 queries' lists in one CTA's shared memory.  Without
 * SOT_CUT_SCALE and SOT_LIMIT, a pair is walked only when a lower bound on its distance (interval means of the two
 * quantile functions) does not exceed the k-th value found so far; skipping it provably cannot change the result.  In
 * the other modes every pair is walked.  `walked` (nullable, device) receives the number of pairs walked, which may
 * vary from call to call; the results do not.  Problem rules as above, except that only batch * rows_u and
 * batch * rows_v (not the pairs) are capped at 2^31 - 1; batch * rows_u == 0 launches no kernel.  No host
 * synchronisation; scratch is stream-ordered (capturable in a CUDA graph). */
int sot_pairwise_knn_device(const sot_pairwise_problem* prob, int32_t k, float* values /* [B, P, k] */,
                            int64_t* indices /* [B, P, k] */, int64_t* walked /* nullable */, void* stream);
/* Exact radius search: every (b, i, j) with dist[b, i, j] <= radius (compared in fp32, so a NaN distance never counts)
 * for dist as sot_pairwise_device gives it.  *count (device) receives their number.  When *count <= capacity, the
 * first *count entries of rows (b * P + i), cols (j) and values (the same bits as the dist entries) are exactly those
 * pairs in ascending (b * P + i, j) order, torch.nonzero's row-major order.  When *count > capacity their contents are
 * unspecified, and nothing is written at or past `capacity` in either case; capacity == 0 is a count-only call (the
 * three arrays may then be NULL).  Without SOT_CUT_SCALE and SOT_LIMIT, a pair is walked only when the lower bound of
 * sot_pairwise_knn_device does not rule it out against the radius; in the other modes every pair is walked, and
 * radius = +inf never prunes.  `walked` (nullable, device) receives the number of pairs walked, which may vary from
 * call to call; count, rows, cols and values do not.  A NaN radius or a negative capacity: SOT_EINVAL.  Problem rules
 * as for sot_pairwise_knn_device; batch * rows_u * rows_v == 0 sets *count = 0 and launches no kernel.  No host
 * synchronisation; scratch is stream-ordered (capturable in a CUDA graph with a fixed capacity). */
int sot_pairwise_radius_device(const sot_pairwise_problem* prob, float radius, int64_t capacity,
                               int64_t* rows /* [capacity] */, int64_t* cols /* [capacity] */,
                               float* values /* [capacity] */, int64_t* count /* device, 1 */,
                               int64_t* walked /* nullable */, void* stream);

/* ---- Wasserstein barycenters (W2) ------------------------------------------------------------------------------
 * out[b, :] = the W2 barycenter of the K rows x[b, 0..K-1, :] with weights w[b, :] (weights_stride K) or w[:] (stride
 * 0), as mass per point of the ascending grid pos_out (each row sums to 1).  Each row is normalised by its own mass
 * (weights = x^2 with SOT_SQUARE), its CDF c_j formed, qs = the stable sort of all K*n CDF entries, and the step
 * qs_k - qs_{k-1} (qs_{-1} = 0) is placed at z_k = sum_j w_j pos[min(searchsorted_left(c_j, qs_k), n-1)] and split
 * linearly between the two grid points around it (below the grid: point 0; at or above its last point: point n_out-1).
 * Weights are used as given and must be non-negative; a barycenter with a negative or non-finite weight or a
 * non-finite input row gives a NaN row (and NaN gradient rows).  Flags: SOT_SQUARE only (anything else: SOT_EINVAL);
 * k, n, n_out >= 1; k * n at most 2^24 per barycenter (else SOT_ETOOBIG); count == 0 launches nothing and returns 0.
 * Deterministic (two calls give the same bits; a barycenter's result does not depend on the others in the call); no
 * host synchronisation; scratch is allocated stream-ordered on `stream` (capturable in a CUDA graph). */
typedef struct sot_barycenter_problem {
    int64_t count;              /* N barycenters */
    int32_t k, n, n_out;        /* rows per barycenter, bins per row, output points */
    const float* x;             /* [N, k, n] contiguous */
    const float* weights;       /* [k] (weights_stride 0) or [N, k] (weights_stride k) */
    int64_t weights_stride;
    const float *pos, *pos_out; /* [n], [n_out], ascending */
    int32_t flags;              /* SOT_SQUARE only */
} sot_barycenter_problem;
int sot_barycenter_device(const sot_barycenter_problem* prob, float* out /* [N, n_out] */, void* stream);
/* grad_x[b, j, :] = d (sum_m upstream[b, m] * out[b, m]) / d x[b, j, :]; the gradient flows through the steps of qs
 * only (z depends on the grid and the weights). */
int sot_barycenter_backward_device(const sot_barycenter_problem* prob, const float* upstream /* [N, n_out] */,
                                   float* grad_x /* [N, k, n] */, void* stream);

/* ---- grouped Wasserstein barycenters (W2) ----------------------------------------------------------------------
 * out[g, :] = the barycenter above of the rows offsets[g] .. offsets[g + 1] - 1 of x, in increasing row order, with
 * their weights weights[row] (or, weights NULL, fl32(1 / K_g) each for a group of K_g rows): bit for bit what
 * sot_barycenter_device gives for those rows alone.  Groups of any size: no padding and no per-group cap; R * n at
 * most 2^31 - 1 per call (else SOT_ETOOBIG).  A group with no rows gets a NaN row, and so does a non-finite row or a
 * negative or non-finite weight for its own group (and its gradient rows).  The offsets table is read on the device
 * only: group g is used when 0 <= offsets[g] <= offsets[g + 1] <= rows and no earlier offset exceeds offsets[g]; any
 * other group gets a NaN row, and no row outside x is read.  Flags: SOT_SQUARE only; n, n_out >= 1; groups, rows >= 0.
 * groups == 0 launches nothing; rows == 0 (every group empty) sets the output rows to NaN with one memset and
 * launches no kernel (the backward does nothing).  Deterministic, independent of the other groups in the call, no
 * host synchronisation; scratch is allocated stream-ordered on `stream` for all the entries at once (about 24 bytes
 * per entry R * n, 28 in the backward; DESIGN.md section 4). */
typedef struct sot_barycenter_groups_problem {
    int64_t groups, rows;        /* G, R */
    int32_t n, n_out;
    const float* x;              /* [R, n]: group g is rows offsets[g] .. offsets[g+1]-1 */
    const int64_t* offsets;      /* [G + 1], device */
    const float* weights;        /* [R], or NULL: 1/K_g within each group */
    const float *pos, *pos_out;  /* [n], [n_out], ascending */
    int32_t flags;               /* SOT_SQUARE only */
} sot_barycenter_groups_problem;
int sot_barycenter_groups_device(const sot_barycenter_groups_problem* prob, float* out /* [G, n_out] */,
                                 void* stream);
/* grad_x[r, :] = d (sum_{g,m} upstream[g, m] * out[g, m]) / d x[r, :]; zero for a row in no group. */
int sot_barycenter_groups_backward_device(const sot_barycenter_groups_problem* prob,
                                          const float* upstream /* [G, n_out] */, float* grad_x /* [R, n] */,
                                          void* stream);

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
 * (see sot_host_release); concurrent calls are serialised. */
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
 * positions in memory the device can reach (else SOT_ETOOBIG).  Shared memory bounds the rest: sot_quantiles_device
 * and the CDF harness take up to 8448 bins, SOT_COMPLEX_INPUT rows up to 4352; longer rows there return SOT_ETOOBIG. */
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
 * if no kernel configuration has that combination.  -1, 0, 0 routes every real-row loss / gradient request through the
 * split-frame path, whatever the row length (tests and benchmarks compare it with the shared-memory kernels). */
int sot_set_tuning(int32_t threads_per_frame, int32_t bins_per_thread, int32_t chains_per_thread);
/* Number of kernel launches issued by this library in the calling process so far. */
int64_t sot_launch_count(void);

#ifdef __cplusplus
}
#endif
#endif /* SOT_B200_H */
